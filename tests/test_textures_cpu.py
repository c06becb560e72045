"""CPU: the statement of image textures on the base colour of Disney materials (include/agpt.h agpt_upload_textures,
statements/agpt_texture_oracle.cpp) against float64 closed forms, and the host mirror's flattening of textured materials.

NOT REFERENCE BEHAVIOUR: the reference has one colour per material."""
import ctypes
import math
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from statements import texture_binding as tb  # noqa: E402

pytestmark = pytest.mark.skipif(not tb.available(), reason="statements/libagpt_texture_oracle.so not built (__graft_entry__.build())")
RNG = np.random.default_rng(12)


def bilinear64(img, uv):
    """float64 bilinear lookup with repeat wrap, texel centres at (i + 0.5) / W, at the texel-space position the statement forms
    in float32 (s = u' * W - 0.5: its rounding moves the sample point by up to W ulps of u, more than the 1e-6 this checks)."""
    H, W, _ = img.shape
    out = np.zeros((len(uv), 3))
    f32 = np.float32
    for i, (u, v) in enumerate(uv):
        u = u - np.floor(u) if np.isfinite(u) else f32(0)
        v = v - np.floor(v) if np.isfinite(v) else f32(0)
        s, t = float(f32(u) * f32(W) - f32(0.5)), float(f32(v) * f32(H) - f32(0.5))
        x0, y0 = math.floor(s), math.floor(t)
        fx, fy = s - x0, t - y0
        T = lambda x, y: img[y % H, x % W].astype(np.float64)
        out[i] = (1 - fy) * ((1 - fx) * T(x0, y0) + fx * T(x0 + 1, y0)) + fy * ((1 - fx) * T(x0, y0 + 1) + fx * T(x0 + 1, y0 + 1))
    return out


@pytest.mark.parametrize("W,H", [(37, 23), (64, 1), (1, 64), (1, 1), (16, 16), (5, 3)])
def test_lookup_equals_float64_bilinear(W, H):
    img = RNG.uniform(0.05, 1.0, (H, W, 3)).astype(np.float32)
    uv = RNG.uniform(-3, 3, (4000, 2)).astype(np.float32)
    got = tb.lookup(img, uv).astype(np.float64)
    want = bilinear64(img, uv)
    assert np.max(np.abs(got - want) / np.maximum(np.abs(want), 1e-6)) < 1e-6


def test_texel_centres_return_the_texel():
    W, H = 37, 23
    img = RNG.uniform(0, 1, (H, W, 3)).astype(np.float32)
    x, y = np.meshgrid(np.arange(W), np.arange(H))
    uv = np.stack([((x + 0.5) / W).ravel(), ((y + 0.5) / H).ravel()], 1).astype(np.float32)
    got = tb.lookup(img, uv)
    # a centre that rounds off in float32 is not a centre: keep the ones whose s, t come out integral
    s = uv[:, 0] * np.float32(W) - np.float32(0.5); t = uv[:, 1] * np.float32(H) - np.float32(0.5)
    ok = (s == np.floor(s)) & (t == np.floor(t))
    assert ok.mean() > 0.5
    assert np.array_equal(got[ok], img.reshape(-1, 3)[ok])


EDGE_UV = np.array([0.0, 1.0, -1e-30, np.nextafter(np.float32(1), np.float32(0)), 1e30, -1e30, np.nan, np.inf, -np.inf, 0.5, -0.25, 7.75],
                   np.float32)


@pytest.mark.parametrize("W,H", [(1, 1), (1, 9), (9, 1), (37, 23), (2048, 2)])
def test_constant_texture_returns_its_colour_exactly(W, H):
    c = np.array([0.3, 0.71, 0.123456], np.float32)
    img = np.broadcast_to(c, (H, W, 3)).copy()
    u, v = np.meshgrid(EDGE_UV, EDGE_UV)
    uv = np.concatenate([np.stack([u.ravel(), v.ravel()], 1), RNG.uniform(-10, 10, (2000, 2)).astype(np.float32)])
    got = tb.lookup(img, uv)
    assert np.array_equal(got.view(np.uint32), np.broadcast_to(c, got.shape).view(np.uint32))


def test_edge_uvs_wrap_into_the_image():
    img = RNG.uniform(0, 1, (5, 7, 3)).astype(np.float32)
    u, v = np.meshgrid(EDGE_UV, EDGE_UV)
    got = tb.lookup(img, np.stack([u.ravel(), v.ravel()], 1))
    assert np.all(np.isfinite(got)) and got.min() >= img.min() - 1e-6 and got.max() <= img.max() + 1e-6


def test_atan2f_port():
    """fdlibm e_atan2f.c: its special cases exactly, everything else within 2 ulp of the float64 atan2."""
    pi, pio2, pio4 = np.float32(3.1415927410e+00), np.float32(1.5707963705e+00), np.float32(7.8539818525e-01)
    cases = [(0.0, 1.0, 0.0), (-0.0, 1.0, -0.0), (0.0, -1.0, pi), (-0.0, -1.0, -pi), (1.0, 0.0, pio2), (-1.0, 0.0, -pio2),
             (np.inf, np.inf, pio4), (-np.inf, np.inf, -pio4), (np.inf, -np.inf, 3 * pio4), (1.0, np.inf, 0.0), (1.0, -np.inf, pi),
             (np.inf, 1.0, pio2), (1.0, 1.0, pio4)]
    y = np.array([c[0] for c in cases], np.float32); x = np.array([c[1] for c in cases], np.float32)
    got = tb.atan2f(y, x)
    assert np.array_equal(got, np.array([c[2] for c in cases], np.float32))
    assert np.isnan(tb.atan2f(np.float32([np.nan]), np.float32([1]))[0])
    y = RNG.normal(0, 1, 200000).astype(np.float32) * np.float32(10) ** RNG.integers(-6, 6, 200000).astype(np.float32)
    x = RNG.normal(0, 1, 200000).astype(np.float32) * np.float32(10) ** RNG.integers(-6, 6, 200000).astype(np.float32)
    got = tb.atan2f(y, x).astype(np.float64)
    want = np.arctan2(y.astype(np.float64), x.astype(np.float64))
    ulp = np.spacing(np.abs(want).astype(np.float32)).astype(np.float64)
    assert np.max(np.abs(got - want) / ulp) <= 2.0


def _host(agpt):
    try:
        agpt.host()
    except Exception as e:      # noqa: BLE001
        pytest.skip(f"host mirror not built: {e}")


def _rays_at(points, origin):
    d = points - origin
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return np.concatenate([np.broadcast_to(origin, points.shape), d, np.full((len(points), 1), 1e30)], 1).astype(np.float32)


def test_surface_uvs_equal_closed_forms(agpt):
    """cfg 12: rays aimed at known points of the floor plane, the spheres and the plain quad grid; uv within 1e-4 of float64."""
    _host(agpt)
    from agpt_b200 import HostScene  # noqa: F401
    hs = agpt.HostScene(12, 0)
    ts = tb.TextureScene(hs)
    O = np.array([0.0, 6.0, -8.0])
    # floor: o = (0, -1, 0), 8 x 8 (half 4 x 4)
    pf = np.stack([RNG.uniform(-3, 3, 200), np.full(200, -1.0), RNG.uniform(-6, -1, 200)], 1)
    r = ts.hit_uv(_rays_at(pf, O))
    hit = r[:, 2] == 0            # (the spheres and grids hide some of the points)
    assert hit.mean() > 0.5
    assert np.allclose(r[hit, 0], (pf[hit, 0] / 4 + 1) / 2, atol=1e-4) and np.allclose(r[hit, 1], (pf[hit, 2] / 4 + 1) / 2, atol=1e-4)
    # sphere 1: centre (-2.4, 0, 0), r 1; points on its camera-facing side
    O2 = np.array([-2.4, 0.3, -6.0])
    th = RNG.uniform(0.3, 2.8, 200); ph = RNG.uniform(np.pi + 0.3, 2 * np.pi - 0.3, 200)
    n = np.stack([np.sin(th) * np.cos(ph), np.sin(th) * np.sin(ph), np.cos(th)], 1)
    ps = np.array([-2.4, 0, 0]) + n
    vis = np.einsum("ij,ij->i", n, O2 - ps) > 0.2
    r = ts.hit_uv(_rays_at(ps[vis], O2))
    hit = r[:, 2] == 1
    assert hit.mean() > 0.5
    m = n[vis][hit]
    phi = np.mod(np.arctan2(m[:, 1], m[:, 0]), 2 * np.pi)
    assert np.allclose(r[hit, 0], phi / (2 * np.pi), atol=1e-4) and np.allclose(r[hit, 1], np.arccos(m[:, 2]) / np.pi, atol=1e-4)
    # plain quad grid (prim 4): centre (-1.2, 1.8, 3), size 2, z = 0.15 (u - .5)(v - .5) * 2, uv = 2 * (u, v)
    u = RNG.uniform(0.05, 0.95, 200); v = RNG.uniform(0.05, 0.95, 200)
    pg = np.stack([-1.2 + (u - .5) * 2, 1.8 + (v - .5) * 2, 3 + .15 * (u - .5) * (v - .5) * 2], 1)
    r = ts.hit_uv(_rays_at(pg, np.array([-1.2, 1.8, -5.0])))
    hit = r[:, 2] == 4
    assert hit.mean() > 0.5
    # within a triangle the surface is flat (the bilinear patch is not): compare with the vertex-interpolated uv, to 1e-2
    assert np.allclose(r[hit, 0], 2 * u[hit], atol=1e-2) and np.allclose(r[hit, 1], 2 * v[hit], atol=1e-2)
    ts.close()


class _Tex(ctypes.Structure):
    _fields_ = [("width", ctypes.c_int), ("height", ctypes.c_int), ("rgb", ctypes.c_void_p)]


class _Env(ctypes.Structure):
    _fields_ = [("width", ctypes.c_int), ("height", ctypes.c_int), ("rgb", ctypes.c_void_p), ("func", ctypes.c_void_p), ("cdf", ctypes.c_void_p),
                ("func_int", ctypes.c_float)]


class _Tables(ctypes.Structure):      # agpt_scene_tables of include/agpt_host.h
    _fields_ = [("prims", ctypes.c_void_p), ("n_prims", ctypes.c_int), ("spheres", ctypes.c_void_p), ("n_spheres", ctypes.c_int),
                ("planes", ctypes.c_void_p), ("n_planes", ctypes.c_int), ("meshes", ctypes.c_void_p), ("n_meshes", ctypes.c_int),
                ("materials", ctypes.c_void_p), ("n_materials", ctypes.c_int), ("lights", ctypes.c_void_p), ("n_lights", ctypes.c_int),
                ("camera", ctypes.c_float * 19), ("envmap", _Env), ("instances", ctypes.c_void_p), ("n_instances", ctypes.c_int),
                ("textures", ctypes.POINTER(_Tex)), ("material_texture", ctypes.POINTER(ctypes.c_int32)), ("n_textures", ctypes.c_int),
                ("n_material_texture", ctypes.c_int)]


def test_flattening_deduplicates_textures_and_binds_materials(agpt):
    _host(agpt)
    assert ctypes.sizeof(_Tables) == 248
    hs = agpt.HostScene(12, 0)
    t = _Tables.from_buffer_copy(hs.tables().raw[:248])
    dims = sorted((t.textures[i].width, t.textures[i].height) for i in range(t.n_textures))
    assert dims == [(37, 23), (64, 1), (2048, 2048)]               # the 37 x 23 and 2048^2 images are shared, flattened once
    bind = [t.material_texture[i] for i in range(t.n_material_texture)]
    assert t.n_material_texture == t.n_materials and bind.count(-1) == 1 and len(set(b for b in bind if b >= 0)) == 3
    mats = np.frombuffer(ctypes.string_at(t.materials, 64 * t.n_materials), np.dtype([("type", np.int32), ("rest", np.uint8, 60)]))
    assert np.all(mats["type"][np.array(bind) >= 0] == 1)          # AGPT_MAT_DISNEY
    cfg1 = _Tables.from_buffer_copy(agpt.HostScene(1, 0).tables().raw[:248])
    assert cfg1.n_textures == 0 and cfg1.n_material_texture == 0 and not cfg1.material_texture
