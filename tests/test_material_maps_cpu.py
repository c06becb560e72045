"""CPU: the statement of roughness-metallic and normal maps on Disney materials (include/agpt.h agpt_upload_material_textures,
statements/agpt_material_maps_oracle.cpp) against float64 geometry and the oracle, and the host mirror's flattening of maps.

NOT REFERENCE BEHAVIOUR except where a map reduces to its material's own values: the reference has neither map."""
import ctypes
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from statements import maps_binding as mb  # noqa: E402
from tests.test_textures_cpu import _Tables as _TexTables  # noqa: E402
from tests.test_gpu_textures import materials, own_colour, bits  # noqa: E402

pytestmark = pytest.mark.skipif(not mb.available(), reason="statements/libagpt_material_maps_oracle.so not built (__graft_entry__.build())")
RNG = np.random.default_rng(13)
LOBE_DIFFUSE, LOBE_RETRO, LOBE_MICROFACET = 1, 2, 4


class _Bind(ctypes.Structure):      # agpt_material_textures
    _fields_ = [("base", ctypes.c_int32), ("roughness_metallic", ctypes.c_int32), ("normal", ctypes.c_int32), ("normal_scale", ctypes.c_float),
                ("color", ctypes.c_float * 3)]


class _Tables(ctypes.Structure):    # agpt_scene_tables: the texture tables' fields, then the map bindings
    _fields_ = _TexTables._fields_ + [("material_textures", ctypes.POINTER(_Bind)), ("n_material_textures", ctypes.c_int)]


def _host(agpt):
    if not os.path.exists(agpt.lib_paths()[1]):
        pytest.skip("libagpt_host.so not built")


def _rays_at(scene_cam_from, targets):
    O = np.broadcast_to(np.float32(scene_cam_from), targets.shape).astype(np.float32)
    D = (targets - O).astype(np.float32)
    D /= np.linalg.norm(D, axis=1, keepdims=True)
    return np.concatenate([O, D, np.full((len(O), 1), 1e30, np.float32)], 1)


def _unit(v):
    v = np.asarray(v, np.float64)
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


# ---- frames -------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def cfg13(agpt):
    _host(agpt)
    hs = agpt.HostScene(13, 1)
    return hs, mb.MapsScene(hs)


def _hits(ms, targets, origin=(0.0, 2.2, -8.5)):
    rows = ms.hit_rows(_rays_at(origin, np.asarray(targets, np.float32)))
    return rows[rows[:, 0] >= 0]


def test_tangents_of_spheres_planes_and_triangles_match_float64_geometry(agpt, cfg13):
    hs, ms = cfg13
    # spheres (cfg 13: centres (-2.2, 0, 0) and (.3, 0, .6), r = 1), near their -z poles too
    for c in ((-2.2, 0.0, 0.0), (0.3, 0.0, 0.6)):
        tg = np.array(c) + RNG.uniform(-.7, .7, (400, 3)) * [1, 1, 0] + [0, 0, -1]
        tg = np.concatenate([tg, np.array(c) + [[1e-4, 2e-4, -1.0], [0, 3e-3, -1.0]]])
        rays = _rays_at((0.0, 2.2, -8.5), tg.astype(np.float32))
        rows = ms.hit_rows(rays)
        # float64 hit point of the same rays on this sphere (r = 1)
        O, D = rays[:, 0:3].astype(np.float64), _unit(rays[:, 3:6])
        oc = O - c
        bq = np.sum(oc * D, 1); disc = bq * bq - (np.sum(oc * oc, 1) - 1)
        t = -bq - np.sqrt(np.maximum(disc, 0))
        p = O + t[:, None] * D - c
        on = (rows[:, 0] >= 0) & (disc > 0) & (np.abs(np.abs(np.sum(rows[:, 3:6] * p, 1)) - 1) < 1e-4)
        on &= np.linalg.norm(p[:, :2], axis=1) > 1e-2                      # (the statement nudges x at the exact pole)
        assert on.sum() > 100 and np.min(p[on, 2]) < -0.99                # hits near the -z pole
        p, rows = p[on], rows[on]
        assert np.max(np.abs(rows[:, 15:17] - 2 * np.pi * np.stack([-p[:, 1], p[:, 0]], 1))) < 1e-4 * 2 * np.pi   # the same points
        theta, phi = np.arccos(np.clip(p[:, 2], -1, 1)), np.arctan2(p[:, 1], p[:, 0])
        want_B = np.pi * np.stack([p[:, 2] * np.cos(phi), p[:, 2] * np.sin(phi), -np.sin(theta)], 1)
        assert np.all(rows[:, 17] == 0)
        keep = np.sin(theta) > 0.1          # (float32 acos near a pole keeps fewer digits of sin(theta))
        assert np.max(np.abs(rows[keep, 18:21] - want_B[keep])) < 1e-3 * np.pi      # (float32 hit points and acos: 1e-3 relative)
    # the floor plane: (1, 0, 0), (0, 0, 1)
    rows = _hits(ms, np.stack([RNG.uniform(-4, 4, 200), np.full(200, -1.0), RNG.uniform(-2, 6, 200)], 1).astype(np.float32))
    plane = rows[np.abs(rows[:, 3:6] - [0, 1, 0]).max(1) < 1e-6]
    assert len(plane) > 50
    assert np.all(plane[:, 15:18] == [1, 0, 0]) and np.all(plane[:, 18:21] == [0, 0, 1])
    # triangles of the quad grid, placed plainly, rotated and scaled, and sheared: T, B against the float64 solve of
    # dp02 = T du02 + B dv02, dp12 = T du12 + B dv12 from the triangle's world-space vertices and uvs
    for centre in ((-1.2, 1.8, 3.0), (1.6, 1.7, 3.2), (-3.6, 2.0, 3.6)):
        tg = np.array(centre) + RNG.uniform(-.6, .6, (300, 3)) * [1, 1, 0]
        rays = _rays_at((0.0, 2.2, -8.5), tg.astype(np.float32))
        rows, tri = ms.hit_rows(rays), ms.hit_triangle(rays)
        on = np.isfinite(tri[:, 0])
        assert on.sum() > 100
        rows, tri = rows[on], tri[on].astype(np.float64)
        v0, v1, v2, uv = tri[:, 0:3], tri[:, 3:6], tri[:, 6:9], tri[:, 9:15]
        du02, dv02, du12, dv12 = uv[:, 0] - uv[:, 4], uv[:, 1] - uv[:, 5], uv[:, 2] - uv[:, 4], uv[:, 3] - uv[:, 5]
        det = du02 * dv12 - dv02 * du12
        want_T = ((dv12 / det)[:, None] * (v0 - v2) - (dv02 / det)[:, None] * (v1 - v2))
        want_B = (-(du12 / det)[:, None] * (v0 - v2) + (du02 / det)[:, None] * (v1 - v2))
        for got, want in ((rows[:, 15:18], want_T), (rows[:, 18:21], want_B)):
            rel = np.linalg.norm(got - want, axis=1) / np.linalg.norm(want, axis=1)
            assert rel.max() < 1e-6, rel.max()
    # the sheared instance's frame is not orthogonal: T . B != 0 there
    rows = _hits(ms, (np.array((-3.6, 2.0, 3.6)) + RNG.uniform(-.5, .5, (50, 3)) * [1, 1, 0]).astype(np.float32))
    assert np.abs(np.sum(rows[:, 15:18].astype(np.float64) * rows[:, 18:21], 1)).max() > 1e-2


def test_mapped_frames_are_orthonormal(agpt, cfg13):
    hs, ms = cfg13
    W, H = 96, 54
    tg = np.stack([RNG.uniform(-4, 4, 3000), RNG.uniform(-1, 3, 3000), RNG.uniform(-1, 4, 3000)], 1).astype(np.float32)
    rows = _hits(ms, tg)
    ns, ss, ts = (rows[:, k:k + 3].astype(np.float64) for k in (6, 9, 12))
    for a in (ns, ss, ts):
        assert np.max(np.abs(np.linalg.norm(a, axis=1) - 1)) < 1e-6
    assert np.max(np.abs(np.sum(ns * ss, 1))) < 1e-6 and np.max(np.abs(np.sum(ns * ts, 1))) < 1e-6 and np.max(np.abs(np.sum(ss * ts, 1))) < 1e-6
    assert np.mean(np.abs(ns - rows[:, 3:6]).max(1) > 1e-3) > 0.3     # most hits are mapped away from the geometric normal


def test_a_constant_tilted_map_gives_the_frame_of_the_tilted_plane():
    N, T, B = np.array([0, 1, 0.]), np.array([1, 0, 0.]), np.array([0, 0, 1.])
    tilt = _unit(RNG.uniform(-1, 1, (500, 3)) * [1, 1, 0] + [0, 0, 1])
    texel = (tilt * 0.5 + 0.5).astype(np.float32)
    sn, sdpdu, changed = mb.frame(np.tile(N, (500, 1)), np.tile(T, (500, 1)), np.tile(B, (500, 1)), texel, 1.0)
    nts = 2 * texel.astype(np.float64) - 1
    want = _unit(nts[:, 0:1] * T + nts[:, 1:2] * B + nts[:, 2:3] * N)     # tangent x -> T, y -> B (increasing v), z -> N
    assert changed.all() and np.max(np.abs(sn - want)) < 1e-6
    assert np.max(np.abs(np.sum(sn * sdpdu, 1))) < 1e-6                    # sdpdu lies in the tilted plane


def test_untouched_cases_leave_the_surface_bit_for_bit():
    n = 64
    N = _unit(RNG.normal(size=(n, 3))).astype(np.float32)
    T = RNG.normal(size=(n, 3)).astype(np.float32)
    B = RNG.normal(size=(n, 3)).astype(np.float32)
    cases = {
        "flat": (np.tile([.5, .5, 1.0], (n, 1)), 1.0),
        "z <= 0": (np.stack([np.full(n, .5), np.full(n, .5), RNG.uniform(0, .5, n)], 1), 1.0),
        "scale 0": (RNG.uniform(0, 1, (n, 3)) * [1, 1, .4] + [0, 0, .6], 0.0),
    }
    for name, (texel, scale) in cases.items():
        sn, sdpdu, changed = mb.frame(N, T, B, texel.astype(np.float32), scale)
        assert not changed.any(), name
        assert np.array_equal(bits(sn), bits(N)) and np.array_equal(bits(sdpdu), bits(T)), name
    sn, sdpdu, changed = mb.frame(N, N * np.float32(3), B, np.tile([.8, .3, .9], (n, 1)).astype(np.float32), 1.0)   # T parallel to N
    exact = np.all(N * np.float32(3) - N * np.sum(N * (N * np.float32(3)), 1, keepdims=True, dtype=np.float32) == 0, 1)
    assert exact.any() and not changed[exact].any() and np.array_equal(bits(sn[exact]), bits(N[exact]))


# ---- per-hit material ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("cfg,level", [(3, 2), (5, 2), (11, 2)])
def test_own_value_maps_give_back_every_disney_record(agpt, cfg, level):
    _host(agpt)
    mats = materials(agpt.HostScene(cfg, level))
    checked = 0
    for m in mats:
        if m["type"] != 1:
            continue
        C = own_colour(m)
        if C is None:
            continue
        for x in (0.0, 0.3, 1.0):
            got = mb.material(m, C, np.array([x, 1, 1], np.float32))
            assert got.tobytes() == m.tobytes()
        checked += 1
    assert checked >= sum(mats["type"] == 1) - 1 and checked > 0


def test_metallic_one_drops_the_diffuse_and_retro_lobes_and_texels_are_clamped(agpt):
    rec = np.zeros(1, mb.MAT_DTYPE)[0]
    rec["type"] = 1; rec["eta"] = 1.5; rec["roughness"] = 0.8; rec["metallic"] = 1.0
    C = np.array([.2, .4, .6], np.float32)
    m = mb.material(rec, C, np.array([0, 1, 1], np.float32))
    assert m["lobes"] == LOBE_MICROFACET and np.all(m["diffuse_r"] == 0) and np.array_equal(m["spec_r0"], C)
    m = mb.material(rec, C, np.array([0, .5, 0], np.float32))
    assert m["lobes"] == LOBE_DIFFUSE | LOBE_RETRO | LOBE_MICROFACET and m["metallic"] == 0
    hi = mb.material(rec, C, np.array([0, 7, 3], np.float32)); one = mb.material(rec, C, np.array([0, 1, 1], np.float32))
    assert hi.tobytes() == one.tobytes()
    lo = mb.material(rec, C, np.array([0, -2, -5], np.float32))
    assert lo["roughness"] == 0 and lo["metallic"] == 0 and lo["alpha_x"] == np.float32(.001) and lo["alpha_y"] == np.float32(.001)


@pytest.mark.parametrize("cfg,level", [(3, 2), (5, 2)])
def test_statement_li_with_own_value_maps_equals_the_oracle(agpt, cfg, level):
    _host(agpt)
    from oracle import port_binding as port
    hs = agpt.HostScene(cfg, level)
    d = agpt.config_defaults(cfg)
    mats = materials(hs)
    images, bind = [np.array([[[.5, .5, 1.0]]], np.float32), np.array([[[.3, 1.0, 1.0]]], np.float32)], []
    for m in mats:
        C = own_colour(m) if m["type"] == 1 else None
        bind.append(agpt.material_textures() if C is None else agpt.material_textures(-1, 1, 0, 1.0, tuple(float(v) for v in C)))
    ms = mb.MapsScene(hs)
    ms.set_textures(images, bind)
    got = ms.render(24, 14, 0, 2, d["max_depth"], d["depth_arg"])
    want, _ = port.PortScene(hs).render(24, 14, 0, 2, d["max_depth"], d["depth_arg"])
    assert np.array_equal(bits(got[..., :3]), bits(want[..., :3]))


# ---- flattening and bindings --------------------------------------------------------------------------------------------

def test_flattening_deduplicates_images_across_the_three_slots(agpt):
    _host(agpt)
    assert ctypes.sizeof(_Tables) == 264
    hs = agpt.HostScene(13, 1)
    t = _Tables.from_buffer_copy(hs.tables().raw[:264])
    dims = sorted((t.textures[i].width, t.textures[i].height) for i in range(t.n_textures))
    # floor checker + height field, ball image + checker + bumps (shared with the grid), mixed normals, grid checker
    assert dims == sorted([(64, 64), (256, 256), (37, 23), (16, 16), (64, 32), (32, 16), (8, 8)])
    assert t.n_material_textures == t.n_materials == t.n_material_texture
    b = [t.material_textures[i] for i in range(t.n_material_textures)]
    assert [x.base for x in b] == [t.material_texture[i] for i in range(t.n_material_texture)]
    normals = [x.normal for x in b if x.normal >= 0]
    assert len(normals) == 4 and len(set(normals)) == 3                          # the bumps image is bound twice, flattened once
    floor = b[0]
    assert floor.base == -1 and floor.roughness_metallic >= 0 and list(floor.color) == [np.float32(.7), np.float32(.62), np.float32(.5)]
    assert agpt.HostScene(13, 2).tables() is not None
    hs12 = agpt.HostScene(12, 0)                 # (the tables borrow the scene's memory)
    cfg12 = _Tables.from_buffer_copy(hs12.tables().raw[:264])
    assert all(cfg12.material_textures[i].roughness_metallic == -1 and cfg12.material_textures[i].normal == -1 for i in range(cfg12.n_material_textures))
    hs1 = agpt.HostScene(1, 0)
    cfg1 = _Tables.from_buffer_copy(hs1.tables().raw[:264])
    assert cfg1.n_material_textures == 0 and not cfg1.material_textures


def test_python_validates_the_bindings(agpt):
    class _NoContext:              # validation happens before the library is called
        _h = None
    up = agpt.Context.upload_material_textures
    img = [np.ones((2, 2, 3), np.float32)]
    for bad in ([agpt.material_textures(normal=1)], [agpt.material_textures(roughness_metallic=-2)],
                [agpt.material_textures(normal=0, normal_scale=float("nan"))], [agpt.material_textures(color=(0, float("inf"), 0))], [(0, -1, -1)]):
        with pytest.raises(agpt.AgptError):
            up(_NoContext(), img, bad)
    with pytest.raises(agpt.AgptError):
        up(_NoContext(), [np.ones((2, 2), np.float32)], [])
