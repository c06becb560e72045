"""CPU: the statements of the denoiser (extension, include/agpt.h agpt_render_guides / agpt_denoise).

The guide statement (oracle/agpt_guides_oracle.cpp) is checked against the oracle's own primary hits and against the
material and normal rules of agpt.h; the filter statement (oracle/denoise.py) against closed forms and edge-stopping
properties on constructed inputs."""
import ctypes
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import denoise as dn  # noqa: E402

F32 = np.float32
W, H, SPP = 96, 54, 4
LEVELS = {1: 0, 5: 2, 8: 3, 9: 2, 10: 2}


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def scene_tables(agpt, hs):
    """prims (PRIM_DTYPE) and materials (agpt_material list) of the flattened scene."""
    from oracle.port_binding import _Tables
    t = _Tables.from_buffer_copy(hs.tables())
    raw = (ctypes.c_byte * (16 * t.n_prims)).from_address(t.prims)
    prims = np.frombuffer(bytes(raw), agpt.PRIM_DTYPE)
    mats = list((agpt.Material * t.n_materials).from_address(t.materials)) if t.n_materials else []
    return prims, mats


def expected_albedo(prims, mats, prim):
    if prim < 0 or prims[prim]["material"] < 0:
        return np.ones(3, F32)
    m = mats[prims[prim]["material"]]
    f = lambda a: np.array(list(a), F32)
    if m.type == agpt_mod().MAT_MIRROR:
        a = f(m.mirror_r)
    elif m.type == agpt_mod().MAT_GLASS:
        a = f(m.mirror_r) + f(m.diffuse_r)
    else:
        a = f(m.diffuse_r) + f(m.spec_r0)
    return np.where(a < 1, a, F32(1)).astype(F32)


def agpt_mod():
    from tests.conftest import load_agpt
    return load_agpt()


@pytest.fixture(scope="module")
def guides():
    from oracle import guides_binding, port_binding
    if not (guides_binding.available() and port_binding.available()):
        pytest.fail("oracle libraries not built: run __graft_entry__.build()")
    agpt = agpt_mod()
    out = {}
    for cfg, level in LEVELS.items():
        hs = agpt.HostScene(cfg, level)
        per, alb, nd = guides_binding.GuideScene(hs).guides(W, H, SPP)
        ps = port_binding.PortScene(hs)
        hits = [ps.primary_hits(W, H, s) for s in range(SPP)]
        out[cfg] = (hs, per, alb, nd, hits)
    return agpt, out


@pytest.mark.parametrize("cfg", list(LEVELS))
def test_guide_samples_are_the_primary_hits(guides, cfg):
    agpt, g = guides
    hs, per, alb, nd, hits = g[cfg]
    for s in range(SPP):
        h = hits[s]
        found = per[s]["prim"] >= 0
        assert np.array_equal(found.astype(np.uint32), h["found"])
        assert np.array_equal(np.where(found, per[s]["prim"], -1), h["prim"])
        assert np.array_equal(bits(per[s]["t"]), bits(h["t"]))
    assert (per["prim"] >= 0).any()


@pytest.mark.parametrize("cfg", list(LEVELS))
def test_guide_normals_and_albedo_follow_the_rules(guides, cfg):
    agpt, g = guides
    hs, per, alb, nd, hits = g[cfg]
    prims, mats = scene_tables(agpt, hs)
    hit = per["prim"] >= 0
    n = per["normal"].astype(np.float64)
    length = np.sqrt((n ** 2).sum(-1))
    assert np.all(np.abs(length[hit] - 1) < 1e-5)
    assert np.all((n * per["dir"]).sum(-1)[hit] <= 0)                 # faces the camera
    assert not per["normal"][~hit].any() and not per["t"][~hit].any() and (per["albedo"][~hit] == 1).all()
    for prim in np.unique(per["prim"]):
        want = expected_albedo(prims, mats, int(prim))
        assert np.array_equal(per["albedo"][per["prim"] == prim], np.broadcast_to(want, (int((per["prim"] == prim).sum()), 3))), prim
    if cfg == 10:
        assert any(m.type == agpt.MAT_GLASS for m in mats)
    if cfg == 9:
        assert (prims["type"][per["prim"][hit]] == agpt.PRIM_INSTANCE).any()


@pytest.mark.parametrize("cfg", [1, 8])
def test_guide_pixels_are_sequential_means(guides, cfg):
    """The per-pixel buffers are the float32 sums of the samples in ascending order, divided as agpt.h states."""
    agpt, g = guides
    hs, per, alb, nd, hits = g[cfg]
    a = np.zeros((W * H, 4), F32); m = np.zeros((W * H, 4), F32)
    for s in range(SPP):
        hit = per[s]["prim"] >= 0
        a[:, :3] += per[s]["albedo"]; a[:, 3] += hit.astype(F32)
        m[:, :3] += per[s]["normal"]; m[:, 3] += np.where(hit, per[s]["t"], F32(0))
    with np.errstate(invalid="ignore", divide="ignore"):
        m[:, 3] = np.where(a[:, 3] > 0, m[:, 3] / a[:, 3], F32(0))
    a /= F32(SPP); m[:, :3] /= F32(SPP)
    flip = lambda x: x.reshape(H, W, 4)[::-1]
    assert np.array_equal(bits(flip(a)), bits(alb)) and np.array_equal(bits(flip(m)), bits(nd))


# ---- the filter statement on constructed inputs -------------------------------------------------------------------------
def uniform(h=32, w=48, n=4, value=(0.3, 0.5, 0.2), spread=0.05, seed=1):
    """A film of n samples per pixel with per-pixel noise, uniform albedo 0.5, normal +z and depth 2."""
    rng = np.random.default_rng(seed)
    c = (np.array(value, F32) * (1 + spread * rng.standard_normal((h, w, n, 3)))).astype(F32)
    film = np.zeros((h, w, 4), F32); mom = np.zeros((h, w, 4), F32)
    for s in range(n):
        film[..., :3] += c[:, :, s]; mom[..., :3] += c[:, :, s] * c[:, :, s]; mom[..., 3] += F32(1)
    alb = np.zeros((h, w, 4), F32); alb[..., :3] = 0.5; alb[..., 3] = 1
    nd = np.zeros((h, w, 4), F32); nd[..., 2] = 1; nd[..., 3] = 2
    return film, mom, alb, nd


def test_constant_image_stays_constant():
    """Bound: 1e-5 relative after 5 iterations (each pass is a weighted mean of equal values; float32 rounding only)."""
    film, mom, alb, nd = uniform(spread=0.0)
    mom[..., :3] += F32(1e-3)                      # some variance, so the luminance stop is not degenerate
    out = dn.denoise(film, mom, alb, nd, 5, 4.0, 0.1, 7)
    want = film[0, 0, :3] / F32(4)
    assert np.all(np.abs(out[..., :3] - want) <= 1e-5 * want)


def test_iterations_zero_returns_the_means():
    film, mom, alb, nd = uniform()
    mom[3, 5] = 0; film[3, 5] = 0
    out = dn.denoise(film, mom, alb, nd, 0, 4.0, 0.1, 7)
    with np.errstate(invalid="ignore"):
        want = np.where(mom[..., 3:4] > 0, film[..., :3] / mom[..., 3:4], F32(0))
    assert np.array_equal(bits(out[..., :3]), bits(want)) and not out[..., 3].any()


@pytest.mark.parametrize("edge", ["hit_miss", "normal_opposite", "normal_orthogonal"])
def test_edges_pass_nothing_across(edge):
    """Whatever the right half holds, the left half's result is the same, bit for bit."""
    film, mom, alb, nd = uniform()
    half = film.shape[1] // 2
    if edge == "hit_miss":
        alb[:, half:, 3] = 0; nd[:, half:, 3] = 0; alb[:, half:, :3] = 1     # normals stay +z: only w_z stops the taps
    else:
        nd[:, half:, :3] = (0, 0, -1) if edge == "normal_opposite" else (1, 0, 0)
    outs = []
    for scale in (1.0, 7.0):
        f = film.copy(); m = mom.copy()
        f[:, half:, :3] *= F32(scale); m[:, half:, :3] *= F32(scale * scale)
        outs.append(dn.denoise(f, m, alb, nd, 5, 1e6, 1e6, 0))
    assert np.array_equal(bits(outs[0][:, :half]), bits(outs[1][:, :half]))
    assert not np.array_equal(bits(outs[0][:, half:]), bits(outs[1][:, half:]))


def test_huge_sigmas_give_the_b3_blur():
    """With every edge stop at 1, one pass is the B3-spline blur h x h over the taps inside the film, normalised by their
    weight, and its variance is sum(h^2 v) / (sum h)^2 (closed forms in float64)."""
    film, mom, alb, nd = uniform(spread=0.2)
    alb[..., :3] = 1
    E, G = dn.prepare(film, mom, alb, nd)
    got = dn.atrous(E, G, 1, 1e15, 1e15, 0)
    h5 = np.array([1, 4, 6, 4, 1], np.float64) / 16
    Hh, Ww = E.shape[:2]
    num = np.zeros((Hh, Ww, 4)); wsum = np.zeros((Hh, Ww)); w2v = np.zeros((Hh, Ww))
    e = E.astype(np.float64)
    for dy in range(-2, 3):
        for dx in range(-2, 3):
            w = h5[dy + 2] * h5[dx + 2]
            ys, xs = np.arange(Hh) + dy, np.arange(Ww) + dx
            ok = ((ys >= 0) & (ys < Hh))[:, None] & ((xs >= 0) & (xs < Ww))[None, :]
            q = e[np.clip(ys, 0, Hh - 1)][:, np.clip(xs, 0, Ww - 1)]
            num[..., :3] += np.where(ok[..., None], w * q[..., :3], 0)
            w2v += np.where(ok, w * w * q[..., 3], 0)
            wsum += np.where(ok, w, 0)
    assert np.allclose(got[..., :3], num[..., :3] / wsum[..., None], rtol=2e-6, atol=0)
    assert np.allclose(got[..., 3], w2v / wsum ** 2, rtol=2e-5, atol=0)


def test_non_finite_pixels_keep_their_value_and_are_skipped():
    """A pixel whose sum of squares overflowed (cfg 8) is invalid: it keeps its demodulated value, and its neighbours' results do
    not depend on it."""
    film, mom, alb, nd = uniform()
    outs = []
    for v in (1.0, 50.0):
        f = film.copy(); m = mom.copy()
        f[10, 10, :3] = F32(v); m[10, 10, 0] = np.inf
        outs.append(dn.denoise(f, m, alb, nd, 3, 4.0, 0.1, 7))
    mask = np.ones(film.shape[:2], bool); mask[10, 10] = False
    assert np.array_equal(bits(outs[0][mask]), bits(outs[1][mask]))
    al = F32(0.5)
    assert np.array_equal(bits(outs[1][10, 10, :3]), bits(((F32(50.0) / F32(4)) / al) * al * np.ones(3, F32)))
    assert np.isfinite(outs[0]).all()
