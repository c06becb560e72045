"""GPU: guide buffers and the a-trous denoiser (agpt_render_guides, agpt_read_guides, agpt_denoise).

NOT REFERENCE BEHAVIOUR: the reference only divides the film by the sample count.  The feature is stated on the CPU in
oracle/agpt_guides_oracle.cpp (guides) and oracle/denoise.py (filter); these tests hold the library to those statements bit for
bit, fed with the film, moments and guides the library itself leaves on the device."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import denoise as dn  # noqa: E402

W, H = 96, 54
LEVELS = {1: 0, 5: 2, 8: 3, 9: 2, 10: 2}


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def same_floats(a, b):
    """Bit-equal, or NaN on both sides."""
    a = np.ascontiguousarray(a, np.float32); b = np.ascontiguousarray(b, np.float32)
    return bool(np.all((bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))))


@pytest.fixture(scope="module")
def dctx(agpt):
    """A context of this file's own: moments and guides are switched on here, other files' contexts stay as they are."""
    if agpt.device_count() == 0:
        pytest.fail("no CUDA device visible: -m gpu tests must run on the GPU box")
    ctx = agpt.Context(0)
    yield ctx
    ctx.close()


def setup(agpt, ctx, cfg, w=W, h=H):
    d = agpt.config_defaults(cfg)
    hs = agpt.HostScene(cfg, LEVELS.get(cfg, 0))
    hs.upload(ctx); ctx.set_film(w, h)
    return d, hs


# 1x1, one row, one column, one 8x4 tile, partial tiles in both axes, tiled films
GUIDE_SHAPES = [pytest.param(c, W, H, id=f"{c}-{H}") for c in LEVELS] + [pytest.param(5, W, 56, id="5-56")] + \
    [pytest.param(c, w, h, id=f"{c}-{w}x{h}") for c, w, h in [(1, 1, 1), (1, 1, 37), (1, 37, 1), (1, 8, 4), (1, 9, 5), (1, 33, 9),
                                                              (1, 97, 55), (1, 104, 60), (5, 33, 9)]]


@pytest.mark.parametrize("cfg,w,h", GUIDE_SHAPES)
def test_guides_equal_the_statement(agpt, dctx, cfg, w, h):
    """At 96x54 the film takes the row-major slot order, at 96x56 (a multiple of the 8x4 tile) the tiled one."""
    from oracle import guides_binding
    d, hs = setup(agpt, dctx, cfg, w, h)
    dctx.render_guides(4)
    alb, nd = dctx.read_guides()
    _, want_alb, want_nd = guides_binding.GuideScene(hs).guides(w, h, 4)
    assert same_floats(alb, want_alb) and same_floats(nd, want_nd)
    # one sample: hit or miss and t are trace_primary(0)'s
    dctx.render_guides(1)
    alb, nd = dctx.read_guides()
    hits = dctx.trace_primary(0).reshape(h, w)[::-1]
    assert np.array_equal(alb[..., 3], hits["found"].astype(np.float32))
    assert np.array_equal(bits(nd[..., 3]), bits(hits["t"]))


def test_guides_leave_the_render_unchanged(agpt, dctx):
    cfg = 5
    d, hs = setup(agpt, dctx, cfg)
    dctx.clear(); dctx.render(0, 2, d["max_depth"], d["depth_arg"]); dctx.render(2, 2, d["max_depth"], d["depth_arg"])
    plain = dctx.read_accum().copy()
    dctx.clear(); dctx.render(0, 2, d["max_depth"], d["depth_arg"]); dctx.render_guides(4); dctx.render(2, 2, d["max_depth"], d["depth_arg"])
    assert np.array_equal(bits(dctx.read_accum()), bits(plain))


def film_for(agpt, ctx, cfg, mode):
    d, hs = setup(agpt, ctx, 5, W, 56) if cfg == "5@96x56" else setup(agpt, ctx, cfg)
    ctx.set_moments(True)
    if mode == "uniform":
        ctx.clear(); ctx.render(0, 8, d["max_depth"], d["depth_arg"])
    else:
        ctx.render_adaptive(agpt.adaptive(4, 32, 4, 0.2, 0.02), d["max_depth"], d["depth_arg"])
    ctx.render_guides(4)
    return d, hs


@pytest.mark.parametrize("mode", ["uniform", "adaptive"])
@pytest.mark.parametrize("cfg", [1, 5, 8, "5@96x56"])
def test_denoise_equals_the_statement(agpt, dctx, cfg, mode):
    """cfg "5@96x56": a film whose size is a multiple of the 8x4 tile, so render, guides and filter use the tiled slot order."""
    film_for(agpt, dctx, cfg, mode)
    film, mom = dctx.read_accum().copy(), dctx.read_moments().copy()
    alb, nd = dctx.read_guides()
    if cfg == 8:
        assert not np.isfinite(mom).all()          # sums of squares that overflowed: the non-finite rule is exercised
    counts = dctx.resolve_counts()
    for it in (0, 1, 5, 10):
        p = agpt.denoise_params(iterations=it)
        out, rgb8 = dctx.denoise(p)
        want = dn.denoise(film, mom, alb, nd, it, p.sigma_luminance, p.sigma_depth, p.normal_power_log2)
        assert same_floats(out, want), it
        if it == 0:
            assert np.array_equal(rgb8, counts)
    # the packed pixels are agpt_resolve's of the denoised floats
    dctx.write_accum(out); dctx.set_moments(False)
    assert np.array_equal(dctx.resolve(1), rgb8)


@pytest.mark.parametrize("mn,mx", [(4, 32), (8, 8)])
def test_host_mirror_render_adaptive_denoised(agpt, dctx, mn, mx):
    cfg, guide_samples = 5, 4
    p, dp = agpt.adaptive(mn, mx, 4, 0.2, 0.02), agpt.denoise_params()
    d, hs = setup(agpt, dctx, cfg)
    dctx.set_moments(True)
    dctx.render_adaptive(p, d["max_depth"], d["depth_arg"])
    dctx.render_guides(guide_samples)
    out, rgb8 = dctx.denoise(dp)
    film, mom = dctx.read_accum().copy(), dctx.read_moments().copy()
    dctx.set_moments(False)
    tr = agpt.HostTracer(d["max_depth"], 0)
    acc = np.full((H, W, 4), 7, np.float32)
    counts, out2, rgb82 = tr.render_adaptive_denoised(hs, W, H, acc, p, dp, guide_samples, d["depth_arg"])
    tr.close()
    assert np.array_equal(bits(acc[..., :3]), bits(film[..., :3])) and np.array_equal(counts, mom[::-1, :, 3].astype(np.int32))
    assert same_floats(out2, out) and np.array_equal(rgb82, rgb8)


def test_refusals_leave_film_moments_and_guides(agpt, dctx):
    cfg = 5
    d, hs = setup(agpt, dctx, cfg)
    dctx.set_moments(True)
    dctx.clear(); dctx.render(0, 4, d["max_depth"], d["depth_arg"]); dctx.render_guides(2)
    state = lambda: (dctx.read_accum().copy(), dctx.read_moments().copy()) + dctx.read_guides()
    before = state()
    nan, inf = float("nan"), float("inf")
    bad = [dict(iterations=-1), dict(iterations=11), dict(sigma_luminance=-1.0), dict(sigma_luminance=inf), dict(sigma_luminance=nan),
           dict(sigma_depth=-0.5), dict(sigma_depth=inf), dict(normal_power_log2=-1), dict(normal_power_log2=11)]
    for b in bad:
        with pytest.raises(agpt.AgptError, match="error -1"):
            dctx.denoise(agpt.denoise_params(**b))
    for n in (0, -3, (1 << 24) + 1):
        with pytest.raises(agpt.AgptError, match="error -1"):
            dctx.render_guides(n)
    after = state()
    assert all(np.array_equal(bits(a), bits(b)) for a, b in zip(before, after))
    p = agpt.denoise_params()
    # stale guides: after set_camera, set_film (even to the same size) and an upload
    for stale in (lambda: dctx.set_camera(hs.camera()), lambda: dctx.set_film(W, H), lambda: hs.upload(dctx)):
        dctx.render_guides(2)
        dctx.denoise(p)
        stale()
        with pytest.raises(agpt.AgptError, match="error -3"):
            dctx.denoise(p)
        with pytest.raises(agpt.AgptError, match="error -3"):
            dctx.read_guides()
    dctx.render_guides(2)
    assert all(np.array_equal(bits(a), bits(b)) for a, b in zip(before, state()))       # same scene, camera and film: same guides
    dctx.set_moments(False)
    with pytest.raises(agpt.AgptError, match="error -3"):
        dctx.denoise(p)
    assert agpt.core().agpt_denoise(dctx.handle, None, None, None) == -1          # NULL params
    fresh = agpt.Context(0)
    with pytest.raises(agpt.AgptError, match="error -3"):
        fresh.render_guides(1)                                # no scene, film or camera
    fresh.set_moments(True)
    with pytest.raises(agpt.AgptError, match="error -3"):
        fresh.denoise(p)                                      # no film
    fresh.set_film(W, H)
    with pytest.raises(agpt.AgptError, match="error -3"):
        fresh.denoise(p)                                      # no guides
    fresh.close()


def test_denoising_halves_the_error(agpt, dctx):
    """cfg 5 at 480x270: the denoised 16-spp film (defaults, 4 guide samples) against a 1024-spp film of the same frame has at most
    half the relative MSE of the raw 16-spp film.  Measured on one B200 (1000 W): raw / denoised = 18.2 with sigma_luminance 4 (DESIGN.md
    section 10)."""
    cfg, w, h = 5, 480, 270
    d, hs = setup(agpt, dctx, cfg, w, h)
    dctx.set_moments(False)
    dctx.clear(); dctx.render(16, 1024, d["max_depth"], d["depth_arg"])
    ref = dctx.read_accum()[..., :3].astype(np.float64) / 1024
    dctx.set_moments(True)
    dctx.clear(); dctx.render(0, 16, d["max_depth"], d["depth_arg"])
    raw = dctx.read_accum()[..., :3].astype(np.float64) / 16
    dctx.render_guides(4)
    out, _ = dctx.denoise(agpt.denoise_params())
    rel = lambda x: float(np.mean((x - ref) ** 2 / (ref ** 2 + 1e-2)))
    factor = rel(raw) / rel(out[..., :3].astype(np.float64))
    print(f"DENOISE_QUALITY cfg5 480x270 16spp: raw {rel(raw):.4e} denoised {rel(out[..., :3]):.4e} factor {factor:.2f}")
    dctx.set_moments(False)
    assert factor >= 2.0


def test_no_failed_device_checks(dctx):
    """Meaningful under AGPT_LIB=libagpt_debug.so (test_debug_build_runs_this_file); a release build runs no checks."""
    s = dctx.debug_status()
    print("DENOISE_DEBUG_STATUS", s["failed"], s["first_code"], s["first_value"], s["checks"])
    assert s["failed"] == 0


def test_debug_build_runs_this_file():
    """The tests above under libagpt_debug.so (path slots in k_guides and tap indices in the filter checked inside the kernels):
    none may fail.  Own process: the library is chosen at load time."""
    lib = os.path.join(ROOT, "ag-pathtracer_b200", "libagpt_debug.so")
    assert os.path.exists(lib)
    env = dict(os.environ, AGPT_LIB=lib)
    out = subprocess.run([sys.executable, "-m", "pytest", "-q", "-s", "-p", "no:cacheprovider", os.path.abspath(__file__), "-k",
                          "not debug_build and not halves and not host_mirror"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if "DENOISE_DEBUG_STATUS" in l][0]
    failed, checks = [int(v) for v in line.split("DENOISE_DEBUG_STATUS")[1].split()[0:4:3]]
    assert checks > 100_000 and failed == 0
