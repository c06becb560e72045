"""GPU: reprojection of the film and its moments across camera moves (agpt_reproject_film).

NOT REFERENCE BEHAVIOUR: the reference clears the film whenever the camera moves.  The feature is stated on the CPU in
oracle/reproject.py; these tests hold the library to that statement bit for bit, fed with the film, moments and guides the library
itself leaves on the device before and after each move."""
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
from oracle import reproject as rp  # noqa: E402

W, H = 96, 54
LEVELS = {1: 0, 5: 2, 7: 0, 8: 3, 9: 2}
PARAMS = dict(max_history=24.0, sigma_depth=0.05, min_normal_dot=0.8)


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def same_floats(a, b):
    """Bit-equal, or NaN on both sides."""
    a = np.ascontiguousarray(a, np.float32); b = np.ascontiguousarray(b, np.float32)
    return bool(np.all((bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))))


@pytest.fixture(scope="module")
def rctx(agpt):
    """A context of this file's own: moments, guides and saved views stay here."""
    if agpt.device_count() == 0:
        pytest.fail("no CUDA device visible: -m gpu tests must run on the GPU box")
    ctx = agpt.Context(0)
    yield ctx
    ctx.close()


def setup(agpt, ctx, cfg, w=W, h=H):
    d = agpt.config_defaults(cfg)
    hs = agpt.HostScene(cfg, LEVELS.get(cfg, 0))
    hs.upload(ctx); ctx.set_film(w, h)           # (an upload drops any saved view)
    ctx.set_moments(True)
    ctx.clear()
    return d, hs


def moves(cam):
    """small orbit, translation, large turn, turn past 90 degrees, lens radius > 0: consecutive moves from `cam`."""
    lf, la, up, aspect, vfov, ap = rp.camera_desc(cam)
    focus = np.linalg.norm(la - lf)
    side = np.cross(up, lf - la); side /= np.linalg.norm(side)
    out, c = [], cam
    for name, f in [("orbit", lambda c: rp.orbit(c, 2.5)), ("translate", lambda c: rp.translate(c, 0.03 * focus * side + 0.01 * focus * up)),
                    ("turn", lambda c: rp.turn(c, 20.0)), ("turn_past_90", lambda c: rp.turn(c, 100.0)),
                    ("lens", lambda c: rp.with_aperture(rp.orbit(c, -1.0), 0.05 * focus))]:
        c = f(c)
        out.append((name, c))
    return out


class Viewer:
    """The viewer loop of agpt.h on a context, checked against the statement at every reprojection."""

    def __init__(self, agpt, ctx, d, params, guide_samples=2, spp=2):
        self.agpt, self.ctx, self.d, self.p = agpt, ctx, d, params
        self.gs, self.spp, self.used = guide_samples, spp, 0
        self.view = None                          # (camera, G) the context saved last
        self.nonfinite = False                    # some reprojection started from non-finite film or moments

    def frame(self, cam, check=True):
        ctx = self.ctx
        ctx.set_camera(cam)
        ctx.render_guides(self.gs)
        film, mom = ctx.read_accum().copy(), ctx.read_moments().copy()
        self.nonfinite |= not (np.isfinite(film).all() and np.isfinite(mom).all())
        alb, nd = ctx.read_guides()
        ctx.reproject_film(self.p)
        got_f, got_m = ctx.read_accum().copy(), ctx.read_moments().copy()
        prev_cam, prev_G = self.view if self.view else (None, None)
        want_f, want_m, G = rp.reproject(prev_cam, prev_G, film, mom, cam, alb, nd, self.p.max_history, self.p.sigma_depth, self.p.min_normal_dot)
        if check:
            assert same_floats(got_f, want_f) and same_floats(got_m, want_m)
        self.view = (np.asarray(cam, np.float32).copy(), G)
        if self.spp:
            ctx.render(self.used, self.spp, self.d["max_depth"], self.d["depth_arg"])
            self.used += self.spp
        return got_f, got_m


SHAPES = [pytest.param(c, W, H, id=f"{c}-{W}x{H}") for c in LEVELS] + [pytest.param(c, W, 56, id=f"{c}-{W}x56") for c in (1, 5)] + \
    [pytest.param(c, w, h, id=f"{c}-{w}x{h}") for c, w, h in [(1, 1, 1), (1, 33, 9), (5, 33, 9)]]


@pytest.mark.parametrize("cfg,w,h", SHAPES)
def test_reprojection_equals_the_statement(agpt, rctx, cfg, w, h):
    """96x54 takes the row-major slot order, 96x56 the tiled one; 1x1 and 33x9 are smaller than a filter block.  cfg 7 has an
    environment sky, cfg 8 non-finite moments, cfg 9 instances.  Five moves in a row: the saved view ping-pongs."""
    d, hs = setup(agpt, rctx, cfg, w, h)
    v = Viewer(agpt, rctx, d, agpt.reproject_params(**PARAMS), spp=8 if cfg == 8 else 2)
    cam0 = hs.camera()
    v.frame(cam0)                                # no saved view: nothing carried
    v.frame(cam0)                                # the same camera: the identity rule
    carried = []
    for name, cam in moves(cam0):
        f, m = v.frame(cam)
        carried.append(float((m[..., 3] > 0).mean()))
    if cfg == 8:
        assert v.nonfinite                           # sums of squares that overflowed: non-finite taps were met
    if w * h > 1:
        assert max(carried) > 0.3, carried          # the moves carry history (the statement decided how much)


def test_synthetic_films_and_moments(agpt, rctx):
    """Films and moments with arithmetic edges (written with write_accum / write_moments) through a real move."""
    d, hs = setup(agpt, rctx, 5)
    p = agpt.reproject_params(max_history=3.0, sigma_depth=0.2, min_normal_dot=0.5)
    rng = np.random.default_rng(11)
    n = rng.integers(0, 8, (H, W)).astype(np.float32)
    n[0, :8] = [0, 1, 2, 3, 1 << 24, 16777215, 5, 7]
    film = (rng.standard_normal((H, W, 4)) * 3).astype(np.float32)
    mom = np.abs(rng.standard_normal((H, W, 4))).astype(np.float32) * 10
    mom[..., 3] = n
    edges = [np.inf, -np.inf, np.nan, -0.0, 1e-40, 3.4e38, -1e-30]
    for i, e in enumerate(edges):
        film[5 + i, 10:40:3, i % 4] = e
        mom[20 + i, 5:60:4, i % 3] = e
    v = Viewer(agpt, rctx, d, p)
    cam0 = hs.camera()
    rctx.set_camera(cam0); rctx.render_guides(2); rctx.reproject_film(p)
    v.view = (cam0, rp.guide_g(*rctx.read_guides()))
    rctx.write_accum(film); rctx.write_moments(mom)
    v.spp = 0
    for _, cam in moves(cam0)[:3]:
        v.frame(cam)


def test_caller_owned_film(agpt, rctx):
    """The same results on a film in caller-owned device memory (agpt_set_accum_dev), which keeps its address."""
    import torch
    cfg = 5
    d, hs = setup(agpt, rctx, cfg)
    p = agpt.reproject_params(**PARAMS)
    cams = [hs.camera()] + [c for _, c in moves(hs.camera())[:3]]
    v = Viewer(agpt, rctx, d, p)
    for c in cams:
        v.frame(c, check=False)
    own = rctx.read_accum().copy(), rctx.read_moments().copy()
    buf = torch.zeros(H * W * 4, dtype=torch.float32, device="cuda")
    d, hs = setup(agpt, rctx, cfg)
    rctx.set_accum_dev(buf.data_ptr()); rctx.clear()
    v = Viewer(agpt, rctx, d, p)
    for c in cams:
        v.frame(c)                                  # checked against the statement
    assert rctx.accum_ptr() == buf.data_ptr()
    torch.cuda.synchronize()
    assert np.array_equal(bits(buf.cpu().numpy().reshape(H, W, 4)), bits(own[0])) and np.array_equal(bits(rctx.read_moments()), bits(own[1]))
    rctx.set_accum_dev(0)


@pytest.mark.parametrize("cfg", [1, 5])
def test_static_camera_accumulates_as_without_reprojection(agpt, rctx, cfg):
    """Frames of k spp with reproject_film between them equal one render of all their samples, bit for bit."""
    d, hs = setup(agpt, rctx, cfg)
    rctx.clear(); rctx.render(0, 12, d["max_depth"], d["depth_arg"])
    want_f, want_m = rctx.read_accum().copy(), rctx.read_moments().copy()
    d, hs = setup(agpt, rctx, cfg)
    p = agpt.reproject_params(**PARAMS)
    for first in range(0, 12, 3):
        rctx.set_camera(hs.camera()); rctx.render_guides(1); rctx.reproject_film(p)
        rctx.render(first, 3, d["max_depth"], d["depth_arg"])
    assert np.array_equal(bits(rctx.read_accum()), bits(want_f)) and np.array_equal(bits(rctx.read_moments()), bits(want_m))


def test_resolve_counts_of_a_carried_film(agpt, rctx):
    """A carried film has fractional counts: resolve_counts divides by them, as the statement's means say."""
    d, hs = setup(agpt, rctx, 5)
    v = Viewer(agpt, rctx, d, agpt.reproject_params(**PARAMS), spp=4)
    v.frame(hs.camera())
    v.frame(rp.orbit(hs.camera(), 3.0))             # disoccluded pixels start again: counts 4 and 8 side by side
    f, m = v.frame(rp.orbit(hs.camera(), 6.0))
    assert (m[..., 3] != np.floor(m[..., 3])).any()
    # (the film now also holds the 4 samples rendered after the move)
    film, mom = rctx.read_accum(), rctx.read_moments()
    out, rgb8 = rctx.denoise(agpt.denoise_params(iterations=0))
    assert same_floats(out[..., :3], dn.means(film, mom))
    assert np.array_equal(rctx.resolve_counts(), rgb8)


def test_saved_view_is_dropped_and_kept(agpt, rctx):
    """Dropped by a film resize, by uploads and by turning moments off (the next call carries nothing); kept by set_camera and by
    set_film at the same size."""
    d, hs = setup(agpt, rctx, 5)
    p = agpt.reproject_params(**PARAMS)
    cam0, cam1 = hs.camera(), rp.orbit(hs.camera(), 3.0)

    def saved_then(change, want_kept):
        rctx.set_camera(cam0); rctx.render_guides(1); rctx.reproject_film(p)
        rctx.clear(); rctx.render(0, 2, d["max_depth"], d["depth_arg"])
        change()
        rctx.set_moments(True)
        rctx.set_camera(cam1); rctx.render_guides(1)
        before = rctx.read_accum().copy(), rctx.read_moments().copy()
        rctx.reproject_film(p)
        after = rctx.read_accum().copy(), rctx.read_moments().copy()
        unchanged = all(np.array_equal(bits(a), bits(b)) for a, b in zip(before, after))
        assert unchanged != want_kept

    saved_then(lambda: None, True)
    saved_then(lambda: rctx.set_camera(cam1), True)
    saved_then(lambda: rctx.set_film(W, H), True)
    saved_then(lambda: hs.upload(rctx), False)
    saved_then(lambda: rctx.set_moments(False), False)
    saved_then(lambda: (rctx.set_film(W + 2, H), rctx.set_film(W, H)), False)


def test_refusals_leave_film_moments_and_view(agpt, rctx):
    d, hs = setup(agpt, rctx, 5)
    p = agpt.reproject_params(**PARAMS)
    cam0, cam1 = hs.camera(), rp.orbit(hs.camera(), 3.0)
    rctx.set_camera(cam0); rctx.render_guides(2); rctx.reproject_film(p)
    rctx.render(0, 4, d["max_depth"], d["depth_arg"])
    rctx.set_camera(cam1); rctx.render_guides(2)
    state = lambda: (rctx.read_accum().copy(), rctx.read_moments().copy())
    before = state()
    nan, inf = float("nan"), float("inf")
    bad = [dict(max_history=0.5), dict(max_history=16777218.0), dict(max_history=nan), dict(max_history=inf), dict(sigma_depth=0.0),
           dict(sigma_depth=-1.0), dict(sigma_depth=inf), dict(sigma_depth=nan), dict(min_normal_dot=-1.01), dict(min_normal_dot=1.01),
           dict(min_normal_dot=nan)]
    for b in bad:
        with pytest.raises(agpt.AgptError, match="error -1"):
            rctx.reproject_film(agpt.reproject_params(**dict(PARAMS, **b)))
    assert agpt.core().agpt_reproject_film(rctx.handle, None) == -1
    # stale guides: after set_camera, and after set_film at the same size
    for stale in (lambda: rctx.set_camera(cam1), lambda: rctx.set_film(W, H)):
        stale()
        with pytest.raises(agpt.AgptError, match="error -3"):
            rctx.reproject_film(p)
    after = state()
    assert all(np.array_equal(bits(a), bits(b)) for a, b in zip(before, after))
    # the saved view is still cam0's: the next call equals the statement from it
    rctx.render_guides(2)
    alb, nd = rctx.read_guides()
    G0 = None
    rctx2 = agpt.Context(0)
    try:
        hs.upload(rctx2); rctx2.set_film(W, H); rctx2.set_camera(cam0); rctx2.render_guides(2)
        G0 = rp.guide_g(*rctx2.read_guides())
    finally:
        rctx2.close()
    rctx.reproject_film(p)
    want_f, want_m, _ = rp.reproject(cam0, G0, before[0], before[1], cam1, alb, nd, p.max_history, p.sigma_depth, p.min_normal_dot)
    assert same_floats(rctx.read_accum(), want_f) and same_floats(rctx.read_moments(), want_m)
    # moments off, no film, no guides
    rctx.set_moments(False)
    with pytest.raises(agpt.AgptError, match="error -3"):
        rctx.reproject_film(p)
    fresh = agpt.Context(0)
    with pytest.raises(agpt.AgptError, match="error -3"):
        fresh.reproject_film(p)                       # moments off, no film
    fresh.set_moments(True)
    with pytest.raises(agpt.AgptError, match="error -3"):
        fresh.reproject_film(p)                       # no film
    fresh.set_film(W, H)
    with pytest.raises(agpt.AgptError, match="error -3"):
        fresh.reproject_film(p)                       # no guides
    fresh.close()


def test_host_mirror_render_temporal(agpt, rctx):
    """CudaPathTracer::RenderTemporal frame by frame equals the Context sequence of agpt.h, bit for bit."""
    cfg, gs, spp = 5, 2, 2
    p, dp = agpt.reproject_params(**PARAMS), agpt.denoise_params()
    d, hs = setup(agpt, rctx, cfg)
    cams = [hs.camera()] + [c for _, c in moves(hs.camera())[:3]]
    want = []
    for i, c in enumerate(cams):
        rctx.set_camera(c); rctx.render_guides(gs); rctx.reproject_film(p)
        rctx.render(i * spp, spp, d["max_depth"], d["depth_arg"])
        want.append((rctx.read_accum().copy(),) + rctx.denoise(dp))
    rctx.set_moments(False)
    tr = agpt.HostTracer(d["max_depth"], 0)
    acc = np.full((H, W, 4), 7, np.float32)
    try:
        for i, c in enumerate(cams):
            out, rgb8 = tr.render_temporal(hs, W, H, acc, i * spp, spp, p, dp, gs, camera=c, depth_arg=d["depth_arg"])
            assert np.array_equal(bits(acc), bits(want[i][0])) and same_floats(out, want[i][1]) and np.array_equal(rgb8, want[i][2]), i
    finally:
        tr.close()


def test_temporal_preview_beats_denoising_alone(agpt, rctx):
    """cfg 5 at 480x270, an 8-frame orbit at 4 spp per frame: reproject + denoise has a lower relative MSE at the last frame
    than denoising the frame's own 4 samples, against a 1024-spp film of that frame's camera.  The bound is conservative: along a
    16-frame orbit at 1080p the measured ratio at the last frame is 8.3 (cfg 3) and 9.7 (cfg 5) on one B200 (DESIGN.md section 10)."""
    cfg, w, h, spp, frames = 5, 480, 270, 4, 8
    d, hs = setup(agpt, rctx, cfg, w, h)
    cams = [rp.orbit(hs.camera(), 0.5 * i) for i in range(frames)]
    rctx.set_moments(False)
    rctx.set_camera(cams[-1]); rctx.clear(); rctx.render(1 << 20, 1024, d["max_depth"], d["depth_arg"])
    ref = rctx.read_accum()[..., :3].astype(np.float64) / 1024
    rel = lambda x: float(np.mean((np.asarray(x, np.float64)[..., :3] - ref) ** 2 / (ref ** 2 + 1e-2)))
    rctx.set_moments(True)
    rctx.clear()                                    # (the film still holds the reference's sums)
    p, dp = agpt.reproject_params(), agpt.denoise_params()
    for i, c in enumerate(cams):
        rctx.set_camera(c); rctx.render_guides(4); rctx.reproject_film(p)
        rctx.render(i * spp, spp, d["max_depth"], d["depth_arg"])
    temporal, _ = rctx.denoise(dp)
    rctx.clear(); rctx.render((frames - 1) * spp, spp, d["max_depth"], d["depth_arg"])
    alone, _ = rctx.denoise(dp)
    ratio = rel(alone) / rel(temporal)
    print(f"TEMPORAL_QUALITY cfg5 480x270 8 frames x 4 spp: denoise alone {rel(alone):.4e} reproject+denoise {rel(temporal):.4e} ratio {ratio:.2f}")
    rctx.set_moments(False)
    assert ratio >= 1.5


def test_no_failed_device_checks(rctx):
    """Meaningful under AGPT_LIB=libagpt_debug.so (test_debug_build_runs_this_file); a release build runs no checks."""
    s = rctx.debug_status()
    print("REPROJECT_DEBUG_STATUS", s["failed"], s["first_code"], s["first_value"], s["checks"])
    assert s["failed"] == 0


def test_debug_build_runs_this_file():
    """The tests above under libagpt_debug.so (history tap indices checked inside the kernel): none may fail.  Own process: the
    library is chosen at load time."""
    lib = os.path.join(ROOT, "ag-pathtracer_b200", "libagpt_debug.so")
    assert os.path.exists(lib)
    env = dict(os.environ, AGPT_LIB=lib)
    out = subprocess.run([sys.executable, "-m", "pytest", "-q", "-s", "-p", "no:cacheprovider", os.path.abspath(__file__), "-k",
                          "not debug_build and not beats and not host_mirror"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if "REPROJECT_DEBUG_STATUS" in l][0]
    failed, checks = [int(v) for v in line.split("REPROJECT_DEBUG_STATUS")[1].split()[0:4:3]]
    assert checks > 10_000 and failed == 0
