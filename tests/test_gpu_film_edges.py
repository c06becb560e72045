"""GPU: adaptive sampling, guides and the denoiser on ragged and tiny films, at the edges of their parameters, over split
batches and on synthetic films and moments.

The kernels (k_adaptive_select, k_generate<true>, k_accumulate<true, *>, k_resolve_counts, k_guides, k_denoise_prepare,
k_denoise_atrous) are held bit for bit (NaN = NaN) to the CPU statements oracle/adaptive.py, oracle/agpt_guides_oracle.cpp and
oracle/denoise.py, here on:
  * films with a partial 32 x 8 filter block or 8 x 4 tile in either axis, films narrower or shorter than the 5 x 5 footprint
    and than the tap spacing (up to 512 at 10 iterations), and tiled films, where k_adaptive_select walks the 8 x 4 tile order;
  * tolerance 0, steps that do not divide max - min or exceed it, min == max and step 1; sigma_luminance 0, sigma_depth 0 and
    normal powers 2^0 and 2^1024 (whose weights fall into float32 subnormals: a flush to zero would show);
  * guides traced over several batches (k_guides carrying sums from one batch to the next);
  * films and moments written from the host with the arithmetic edges of the convergence test and of k_denoise_prepare
    (n = 0, 1, 2, 3, 2^24, d = 0 and d < 0, inf, NaN, negative and subnormal sums).
The float64 check of the convergence test (tests/test_film_edges_cpu.py) runs here against the device."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import adaptive as st  # noqa: E402
from oracle import denoise as dn  # noqa: E402
from tests.test_film_edges_cpu import convergence_f64  # noqa: E402

F32 = np.float32
LEVELS = {1: 0, 5: 2}
TOL, FLOOR = 0.2, 0.02
# (cfg, W, H): 1x1, one row, one column; exactly one 8x4 tile; partial blocks and tiles in both axes; tiled films
SHAPES = [(1, 1, 1), (1, 1, 37), (1, 37, 1), (1, 8, 4), (1, 9, 5), (1, 33, 9), (1, 97, 55), (1, 96, 56), (1, 104, 60),
          (5, 33, 9), (5, 96, 56)]
EDGE_SIZES = [(33, 9), (96, 56)]
shape_id = lambda s: f"cfg{s[0]}-{s[1]}x{s[2]}"


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def same_floats(a, b):
    """Bit-equal, or NaN on both sides."""
    a = np.ascontiguousarray(a, np.float32); b = np.ascontiguousarray(b, np.float32)
    return bool(np.all((bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))))


@pytest.fixture(scope="module")
def ectx(agpt):
    """A context of this file's own: moments are switched on and off here, other files' contexts stay as they are."""
    if agpt.device_count() == 0:
        pytest.fail("no CUDA device visible: -m gpu tests must run on the GPU box")
    ctx = agpt.Context(0)
    yield ctx
    ctx.close()


def setup(agpt, ctx, cfg, w, h):
    """cfg uploaded, a w x h film, moments on: (defaults, host scene, li(xs, ys, ss) = the library's single-path radiances)."""
    d = agpt.config_defaults(cfg)
    hs = agpt.HostScene(cfg, LEVELS[cfg])
    hs.upload(ctx); ctx.set_film(w, h); ctx.set_moments(True)
    li = lambda xs, ys, ss: ctx.li_pixels(xs, ys, ss, d["max_depth"], d["depth_arg"])
    return d, hs, li


def check_render_adaptive(agpt, ctx, d, li, w, h, p):
    """render_adaptive equals the statement (film, moments, rounds, paths); returns the device's film, moments and rounds."""
    rounds, paths = ctx.render_adaptive(p, d["max_depth"], d["depth_arg"])
    film, mom = ctx.read_accum(), ctx.read_moments()
    want_film, want_mom, want_rounds, want_paths, _ = st.render_adaptive(li, w, h, p)
    assert same_floats(film[..., :3], want_film[..., :3]) and same_floats(mom, want_mom)
    assert (rounds, paths) == (want_rounds, want_paths)
    n = mom[..., 3].astype(np.int64)
    assert n.min() >= p.min_samples and n.max() <= p.max_samples and ((n - p.min_samples) % p.step == 0).all()
    assert paths == n.sum() and rounds <= (p.max_samples - p.min_samples) // p.step
    assert ctx.adaptive_select(p)[0] == 0
    return film, mom, rounds


# ---- film shapes ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", SHAPES, ids=shape_id)
def test_select_on_film_shapes(agpt, ectx, shape):
    cfg, w, h = shape
    d, _, _ = setup(agpt, ectx, cfg, w, h)
    p = agpt.adaptive(4, 32, 4, TOL, FLOOR)
    ectx.clear(); ectx.render(0, p.min_samples, d["max_depth"], d["depth_arg"])
    film, mom = ectx.read_accum(), ectx.read_moments()
    n, pix = ectx.adaptive_select(p)
    want = st.selected_pixels(film, mom, p)
    assert n == len(want) and np.array_equal(np.sort(pix), want)


@pytest.mark.parametrize("shape", SHAPES, ids=shape_id)
def test_render_adaptive_on_film_shapes(agpt, ectx, shape):
    """The statement's frame, and per final count k the pixels of a plain render(0, k) and resolve(k)."""
    cfg, w, h = shape
    d, _, li = setup(agpt, ectx, cfg, w, h)
    film, mom, rounds = check_render_adaptive(agpt, ectx, d, li, w, h, agpt.adaptive(4, 32, 4, TOL, FLOOR))
    n = mom[..., 3].astype(np.int64)
    print(f"{shape_id(shape)}: {rounds} rounds, counts {dict(zip(*np.unique(n, return_counts=True)))}")
    packed = ectx.resolve_counts()
    ectx.set_moments(False)
    for k in np.unique(n):
        ectx.clear(); ectx.render(0, int(k), d["max_depth"], d["depth_arg"])
        m = n == k
        assert np.array_equal(bits(ectx.read_accum()[m]), bits(film[m])), k
        assert np.array_equal(ectx.resolve(int(k))[m], packed[m]), k


@pytest.mark.parametrize("shape", SHAPES, ids=shape_id)
def test_denoise_on_film_shapes(agpt, ectx, shape):
    """An adaptive film denoised at 0, 1, 5 and 10 iterations (tap spacing up to 512, beyond every film here)."""
    cfg, w, h = shape
    d, _, _ = setup(agpt, ectx, cfg, w, h)
    ectx.render_adaptive(agpt.adaptive(4, 32, 4, TOL, FLOOR), d["max_depth"], d["depth_arg"])
    ectx.render_guides(4)
    film, mom = ectx.read_accum(), ectx.read_moments()
    alb, nd = ectx.read_guides()
    counts = ectx.resolve_counts()
    for it in (0, 1, 5, 10):
        p = agpt.denoise_params(iterations=it)
        out, rgb8 = ectx.denoise(p)
        assert same_floats(out, dn.denoise(film, mom, alb, nd, it, p.sigma_luminance, p.sigma_depth, p.normal_power_log2)), it
        if it == 0:
            assert np.array_equal(rgb8, counts)


# ---- parameter edges (cfg 5) ----------------------------------------------------------------------------------------------
ADAPTIVE_EDGES = {"tol0-floor0": (4, 32, 4, 0.0, 0.0), "step-not-dividing": (4, 30, 4, TOL, FLOOR), "step-over-range": (4, 6, 4, TOL, FLOOR),
                  "min-eq-max": (8, 8, 1, TOL, FLOOR), "step1": (2, 9, 1, TOL, FLOOR)}


@pytest.mark.parametrize("size", EDGE_SIZES, ids=lambda s: f"{s[0]}x{s[1]}")
@pytest.mark.parametrize("edge", list(ADAPTIVE_EDGES))
def test_adaptive_parameter_edges(agpt, ectx, edge, size):
    w, h = size
    d, _, li = setup(agpt, ectx, 5, w, h)
    p = agpt.adaptive(*ADAPTIVE_EDGES[edge])
    _, mom, rounds = check_render_adaptive(agpt, ectx, d, li, w, h, p)
    if edge in ("step-over-range", "min-eq-max"):
        assert rounds == 0 and (mom[..., 3] == p.min_samples).all()
    if edge == "tol0-floor0":
        assert rounds == 7                           # a noisy pixel is never within tolerance 0: it runs to the cap


DENOISE_EDGES = {"sigma_l0": dict(sigma_luminance=0.0), "sigma_z0": dict(sigma_depth=0.0), "npow0": dict(normal_power_log2=0),
                 "npow10": dict(normal_power_log2=10)}


@pytest.mark.parametrize("size", EDGE_SIZES, ids=lambda s: f"{s[0]}x{s[1]}")
@pytest.mark.parametrize("edge", list(DENOISE_EDGES))
def test_denoise_parameter_edges(agpt, ectx, edge, size):
    w, h = size
    d, _, _ = setup(agpt, ectx, 5, w, h)
    ectx.clear(); ectx.render(0, 8, d["max_depth"], d["depth_arg"])
    ectx.render_guides(4)
    film, mom = ectx.read_accum(), ectx.read_moments()
    alb, nd = ectx.read_guides()
    for it in (1, 5):
        p = agpt.denoise_params(iterations=it, **DENOISE_EDGES[edge])
        out, _ = ectx.denoise(p)
        assert same_floats(out, dn.denoise(film, mom, alb, nd, it, p.sigma_luminance, p.sigma_depth, p.normal_power_log2)), it
        if edge == "npow10":
            assert subnormal_normal_weights(nd, p.normal_power_log2) > 0
        if edge == "sigma_z0":
            # the filter is off (agpt.h): every pixel comes back as its demodulated and remodulated mean
            al = dn.demodulation_albedo(alb)
            assert np.array_equal(bits(out[..., :3]), bits((dn.means(film, mom) / al) * al))


def subnormal_normal_weights(nd, normal_power_log2):
    """Taps at spacing 1 whose w_n (float32, as oracle/denoise.py forms it) is a subnormal: the case a flush to zero changes."""
    n = nd[..., :3]
    h, w = n.shape[:2]
    count = 0
    for dy in range(-2, 3):
        for dx in range(-2, 3):
            a = n[max(0, -dy):h - max(0, dy), max(0, -dx):w - max(0, dx)]
            b = n[max(0, dy):h + min(0, dy), max(0, dx):w + min(0, dx)]
            m = (a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1]) + a[..., 2] * b[..., 2]
            m = np.where(m > 0, m, F32(0)).astype(F32)
            with np.errstate(under="ignore"):
                for _ in range(normal_power_log2):
                    m = m * m
            count += int(((m > 0) & (m < np.finfo(F32).tiny)).sum())
    return count


# ---- guides over split batches ----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def small_batch_ctx(agpt):
    """A context whose batches hold 2^10 paths (AGPT_BATCH_LOG2 is read when a context is created)."""
    old = os.environ.get("AGPT_BATCH_LOG2")
    os.environ["AGPT_BATCH_LOG2"] = "10"
    try:
        ctx = agpt.Context(0)
    finally:
        if old is None:
            os.environ.pop("AGPT_BATCH_LOG2", None)
        else:
            os.environ["AGPT_BATCH_LOG2"] = old
    yield ctx
    ctx.close()


@pytest.mark.parametrize("w,h,n,batches", [(96, 54, 4, 4), (96, 54, 5, 5), (24, 16, 5, 3)])
def test_guides_over_split_batches(agpt, ectx, small_batch_ctx, w, h, n, batches):
    """96x54 with 2^10-path batches: one sample per batch; 24x16 (tiled, 384 pixels): batches of 2, 2 and 1 samples.  The guides
    equal the one-batch guides and the statement, and so does the denoised frame."""
    from oracle import guides_binding
    outs = []
    for ctx in (ectx, small_batch_ctx):
        d, hs, _ = setup(agpt, ctx, 5, w, h)
        ctx.clear(); ctx.render(0, 8, d["max_depth"], d["depth_arg"])
        ctx.reset_stats()
        ctx.render_guides(n)
        outs.append((ctx.stats().launches_closest, ctx.read_guides(), ctx.read_accum(), ctx.read_moments(), ctx.denoise(agpt.denoise_params())))
    (b1, g1, f1, m1, o1), (b2, g2, f2, m2, o2) = outs
    assert (b1, b2) == (1, batches)
    _, want_alb, want_nd = guides_binding.GuideScene(hs).guides(w, h, n)
    assert same_floats(g1[0], want_alb) and same_floats(g1[1], want_nd)
    assert np.array_equal(bits(g2[0]), bits(g1[0])) and np.array_equal(bits(g2[1]), bits(g1[1]))
    assert np.array_equal(bits(f2), bits(f1)) and np.array_equal(bits(m2), bits(m1))
    assert same_floats(o2[0], o1[0]) and np.array_equal(o2[1], o1[1])
    p = agpt.denoise_params()
    assert same_floats(o1[0], dn.denoise(f1, m1, want_alb, want_nd, p.iterations, p.sigma_luminance, p.sigma_depth, p.normal_power_log2))


# ---- synthetic film and moments ---------------------------------------------------------------------------------------------
ABOVE_2_24 = np.nextafter(F32(1 << 24), F32(np.inf))       # 2^24 + 2: 2^24 + 1 has no float32


def synthetic(w, h, seed):
    """(film, moments, edge pixel count) in film row order: random sums, with the edge table written over some pixels."""
    rng = np.random.default_rng(seed)
    N = w * h
    n = rng.integers(0, 41, N).astype(F32)
    mean = rng.uniform(0, 2, (N, 3)).astype(F32)
    a = (mean * n[:, None]).astype(F32)
    q = (a * mean * rng.uniform(0.9, 1.5, (N, 3)).astype(F32)).astype(F32)
    rows = []                                           # (n, a, q) with a and q per channel
    for k in (0, 1, 2, 3, 1 << 24):
        rows.append((k, mean[len(rows)] * F32(k), mean[len(rows)] * mean[len(rows)] * F32(k) * F32(1.2)))
    with np.errstate(over="ignore", invalid="ignore"):
        for k in (2, 3, 4, 7):
            for c in range(3):
                av = np.full(3, F32(1.7) * F32(k), F32) * rng.uniform(0.5, 1.5, 3).astype(F32)
                qv = av * (av / F32(k)) * F32(1.3)
                exact = av.copy(); qx = qv.copy(); qx[c] = av[c] * (av[c] / F32(k))                   # d = 0
                rows.append((k, exact, qx))
                qb = qx.copy(); qb[c] = np.nextafter(qx[c], F32(0))                                  # d one ulp below 0
                rows.append((k, av, qb))
                for av_c, qv_c in ((av[c], F32(np.inf)), (F32(np.inf), qv[c]), (F32(-np.inf), qv[c]), (F32(np.nan), qv[c]),
                                   (F32(-1.5), qv[c]), (F32(-1.5), F32(0.1)), (F32(1e-40), F32(1e-42)), (F32(1e-40), qv[c]),
                                   (av[c], F32(1e-42)), (F32(np.inf), F32(np.inf))):
                    ai = av.copy(); qi = qv.copy(); ai[c] = av_c; qi[c] = qv_c
                    rows.append((k, ai, qi))
    at = rng.permutation(N)[:len(rows)]
    assert len(rows) <= N
    for i, (k, av, qv) in zip(at, rows):
        n[i], a[i], q[i] = k, av, qv
    film = np.zeros((h, w, 4), F32); mom = np.zeros((h, w, 4), F32)
    film[..., :3] = a.reshape(h, w, 3); mom[..., :3] = q.reshape(h, w, 3); mom[..., 3] = n.reshape(h, w)
    return film, mom


SYNTH_PARAMS = [(2, 64, 4, TOL, FLOOR), (2, 1 << 24, 1, 0.0, 0.0), (2, 40, 8, 1.0, 0.5)]


@pytest.mark.parametrize("size", EDGE_SIZES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_synthetic_film_and_moments(agpt, ectx, size):
    """select, resolve_counts and denoise on written film and moments with the arithmetic edges; guides of cfg 1 stay fresh
    across agpt_write_accum and agpt_write_moments."""
    w, h = size
    setup(agpt, ectx, 1, w, h)
    ectx.render_guides(4)
    film, mom = synthetic(w, h, seed=w)
    ectx.write_accum(film); ectx.write_moments(mom)
    assert np.array_equal(bits(ectx.read_accum()), bits(film)) and np.array_equal(bits(ectx.read_moments()), bits(mom))
    alb, nd = ectx.read_guides()
    for q in SYNTH_PARAMS:
        p = agpt.adaptive(*q)
        n, pix = ectx.adaptive_select(p)
        want = st.selected_pixels(film, mom, p)
        assert n == len(want) and np.array_equal(np.sort(pix), want), q
    packed = ectx.resolve_counts()
    cnt = mom[..., 3]
    assert not packed[cnt == 0].any()
    for k in np.unique(cnt[cnt > 0]):
        assert np.array_equal(ectx.resolve(int(k))[cnt == k], packed[cnt == k]), k
    for it in (0, 1):
        p = agpt.denoise_params(iterations=it)
        out, rgb8 = ectx.denoise(p)
        assert same_floats(out, dn.denoise(film, mom, alb, nd, it, p.sigma_luminance, p.sigma_depth, p.normal_power_log2)), it
        if it == 0:
            assert np.array_equal(rgb8, packed)


def test_write_moments_refusals(agpt, ectx):
    """Counts that are negative, fractional, NaN, infinite or above 2^24 are refused, and so is any write with moments off; film
    and moments stay as they were."""
    w, h = EDGE_SIZES[0]
    setup(agpt, ectx, 1, w, h)
    film, mom = synthetic(w, h, seed=1)
    ectx.write_accum(film); ectx.write_moments(mom)
    for v in (-1.0, 2.5, np.nan, np.inf, ABOVE_2_24):
        bad = mom.copy(); bad[h // 2, w // 2, 3] = v
        with pytest.raises(agpt.AgptError, match="error -1"):
            ectx.write_moments(bad)
        assert np.array_equal(bits(ectx.read_accum()), bits(film)) and np.array_equal(bits(ectx.read_moments()), bits(mom)), v
    edge = mom.copy(); edge[0, 0, 3] = F32(1 << 24)
    ectx.write_moments(edge)                                  # 2^24 itself is a count
    ectx.set_moments(False)
    with pytest.raises(agpt.AgptError, match="error -3"):
        ectx.write_moments(mom)
    assert np.array_equal(bits(ectx.read_accum()), bits(film))


# ---- the convergence test against float64 -----------------------------------------------------------------------------------
def test_convergence_test_equals_float64(agpt, ectx):
    """cfg 5 at 96x54, 8 samples: the device's selection agrees with the float64 test from the library's own samples on every
    pixel whose se / thr is not within 1e-3 of 1, and fewer than 1 % of the pixels are that close."""
    w, h, spp = 96, 54, 8
    d, _, li = setup(agpt, ectx, 5, w, h)
    ectx.clear(); ectx.render(0, spp, d["max_depth"], d["depth_arg"])
    ys, xs = np.divmod(np.arange(w * h, dtype=np.int32), w)
    samples = np.stack([li(xs, ys, np.full(w * h, s, np.int32)) for s in range(spp)], axis=1)
    _, pix = ectx.adaptive_select(agpt.adaptive(4, 32, 4, TOL, FLOOR))
    got = np.zeros(w * h, bool); got[pix] = True
    want, border = convergence_f64(samples, TOL, FLOOR)
    print(f"convergence f64 vs device: {int(border.sum())} borderline of {w * h}, {int(want.sum())} unconverged")
    assert 0 < want.sum() < w * h and border.sum() < 0.01 * w * h
    assert np.array_equal(got[~border], want[~border])


# ---- the debug build -----------------------------------------------------------------------------------------------------------
def test_no_failed_device_checks(ectx):
    """Meaningful under AGPT_LIB=libagpt_debug.so (test_debug_build_runs_this_file); a release build runs no checks."""
    s = ectx.debug_status()
    print("FILM_EDGES_DEBUG_STATUS", s["failed"], s["first_code"], s["first_value"], s["checks"])
    assert s["failed"] == 0


def test_debug_build_runs_this_file():
    """The tests above under libagpt_debug.so (list, slot, sample-range and tap indices checked inside the kernels): none may
    fail.  Own process: the library is chosen at load time."""
    lib = os.path.join(ROOT, "ag-pathtracer_b200", "libagpt_debug.so")
    assert os.path.exists(lib)
    env = dict(os.environ, AGPT_LIB=lib)
    out = subprocess.run([sys.executable, "-m", "pytest", "-q", "-s", "-p", "no:cacheprovider", os.path.abspath(__file__), "-k",
                          "not debug_build"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if "FILM_EDGES_DEBUG_STATUS" in l][0]
    failed, checks = [int(v) for v in line.split("FILM_EDGES_DEBUG_STATUS")[1].split()[0:4:3]]
    assert checks > 100_000 and failed == 0
