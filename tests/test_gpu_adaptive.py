"""GPU: adaptive sampling (agpt_set_moments, agpt_adaptive_select, agpt_render_adaptive, agpt_resolve_counts).

NOT REFERENCE BEHAVIOUR: the reference gives every pixel the same number of samples.  The feature is stated on the CPU in
oracle/adaptive.py; these tests hold the library to that statement bit for bit, driven by the library's own single-path
radiances (agpt_li_pixels), and to the property the design makes exact: each pixel of an adaptive film equals the same pixel of
a plain agpt_render(0, n_p) film, n_p being the samples that pixel received."""
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

W, H = 96, 54
LEVELS = {1: 0, 5: 2, 8: 3}
# tolerance and floor: on each of these films they leave at least three distinct final counts, some pixels at min and some at max
TOL, FLOOR = 0.2, 0.02


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def same_floats(a, b):
    """Bit-equal, or NaN on both sides."""
    a = np.ascontiguousarray(a, np.float32); b = np.ascontiguousarray(b, np.float32)
    return bool(np.all((bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))))


@pytest.fixture(scope="module")
def actx(agpt):
    """A context of this file's own: moments are switched on and off here, other files' contexts stay as they are."""
    if agpt.device_count() == 0:
        pytest.fail("no CUDA device visible: -m gpu tests must run on the GPU box")
    ctx = agpt.Context(0)
    yield ctx
    ctx.close()


def setup(agpt, ctx, cfg):
    d = agpt.config_defaults(cfg)
    hs = agpt.HostScene(cfg, LEVELS[cfg])
    hs.upload(ctx); ctx.set_film(W, H)
    li = lambda xs, ys, ss: ctx.li_pixels(xs, ys, ss, d["max_depth"], d["depth_arg"])
    return d, hs, li


def params(agpt, mn=4, mx=32, step=4):
    return agpt.adaptive(mn, mx, step, TOL, FLOOR)


def adaptive_run(agpt, ctx, cfg):
    """render_adaptive of cfg at W x H: film, moments, rounds, paths."""
    d, hs, _ = setup(agpt, ctx, cfg)
    ctx.set_moments(True)
    rounds, paths = ctx.render_adaptive(params(agpt), d["max_depth"], d["depth_arg"])
    return ctx.read_accum().copy(), ctx.read_moments().copy(), rounds, paths


@pytest.mark.parametrize("cfg", [5, 8])
def test_moments_change_no_film_and_match_the_statement(agpt, actx, cfg):
    spp = 6
    d, hs, li = setup(agpt, actx, cfg)
    actx.set_moments(False)
    actx.clear(); actx.render(0, spp, d["max_depth"], d["depth_arg"])
    plain = actx.read_accum().copy()
    actx.set_moments(True)
    actx.clear(); actx.render(0, 2, d["max_depth"], d["depth_arg"]); actx.render(2, spp - 2, d["max_depth"], d["depth_arg"])
    film, mom = actx.read_accum().copy(), actx.read_moments().copy()
    assert np.array_equal(bits(film), bits(plain))
    want_film, want_mom = st.render_uniform(li, W, H, 0, spp)
    assert same_floats(film[..., :3], want_film[..., :3])
    assert same_floats(mom, want_mom)
    assert (mom[..., 3] == spp).all()
    actx.clear()
    assert not actx.read_moments().any()
    actx.set_moments(False)


@pytest.mark.parametrize("cfg", [1, 5, 8])
def test_select_equals_the_statement(agpt, actx, cfg):
    d, hs, li = setup(agpt, actx, cfg)
    actx.set_moments(True)
    p = params(agpt)
    actx.clear(); actx.render(0, p.min_samples, d["max_depth"], d["depth_arg"])
    film, mom = actx.read_accum(), actx.read_moments()
    n, pix = actx.adaptive_select(p)
    want = st.selected_pixels(film, mom, p)
    assert n == len(pix) == len(want) and 0 < n < W * H
    assert np.array_equal(np.sort(pix), want)
    assert actx.adaptive_select(p, want_pixels=False)[0] == n
    # the list keeps the 8x4 tiles together: consecutive entries are mostly neighbours
    ys, xs = np.divmod(pix, W)
    near = (np.abs(np.diff(xs)) <= 7) & (np.abs(np.diff(ys)) <= 3)
    assert near.mean() > 0.5
    actx.set_moments(False)


@pytest.mark.parametrize("cfg", [1, 5, 8])
def test_render_adaptive(agpt, actx, cfg):
    """Film, moments, rounds and paths equal the statement's; counts in [min, max]; nothing selected at the end; per count k
    the pixels equal a plain agpt_render(0, k) film and agpt_resolve(k) byte for byte."""
    d, hs, li = setup(agpt, actx, cfg)
    p = params(agpt)
    film, mom, rounds, paths = adaptive_run(agpt, actx, cfg)
    want_film, want_mom, want_rounds, want_paths, sizes = st.render_adaptive(li, W, H, p)
    assert same_floats(film[..., :3], want_film[..., :3])
    assert same_floats(mom, want_mom)
    assert (rounds, paths) == (want_rounds, want_paths)
    n = mom[..., 3].astype(np.int64)
    print(f"cfg{cfg}: rounds {rounds} of sizes {sizes}, counts {dict(zip(*np.unique(n, return_counts=True)))}")
    assert n.min() == p.min_samples and n.max() == p.max_samples and len(np.unique(n)) >= 3
    assert ((n - p.min_samples) % p.step == 0).all() and paths == n.sum()
    assert rounds <= (p.max_samples - p.min_samples) // p.step
    assert actx.adaptive_select(p)[0] == 0
    packed = actx.resolve_counts()
    actx.set_moments(False)
    for k in np.unique(n):
        actx.clear(); actx.render(0, int(k), d["max_depth"], d["depth_arg"])
        m = n == k
        assert np.array_equal(bits(actx.read_accum()[m]), bits(film[m])), k
        assert np.array_equal(actx.resolve(int(k))[m], packed[m]), k                  # (both in film row order, like m)


def test_host_mirror_render_adaptive(agpt, actx):
    cfg = 5
    film, mom, _, _ = adaptive_run(agpt, actx, cfg)
    actx.set_moments(False)
    d = agpt.config_defaults(cfg)
    hs = agpt.HostScene(cfg, LEVELS[cfg])
    tr = agpt.HostTracer(d["max_depth"], 0)
    acc = np.full((H, W, 4), 7, np.float32)
    counts = tr.render_adaptive(hs, W, H, acc, params(agpt), d["depth_arg"])
    tr.close()
    assert np.array_equal(bits(acc[..., :3]), bits(film[..., :3]))
    assert np.array_equal(counts, mom[::-1, :, 3].astype(np.int32))


def _dump(path):
    """Subprocess body of test_rounds_split_into_batches: the render_adaptive cases into an npz."""
    from tests.conftest import load_agpt
    agpt = load_agpt()
    ctx = agpt.Context(0)
    out = {}
    for cfg in LEVELS:
        film, mom, rounds, paths = adaptive_run(agpt, ctx, cfg)
        out[f"film{cfg}"], out[f"mom{cfg}"], out[f"rp{cfg}"] = film, mom, np.array([rounds, paths])
    ctx.close()
    np.savez(path, **out)


def test_rounds_split_into_batches(agpt, actx, tmp_path):
    """With batches of 2^10 paths a round of more than 256 pixels at step 4 runs in several batches of whole pixels: the
    results are identical to one batch per round."""
    path = str(tmp_path / "batched.npz")
    env = dict(os.environ, AGPT_BATCH_LOG2="10")
    out = subprocess.run([sys.executable, os.path.abspath(__file__), path], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1200)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    got = np.load(path)
    split = False
    for cfg in LEVELS:
        film, mom, rounds, paths = adaptive_run(agpt, actx, cfg)
        assert np.array_equal(bits(got[f"film{cfg}"]), bits(film)) and np.array_equal(bits(got[f"mom{cfg}"]), bits(mom))
        assert got[f"rp{cfg}"].tolist() == [rounds, paths]
        split = split or (rounds > 0 and (paths - W * H * 4) // 4 > 256 * rounds)     # a round of more than one batch's pixels
    assert split
    actx.set_moments(False)


def test_refusals_leave_film_and_moments(agpt, actx):
    cfg = 5
    d, hs, _ = setup(agpt, actx, cfg)
    actx.set_moments(True)
    actx.clear(); actx.render(0, 4, d["max_depth"], d["depth_arg"])
    film, mom = actx.read_accum().copy(), actx.read_moments().copy()
    good = dict(min_samples=4, max_samples=32, step=4, tolerance=0.1, floor=0.0)
    bad = [dict(min_samples=1), dict(min_samples=40), dict(max_samples=(1 << 24) + 1), dict(step=0), dict(tolerance=-0.1),
           dict(floor=-1.0), dict(tolerance=float("inf")), dict(floor=float("nan"))]
    for b in bad:
        q = dict(good, **b)
        p = agpt.adaptive(q["min_samples"], q["max_samples"], q["step"], q["tolerance"], q["floor"])
        with pytest.raises(agpt.AgptError, match="error -1"):
            actx.adaptive_select(p)
        with pytest.raises(agpt.AgptError, match="error -1"):
            actx.render_adaptive(p, d["max_depth"], d["depth_arg"])
    assert np.array_equal(bits(actx.read_accum()), bits(film)) and np.array_equal(bits(actx.read_moments()), bits(mom))
    p = agpt.adaptive(**good)
    fresh = agpt.Context(0)                                    # no film, scene or camera yet
    fresh.set_moments(True)
    with pytest.raises(agpt.AgptError, match="error -3"):
        fresh.render_adaptive(p, d["max_depth"])
    fresh.set_film(W, H)
    with pytest.raises(agpt.AgptError, match="error -3"):
        fresh.render_adaptive(p, d["max_depth"])               # no scene
    fresh.close()
    actx.set_moments(False)                                    # moments off: state errors, film untouched
    for call in (lambda: actx.render_adaptive(p, d["max_depth"]), lambda: actx.adaptive_select(p), actx.read_moments, actx.resolve_counts):
        with pytest.raises(agpt.AgptError, match="error -3"):
            call()
    assert np.array_equal(bits(actx.read_accum()), bits(film))


def test_no_failed_device_checks(actx):
    """Meaningful under AGPT_LIB=libagpt_debug.so (test_debug_build_runs_this_file); a release build runs no checks."""
    s = actx.debug_status()
    print("ADAPTIVE_DEBUG_STATUS", s["failed"], s["first_code"], s["first_value"], s["checks"])
    assert s["failed"] == 0


def test_debug_build_runs_this_file():
    """The tests above under libagpt_debug.so (list indices and per-pixel sample ranges checked inside the new kernels): none
    may fail.  Own process: the library is chosen at load time."""
    lib = os.path.join(ROOT, "ag-pathtracer_b200", "libagpt_debug.so")
    assert os.path.exists(lib)
    env = dict(os.environ, AGPT_LIB=lib)
    out = subprocess.run([sys.executable, "-m", "pytest", "-q", "-s", "-p", "no:cacheprovider", os.path.abspath(__file__), "-k",
                          "not debug_build and not batches and not host_mirror"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if "ADAPTIVE_DEBUG_STATUS" in l][0]
    failed, checks = [int(v) for v in line.split("ADAPTIVE_DEBUG_STATUS")[1].split()[0:4:3]]
    assert checks > 100_000 and failed == 0


if __name__ == "__main__":
    _dump(sys.argv[1])
