"""CPU: the statement of adaptive sampling (oracle/adaptive.py) -- the convergence test on constructed inputs, and its film
sums tied to the oracle port's own render bit for bit."""
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import adaptive as st

F32 = np.float32


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def one_pixel(samples):
    """film and moments [1, 1, 4] of one pixel that received `samples` ([k, 3])."""
    film = np.zeros((1, 1, 4), F32); mom = np.zeros((1, 1, 4), F32)
    st.accumulate(film, mom, np.array([0]), np.array([0]), np.asarray(samples, F32)[None])
    return film, mom


def sel(film, mom, mn=2, mx=64, step=4, tol=0.05, floor=0.0):
    return bool(st.selected(film, mom, mn, mx, step, tol, floor)[0, 0])


def test_zero_variance_is_not_selected():
    for v in (0.0, 0.3, 1.7, 123.0):
        film, mom = one_pixel(np.full((2, 3), v))
        assert not sel(film, mom, tol=0.0 if v else 0.05)
    # a black sky pixel: mu = 0 = floor, se = 0 <= 0
    film, mom = one_pixel(np.zeros((2, 3)))
    assert not sel(film, mom, tol=0.0, floor=0.0)


def test_rounding_below_zero_is_not_selected():
    """Equal samples whose sum of squares rounds below a * mu: d < 0, v is clamped to 0, se = 0."""
    found = 0
    rng = np.random.default_rng(3)
    for v in rng.uniform(0.01, 10, 2000).astype(F32):
        for k in (3, 5, 7):
            film, mom = one_pixel(np.full((k, 3), v))
            a, q, n = film[0, 0, 0], mom[0, 0, 0], mom[0, 0, 3]
            if q - a * (a / n) < 0:
                found += 1
                assert not sel(film, mom, tol=0.0)
    assert found > 10


def test_non_finite_sums_are_selected_until_max():
    """Sums of finite samples that overflow (cfg 8's 3e38 light): squares past FLT_MAX, or film and squares both, make se
    infinite or NaN; a NaN anywhere does too.  Such a pixel samples on whatever the tolerance, up to the cap."""
    film, mom = one_pixel(np.array([[1, 1, 1], [2, 2, 2]], F32))
    cases = []
    m = mom.copy(); m[0, 0, 2] = np.inf; cases.append((film, m))                        # d = inf
    f = film.copy(); f[0, 0, 1] = np.inf; m = mom.copy(); m[0, 0, 1] = np.inf
    cases.append((f, m))                                                                 # d = inf - inf = NaN
    f = film.copy(); f[0, 0, 0] = np.nan; cases.append((f, mom))
    m = mom.copy(); m[0, 0, 1] = np.nan; cases.append((film, m))
    for f, m in cases:
        assert sel(f, m, tol=1e3, floor=1e3)
        m = m.copy(); m[0, 0, 3] = 61
        assert not sel(f, m, mx=64, step=4, tol=1e3, floor=1e3)      # the cap still holds


def test_the_sample_cap():
    film, mom = one_pixel(np.array([[0, 0, 0], [5, 5, 5]], F32))        # very noisy
    for n, mx, step, want in ((2, 64, 4, True), (60, 64, 4, True), (61, 64, 4, False), (64, 64, 1, False), (63, 64, 1, True)):
        m = mom.copy(); m[0, 0, 3] = n
        assert sel(film, m, mx=mx, step=step) == want, (n, mx, step)


def test_the_floor_for_dark_pixels():
    """A dark pixel with a small absolute error: selected against its own mean, not against a floor above its mean."""
    film, mom = one_pixel(np.array([[0.001, 0.001, 0.001], [0.003, 0.003, 0.003]], F32))
    assert sel(film, mom, tol=0.1, floor=0.0)                           # se / mu = 0.5
    assert not sel(film, mom, tol=0.1, floor=0.02)                      # se = 0.001 <= 0.1 * 0.02
    assert sel(film, mom, tol=0.1, floor=0.005)                         # 0.001 > 0.0005


def test_every_channel_counts():
    film, mom = one_pixel(np.array([[1, 1, 0], [1, 1, 4]], F32))
    assert sel(film, mom, tol=0.01)
    film, mom = one_pixel(np.array([[1, 1, 0], [1, 1, 0]], F32))
    assert not sel(film, mom, tol=0.0)


def test_filter_zeroes_and_counts():
    film, mom = one_pixel(np.array([[np.nan, 1, 1], [1, 2, 3], [np.inf, 0, 0]], F32))
    assert film[0, 0, :3].tolist() == [1, 2, 3]
    assert mom[0, 0, :3].tolist() == [1, 4, 9] and mom[0, 0, 3] == 3


@pytest.fixture(scope="module")
def port():
    from oracle import port_binding
    if not port_binding.available():
        pytest.fail("oracle/libagpt_oracle.so is not built (build())")
    return port_binding


@pytest.mark.parametrize("cfg,level,W,H,spp", [(5, 2, 32, 20, 6), (8, 3, 40, 24, 6)])
def test_uniform_statement_equals_the_port_render(agpt, port, cfg, level, W, H, spp):
    """The statement's film of per-path li_pixels radiances == the port's own render, bit for bit (same filter, same order);
    cfg 8 has inf and NaN samples."""
    d = agpt.config_defaults(cfg)
    hs = agpt.HostScene(cfg, level); ps = port.PortScene(hs)
    li = lambda xs, ys, ss: ps.li_pixels(W, H, xs, ys, ss, d["max_depth"], d["depth_arg"])[0]
    film, mom = st.render_uniform(li, W, H, 0, spp)
    want, _ = ps.render(W, H, 0, spp, d["max_depth"], d["depth_arg"])
    assert np.array_equal(bits(film[..., :3]), bits(want[..., :3]))
    assert (mom[..., 3] == spp).all()
    if cfg == 8:
        ys, xs = np.divmod(np.arange(W * H, dtype=np.int32), W)
        raw = np.stack([li(xs, ys, np.full(W * H, s, np.int32)) for s in range(spp)])
        assert not np.isfinite(raw).all(), "cfg 8 produces inf and NaN samples"


def test_round_loop_on_a_synthetic_radiance():
    """The round loop: every count in [min, max], final state selects nothing, counts step by `step`, and the film of each
    pixel is the uniform film of its own count."""
    W, H = 16, 8
    P = SimpleNamespace(min_samples=4, max_samples=32, step=4, tolerance=0.05, floor=0.01)

    def li(xs, ys, ss):
        # noise that grows to the right, a black column at x = 0, a NaN in some samples of x = 3
        u = ((xs * 7919 + ys * 104729 + ss * 1299709) % 1000).astype(F32) / F32(1000)
        v = (F32(0.5) + (xs.astype(F32) / F32(W)) * (u - F32(0.5))).astype(F32)
        v = np.where(xs == 0, F32(0), v)
        out = np.repeat(v[:, None], 3, 1).astype(F32)
        out[(xs == 3) & (ss % 5 == 0), 1] = np.nan
        return out
    film, mom, rounds, paths, sizes = st.render_adaptive(li, W, H, P)
    n = mom[..., 3]
    assert n.min() >= P.min_samples and n.max() <= P.max_samples and ((n - P.min_samples) % P.step == 0).all()
    assert len(st.selected_pixels(film, mom, P)) == 0
    assert rounds == len(sizes) <= (P.max_samples - P.min_samples) // P.step
    assert paths == n.sum()
    assert len(np.unique(n)) >= 3
    for k in np.unique(n):
        f, _ = st.render_uniform(li, W, H, 0, int(k))
        m = n == k
        assert np.array_equal(bits(f[m]), bits(film[m]))
