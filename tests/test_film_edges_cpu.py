"""CPU: the float32 statements of adaptive sampling (oracle/adaptive.py) and of the denoiser (oracle/denoise.py) against plain
float64 computations of the same quantities.

The kernels match the statements bit for bit, but the statements were written with the kernels, so a slip they share (the
variance divided by n instead of n - 1, a tap weight off by a factor) would pass every bit-exact test.  The references here are
written from the formulas of include/agpt.h alone: the convergence test from the raw samples (two-pass variance), the
denoiser's prepare step and a-trous passes as explicit per-pixel tap loops.  tests/test_gpu_film_edges.py runs the same
convergence check against the device."""
import os
import sys
import time

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import adaptive as st  # noqa: E402
from oracle import denoise as dn  # noqa: E402

F32 = np.float32
W, H, SPP, GUIDE_SPP = 48, 27, 8, 4
TOL, FLOOR = 0.2, 0.02
BAND = 1e-3          # se / thr this close to 1: float32 rounding may decide either way


# ---- float64 references ----------------------------------------------------------------------------------------------------
def convergence_f64(samples, tolerance, floor):
    """samples: [N, n, 3] radiance of N pixels (n samples each).  Per channel in float64 from the samples the film adds: the mean,
    the unbiased variance (two-pass), se = sqrt(var / n) and thr = tolerance * max(mean, floor).  Returns (unconverged [N]: some
    channel's se > thr, borderline [N]: some channel's se / thr within BAND of 1).  tolerance and floor are taken as the float32
    values the device receives."""
    c = st.filter_samples(samples).astype(np.float64)
    n = c.shape[1]
    mean = c.mean(axis=1)
    var = c.var(axis=1, ddof=1)
    se = np.sqrt(var / n)
    thr = float(F32(tolerance)) * np.maximum(mean, float(F32(floor)))
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = se / thr
    return (se > thr).any(axis=-1), (np.abs(ratio - 1) <= BAND).any(axis=-1)


LUM64 = (0.212671, 0.715160, 0.072169)
H64 = (1 / 16, 1 / 4, 3 / 8, 1 / 4, 1 / 16)


def prepare_f64(film, moments, albedo, normal_depth):
    """include/agpt.h's per-pixel quantities in float64: E = (e.rgb, v_l), normal, depth and the miss flag."""
    a, q, n = film[..., :3].astype(np.float64), moments[..., :3].astype(np.float64), moments[..., 3:4].astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        mu = np.where(n > 0, a / n, 0.0)
        var_of_mean = np.where(n >= 2, np.maximum((q - n * mu * mu) / (n - 1), 0.0) / n, 0.0)
    al = np.maximum(albedo[..., :3].astype(np.float64), 0.01)
    E = np.empty(film.shape, np.float64)
    E[..., :3] = mu / al
    E[..., 3] = sum(LUM64[c] ** 2 * var_of_mean[..., c] / al[..., c] ** 2 for c in range(3))
    return E, normal_depth[..., :3].astype(np.float64), normal_depth[..., 3].astype(np.float64), albedo[..., 3] == 0, al


def atrous_f64(E, normal, depth, missed, step, sigma_l, sigma_z, normal_power_log2):
    """One a-trous pass over every pixel with explicit tap loops (a tap outside the film, a non-finite tap or weight is skipped;
    a pixel without weight keeps its value).  Returns (the new E, underflow [H, W]: some tap whose share of the pixel's weight
    is above 1e-7 has a weight w with w * w below FLT_MIN, where float32 keeps fewer bits of the variance's weights or none --
    the normal power 2^128 of a mean normal shorter than about 0.8 does that)."""
    Hh, Ww = E.shape[:2]
    out = E.copy()
    underflow = np.zeros((Hh, Ww), bool)
    lum = lambda e: LUM64[0] * e[0] + LUM64[1] * e[1] + LUM64[2] * e[2]
    for r in range(Hh):
        for x in range(Ww):
            ep = E[r, x]
            if not np.isfinite(ep).all():
                continue
            sw, sv, se, tiny = 0.0, 0.0, np.zeros(3), 0.0
            for dy in range(-2, 3):
                for dx in range(-2, 3):
                    rq, xq = r + dy * step, x + dx * step
                    if not (0 <= rq < Hh and 0 <= xq < Ww) or not np.isfinite(E[rq, xq]).all():
                        continue
                    eq = E[rq, xq]
                    wl = 1 / (1 + (lum(ep) - lum(eq)) ** 2 / (sigma_l ** 2 * ep[3] + 1e-4))
                    wn = max(float(normal[r, x] @ normal[rq, xq]), 0.0) ** (2 ** normal_power_log2)
                    if missed[r, x] or missed[rq, xq]:
                        wz = 1.0 if missed[r, x] and missed[rq, xq] else 0.0
                    else:
                        with np.errstate(divide="ignore", invalid="ignore"):
                            wz = 1 / (1 + np.float64(abs(depth[r, x] - depth[rq, xq])) / (sigma_z * depth[r, x]))
                    w = H64[dx + 2] * H64[dy + 2] * wl * wn * wz
                    if not np.isfinite(w):
                        continue
                    sw += w; se += w * eq[:3]; sv += w * w * eq[3]
                    if 0 < w < SQRT_FLT_MIN:
                        tiny = max(tiny, w)
            underflow[r, x] = tiny > 1e-7 * sw
            if sw > 0:
                out[r, x, :3], out[r, x, 3] = se / sw, sv / sw ** 2
    return out, underflow


SQRT_FLT_MIN = float(np.sqrt(np.finfo(F32).tiny))


# ---- inputs: the oracle port's radiance of cfg 5 --------------------------------------------------------------------------
@pytest.fixture(scope="module")
def scene(agpt):
    from oracle import guides_binding, port_binding
    if not (port_binding.available() and guides_binding.available()):
        pytest.fail("oracle libraries not built: run __graft_entry__.build()")
    cfg = 5
    d = agpt.config_defaults(cfg)
    hs = agpt.HostScene(cfg, 2)
    ps = port_binding.PortScene(hs)
    li = lambda xs, ys, ss: ps.li_pixels(W, H, xs, ys, ss, d["max_depth"], d["depth_arg"])[0]
    ys, xs = np.divmod(np.arange(W * H, dtype=np.int32), W)
    samples = np.stack([li(xs, ys, np.full(W * H, s, np.int32)) for s in range(SPP)], axis=1)     # [W*H, SPP, 3], image order
    film, mom = st.render_uniform(li, W, H, 0, SPP)
    _, alb, nd = guides_binding.GuideScene(hs).guides(W, H, GUIDE_SPP)
    return samples, film, mom, alb, nd


def test_convergence_test_equals_float64(scene):
    """The statement's selection (float32, from film and moments) agrees with the float64 test (from the samples) on every pixel
    whose se / thr is not within 1e-3 of 1.  Dividing by n instead of n - 1 moves se by sqrt(7/8) at 8 samples: it fails here."""
    samples, film, mom, _, _ = scene
    want, border = convergence_f64(samples, TOL, FLOOR)                      # (n = 8: the cap of 32 is far)
    got = st.selected(film, mom, 4, 32, 4, TOL, FLOOR)[::-1].reshape(-1)      # film row order -> image order
    print(f"convergence f64 vs statement: {int(border.sum())} borderline of {W * H}, {int(want.sum())} unconverged")
    assert 0 < want.sum() < W * H
    assert border.sum() < 0.01 * W * H
    assert np.array_equal(got[~border], want[~border])


def rel_diff(got, want):
    """|got - want| relative to |want|, values below 1e-3 of the mean magnitude measured against that floor instead."""
    return np.abs(got - want) / np.maximum(np.abs(want), 1e-3 * np.abs(want).mean())


# Per pass, the largest relative difference between the float32 statement and the float64 pass fed the statement's own input,
# over the pixels whose weights stay in float32's normal range (e.rgb and v_l of the pass).  Measured on this film: 6.0e-6 at
# 1 and at 5 passes; 2.5 % (1 pass) and 3.2 % (5 passes) of the pixel passes underflow and are left out.
PASS_REL_TOL = 1e-4


@pytest.mark.parametrize("iterations", [1, 5])
def test_denoise_equals_float64(scene, iterations):
    """The float32 statement against the float64 restatement (defaults: sigma_l 8, sigma_z 0.1, normal power 2^7): prepare,
    then each a-trous pass fed the statement's own input, so a pass's rounding is measured alone.  The luminance variance of
    prepare is compared directly: divided by n instead of n - 1 it is 8/7 of the right one at 8 samples.  The chain of passes is
    denoise.denoise's output."""
    _, film, mom, alb, nd = scene
    E32, G = dn.prepare(film, mom, alb, nd)
    E64, normal, depth, missed, al = prepare_f64(film, mom, alb, nd)
    assert np.isfinite(E32).all()
    assert rel_diff(E32, E64).max() <= 1e-5
    t0 = time.time()
    worst, lost = 0.0, 0
    for i in range(iterations):
        nxt32 = dn.atrous(E32, G, 1 << i, 8.0, 0.1, 7)
        nxt64, underflow = atrous_f64(E32.astype(np.float64), normal, depth, missed, 1 << i, 8.0, 0.1, 7)
        worst = max(worst, float(rel_diff(nxt32, nxt64)[~underflow].max()))
        lost += int(underflow.sum())
        assert not np.array_equal(nxt32, E32)                                  # the pass did something
        E32 = nxt32
    print(f"denoise f64 vs statement, {iterations} passes: max rel per pass {worst:.2e}, {lost} pixel passes underflow of "
          f"{iterations * W * H}, {time.time() - t0:.1f} s")
    assert worst <= PASS_REL_TOL and lost < 0.05 * iterations * W * H
    got = dn.denoise(film, mom, alb, nd, iterations, 8.0, 0.1, 7)
    assert np.array_equal(got[..., :3], E32[..., :3] * dn.demodulation_albedo(alb))
