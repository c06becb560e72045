"""The a-trous denoiser (extension, include/agpt.h agpt_denoise) stated on the CPU -- TEST INFRASTRUCTURE.

numpy, float32 throughout, every operation rounded on its own (numpy never fuses a multiply into an add), so each step is the
device's step bit for bit.  The filter loops over the 25 taps, dy outer and dx inner, and adds one tap to every pixel's sums per
step: each pixel's sums run in the stated order (no np.sum, no reordering).

Inputs are what the library keeps and returns: film, moments, albedo and normal/depth guides, each [H, W, 4] float32 in the
film's row order (row H-1-y holds image row y).  Taps are offsets in those buffer rows and columns.
"""
import numpy as np

F32 = np.float32
EPS_A = F32(0.01)          # albedo floor of the demodulation
EPS_L = F32(1e-4)          # luminance edge stop floor
LUM = (F32(0.212671), F32(0.715160), F32(0.072169))
H5 = (F32(1 / 16), F32(1 / 4), F32(3 / 8), F32(1 / 4), F32(1 / 16))


def lum(e):
    return (LUM[0] * e[..., 0] + LUM[1] * e[..., 1]) + LUM[2] * e[..., 2]


def means(film, moments):
    """mu = a / n per channel, 0 where n = 0 (k_resolve_counts' division)."""
    n = moments[..., 3:4]
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        return np.where(n > 0, film[..., :3] / n, F32(0)).astype(F32)


def variance_of_mean(film, moments):
    """v / n per channel with the convergence test's arithmetic (oracle/adaptive.py), 0 where n < 2."""
    a, q, n = film[..., :3], moments[..., :3], moments[..., 3:4]
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        mu = a / n
        d = q - a * mu
        v = d / (n - F32(1))
        v = np.where(v < 0, F32(0), v)
        var = v / n
    return np.where(n >= 2, var, F32(0)).astype(F32)


def demodulation_albedo(albedo):
    al = albedo[..., :3]
    return np.where(al > EPS_A, al, EPS_A).astype(F32)


def prepare(film, moments, albedo, normal_depth):
    """(E = [H, W, 4] (e.rgb, v_l), G = [H, W, 4] (normal, depth or -1 for a pixel that missed)), as k_denoise_prepare."""
    mu = means(film, moments)
    var = variance_of_mean(film, moments)
    al = demodulation_albedo(albedo)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        t = [((LUM[c] * LUM[c]) * var[..., c]) / (al[..., c] * al[..., c]) for c in range(3)]
        vl = (t[0] + t[1]) + t[2]
        E = np.concatenate([mu / al, vl[..., None]], axis=-1).astype(F32)
    G = normal_depth.astype(F32).copy()
    G[..., 3] = np.where(albedo[..., 3] == 0, F32(-1), normal_depth[..., 3])
    return E, G


def finite4(x):
    return np.isfinite(x).all(axis=-1)


def atrous(E, G, step, sigma_l, sigma_z, normal_pow):
    """One pass of k_denoise_atrous at tap spacing `step`: the new E."""
    Hh, W = E.shape[:2]
    sl, sz = F32(sigma_l), F32(sigma_z)
    valid_p = finite4(E)
    lp = lum(E)
    miss_p = G[..., 3] < 0
    sw = np.zeros((Hh, W), F32)
    sv = np.zeros((Hh, W), F32)
    se = np.zeros((Hh, W, 3), F32)
    rows, cols = np.meshgrid(np.arange(Hh), np.arange(W), indexing="ij")
    with np.errstate(divide="ignore", invalid="ignore", over="ignore", under="ignore"):
        den = (sl * sl) * E[..., 3] + EPS_L
        for dy in range(-2, 3):
            for dx in range(-2, 3):
                rq, xq = rows + dy * step, cols + dx * step
                inside = (rq >= 0) & (rq < Hh) & (xq >= 0) & (xq < W)
                rqc, xqc = np.clip(rq, 0, Hh - 1), np.clip(xq, 0, W - 1)
                eq, gq = E[rqc, xqc], G[rqc, xqc]
                dl = lp - lum(eq)
                wl = F32(1) / (F32(1) + (dl * dl) / den)
                m = (G[..., 0] * gq[..., 0] + G[..., 1] * gq[..., 1]) + G[..., 2] * gq[..., 2]
                m = np.where(m > 0, m, F32(0)).astype(F32)
                for _ in range(normal_pow):
                    m = m * m
                miss_q = gq[..., 3] < 0
                wz_hit = F32(1) / (F32(1) + np.abs(G[..., 3] - gq[..., 3]) / (sz * G[..., 3]))
                wz = np.where(miss_p & miss_q, F32(1), np.where(miss_p != miss_q, F32(0), wz_hit)).astype(F32)
                w = (((H5[dx + 2] * H5[dy + 2]) * wl) * m) * wz
                take = valid_p & inside & finite4(eq) & np.isfinite(w)
                w = np.where(take, w, F32(0)).astype(F32)
                sw = np.where(take, sw + w, sw)
                for c in range(3):
                    se[..., c] = np.where(take, se[..., c] + w * eq[..., c], se[..., c])
                sv = np.where(take, sv + (w * w) * eq[..., 3], sv)
        e2 = np.concatenate([se / sw[..., None], (sv / (sw * sw))[..., None]], axis=-1).astype(F32)
    keep = ~valid_p | ~(sw > 0) | ~finite4(e2)
    return np.where(keep[..., None], E, e2).astype(F32)


def denoise(film, moments, albedo, normal_depth, iterations, sigma_luminance, sigma_depth, normal_power_log2):
    """agpt_denoise's float output [H, W, 4] (out.w = 0)."""
    if iterations == 0:
        out = np.zeros_like(film, dtype=F32)
        out[..., :3] = means(film, moments)
        return out
    E, G = prepare(film, moments, albedo, normal_depth)
    for i in range(iterations):
        E = atrous(E, G, 1 << i, sigma_luminance, sigma_depth, normal_power_log2)
    out = np.zeros_like(film, dtype=F32)
    with np.errstate(over="ignore", invalid="ignore"):
        out[..., :3] = E[..., :3] * demodulation_albedo(albedo)
    return out
