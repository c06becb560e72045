"""Adaptive sampling (extension, include/agpt.h agpt_adaptive) stated on the CPU -- TEST INFRASTRUCTURE.

numpy, float32 throughout, every operation rounded on its own (numpy never fuses a multiply into an add), so each step is the
device's step bit for bit:
  * the film filter of k_accumulate (myapp.cpp:169-172): a sample with a NaN channel or an infinite luminance becomes 0;
  * film and moments as sequential float32 sums in ascending sample order: film.xyz += c, moments.xyz += c * c, moments.w += 1;
  * the convergence test of agpt_adaptive_select, element for element;
  * the round loop of agpt_render_adaptive, driven by a function li(xs, ys, ss) -> float32 [N, 3] that returns the radiance of
    the camera paths (pixel xs[i], ys[i], sample ss[i]) -- the oracle port's or the library's own li_pixels.

Films and moments are [H, W, 4] float32 in the film's row order (row H-1-y holds image row y), as the library keeps them.
"""
import numpy as np

F32 = np.float32


def filter_samples(c):
    """c: [..., 3] float32 radiance -> the sample the film adds (NaN channel or infinite luminance -> 0)."""
    c = np.asarray(c, F32)
    with np.errstate(over="ignore", invalid="ignore"):
        lum = (F32(0.212671) * c[..., 0] + F32(0.715160) * c[..., 1]) + F32(0.072169) * c[..., 2]
    bad = np.isnan(c).any(axis=-1) | np.isinf(lum)
    return np.where(bad[..., None], F32(0), c).astype(F32)


def accumulate(film, moments, rows, cols, samples):
    """Adds samples [N, k, 3] (k per pixel, ascending sample order) of the film pixels (rows[i], cols[i]) to film and moments
    (moments may be None).  One add per pixel per step, so every pixel's sum runs in sample order."""
    c = filter_samples(samples)
    with np.errstate(over="ignore", invalid="ignore"):
        for j in range(c.shape[1]):
            cj = c[:, j, :]
            film[rows, cols, :3] += cj
            if moments is not None:
                moments[rows, cols, :3] += cj * cj
                moments[rows, cols, 3] += F32(1)


def selected(film, moments, min_samples, max_samples, step, tolerance, floor):
    """The convergence test: bool [H, W] in film row order, True = the pixel needs `step` more samples."""
    a = film[..., :3].astype(F32)
    q = moments[..., :3].astype(F32)
    n = moments[..., 3:4].astype(F32)
    tol, flo = F32(tolerance), F32(floor)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        mu = a / n
        d = q - a * mu
        v = d / (n - F32(1))
        v = np.where(v < 0, F32(0), v)            # a NaN stays NaN
        se = np.sqrt(v / n)
        thr = tol * np.where(mu > flo, mu, flo)
        unconverged = ~(se <= thr)
    return (moments[..., 3].astype(np.int64) + step <= max_samples) & unconverged.any(axis=-1)


def selected_pixels(film, moments, params):
    """Sorted film pixel indices y*W + x of the selected pixels (the device's list, sorted)."""
    H = film.shape[0]
    sel = selected(film, moments, params.min_samples, params.max_samples, params.step, params.tolerance, params.floor)
    r, x = np.nonzero(sel)
    return np.sort((H - 1 - r) * film.shape[1] + x)


def render_uniform(li, W, H, first, num, moments=True, film=None, mom=None):
    """agpt_render(first, num) of a W x H film (with moments): returns (film, moments)."""
    film = np.zeros((H, W, 4), F32) if film is None else film
    mom = (np.zeros((H, W, 4), F32) if mom is None else mom) if moments else None
    ys, xs = np.divmod(np.arange(W * H, dtype=np.int32), W)
    samples = np.empty((W * H, num, 3), F32)
    for k in range(num):
        samples[:, k] = li(xs, ys, np.full(W * H, first + k, np.int32))
    accumulate(film, mom, H - 1 - ys, xs, samples)
    return film, mom


def render_adaptive(li, W, H, params):
    """agpt_render_adaptive: returns (film, moments, rounds, paths, per-round selected counts)."""
    film, mom = render_uniform(li, W, H, 0, params.min_samples)
    rounds, paths, sizes = 0, W * H * params.min_samples, []
    while True:
        pix = selected_pixels(film, mom, params)
        if len(pix) == 0:
            break
        ys, xs = np.divmod(pix.astype(np.int32), W)
        have = mom[H - 1 - ys, xs, 3].astype(np.int32)
        samples = np.empty((len(pix), params.step, 3), F32)
        for j in range(params.step):
            samples[:, j] = li(xs, ys, have + j)
        accumulate(film, mom, H - 1 - ys, xs, samples)
        rounds += 1
        paths += len(pix) * params.step
        sizes.append(len(pix))
    return film, mom, rounds, paths, sizes


def counts_image(moments):
    """Per-pixel sample counts [H, W] in image order (row 0 = top), from moments in film row order."""
    return moments[::-1, :, 3].astype(np.int64)
