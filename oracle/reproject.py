"""Reprojection of the film and its moments across a camera move (extension, include/agpt.h agpt_reproject_film) stated on the
CPU -- TEST INFRASTRUCTURE.

numpy, float32 throughout, every operation rounded on its own (numpy never fuses a multiply into an add), so each step is the
device's step bit for bit.  The four taps are added one after another to every pixel's sums, in the stated tap order.

Buffers are what the library keeps and returns, [H, W, 4] float32 in the film's row order (row H-1-y holds image row y):
film, moments, the guides (albedo, normal_depth) and the saved view's G.  Cameras are the 19 floats of agpt_camera
(origin, lower_left_corner, horizontal, vertical, u, v, lens_radius).
"""
import numpy as np

F32 = np.float32


def guide_g(albedo, normal_depth):
    """The saved view's G of the current guides: mean normal, and the mean depth or -1 where no guide sample hit."""
    G = np.ascontiguousarray(normal_depth, F32).copy()
    G[..., 3] = np.where(albedo[..., 3] == 0, F32(-1), normal_depth[..., 3])
    return G


def _vecs(cam):
    cam = np.asarray(cam, F32)
    return cam[0:3], cam[3:6], cam[6:9], cam[9:12]


def dot(a, b):
    return (a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1]) + a[..., 2] * b[..., 2]


def centre_rays(cam, W, H):
    """D [H, W, 3] in film row order: CameraRay's direction for the pixel centre, without lens offset."""
    O, L, Hz, Vt = _vecs(cam)
    r = np.arange(H)
    y = (H - 1 - r).astype(F32)
    x = np.arange(W).astype(F32)
    s = (x + F32(0.5)) / F32(W)
    t = (y + F32(0.5)) / F32(H)
    p = (L + s[None, :, None] * Hz) + t[:, None, None] * Vt
    v = p - O
    inv = F32(1) / np.sqrt(dot(v, v))
    return v * inv[..., None]


def project(d, prev_cam, W, H):
    """(px, py, ok) of points or directions d [..., 3] relative to the saved camera's origin: where they land on its film
    (image pixel coordinates, pixel centres at integers), ok = False where den = dot(d, f) is not > 0."""
    O1, L1, H1, V1 = _vecs(prev_cam)
    f = ((L1 + F32(0.5) * H1) + F32(0.5) * V1) - O1
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        den = dot(d, f)
        lam = dot(f, f) / den
        u = F32(0.5) + (lam * dot(d, H1)) / dot(H1, H1)
        v = F32(0.5) + (lam * dot(d, V1)) / dot(V1, V1)
        px = u * F32(W) - F32(0.5)
        py = v * F32(H) - F32(0.5)
    return px.astype(F32), py.astype(F32), den > 0


def reproject(prev_cam, prev_G, film, moments, cam, albedo, normal_depth, max_history, sigma_depth, min_normal_dot):
    """agpt_reproject_film: (film, moments, the saved G) after the call.  prev_cam None: no saved view."""
    Hh, W = film.shape[:2]
    G = guide_g(albedo, normal_depth)
    film, moments = np.asarray(film, F32), np.asarray(moments, F32)
    prev_G = None if prev_G is None else np.asarray(prev_G, F32)
    if prev_cam is None or np.array_equal(np.asarray(prev_cam, F32).view(np.uint32), np.asarray(cam, F32).view(np.uint32)):
        return film.copy(), moments.copy(), G
    O, _, _, _ = _vecs(cam)
    O1 = _vecs(prev_cam)[0]
    mh, sz, mnd = F32(max_history), F32(sigma_depth), F32(min_normal_dot)
    D = centre_rays(cam, W, Hh)
    hit = G[..., 3] >= 0
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        X = O + G[..., 3:4] * D
        dh = X - O1
        z = np.sqrt(dot(dh, dh))
        d = np.where(hit[..., None], dh, D).astype(F32)
        z = np.where(hit, z, F32(0)).astype(F32)
        px, py, ok = project(d, prev_cam, W, Hh)
        x0, y0 = np.floor(px), np.floor(py)
        ok = ok & (x0 >= -1) & (x0 <= F32(W) - F32(1)) & (y0 >= -1) & (y0 <= F32(Hh) - F32(1))
        fx, fy = (px - x0).astype(F32), (py - y0).astype(F32)
    ix = np.where(ok, x0, 0).astype(np.int64)
    iy = np.where(ok, y0, 0).astype(np.int64)
    wx = ((F32(1) - fx), fx)
    wy = ((F32(1) - fy), fy)
    sw = np.zeros((Hh, W), F32)
    S = np.zeros((Hh, W, 4), F32)
    Q = np.zeros((Hh, W, 4), F32)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore", under="ignore"):
        for k in range(4):
            tx, ty = ix + (k & 1), iy + (k >> 1)
            w = (wx[k & 1] * wy[k >> 1]).astype(F32)
            inside = ok & (tx >= 0) & (tx < W) & (ty >= 0) & (ty < Hh)
            rows = np.clip(Hh - 1 - ty, 0, Hh - 1)
            cols = np.clip(tx, 0, W - 1)
            a, q, g = film[rows, cols], moments[rows, cols], prev_G[rows, cols]
            hit_q = g[..., 3] >= 0
            geo = (np.abs(g[..., 3] - z) <= sz * z) & ((G[..., 0] * g[..., 0] + G[..., 1] * g[..., 1]) + G[..., 2] * g[..., 2] >= mnd)
            take = inside & (w > 0) & np.isfinite(a).all(-1) & np.isfinite(q).all(-1) & (hit_q == hit) & (~hit | geo)
            sw = np.where(take, sw + w, sw).astype(F32)
            S = np.where(take[..., None], S + w[..., None] * a, S).astype(F32)
            Q = np.where(take[..., None], Q + w[..., None] * q, Q).astype(F32)
        a2 = (S / sw[..., None]).astype(F32)
        q2 = (Q / sw[..., None]).astype(F32)
        cap = q2[..., 3] > mh
        k = (mh / q2[..., 3]).astype(F32)
        a2 = np.where(cap[..., None], a2 * k[..., None], a2).astype(F32)
        q2c = q2.copy()
        q2c[..., :3] = q2[..., :3] * k[..., None]
        q2c[..., 3] = mh
        q2 = np.where(cap[..., None], q2c, q2).astype(F32)
    have = sw > 0
    a2 = np.where(have[..., None], a2, F32(0)).astype(F32)
    q2 = np.where(have[..., None], q2, F32(0)).astype(F32)
    return a2, q2, G


def camera_look_at(lookfrom, lookat, vup, aspect, vfov, aperture=0.0):
    """agpt_camera (19 float32) of Camera(lookfrom, lookat, vup, aspect, vfov, aperture), float32 arithmetic as host/camera.h."""
    lf, la, up = (np.asarray(v, F32) for v in (lookfrom, lookat, vup))
    half = F32(np.tan(F32(np.radians(F32(vfov))) / F32(2)))
    vh = F32(2) * half
    vw = F32(aspect) * vh
    norm = lambda v: v * (F32(1) / np.sqrt(dot(v, v)))
    focus = np.sqrt(dot(la - lf, la - lf))
    w = norm(lf - la)
    u = norm(np.cross(up, w).astype(F32))
    v = np.cross(w, u).astype(F32)
    hz = (focus * vw) * u
    vt = (focus * vh) * v
    llc = ((lf - hz / F32(2)) - vt / F32(2)) - focus * w
    return np.concatenate([lf, llc, hz, vt, u, v, [F32(aperture) / F32(2)]]).astype(F32)


def camera_desc(cam):
    """(lookfrom, lookat, vup, aspect, vfov, aperture) of a camera built by camera_look_at or host/camera.h, in float64."""
    c = np.asarray(cam, np.float64)
    O, L, Hz, Vt = c[0:3], c[3:6], c[6:9], c[9:12]
    centre = L + Hz / 2 + Vt / 2
    focus = np.linalg.norm(centre - O)
    vup = Vt / np.linalg.norm(Vt)
    vfov = np.degrees(2 * np.arctan(np.linalg.norm(Vt) / focus / 2))
    return O, centre, vup, np.linalg.norm(Hz) / np.linalg.norm(Vt), vfov, 2 * c[18]


def _rotate(v, axis, deg):
    axis = axis / np.linalg.norm(axis)
    a = np.radians(deg)
    return v * np.cos(a) + np.cross(axis, v) * np.sin(a) + axis * np.dot(axis, v) * (1 - np.cos(a))


def orbit(cam, deg):
    """The camera moved on a circle around its look-at point, about its up vector, by deg degrees."""
    lf, la, up, aspect, vfov, ap = camera_desc(cam)
    return camera_look_at(la + _rotate(lf - la, up, deg), la, up, aspect, vfov, ap)


def turn(cam, deg):
    """The camera turned in place about its up vector by deg degrees."""
    lf, la, up, aspect, vfov, ap = camera_desc(cam)
    return camera_look_at(lf, lf + _rotate(la - lf, up, deg), up, aspect, vfov, ap)


def translate(cam, offset):
    """The camera and its look-at point moved by offset (world units)."""
    lf, la, up, aspect, vfov, ap = camera_desc(cam)
    return camera_look_at(lf + offset, la + offset, up, aspect, vfov, ap)


def with_aperture(cam, aperture):
    lf, la, up, aspect, vfov, _ = camera_desc(cam)
    return camera_look_at(lf, la, up, aspect, vfov, aperture)
