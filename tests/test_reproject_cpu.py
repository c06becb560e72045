"""CPU: the statement of the film reprojection (extension, include/agpt.h agpt_reproject_film, oracle/reproject.py) on synthetic
guides and cameras: the projection against float64 geometry, whole-pixel translations, the identity rule, and every rejection."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import reproject as rp  # noqa: E402

F32 = np.float32
W, H = 48, 27


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def front_camera(origin=(0.0, 0.0, 0.0), aperture=0.0):
    """Looking down -z with +y up, image plane at distance 1."""
    o = np.asarray(origin, np.float64)
    return rp.camera_look_at(o, o + (0, 0, -1), (0, 1, 0), W / H, 45, aperture)


def plane_guides(cam, depth_z, normal=(0.0, 0.0, 1.0)):
    """Guides of the plane z = -depth_z seen by `cam`: every pixel hits it, at the hit distance along its centre ray."""
    D = rp.centre_rays(cam, W, H).astype(np.float64)
    o = np.asarray(cam[0:3], np.float64)
    t = (o[2] + depth_z) / -D[..., 2]
    albedo = np.ones((H, W, 4), F32)
    nd = np.zeros((H, W, 4), F32)
    nd[..., :3] = normal
    nd[..., 3] = t
    return albedo, nd


def random_film(seed, n_max=64):
    rng = np.random.default_rng(seed)
    n = rng.integers(1, n_max, (H, W)).astype(F32)
    film = np.zeros((H, W, 4), F32)
    film[..., :3] = (rng.random((H, W, 3)) * n[..., None]).astype(F32)
    mom = np.zeros((H, W, 4), F32)
    mom[..., :3] = (rng.random((H, W, 3)) * n[..., None]).astype(F32)
    mom[..., 3] = n
    return film, mom


def test_projection_equals_float64_geometry():
    """Known world points through cameras built like host/camera.h land where a float64 solve puts them, within 1e-4 px."""
    rng = np.random.default_rng(1)
    for k in range(20):
        lf = rng.uniform(-3, 3, 3)
        la = lf + rng.uniform(-1, 1, 3) * 2 + (0, 0, -2)
        cam = rp.camera_look_at(lf, la, (0, 1, 0), W / H, rng.uniform(20, 90))
        c = cam.astype(np.float64)
        O, L, Hz, Vt = c[0:3], c[3:6], c[6:9], c[9:12]
        # points in front of the camera, inside and outside the frame
        a, b, dist = rng.uniform(-0.4, 1.4, 50), rng.uniform(-0.4, 1.4, 50), rng.uniform(0.5, 20, 50)
        P = O + dist[:, None] * ((L + a[:, None] * Hz + b[:, None] * Vt) - O)
        d = (P - O).astype(F32)
        px, py, ok = rp.project(d, cam, W, H)
        f = (L + Hz / 2 + Vt / 2) - O
        sol = np.linalg.solve(np.stack([f, Hz, Vt], axis=1)[None].repeat(50, 0), (P - O)[..., None])[..., 0]
        want_x = (0.5 + sol[:, 1] / sol[:, 0]) * W - 0.5
        want_y = (0.5 + sol[:, 2] / sol[:, 0]) * H - 0.5
        assert ok.all()
        assert np.abs(px - want_x).max() <= 1e-4 and np.abs(py - want_y).max() <= 1e-4, k


def test_whole_pixel_translation_carries_the_neighbour():
    """A fronto-parallel plane, the camera moved by exactly (kx, ky) pixels at the plane's depth: every interior pixel takes the
    sums of the pixel that far away; rounding leaves the other taps at most 1e-4 of the weight."""
    depth_z = 5.0
    prev = front_camera()
    alb, nd = plane_guides(prev, depth_z)
    G = rp.guide_g(alb, nd)
    film, mom = random_film(2)
    pix = np.linalg.norm(prev[6:9].astype(np.float64)) * depth_z / W          # world size of a pixel at the plane
    for kx, ky in [(1, 0), (0, 1), (-3, 2), (5, -4)]:
        cam = front_camera((kx * pix, ky * pix, 0.0))
        alb2, nd2 = plane_guides(cam, depth_z)
        a2, q2, G2 = rp.reproject(prev, G, film, mom, cam, alb2, nd2, 1 << 24, 0.01, 0.9)
        assert np.array_equal(bits(G2), bits(rp.guide_g(alb2, nd2)))
        for r in range(H):
            y = H - 1 - r
            for x in range(W):
                xs, ys = x + kx, y + ky
                if not (1 <= xs < W - 1 and 1 <= ys < H - 1):
                    continue
                rs = H - 1 - ys
                tol = 1e-4 * (np.abs(film).max() + 1)
                assert np.allclose(a2[r, x], film[rs, xs], rtol=0, atol=tol), (kx, ky, x, y)
                assert np.allclose(q2[r, x], mom[rs, xs], rtol=0, atol=1e-4 * (np.abs(mom).max() + 1)), (kx, ky, x, y)


def test_identical_camera_leaves_everything():
    cam = front_camera()
    alb, nd = plane_guides(cam, 4.0)
    film, mom = random_film(3)
    film[0, 0, 0] = np.inf
    mom[1, 1, 2] = np.nan
    prev_G = np.full((H, W, 4), 7, F32)
    a2, q2, G2 = rp.reproject(cam.copy(), prev_G, film, mom, cam, alb, nd, 2.0, 0.01, 0.9)
    assert np.array_equal(bits(a2), bits(film)) and np.array_equal(bits(q2), bits(mom))
    assert np.array_equal(bits(G2), bits(rp.guide_g(alb, nd)))
    # no saved view: the same
    a2, q2, _ = rp.reproject(None, None, film, mom, cam, alb, nd, 2.0, 0.01, 0.9)
    assert np.array_equal(bits(a2), bits(film)) and np.array_equal(bits(q2), bits(mom))


def small_move():
    prev = front_camera()
    cam = front_camera((0.013, -0.007, 0.02))
    return prev, cam


def test_depth_steps_and_normal_flips_are_rejected():
    prev, cam = small_move()
    alb_p, nd_p = plane_guides(prev, 5.0)
    alb, nd = plane_guides(cam, 5.0)
    film, mom = random_film(4)
    base, qb, _ = rp.reproject(prev, rp.guide_g(alb_p, nd_p), film, mom, cam, alb, nd, 1 << 24, 0.05, 0.9)
    assert (qb[..., 3] > 0).mean() > 0.9
    # the saved view 30 % deeper: nothing passes a 5 % depth test
    nd_far = nd_p.copy(); nd_far[..., 3] *= F32(1.3)
    a2, q2, _ = rp.reproject(prev, rp.guide_g(alb_p, nd_far), film, mom, cam, alb, nd, 1 << 24, 0.05, 0.9)
    assert not a2.any() and not q2.any()
    # ... but a 50 % tolerance takes them
    a2, q2, _ = rp.reproject(prev, rp.guide_g(alb_p, nd_far), film, mom, cam, alb, nd, 1 << 24, 0.5, 0.9)
    assert np.array_equal(bits(a2), bits(base)) and np.array_equal(bits(q2), bits(qb))
    # flipped normals in the saved view
    nd_flip = nd_p.copy(); nd_flip[..., :3] *= F32(-1)
    a2, q2, _ = rp.reproject(prev, rp.guide_g(alb_p, nd_flip), film, mom, cam, alb, nd, 1 << 24, 0.05, 0.9)
    assert not a2.any() and not q2.any()
    # min_normal_dot = -1 accepts any normal
    a2, q2, _ = rp.reproject(prev, rp.guide_g(alb_p, nd_flip), film, mom, cam, alb, nd, 1 << 24, 0.05, -1.0)
    assert np.array_equal(bits(a2), bits(base))
    # one saved pixel deeper: the pixels that had a tap on it lose that tap's weight only
    nd_step = nd_p.copy(); nd_step[10, 20, 3] *= F32(2)
    a2, q2, _ = rp.reproject(prev, rp.guide_g(alb_p, nd_step), film, mom, cam, alb, nd, 1 << 24, 0.05, 0.9)
    changed = np.argwhere((bits(q2) != bits(qb)).any(-1))
    assert 1 <= len(changed) <= 4 and all(abs(r - 10) <= 1 and abs(x - 20) <= 1 for r, x in changed)


def test_sky_follows_direction_and_never_takes_hit_taps():
    prev = front_camera((0, 0, 0))
    cam = rp.turn(prev, 4.0)
    cam_moved = rp.translate(cam, np.array([50.0, 0, 0]))      # a translation does not move points at infinity
    sky_alb = np.zeros((H, W, 4), F32)
    sky_nd = np.zeros((H, W, 4), F32)
    film, mom = random_film(5)
    a1, q1, G1 = rp.reproject(prev, rp.guide_g(sky_alb, sky_nd), film, mom, cam, sky_alb, sky_nd, 1 << 24, 0.05, 0.9)
    assert (G1[..., 3] == -1).all() and (q1[..., 3] > 0).mean() > 0.8
    # the same turn from a far-away position carries the same taps: only the direction counts
    prev_moved = rp.translate(prev, np.array([50.0, 0, 0]))
    a2, q2, _ = rp.reproject(prev_moved, rp.guide_g(sky_alb, sky_nd), film, mom, cam_moved, sky_alb, sky_nd, 1 << 24, 0.05, 0.9)
    assert np.allclose(q2, q1, atol=1e-3 * np.abs(mom).max()) and np.allclose(a2, a1, atol=1e-3 * np.abs(film).max())
    # a saved view that hit everywhere gives a sky pixel nothing, and a hit pixel never takes a sky tap
    alb_hit, nd_hit = plane_guides(prev, 5.0)
    a3, q3, _ = rp.reproject(prev, rp.guide_g(alb_hit, nd_hit), film, mom, cam, sky_alb, sky_nd, 1 << 24, 0.05, 0.9)
    assert not a3.any() and not q3.any()
    alb_c, nd_c = plane_guides(cam, 5.0)
    a4, q4, _ = rp.reproject(prev, rp.guide_g(sky_alb, sky_nd), film, mom, cam, alb_c, nd_c, 1 << 24, 0.05, 0.9)
    assert not a4.any() and not q4.any()


def test_points_behind_the_saved_camera_get_no_history():
    prev = front_camera()
    back = rp.turn(prev, 180.0)
    alb, nd = plane_guides(prev, 5.0)
    # the current camera looks at +z: hits there are behind the saved camera
    D = rp.centre_rays(back, W, H)
    nd_b = np.zeros((H, W, 4), F32); nd_b[..., 2] = -1; nd_b[..., 3] = F32(3) / D[..., 2]
    film, mom = random_film(6)
    a2, q2, _ = rp.reproject(prev, rp.guide_g(alb, nd), film, mom, back, alb, nd_b, 1 << 24, 10.0, -1.0)
    assert not a2.any() and not q2.any()
    # and the projection says why
    X = back[0:3] + nd_b[..., 3:4] * D
    _, _, ok = rp.project((X - prev[0:3]).astype(F32), prev, W, H)
    assert not ok.any()


def test_max_history_scales_sums_and_counts():
    prev, cam = small_move()
    alb_p, nd_p = plane_guides(prev, 5.0)
    alb, nd = plane_guides(cam, 5.0)
    film, mom = random_film(7, n_max=2)          # n = 1 everywhere
    mom[..., 3] = 100
    a1, q1, _ = rp.reproject(prev, rp.guide_g(alb_p, nd_p), film, mom, cam, alb, nd, 1 << 24, 0.05, 0.9)
    a2, q2, _ = rp.reproject(prev, rp.guide_g(alb_p, nd_p), film, mom, cam, alb, nd, 10.0, 0.05, 0.9)
    have = q1[..., 3] > 0
    assert have.mean() > 0.9
    assert (q2[have, 3] == 10).all()
    k = (F32(10) / q1[..., 3]).astype(F32)
    assert np.array_equal(bits(a2[have]), bits((a1 * k[..., None])[have]))
    assert np.array_equal(bits(q2[have, :3]), bits((q1[..., :3] * k[..., None])[have]))
    # means are kept (to rounding)
    assert np.allclose(a2[have, :3] / q2[have, 3:4], a1[have, :3] / q1[have, 3:4], rtol=1e-5)
    # a cap above every count changes nothing (an interpolated 100 may round to just above 100)
    a3, q3, _ = rp.reproject(prev, rp.guide_g(alb_p, nd_p), film, mom, cam, alb, nd, 101.0, 0.05, 0.9)
    assert np.array_equal(bits(a3), bits(a1)) and np.array_equal(bits(q3), bits(q1))


def test_non_finite_taps_are_rejected():
    prev, cam = small_move()
    alb_p, nd_p = plane_guides(prev, 5.0)
    alb, nd = plane_guides(cam, 5.0)
    film, mom = random_film(8)
    G = rp.guide_g(alb_p, nd_p)
    a1, q1, _ = rp.reproject(prev, G, film, mom, cam, alb, nd, 1 << 24, 0.05, 0.9)
    for which, val in [("film", np.inf), ("film", np.nan), ("mom", np.inf), ("mom", np.nan), ("mom_n", np.inf)]:
        f2, m2 = film.copy(), mom.copy()
        if which == "film":
            f2[10, 20, 1] = val
        elif which == "mom":
            m2[10, 20, 0] = val
        else:
            m2[10, 20, 3] = val
        a2, q2, _ = rp.reproject(prev, G, f2, m2, cam, alb, nd, 1 << 24, 0.05, 0.9)
        assert np.isfinite(a2).all() and np.isfinite(q2).all(), which
        changed = np.argwhere((bits(q2) != bits(q1)).any(-1))
        assert 1 <= len(changed) <= 4 and all(abs(r - 10) <= 1 and abs(x - 20) <= 1 for r, x in changed), which
