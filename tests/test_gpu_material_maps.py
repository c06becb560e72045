"""GPU: roughness-metallic and normal maps on Disney materials (include/agpt.h agpt_upload_material_textures).

NOT REFERENCE BEHAVIOUR except where a map reduces to its material's own values: the reference has neither map.  The extension
is stated on the CPU in statements/agpt_material_maps_oracle.cpp; these tests hold the library to it bit for bit on cfg 13
(every shape's tangent frame, per-hit lobe sets, the rules that leave a surface as it is), and to the reference-pinned unmapped
films where each material's maps are 1x1 images of its own values."""
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
from statements import maps_binding as mb  # noqa: E402
from tests.test_gpu_textures import bits, materials, own_colour, same_floats  # noqa: E402

FLAT = np.array([[[.5, .5, 1.0]]], np.float32)         # a flat normal-map texel
ONES = np.array([[[.3, 1.0, 1.0]]], np.float32)         # roughness and metallic factors of 1


@pytest.fixture(scope="module")
def mctx(agpt):
    if agpt.device_count() == 0:
        pytest.fail("no CUDA device visible: -m gpu tests must run on the GPU box")
    ctx = agpt.Context(0)
    yield ctx
    ctx.close()


@pytest.fixture(scope="module")
def cfg13(agpt):
    hs = agpt.HostScene(13, 1)
    return hs, mb.MapsScene(hs), mb.MapsScene(hs, rr_by_bounce=True)


def own_value_bindings(agpt, hs):
    """Every Disney material: a flat normal map, an (x, 1, 1) roughness-metallic map and its own colour."""
    images, bind = [FLAT, ONES], []
    for m in materials(hs):
        C = own_colour(m) if m["type"] == 1 else None
        bind.append(agpt.material_textures() if C is None else agpt.material_textures(-1, 1, 0, 1.0, tuple(float(v) for v in C)))
    return images, bind


# cfg 3 (reduced level) and cfg 5 run <false, false, false, 2>; cfg 10 (rough glass) and cfg 11 (sampled shape lights)
# <true, true, true, 2>.
@pytest.mark.parametrize("cfg,level", [(3, 2), (5, 2), (10, 2), (11, 2)])
def test_own_value_maps_leave_the_film_unchanged(agpt, mctx, cfg, level):
    d = agpt.config_defaults(cfg)
    hs = agpt.HostScene(cfg, level)
    hs.upload(mctx); mctx.set_film(96, 54); mctx.clear()
    flags = agpt.FLAG_RR_BY_BOUNCE if cfg == 10 else 0
    mctx.render(0, 2, d["max_depth"], d["depth_arg"], flags)
    want = mctx.read_accum().copy()
    images, bind = own_value_bindings(agpt, hs)
    assert sum(b.normal >= 0 for b in bind) >= sum(materials(hs)["type"] == 1) - 1
    mctx.upload_material_textures(images, bind)
    mctx.clear()
    mctx.render(0, 2, d["max_depth"], d["depth_arg"], flags)
    got = mctx.read_accum()
    mctx.upload_textures([], [])
    assert np.array_equal(bits(got), bits(want))


def test_base_colour_scene_through_the_maps_path_equals_the_base_colour_path(agpt, mctx):
    """cfg 12 with one own-value roughness-metallic map runs <..., 2>; its film is the <..., 1> film."""
    hs = agpt.HostScene(12, 0)
    hs.upload(mctx); mctx.set_film(96, 54); mctx.clear()
    mctx.render(0, 2, 8)
    want = mctx.read_accum().copy()
    from tests.test_material_maps_cpu import _Tables
    import ctypes
    t = _Tables.from_buffer_copy(hs.tables().raw[:ctypes.sizeof(_Tables)])
    imgs = [np.ctypeslib.as_array(ctypes.cast(t.textures[i].rgb, ctypes.POINTER(ctypes.c_float)), (t.textures[i].height, t.textures[i].width, 3)).copy()
            for i in range(t.n_textures)]
    mats = materials(hs)
    bind = []
    for i in range(t.n_material_textures):
        base = t.material_texture[i]
        C = own_colour(mats[i]) if base < 0 and mats[i]["type"] == 1 else None
        bind.append(agpt.material_textures(base) if C is None else agpt.material_textures(-1, len(imgs), -1, 1.0, tuple(float(v) for v in C)))
    assert any(b.roughness_metallic >= 0 for b in bind)
    mctx.upload_material_textures(imgs + [ONES], bind)
    mctx.clear()
    mctx.render(0, 2, 8)
    got = mctx.read_accum()
    assert np.array_equal(bits(got), bits(want))


@pytest.mark.parametrize("w,h", [(96, 54), (96, 56)])
@pytest.mark.parametrize("depth,flags", [(1, 0), (8, 0), (8, 16)])
def test_cfg13_film_and_ray_accounting_equal_the_statement(agpt, mctx, cfg13, w, h, depth, flags):
    """96x54: row-major slots, 96x56: tiled.  flags 16: roulette by bounce.  The per-hit lobe sets decide which vertices are
    perfectly specular and which MIS rays are culled: rays traced + rays proven useless == the rays the statement issues."""
    hs, ms, ms_rr = cfg13
    hs.upload(mctx); mctx.set_film(w, h); mctx.clear(); mctx.reset_stats()
    mctx.render(0, 2, depth, 0, flags | agpt.FLAG_COUNTERS)         # exact ray accounting needs the counting mode
    got = mctx.read_accum()
    st = mctx.stats()
    want, cnt = (ms_rr if flags else ms).render(w, h, 0, 2, depth, 0, counters=True)
    assert np.array_equal(bits(got[..., :3]), bits(want[..., :3]))
    assert st.rays_shadow == cnt["rays_any"]
    assert st.rays_closest + st.rays_mis + st.rays_mis_culled + st.rays_tail_culled == cnt["rays_closest"]
    mctx.clear()
    mctx.render(0, 2, depth, 0, flags)                             # the film does not depend on the counting mode
    assert np.array_equal(bits(mctx.read_accum()[..., :3]), bits(want[..., :3]))


def test_cfg13_with_rough_glass_equals_the_statement(agpt, mctx):
    """Level 2 adds a rough glass sphere: <true, true, true, 2> runs."""
    hs = agpt.HostScene(13, 2)
    ms = mb.MapsScene(hs)
    hs.upload(mctx); mctx.set_film(96, 54); mctx.clear()
    mctx.render(0, 2, 8)
    assert np.array_equal(bits(mctx.read_accum()[..., :3]), bits(ms.render(96, 54, 0, 2, 8, 0)[..., :3]))


def test_li_pixels_equal_the_statement(agpt, mctx, cfg13):
    hs, ms, _ = cfg13
    hs.upload(mctx); mctx.set_film(96, 54)
    rng = np.random.default_rng(5)
    xs = rng.integers(0, 96, 400); ys = rng.integers(0, 54, 400); ss = rng.integers(0, 50, 400)
    got = mctx.li_pixels(xs, ys, ss, 8)
    want = ms.li_pixels(96, 54, xs, ys, ss, 8, 0)
    assert np.array_equal(bits(got), bits(want))


@pytest.mark.parametrize("w,h", [(96, 54), (96, 56)])
@pytest.mark.parametrize("depth,flags", [(1, 0), (8, 0), (8, 16)])
def test_guides_and_denoise_equal_the_statement(agpt, mctx, cfg13, w, h, depth, flags):
    hs, ms, _ = cfg13
    hs.upload(mctx); mctx.set_film(w, h); mctx.set_moments(True); mctx.clear()
    mctx.render(0, 4, depth, 0, flags)
    mctx.render_guides(3)
    alb, nd = mctx.read_guides()
    walb, wnd = ms.guides(w, h, 3)
    assert np.array_equal(bits(alb), bits(walb)) and np.array_equal(bits(nd), bits(wnd))
    film, mom = mctx.read_accum(), mctx.read_moments()
    for it in (0, 1, 5):
        p = agpt.denoise_params(iterations=it)
        out, _ = mctx.denoise(p)
        want = dn.denoise(film, mom, alb, nd, it, p.sigma_luminance, p.sigma_depth, p.normal_power_log2)
        assert same_floats(out, want), it
    mctx.set_moments(False)


def test_reprojection_follows_the_mapped_guides(agpt, mctx, cfg13):
    """One camera move of agpt_reproject_film on cfg 13: the first frame's guides are the statement's (mapped normals, per-hit
    albedo), and the carried film and moments are oracle/reproject.py's, fed with the library's guides."""
    from oracle import reproject as rp
    hs, ms, _ = cfg13
    hs.upload(mctx); mctx.set_film(96, 54); mctx.set_moments(True); mctx.clear()
    p = agpt.reproject_params()
    cam0 = hs.camera()
    mctx.set_camera(cam0)
    mctx.render_guides(2)
    alb0, nd0 = mctx.read_guides()
    walb, wnd = ms.guides(96, 54, 2)
    assert np.array_equal(bits(alb0), bits(walb)) and np.array_equal(bits(nd0), bits(wnd))
    mctx.reproject_film(p)                                             # saves the view
    _, _, G0 = rp.reproject(None, None, mctx.read_accum().copy(), mctx.read_moments().copy(), cam0, alb0, nd0, p.max_history, p.sigma_depth,
                            p.min_normal_dot)
    mctx.render(0, 4, 8)
    cam1 = rp.orbit(cam0, 2.5)
    mctx.set_camera(cam1)
    mctx.render_guides(2)
    film, mom = mctx.read_accum().copy(), mctx.read_moments().copy()
    alb, nd = mctx.read_guides()
    mctx.reproject_film(p)
    want_f, want_m, _ = rp.reproject(np.asarray(cam0, np.float32), G0, film, mom, cam1, alb, nd, p.max_history, p.sigma_depth, p.min_normal_dot)
    got_m = mctx.read_moments()
    assert same_floats(mctx.read_accum(), want_f) and same_floats(got_m, want_m)
    assert (got_m[..., 3] > 0).mean() > 0.3                          # the move carries history
    mctx.set_moments(False)


def test_probe_rows_equal_the_statement(agpt, mctx, cfg13):
    """agpt_probe_material_maps against the statement's per-hit rows: the floor, both spheres (near their -z poles too), the
    plain grid and its rotated-and-scaled and sheared instances."""
    hs, ms, _ = cfg13
    hs.upload(mctx)
    rng = np.random.default_rng(11)
    groups = {
        "floor": np.stack([rng.uniform(-5, 5, 400), np.full(400, -1.0), rng.uniform(-3, 7, 400)], 1),
        "sphere_textured": np.array([-2.2, 0, 0]) + rng.uniform(-.8, .8, (400, 3)) * [1, 1, 0] + [0, 0, -1],
        "sphere_mixed": np.array([.3, 0, .6]) + rng.uniform(-.8, .8, (400, 3)) * [1, 1, 0] + [0, 0, -1],
        "poles": np.array([[-2.2 + 1e-4, 2e-4, -1.0], [.3, 3e-3, -.4], [-2.2, 0, -1.0], [.3, 0, -.4]]),
        "grid": np.array([-1.2, 1.8, 3.0]) + rng.uniform(-.9, .9, (400, 3)) * [1, 1, 0],
        "instance": np.array([1.6, 1.7, 3.2]) + rng.uniform(-.9, .9, (400, 3)) * [1, 1, 0],
        "sheared": np.array([-3.6, 2.0, 3.6]) + rng.uniform(-.9, .9, (400, 3)) * [1, 1, 0],
    }
    for name, tg in groups.items():
        O = np.broadcast_to(np.float32([0, 2.2, -8.5]), tg.shape).astype(np.float32)
        D = (tg - O).astype(np.float32)
        rays = np.concatenate([O, D, np.full((len(O), 1), 1e30, np.float32)], 1)
        got, want = mctx.probe_material_maps(rays), ms.hit_rows(rays)
        assert (want[:, 0] >= 0).sum() > len(rays) // 2, name
        assert same_floats(got, want), name
    hs1 = agpt.HostScene(1, 0)
    hs1.upload(mctx)
    with pytest.raises(agpt.AgptError):                                # no material has a map
        mctx.probe_material_maps(rays)


def test_adaptive_pixels_equal_plain_renders(agpt, mctx, cfg13):
    hs, _, _ = cfg13
    hs.upload(mctx); mctx.set_film(48, 27); mctx.set_moments(True)
    mctx.render_adaptive(agpt.adaptive(2, 8, 2, 0.05), 8)
    film, counts = mctx.read_accum().copy(), mctx.read_moments()[..., 3].copy()
    for k in np.unique(counts):
        mctx.clear(); mctx.render(0, int(k), 8)
        plain = mctx.read_accum()
        sel = counts == k
        assert np.array_equal(bits(film[sel]), bits(plain[sel]))
    mctx.set_moments(False)


def test_host_mirror_equals_the_context(agpt, mctx, cfg13):
    hs, _, _ = cfg13
    tr = agpt.HostTracer(8, 0)
    acc = np.zeros((54, 96, 4), np.float32)
    tr.render(hs, 96, 54, acc, 0, 2)
    hs.upload(mctx); mctx.set_film(96, 54); mctx.clear(); mctx.render(0, 2, 8)
    assert np.array_equal(bits(acc), bits(mctx.read_accum()))
    tr.close()


def test_refusals(agpt, mctx, cfg13):
    hs, _, _ = cfg13
    hs.upload(mctx); mctx.set_film(32, 18); mctx.clear()
    n = len(materials(hs))
    img = [np.ones((2, 3, 3), np.float32)]
    before = mctx.scene_bytes()
    core = agpt.binding.core()
    T, MT = agpt.binding.Texture, agpt.binding.MaterialTextures
    for bad in (agpt.material_textures(normal=1), agpt.material_textures(roughness_metallic=-2), agpt.material_textures(base=5),
                agpt.material_textures(normal=0, normal_scale=float("nan")), agpt.material_textures(normal=0, normal_scale=float("inf")),
                agpt.material_textures(roughness_metallic=0, color=(0, float("nan"), 0))):
        rows = (T * 1)(T(3, 2, agpt.binding._fptr(img[0])))
        with pytest.raises(agpt.AgptError):                          # the library's own checks (Python's are skipped here)
            agpt.binding._check(core.agpt_upload_material_textures(mctx.handle, rows, 1, (MT * n)(*([bad] * n)), n))
        assert mctx.scene_bytes() == before                            # refused: resident textures as they were
    # wrong binding count, and a map on a mirror material: refused at render time
    mctx.upload_material_textures(img, [agpt.material_textures(normal=0)] * (n + 1))
    with pytest.raises(agpt.AgptError):
        mctx.render(0, 1, 2)
    hs1 = agpt.HostScene(1, 0)                                         # cfg 1: material 1 is a mirror
    hs1.upload(mctx)
    m1 = materials(hs1)
    for key in ("roughness_metallic", "normal"):
        bind = [agpt.material_textures() for _ in m1]
        setattr(bind[int(np.nonzero(m1["type"] == 2)[0][0])], key, 0)
        mctx.upload_material_textures(img, bind)
        with pytest.raises(agpt.AgptError):
            mctx.render(0, 1, 2)
    mctx.upload_textures([], [])
    # an upload makes the guides stale and drops the saved reprojection view
    hs.upload(mctx); mctx.set_moments(True); mctx.clear()
    mctx.render(0, 1, 2); mctx.render_guides(1)
    mctx.reproject_film(agpt.reproject_params())                       # saves the view
    mctx.upload_material_textures([], [])
    with pytest.raises(agpt.AgptError):
        mctx.denoise(agpt.denoise_params())
    mctx.render_guides(1)
    film = mctx.read_accum().copy()
    cam = hs.camera().copy(); cam[0] += 0.1
    mctx.set_camera(cam)
    mctx.render_guides(1)
    mctx.reproject_film(agpt.reproject_params())                       # no saved view after the upload: film left as it is
    assert np.array_equal(bits(mctx.read_accum()), bits(film))
    mctx.set_moments(False)


def test_no_failed_device_checks(mctx):
    """Meaningful under AGPT_LIB=libagpt_debug.so (test_debug_build_runs_this_file); a release build runs no checks."""
    s = mctx.debug_status()
    print("MAPS_DEBUG_STATUS", s["failed"], s["first_code"], s["first_value"], s["checks"])
    assert s["failed"] == 0


def test_debug_build_runs_this_file():
    """The tests above under libagpt_debug.so (map, texture and texel indices checked inside the kernels): none may fail."""
    lib = os.path.join(ROOT, "ag-pathtracer_b200", "libagpt_debug.so")
    assert os.path.exists(lib)
    env = dict(os.environ, AGPT_LIB=lib)
    out = subprocess.run([sys.executable, "-m", "pytest", "-q", "-s", "-p", "no:cacheprovider", os.path.abspath(__file__), "-k",
                          "not debug_build and not host_mirror"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if "MAPS_DEBUG_STATUS" in l][0]
    failed, checks = [int(v) for v in line.split("MAPS_DEBUG_STATUS")[1].split()[0:4:3]]
    assert checks > 100_000 and failed == 0
