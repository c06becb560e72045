"""GPU: emissive materials (include/agpt.h agpt_upload_emission).

NOT REFERENCE BEHAVIOUR: the reference's only emitters are AreaLights around null-material shapes.  cfg 15, built to use every
uv rule of the emission lookup beside next-event estimation (level 1), with no light and an alpha-masked sign (level 2), must
equal the CPU statement (statements/agpt_emission_oracle.cpp) bit for bit.  Relations that need no statement hold too: a closed
mirror cube's geometric series, linearity in the factors, a constant texture against its colour, and an emitting row no
primitive uses, which runs k_shade_a_emit and traces the tail rays beside every k_shade_b variant yet changes no pixel."""
import ctypes
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
from statements import emission_binding as eb  # noqa: E402
from tests.test_emission_cpu import closed_cube  # noqa: E402
from tests.test_gpu_alpha_masks import scene_textures, table_rows  # noqa: E402
from tests.test_gpu_textures import bits, same_floats  # noqa: E402
from tests.test_material_maps_cpu import _Tables  # noqa: E402

W, H = 96, 54


@pytest.fixture(scope="module")
def ectx(agpt):
    if agpt.device_count() == 0:
        pytest.fail("no CUDA device visible: -m gpu tests must run on the GPU box")
    ctx = agpt.Context(0)
    yield ctx
    ctx.close()


@pytest.fixture(scope="module")
def cfg15(agpt):
    return {level: agpt.HostScene(15, level) for level in (1, 2)}


def materials(agpt, hs):
    t = _Tables.from_buffer_copy(hs.tables().raw[:ctypes.sizeof(_Tables)])
    return [agpt.Material.from_buffer_copy(ctypes.string_at(t.materials + 64 * i, 64)) for i in range(t.n_materials)]


def counts(st):
    return (st.rays_closest, st.rays_shadow, st.rays_mis, st.rays_mis_culled, st.rays_tail_culled)


@pytest.mark.parametrize("level", [1, 2])
@pytest.mark.parametrize("h", [54, 56])
@pytest.mark.parametrize("depth,flags", [(0, 0), (1, 0), (8, 0), (8, 16)])
def test_cfg15_film_and_ray_accounting_equal_the_statement(agpt, ectx, cfg15, level, h, depth, flags):
    hs = cfg15[level]
    hs.upload(ectx); ectx.set_film(W, h); ectx.clear(); ectx.reset_stats()
    ectx.render(0, 2, depth, 0, flags | agpt.FLAG_COUNTERS)
    got = ectx.read_accum().copy()
    st = ectx.stats()
    want, cnt = eb.EmissionScene(hs, rr_by_bounce=bool(flags & agpt.FLAG_RR_BY_BOUNCE)).render(W, h, 0, 2, depth, 0, counters=True)
    assert np.array_equal(bits(got[..., :3]), bits(want[..., :3]))
    assert st.rays_tail_culled == 0
    assert st.rays_shadow == cnt["rays_any"]
    assert st.rays_closest + st.rays_mis + st.rays_mis_culled + st.rays_tail_culled == cnt["rays_closest"]
    if level == 2:
        assert st.rays_shadow == 0 and st.rays_mis == 0
    ectx.clear()
    ectx.render(0, 2, depth, 0, flags)
    assert np.array_equal(bits(ectx.read_accum()[..., :3]), bits(want[..., :3]))


@pytest.mark.parametrize("level", [1, 2])
@pytest.mark.parametrize("h", [54, 56])
def test_cfg15_paths_and_rays_equal_the_statement(agpt, ectx, cfg15, level, h):
    hs = cfg15[level]
    d = agpt.config_defaults(15)
    es = eb.EmissionScene(hs)
    hs.upload(ectx); ectx.set_film(W, h)
    rng = np.random.default_rng(level * 100 + h)
    xs, ys, ss = rng.integers(0, W, 200), rng.integers(0, h, 200), rng.integers(0, 64, 200)
    for depth in (0, 1, d["max_depth"]):
        got = ectx.li_pixels(xs, ys, ss, depth, d["depth_arg"])
        assert np.array_equal(bits(got), bits(es.li_pixels(W, h, xs, ys, ss, depth, d["depth_arg"]))), depth
    # caller rays from the camera towards the screen, the ball, the strip, the icospheres and the mirror
    cam = hs.camera()
    targets = np.concatenate([rng.uniform([-1.2, .15, 5.4], [1.2, 2.55, 5.6], (300, 3)), rng.uniform([1.8, -1, 1.2], [3.4, .6, 2.8], (200, 3)),
                              rng.uniform([-3, 4.85, .8], [3, 4.95, 1.2], (200, 3)), rng.uniform([-3.1, -1, -.9], [-.5, 0, 2], (200, 3)),
                              rng.uniform([-4.8, -.5, -1], [-4.8, 3, 3.5], (200, 3))])
    dirs = targets - cam[0:3]
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    rays7 = np.concatenate([np.broadcast_to(cam[0:3], dirs.shape), dirs, np.full((len(dirs), 1), 1e30)], 1).astype(np.float32)
    states = rng.integers(1, 2 ** 32, len(rays7), dtype=np.uint32)
    got = ectx.li_rays(rays7, states, d["max_depth"], d["depth_arg"])
    want = es.li_rays(rays7, states, d["max_depth"], d["depth_arg"])
    assert np.array_equal(bits(got), bits(want))
    assert np.count_nonzero(want.sum(1)) > len(rays7) // 2


def test_cfg15_batches_equal_one_batch(agpt, ectx, cfg15):
    d = agpt.config_defaults(15)
    for level in (1, 2):
        hs = cfg15[level]
        hs.upload(ectx); ectx.set_film(W, H); ectx.clear()
        ectx.render(0, 4, d["max_depth"], d["depth_arg"])
        one = ectx.read_accum().copy()
        os.environ["AGPT_BATCH_LOG2"] = "10"
        try:
            ctx = agpt.Context(0)
            hs.upload(ctx); ctx.set_film(W, H); ctx.clear()
            ctx.render(0, 4, d["max_depth"], d["depth_arg"])
            assert np.array_equal(bits(ctx.read_accum()), bits(one)), level
            ctx.close()
        finally:
            del os.environ["AGPT_BATCH_LOG2"]


def test_cfg15_host_mirror_equals_the_context_sequence(agpt, ectx, cfg15):
    d = agpt.config_defaults(15)
    for level in (1, 2):
        hs = cfg15[level]
        hs.upload(ectx); ectx.set_film(W, H); ectx.clear()
        ectx.render(0, 2, d["max_depth"], d["depth_arg"])
        want = ectx.read_accum().copy()
        tracer = agpt.HostTracer(d["max_depth"], 0)
        film = np.zeros((H, W, 4), np.float32)
        tracer.render(hs, W, H, film, 0, 2, d["depth_arg"])
        assert np.array_equal(bits(film[..., :3]), bits(want[..., :3])), level
        tracer.close()


def test_cfg15_two_gpus_equal_one(agpt, cfg15):
    if agpt.device_count() < 2:
        pytest.skip("one GPU visible")
    hs = cfg15[1]
    d = agpt.config_defaults(15)
    one, two = agpt.HostTracer(d["max_depth"], 0), agpt.HostTracer(d["max_depth"], devices=[0, 1])
    a = np.zeros((H, W, 4), np.float32); b = np.zeros((H, W, 4), np.float32)
    one.render(hs, W, H, a, 0, 4); two.render(hs, W, H, b, 0, 4)
    assert np.allclose(a, b, rtol=1e-5, atol=1e-6)
    one.close(); two.close()


def test_cfg15_adaptive_pixels_equal_plain_renders(agpt, ectx, cfg15):
    hs = cfg15[1]
    d = agpt.config_defaults(15)
    hs.upload(ectx); ectx.set_film(48, 27); ectx.set_moments(True)
    ectx.render_adaptive(agpt.adaptive(2, 8, 2, 0.05), d["max_depth"])
    film, cnt = ectx.read_accum().copy(), ectx.read_moments()[..., 3].copy()
    assert len(np.unique(cnt)) > 1
    for k in np.unique(cnt):
        ectx.clear(); ectx.render(0, int(k), d["max_depth"])
        plain = ectx.read_accum()
        sel = cnt == k
        assert np.array_equal(bits(film[sel]), bits(plain[sel]))
    ectx.set_moments(False)


def test_cfg15_guides_and_denoise(agpt, ectx, cfg15):
    """Guides ignore emission (they equal the guides with the table cleared); denoise at 0 and 5 iterations equals the oracle."""
    hs = cfg15[2]
    d = agpt.config_defaults(15)
    hs.upload(ectx); ectx.set_film(W, H); ectx.set_moments(True); ectx.clear()
    ectx.render(0, 4, d["max_depth"], d["depth_arg"])
    ectx.render_guides(3)
    alb, nd = [g.copy() for g in ectx.read_guides()]
    film, mom = ectx.read_accum().copy(), ectx.read_moments().copy()
    want_film = eb.EmissionScene(hs).render(W, H, 0, 4, d["max_depth"], d["depth_arg"])
    assert np.array_equal(bits(film[..., :3]), bits(want_film[..., :3]))
    for it in (0, 5):
        p = agpt.denoise_params(iterations=it)
        out, _ = ectx.denoise(p)
        want = dn.denoise(film, mom, alb, nd, it, p.sigma_luminance, p.sigma_depth, p.normal_power_log2)
        assert same_floats(out, want), it
    ectx.upload_emission([])
    ectx.render_guides(3)
    for g, w in zip(ectx.read_guides(), (alb, nd)):
        assert np.array_equal(bits(g), bits(w))
    ectx.set_moments(False)


def test_cfg15_reprojection(agpt, ectx, cfg15):
    from oracle import reproject as rp
    hs = cfg15[1]
    d = agpt.config_defaults(15)
    hs.upload(ectx); ectx.set_film(W, H); ectx.set_moments(True); ectx.clear()
    p = agpt.reproject_params()
    cam0 = hs.camera()
    ectx.set_camera(cam0)
    ectx.render_guides(2)
    alb0, nd0 = ectx.read_guides()
    ectx.reproject_film(p)                                             # saves the view
    _, _, G0 = rp.reproject(None, None, ectx.read_accum().copy(), ectx.read_moments().copy(), cam0, alb0, nd0, p.max_history, p.sigma_depth,
                            p.min_normal_dot)
    ectx.render(0, 4, d["max_depth"])
    cam1 = rp.orbit(cam0, 2.5)
    ectx.set_camera(cam1)
    ectx.render_guides(2)
    film, mom = ectx.read_accum().copy(), ectx.read_moments().copy()
    alb, nd = ectx.read_guides()
    ectx.reproject_film(p)
    want_f, want_m, _ = rp.reproject(np.asarray(cam0, np.float32), G0, film, mom, cam1, alb, nd, p.max_history, p.sigma_depth, p.min_normal_dot)
    got_m = ectx.read_moments()
    assert same_floats(ectx.read_accum(), want_f) and same_floats(got_m, want_m)
    assert (got_m[..., 3] > 0).mean() > 0.3
    ectx.set_moments(False)
    ectx.set_camera(cam0)


@pytest.mark.parametrize("depth", [0, 1, 2, 8])
def test_closed_mirror_cube_is_a_geometric_series(agpt, ectx, depth):
    r, e, spp = .5, .75, 4
    prims, mesh, mat, cam, row = closed_cube(agpt, r, e)
    ctx = agpt.Context(0)                       # nothing resident but the cube
    ctx.upload_meshes([mesh])
    ctx.upload_table("materials", [mat])
    ctx.upload_table("primitives", prims)
    ctx.upload_emission([row])
    ctx.set_camera(cam); ctx.set_film(48, 27); ctx.clear()
    ctx.render(0, spp, depth, 0)
    film = ctx.read_accum()[..., :3].astype(np.float64)
    ctx.close()
    want = e * spp * sum(r ** k for k in range(depth + 1))
    if depth == 0:
        assert (film == e * spp).all()
    assert np.abs(film / want - 1).max() < 1e-5


def test_doubling_every_factor_doubles_the_film_without_lights(agpt, ectx, cfg15):
    hs = cfg15[2]
    d = agpt.config_defaults(15)
    hs.upload(ectx); ectx.set_film(W, H); ectx.clear()
    ectx.render(0, 2, d["max_depth"], d["depth_arg"])
    one = ectx.read_accum().copy()
    ectx.upload_emission([agpt.emission(r.texture, tuple(2 * f for f in r.factor)) for r in hs.emission()])
    ectx.clear()
    ectx.render(0, 2, d["max_depth"], d["depth_arg"])
    assert np.array_equal(bits(ectx.read_accum()), bits(2 * one))


def test_a_constant_texture_equals_its_colour(agpt, ectx, cfg15):
    """Every emitting row of cfg 15 level 1 as factor (1, 1, 1) times a 1 x 1 image of colour c, against factor c."""
    hs = cfg15[1]
    d = agpt.config_defaults(15)
    images, binds, _, _ = scene_textures(agpt, hs)
    colours = [(.5, .25, 2.), (3., 1., .125), (.75, .75, .75), (1.5, 0., 4.)]
    rows = hs.emission()
    emitting = [i for i, r in enumerate(rows) if max(r.factor) > 0]
    hs.upload(ectx); ectx.set_film(W, H)

    def film():
        ectx.clear(); ectx.render(0, 2, d["max_depth"], d["depth_arg"])
        return ectx.read_accum().copy()
    ectx.upload_material_textures(images + [np.full((1, 1, 3), c, np.float32) for c in colours], binds)
    textured = list(rows)
    for k, i in enumerate(emitting):
        textured[i] = agpt.emission(len(images) + k, (1., 1., 1.))
    ectx.upload_emission(textured)
    a = film()
    plain = list(rows)
    for k, i in enumerate(emitting):
        plain[i] = agpt.emission(-1, colours[k])
    ectx.upload_emission(plain)
    assert np.array_equal(bits(a), bits(film()))


UNSEEN = [(3, 2), (5, 2), (7, 0), (9, 2), (10, 2), (11, 1), (11, 2), (12, 0), (13, 1), (14, 1)]


def unseen_emitter(agpt, ctx, hs):
    """One extra material, used by no primitive, with factor (1, 1, 1); the scene's texture bindings and masks extended by a row."""
    mats = materials(agpt, hs)
    images, binds, _, _ = scene_textures(agpt, hs)
    ctx.upload_table("materials", mats + [mats[0]])
    if binds:
        ctx.upload_material_textures(images, binds + [agpt.material_textures()])
    masks = hs.alpha_masks()
    if masks:
        ctx.upload_alpha_masks(masks + [agpt.alpha_mask()])
    ctx.upload_emission([agpt.emission() for _ in mats] + [agpt.emission(-1, (1., 1., 1.))])


@pytest.mark.parametrize("cfg,level", UNSEEN)
def test_an_emitter_nobody_sees_changes_no_pixel(agpt, ectx, cfg, level):
    """k_shade_a_emit, and the tail rays traced, beside every k_shade_b variant (environment map, instances, glass, sampled shape
    lights, textures, maps) and the masked trace: film and guides bit-identical, the tail rays moved into rays_closest."""
    hs = agpt.HostScene(cfg, level)
    d = agpt.config_defaults(cfg)
    flags = agpt.FLAG_RR_BY_BOUNCE if cfg == 10 else 0

    def run():
        ectx.set_film(W, H); ectx.clear(); ectx.reset_stats()
        ectx.render(0, 2, d["max_depth"], d["depth_arg"], flags | agpt.FLAG_COUNTERS)
        film = ectx.read_accum().copy()
        c = counts(ectx.stats())
        ectx.clear(); ectx.render(0, 2, d["max_depth"], d["depth_arg"], flags)
        assert np.array_equal(bits(ectx.read_accum()), bits(film))
        ectx.render_guides(2)
        return film, c, [g.copy() for g in ectx.read_guides()]
    hs.upload(ectx)
    plain = run()
    unseen_emitter(agpt, ectx, hs)
    emit = run()
    assert np.array_equal(bits(emit[0]), bits(plain[0])), "film"
    for g, w in zip(emit[2], plain[2]):
        assert np.array_equal(bits(g), bits(w)), "guides"
    closest, shadow, mis, mis_culled, tail = plain[1]
    assert tail > 0
    assert emit[1] == (closest + tail, shadow, mis, mis_culled, 0)


def test_an_all_zero_table_runs_the_old_path(agpt, ectx):
    hs = agpt.HostScene(5, 2)
    d = agpt.config_defaults(5)
    hs.upload(ectx); ectx.set_film(W, H); ectx.clear(); ectx.reset_stats()
    ectx.render(0, 2, d["max_depth"], d["depth_arg"], agpt.FLAG_COUNTERS)
    want, wc = ectx.read_accum().copy(), counts(ectx.stats())
    ectx.upload_emission([agpt.emission() for _ in materials(agpt, hs)])
    ectx.clear(); ectx.reset_stats()
    ectx.render(0, 2, d["max_depth"], d["depth_arg"], agpt.FLAG_COUNTERS)
    assert np.array_equal(bits(ectx.read_accum()), bits(want))
    assert counts(ectx.stats()) == wc and wc[4] > 0


def test_refusals_and_state(agpt, ectx, cfg15):
    hs = cfg15[1]
    d = agpt.config_defaults(15)
    hs.upload(ectx); ectx.set_film(W, H)
    images, binds, _, n_mat = scene_textures(agpt, hs)
    rows = hs.emission()
    core = agpt.core()
    before = ectx.scene_bytes()
    for bad in (agpt.emission(len(images), (1, 1, 1)), agpt.emission(-2, (1, 1, 1)), agpt.emission(-1, (-1, 1, 1)),
                agpt.emission(-1, (1, float("nan"), 1)), agpt.emission(0, (1, 1, float("inf"))), agpt.emission(-1, (-0.5, 0, 0))):
        t = (agpt.Emission * n_mat)(*rows)
        t[0] = bad
        assert core.agpt_upload_emission(ectx.handle, t, n_mat) == -1
    assert core.agpt_upload_emission(ectx.handle, None, 1) == -1
    assert core.agpt_upload_emission(ectx.handle, (agpt.Emission * n_mat)(*rows), -1) == -1
    assert ectx.scene_bytes() == before                        # the resident table stays
    ectx.clear(); ectx.render(0, 1, d["max_depth"], d["depth_arg"])
    want = eb.EmissionScene(hs).render(W, H, 0, 1, d["max_depth"], d["depth_arg"])
    assert np.array_equal(bits(ectx.read_accum()[..., :3]), bits(want[..., :3]))
    # the table is counted: 16 bytes per material
    ectx.upload_emission([])
    assert before - ectx.scene_bytes() == 16 * n_mat
    # a different material count: refused at render time
    ectx.upload_emission(rows[:-1])
    with pytest.raises(agpt.AgptError, match="number of materials"):
        ectx.render(0, 1, 1, 0)
    # a texture upload clears the table: the scene renders as without it
    ectx.upload_emission(rows)
    ectx.upload_material_textures(images, binds)
    ectx.clear(); ectx.reset_stats(); ectx.render(0, 1, d["max_depth"], d["depth_arg"])
    want = eb.EmissionScene(hs, rows=[]).render(W, H, 0, 1, d["max_depth"], d["depth_arg"])
    assert np.array_equal(bits(ectx.read_accum()[..., :3]), bits(want[..., :3]))
    assert ectx.stats().rays_tail_culled > 0
    # an emission upload makes the guides stale and drops the saved reprojection view
    ectx.set_moments(True); ectx.clear()
    ectx.render(0, 1, 2); ectx.render_guides(1)
    ectx.reproject_film(agpt.reproject_params())                       # saves the view
    ectx.upload_emission(rows)
    with pytest.raises(agpt.AgptError):
        ectx.read_guides()
    with pytest.raises(agpt.AgptError):
        ectx.denoise(agpt.denoise_params())
    ectx.render_guides(1)
    film = ectx.read_accum().copy()
    cam = hs.camera().copy(); cam[0] += 0.1
    ectx.set_camera(cam)
    ectx.render_guides(1)
    ectx.reproject_film(agpt.reproject_params())                       # no saved view after the upload: film left as it is
    assert np.array_equal(bits(ectx.read_accum()), bits(film))
    ectx.set_moments(False)
    ectx.set_camera(hs.camera())


def test_an_emitter_on_an_area_light_is_refused(agpt, ectx):
    """cfg 5's light sphere given material 0, which emits: refused at render time; without the emission it renders."""
    hs = agpt.HostScene(5, 2)
    hs.upload(ectx); ectx.set_film(32, 18)
    prims, _ = table_rows(agpt, hs)
    light = int(np.nonzero(prims["area_light"] >= 0)[0][0])
    prims["material"][light] = 0
    ectx.upload_table("primitives", prims)
    n_mat = len(materials(agpt, hs))
    ectx.upload_emission([agpt.emission(-1, (1, 1, 1))] + [agpt.emission() for _ in range(n_mat - 1)])
    with pytest.raises(agpt.AgptError, match="area light"):
        ectx.render(0, 1, 2)
    ectx.upload_emission([agpt.emission(-1, (0, 0, 0))] + [agpt.emission(-1, (1, 1, 1)) for _ in range(n_mat - 1)])
    ectx.render(0, 1, 2)
    ectx.upload_emission([])


def test_no_failed_device_checks(ectx):
    """Meaningful under AGPT_LIB=libagpt_debug.so (test_debug_build_runs_this_file); a release build runs no checks."""
    s = ectx.debug_status()
    print("EMISSION_DEBUG_STATUS", s["failed"], s["first_code"], s["first_value"], s["checks"])
    assert s["failed"] == 0


def test_debug_build_runs_this_file():
    """This module under libagpt_debug.so (emission row, texture and texel indices checked inside k_shade_a_emit)."""
    lib = os.path.join(ROOT, "ag-pathtracer_b200", "libagpt_debug.so")
    assert os.path.exists(lib)
    env = dict(os.environ, AGPT_LIB=lib)
    out = subprocess.run([sys.executable, "-m", "pytest", "-q", "-s", "-p", "no:cacheprovider", os.path.abspath(__file__), "-k",
                          "not debug_build and not two_gpus and not batches and not host_mirror"], cwd=ROOT, env=env,
                         capture_output=True, text=True, timeout=1800)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if "EMISSION_DEBUG_STATUS" in l][0]
    failed, checks = [int(v) for v in line.split("EMISSION_DEBUG_STATUS")[1].split()[0:4:3]]
    assert checks > 100_000 and failed == 0
