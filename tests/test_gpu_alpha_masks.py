"""GPU: alpha-masked cutout geometry (include/agpt.h agpt_upload_alpha_masks).

NOT REFERENCE BEHAVIOUR: the reference has no masks.  Two kinds of checks: masks that keep every hit (a constant 1 at cutoff 0.5)
must leave every output of the unmasked scene bit for bit -- they run the MASK trace instantiations, so this shows their non-mask
code is the old code -- and cfg 14, built to use every masked path of the walk, must equal the CPU statement
(statements/agpt_alpha_oracle.cpp) bit for bit."""
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
from statements import alpha_binding as ab  # noqa: E402
from tests.test_gpu_textures import bits, same_floats  # noqa: E402
from tests.test_material_maps_cpu import _Tables  # noqa: E402

ONES = np.ones((1, 1, 3), np.float32)
W, H = 96, 54


@pytest.fixture(scope="module")
def actx(agpt):
    if agpt.device_count() == 0:
        pytest.fail("no CUDA device visible: -m gpu tests must run on the GPU box")
    ctx = agpt.Context(0)
    yield ctx
    ctx.close()


def scene_textures(agpt, hs):
    """The flattened scene's images (H, W, 3), per-material bindings as the host mirror uploads them, primitive rows and the
    material count."""
    t = _Tables.from_buffer_copy(hs.tables().raw[:ctypes.sizeof(_Tables)])
    images = []
    for i in range(t.n_textures):
        tx = t.textures[i]
        rgb = ctypes.cast(tx.rgb, ctypes.POINTER(ctypes.c_float))
        images.append(np.ctypeslib.as_array(rgb, (tx.height * tx.width * 3,)).reshape(tx.height, tx.width, 3).copy())
    binds = [t.material_textures[i] for i in range(t.n_material_textures)]
    binds = [agpt.material_textures(b.base, b.roughness_metallic, b.normal, b.normal_scale, tuple(b.color)) for b in binds]
    prims = np.ctypeslib.as_array(ctypes.cast(t.prims, ctypes.POINTER(ctypes.c_int32)), (4 * t.n_prims,)).reshape(-1, 4).copy()
    return images, binds, prims, t.n_materials


def bind_ones(agpt, ctx, hs):
    """Uploads the scene's images plus a constant 1, and masks every material that may carry one (not on spheres, not on
    emitters) with it at cutoff 0.5.  Returns the number of masked materials."""
    images, binds, prims, n_mat = scene_textures(agpt, hs)
    if not binds:
        binds = [agpt.material_textures() for _ in range(n_mat)]
    ctx.upload_material_textures(images + [ONES], binds)
    excluded = {int(p[2]) for p in prims if p[0] == agpt.PRIM_SPHERE or p[3] >= 0}
    masks = [agpt.alpha_mask(len(images), 1, .5) if i not in excluded else agpt.alpha_mask() for i in range(n_mat)]
    ctx.upload_alpha_masks(masks)
    return sum(m.texture >= 0 for m in masks)


def outputs(agpt, ctx, d, flags):
    ctx.set_film(W, H); ctx.clear(); ctx.reset_stats()
    ctx.set_moments(True)
    ctx.render(0, 2, d["max_depth"], d["depth_arg"], flags | agpt.FLAG_COUNTERS)
    film = ctx.read_accum().copy()
    st = ctx.stats()
    # walk counters of both kernel kinds; not the analytic records, which sphere runs read where any lane of a warp may hit the
    # run's box, so that past the camera rays their count depends on the order of queue appends
    rays = (st.rays_closest, st.rays_shadow, st.rays_mis, st.rays_mis_culled, st.rays_tail_culled,
            *[tuple(getattr(st, f)) for f in ("node_visits", "box_tests", "tri_tests")])
    hits = ctx.trace_primary(1).copy()
    ctx.render_guides(2)
    guides = ctx.read_guides()
    den, _ = ctx.denoise(agpt.denoise_params())
    ctx.set_moments(False)
    return film, rays, hits, guides, den


@pytest.mark.parametrize("cfg,level", [(3, 2), (5, 2), (7, 0), (9, 2), (10, 2), (11, 2), (12, 0), (13, 1)])
def test_all_ones_masks_leave_every_output_unchanged(agpt, actx, cfg, level):
    d = agpt.config_defaults(cfg)
    flags = agpt.FLAG_RR_BY_BOUNCE if cfg == 10 else 0
    hs = agpt.HostScene(cfg, level)
    hs.upload(actx)
    want = outputs(agpt, actx, d, flags)
    assert bind_ones(agpt, actx, hs) > 0
    got = outputs(agpt, actx, d, flags)
    assert np.array_equal(bits(got[0]), bits(want[0])), "film"
    assert got[1] == want[1], "ray counts and walk counters"
    for f in ("found", "prim", "tri"):
        assert np.array_equal(got[2][f], want[2][f]), f
    assert np.array_equal(bits(got[2]["t"]), bits(want[2]["t"]))
    for g, w in zip(got[3], want[3]):
        assert np.array_equal(bits(g), bits(w)), "guides"
    assert np.array_equal(bits(got[4]), bits(want[4])), "denoised"


CHECKER = np.kron(np.indices((4, 4)).sum(0) % 2, np.ones((2, 2)))[..., None].repeat(3, 2).astype(np.float32)     # 8 x 8 of 0 and 1


@pytest.mark.parametrize("cfg,level,h", [(7, 0, 54), (9, 2, 54), (10, 2, 54), (12, 0, 54), (13, 1, 54), (13, 2, 54), (13, 1, 56)])
def test_checker_masks_beside_every_shade_variant_equal_the_statement(agpt, actx, cfg, level, h):
    """A checker mask on every material that may carry one, appended to the scene's own images: the masked trace beside the
    environment map (cfg 7), instances (9), glass with roulette by bounce (10), textures (12) and maps (13).  Film, ray accounting,
    single paths, primary hits and guides equal the statement's, and the mask does remove primary hits."""
    hs = agpt.HostScene(cfg, level)
    d = agpt.config_defaults(cfg)
    rr = cfg == 10
    flags = agpt.FLAG_RR_BY_BOUNCE if rr else 0
    images, binds, prims, n_mat = scene_textures(agpt, hs)
    binds = binds or [agpt.material_textures() for _ in range(n_mat)]
    excluded = {int(p[2]) for p in prims if p[0] == agpt.PRIM_SPHERE or p[3] >= 0}
    masks = [agpt.alpha_mask(len(images), 0, .5) if i not in excluded else agpt.alpha_mask() for i in range(n_mat)]
    assert sum(m.texture >= 0 for m in masks) > 0
    hs.upload(actx)
    actx.upload_material_textures(images + [CHECKER], binds)
    actx.upload_alpha_masks(masks)
    st = ab.AlphaScene(hs, masks=[], rr_by_bounce=rr)
    st.set_textures(images + [CHECKER], binds)
    st.set_masks(masks)
    actx.set_film(W, h); actx.clear(); actx.reset_stats()
    actx.render(0, 2, d["max_depth"], d["depth_arg"], flags | agpt.FLAG_COUNTERS)
    s = actx.stats()
    want, cnt = st.render(W, h, 0, 2, d["max_depth"], d["depth_arg"], counters=True)
    assert np.array_equal(bits(actx.read_accum()[..., :3]), bits(want[..., :3])), "film"
    assert s.rays_shadow == cnt["rays_any"]
    assert s.rays_closest + s.rays_mis + s.rays_mis_culled + s.rays_tail_culled == cnt["rays_closest"]
    rng = np.random.default_rng(cfg + level)
    xs, ys, ss = rng.integers(0, W, 200), rng.integers(0, h, 200), rng.integers(0, 64, 200)
    got = actx.li_pixels(xs, ys, ss, d["max_depth"], d["depth_arg"], flags)
    assert np.array_equal(bits(got), bits(st.li_pixels(W, h, xs, ys, ss, d["max_depth"], d["depth_arg"]))), "paths"
    got = actx.trace_primary(1)
    want = st.primary_hits(W, h, 1).reshape(-1)
    for f in ("found", "prim", "tri"):
        assert np.array_equal(got[f], want[f]), f
    assert np.array_equal(bits(got["t"]), bits(want["t"]))
    bare = ab.AlphaScene(hs, masks=[]).primary_hits(W, h, 1).reshape(-1)
    assert np.count_nonzero((bare["prim"] != want["prim"]) | (bits(bare["t"]) != bits(want["t"]))) > 50, "the mask removes primary hits"
    actx.render_guides(2)
    for g, w in zip(actx.read_guides(), st.guides(W, h, 2)):
        assert np.array_equal(bits(g), bits(w)), "guides"


@pytest.fixture(scope="module")
def cfg14(agpt):
    return {level: agpt.HostScene(14, level) for level in (1, 2)}


@pytest.mark.parametrize("level", [1, 2])
@pytest.mark.parametrize("h", [54, 56])
@pytest.mark.parametrize("depth,flags", [(1, 0), (None, 0), (None, 16), (None, 4), (None, 4 | 16)])
def test_cfg14_film_and_ray_accounting_equal_the_statement(agpt, actx, cfg14, level, h, depth, flags):
    hs = cfg14[level]
    d = agpt.config_defaults(14)
    depth = d["max_depth"] if depth is None else depth
    hs.upload(actx); actx.set_film(W, h); actx.clear(); actx.reset_stats()
    actx.render(0, 2, depth, 0, flags | agpt.FLAG_COUNTERS)
    got = actx.read_accum()
    st = actx.stats()
    want, cnt = ab.AlphaScene(hs, rr_by_bounce=bool(flags & agpt.FLAG_RR_BY_BOUNCE)).render(W, h, 0, 2, depth, 0, counters=True)
    assert np.array_equal(bits(got[..., :3]), bits(want[..., :3]))
    assert st.rays_shadow == cnt["rays_any"]
    assert st.rays_closest + st.rays_mis + st.rays_mis_culled + st.rays_tail_culled == cnt["rays_closest"]
    actx.clear()
    actx.render(0, 2, depth, 0, flags)
    assert np.array_equal(bits(actx.read_accum()[..., :3]), bits(want[..., :3]))


@pytest.mark.parametrize("level", [1, 2])
def test_cfg14_paths_hits_and_guides_equal_the_statement(agpt, actx, cfg14, level):
    hs = cfg14[level]
    d = agpt.config_defaults(14)
    st = ab.AlphaScene(hs)
    hs.upload(actx); actx.set_film(W, H)
    # single paths
    rng = np.random.default_rng(level)
    xs, ys, ss = rng.integers(0, W, 400), rng.integers(0, H, 400), rng.integers(0, 64, 400)
    got = actx.li_pixels(xs, ys, ss, d["max_depth"], d["depth_arg"])
    assert np.array_equal(bits(got), bits(st.li_pixels(W, H, xs, ys, ss, d["max_depth"], d["depth_arg"])))
    # camera rays
    for sample in (0, 3):
        got = actx.trace_primary(sample)
        want = st.primary_hits(W, H, sample).reshape(-1)
        for f in ("found", "prim", "tri"):
            assert np.array_equal(got[f], want[f]), f
        assert np.array_equal(bits(got["t"]), bits(want["t"]))
    # caller rays aimed through the leaf cloud, the grate (shadow side), the checker quad and the mirror
    targets = np.concatenate([rng.uniform([-2.5, 1, -1], [-.5, 3.2, 1], (3000, 3)), rng.uniform([-3, 4, -3], [3, 4, 3], (2000, 3)),
                              rng.uniform([1, -1, -1.5], [3, 1, -1.2], (1000, 3)), rng.uniform([-4.2, -1, 1.4], [-2.4, 1.5, 2], (1000, 3))])
    origins = np.where(targets[:, 1:2] > 3.9, np.array([.2, 5.3, .4]), np.array([.3, 2.0, -8.5]))     # under the light, or the camera
    dirs = targets - origins
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    rays7 = np.concatenate([origins, dirs, np.full((len(dirs), 1), 1e30)], 1).astype(np.float32)
    for flags in (0, agpt.FLAG_COUNTERS | agpt.FLAG_STRICT_BOXES):
        for any_hit in (False, True):
            actx.reset_stats()
            got = actx.trace_rays(rays7, any_hit, flags)
            want, cnt = st.trace_rays(rays7, any_hit, counters=True)
            for f in ("found", "prim", "tri"):
                assert np.array_equal(got[f], want[f]), (flags, any_hit, f)
            assert np.array_equal(bits(got["t"]), bits(want["t"]))
            if flags and not any_hit:       # the any-hit kernels count two boxes per visit: not the statement's count
                s = actx.stats()
                assert (s.node_visits[0], s.box_tests[0], s.tri_tests[0]) == (cnt["interior"], cnt["boxes"], cnt["tris"])
    # some of those rays pass through holes: without the masks they would all stop at the first geometric hit
    nomask = ab.AlphaScene(hs, masks=[]).trace_rays(rays7)
    assert np.count_nonzero(nomask["prim"] != actx.trace_rays(rays7)["prim"]) > 100
    # guides
    actx.render_guides(3)
    for g, w in zip(actx.read_guides(), st.guides(W, H, 3)):
        assert np.array_equal(bits(g), bits(w))


def test_cfg14_batches_equal_one_batch(agpt, actx, cfg14):
    hs = cfg14[1]
    d = agpt.config_defaults(14)
    hs.upload(actx); actx.set_film(W, H); actx.clear()
    actx.render(0, 4, d["max_depth"], d["depth_arg"])
    one = actx.read_accum().copy()
    os.environ["AGPT_BATCH_LOG2"] = "10"
    try:
        ctx = agpt.Context(0)
        hs.upload(ctx); ctx.set_film(W, H); ctx.clear()
        ctx.render(0, 4, d["max_depth"], d["depth_arg"])
        assert np.array_equal(bits(ctx.read_accum()), bits(one))
        ctx.close()
    finally:
        del os.environ["AGPT_BATCH_LOG2"]


def test_host_mirror_equals_the_context_sequence(agpt, actx, cfg14):
    hs = cfg14[2]
    d = agpt.config_defaults(14)
    hs.upload(actx); actx.set_film(W, H); actx.clear()
    actx.render(0, 2, d["max_depth"], d["depth_arg"])
    want = actx.read_accum().copy()
    tracer = agpt.HostTracer(d["max_depth"], 0)
    film = np.zeros((H, W, 4), np.float32)
    tracer.render(hs, W, H, film, 0, 2, d["depth_arg"])
    assert np.array_equal(bits(film[..., :3]), bits(want[..., :3]))
    tracer.close()


def test_refusals_and_state(agpt, actx, cfg14):
    hs = cfg14[1]
    d = agpt.config_defaults(14)
    hs.upload(actx); actx.set_film(W, H)
    images, binds, prims, n_mat = scene_textures(agpt, hs)
    masks = hs.alpha_masks()
    n_tex = len(images)
    core = agpt.core()
    table = (agpt.AlphaMask * n_mat)(*masks)
    before = actx.scene_bytes()
    for bad in (agpt.AlphaMask(n_tex, 0, .5, 0), agpt.AlphaMask(-2, 0, .5, 0), agpt.AlphaMask(0, 3, .5, 0), agpt.AlphaMask(0, -1, .5, 0),
                agpt.AlphaMask(0, 0, float("nan"), 0), agpt.AlphaMask(0, 0, float("-inf"), 0)):
        t = (agpt.AlphaMask * n_mat)(*masks)
        t[0] = bad
        assert core.agpt_upload_alpha_masks(actx.handle, t, n_mat) == -1
    assert actx.scene_bytes() == before                        # the resident masks stay
    actx.clear(); actx.render(0, 1, d["max_depth"], d["depth_arg"])
    want = ab.AlphaScene(hs).render(W, H, 0, 1, d["max_depth"], d["depth_arg"])
    assert np.array_equal(bits(actx.read_accum()[..., :3]), bits(want[..., :3]))
    # the mask table is counted: 16 bytes per material
    actx.upload_alpha_masks([])
    assert before - actx.scene_bytes() == 16 * n_mat
    # a different material count, a masked sphere or emitter: refused at render time
    actx.upload_alpha_masks(masks[:-1])
    with pytest.raises(agpt.AgptError):
        actx.render(0, 1, 1, 0)
    # a texture upload clears the masks: the scene renders as without them
    actx.upload_alpha_masks(masks)
    actx.upload_material_textures(images, binds)
    actx.clear(); actx.render(0, 1, d["max_depth"], d["depth_arg"])
    want = ab.AlphaScene(hs, masks=[]).render(W, H, 0, 1, d["max_depth"], d["depth_arg"])
    assert np.array_equal(bits(actx.read_accum()[..., :3]), bits(want[..., :3]))
    # a mask upload makes the guides stale and drops the saved reprojection view
    actx.set_moments(True); actx.clear()
    actx.render(0, 1, 2); actx.render_guides(1)
    actx.reproject_film(agpt.reproject_params())                       # saves the view
    actx.upload_alpha_masks(masks)
    with pytest.raises(agpt.AgptError):
        actx.read_guides()
    with pytest.raises(agpt.AgptError):
        actx.denoise(agpt.denoise_params())
    actx.render_guides(1)
    film = actx.read_accum().copy()
    cam = hs.camera().copy(); cam[0] += 0.1
    actx.set_camera(cam)
    actx.render_guides(1)
    actx.reproject_film(agpt.reproject_params())                       # no saved view after the upload: film left as it is
    assert np.array_equal(bits(actx.read_accum()), bits(film))
    actx.set_moments(False)


def table_rows(agpt, hs):
    """The flattened scene's primitive and light rows."""
    t = _Tables.from_buffer_copy(hs.tables().raw[:ctypes.sizeof(_Tables)])
    prims = np.frombuffer(ctypes.string_at(t.prims, agpt.PRIM_DTYPE.itemsize * t.n_prims), agpt.PRIM_DTYPE).copy()
    lights = np.frombuffer(ctypes.string_at(t.lights, agpt.LIGHT_DTYPE.itemsize * t.n_lights), agpt.LIGHT_DTYPE).copy()
    return prims, lights


def test_masked_sphere_and_masked_emitter_are_refused(agpt, actx):
    """Render-time refusals with the masks resident: a mask on a sphere's material (cfg 12's textured spheres), and a mask on the
    material of an emitting plane (cfg 11's plane light, given a material)."""
    hs = agpt.HostScene(12, 0)
    hs.upload(actx); actx.set_film(32, 18)
    images, binds, prims, n_mat = scene_textures(agpt, hs)
    actx.upload_material_textures(images + [ONES], binds)
    sphere_mat = int(prims[(prims[:, 0] == agpt.PRIM_SPHERE) & (prims[:, 2] >= 0)][0, 2])
    masks = [agpt.alpha_mask() for _ in range(n_mat)]
    masks[sphere_mat] = agpt.alpha_mask(len(images), 0, .5)
    actx.upload_alpha_masks(masks)
    with pytest.raises(agpt.AgptError, match="sphere"):
        actx.render(0, 1, 2)
    with pytest.raises(agpt.AgptError, match="sphere"):
        actx.trace_primary(0)
    masks[sphere_mat] = agpt.alpha_mask()
    actx.upload_alpha_masks(masks)
    actx.render(0, 1, 2)                                               # the same scene without that mask renders

    hs = agpt.HostScene(11, 2)
    hs.upload(actx); actx.set_film(32, 18)
    rows, _ = table_rows(agpt, hs)
    plane_light = int(np.nonzero((rows["type"] == agpt.PRIM_PLANE) & (rows["area_light"] >= 0))[0][0])
    n_mat = scene_textures(agpt, hs)[3]
    rows["material"][plane_light] = 0
    actx.upload_table("primitives", rows)
    actx.upload_material_textures([ONES], [agpt.material_textures() for _ in range(n_mat)])
    actx.upload_alpha_masks([agpt.alpha_mask(0, 0, .5)] + [agpt.alpha_mask() for _ in range(n_mat - 1)])
    with pytest.raises(agpt.AgptError, match="emitter"):
        actx.render(0, 1, 2)
    actx.upload_alpha_masks([])
    actx.render(0, 1, 2)


ZERO = np.zeros((1, 1, 3), np.float32)
QUARTER = np.full((1, 1, 3), .25, np.float32)


@pytest.mark.parametrize("kind", ["mesh", "instance", "plane", "shape_lights"])
def test_all_zero_mask_equals_the_scene_without_that_primitive(agpt, actx, cfg14, kind):
    """A mask that keeps no hit (a constant 0, or a constant 0.25 at cutoff 0.5 on the plane) on the material of one primitive,
    whose scene's other masks stay bound: film, ray counts, guides and hit tables equal those of the scene with that primitive
    deleted (later primitives and the lights' primitive indices renumbered).  That scene runs the kernels without the mask test,
    so the reference here is not the statement.  cfg 14 level 1: the mirror quad (a plain TriangleMesh), the instance with its
    own material, and the grate plane.  cfg 11 level 2 (shape_lights): a non-emitting BVH mesh of the room lit by sampled plane
    and mesh lights, which have no CPU statement with masks; this puts the masked trace beside the shade kernels that sample
    shape lights."""
    cfg = 11 if kind == "shape_lights" else 14
    hs = agpt.HostScene(11, 2) if cfg == 11 else cfg14[1]
    d = agpt.config_defaults(cfg)
    images, binds, _, n_mat = scene_textures(agpt, hs)
    binds = binds or [agpt.material_textures() for _ in range(n_mat)]
    prims, lights = table_rows(agpt, hs)
    want_type = {"mesh": agpt.PRIM_MESH, "instance": agpt.PRIM_INSTANCE, "plane": agpt.PRIM_PLANE, "shape_lights": agpt.PRIM_BVH_MESH}[kind]
    k = int([i for i in np.nonzero(prims["type"] == want_type)[0]
             if prims["area_light"][i] < 0 and np.count_nonzero(prims["material"] == prims["material"][i]) == 1][-1])
    rng = np.random.default_rng(7)
    targets = np.concatenate([rng.uniform([-4, -1, -2], [4, 4.2, 5], (3000, 3)), rng.uniform([-3, 3.9, -3], [3, 4.1, 3], (1000, 3))])
    origins = np.where(targets[:, 1:2] > 3.8, np.array([.2, 5.3, .4]), np.array([.3, 2.0, -8.5]))
    dirs = targets - origins
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    rays7 = np.concatenate([origins, dirs, np.full((len(dirs), 1), 1e30)], 1).astype(np.float32)

    def run(flags=0):
        actx.set_film(W, H); actx.clear(); actx.reset_stats()
        actx.render(0, 2, d["max_depth"], d["depth_arg"], flags | agpt.FLAG_COUNTERS)
        st = actx.stats()
        film = actx.read_accum().copy()
        actx.render_guides(2)
        return (film, (st.rays_closest, st.rays_shadow, st.rays_mis, st.rays_mis_culled, st.rays_tail_culled), actx.read_guides(),
                actx.trace_primary(1).copy(), actx.trace_rays(rays7).copy(), actx.trace_rays(rays7, True).copy())

    # masked: the scene's own masks, that primitive's replaced by one that keeps nothing (the texture indices stay as they were)
    hs.upload(actx)
    actx.upload_material_textures(images + [ZERO, QUARTER], binds)
    masks = hs.alpha_masks() or [agpt.alpha_mask() for _ in range(n_mat)]
    masks[int(prims["material"][k])] = agpt.alpha_mask(len(images) + (1 if kind == "plane" else 0), 2, .5)
    actx.upload_alpha_masks(masks)
    got = run()
    # deleted: the scene as the host mirror uploads it (its own masks), without that primitive
    hs.upload(actx)
    rows = np.delete(prims, k)
    lt = lights.copy()
    lt["prim"] = np.where(lt["prim"] > k, lt["prim"] - 1, lt["prim"])
    actx.upload_table("lights", lt)
    actx.upload_table("primitives", rows)
    want = run()
    assert np.array_equal(bits(got[0]), bits(want[0])), "film"
    assert got[1] == want[1], "ray counts"
    for g, w in zip(got[2], want[2]):
        assert np.array_equal(bits(g), bits(w)), "guides"
    renum = lambda p: np.where(p >= k, p + 1, p)
    for g, w in zip(got[3:], want[3:]):
        assert np.array_equal(g["found"], w["found"])
        assert np.array_equal(g["prim"], np.where(w["prim"] >= 0, renum(w["prim"]), w["prim"]))
        assert np.array_equal(g["tri"], w["tri"]) and np.array_equal(bits(g["t"]), bits(w["t"]))
        assert not np.any(g["prim"] == k)
    # without its mask the primitive does stand in the way of some of these rays
    assert np.any(ab.AlphaScene(hs, masks=[]).trace_rays(rays7)["prim"] == k)
    actx.upload_alpha_masks([])


@pytest.mark.parametrize("level", [1, 2])
def test_cfg14_at_96x56_paths_and_guides_equal_the_statement(agpt, actx, cfg14, level):
    hs = cfg14[level]
    d = agpt.config_defaults(14)
    st = ab.AlphaScene(hs)
    hs.upload(actx); actx.set_film(W, 56)
    rng = np.random.default_rng(5 + level)
    xs, ys, ss = rng.integers(0, W, 300), rng.integers(0, 56, 300), rng.integers(0, 64, 300)
    for depth in (1, d["max_depth"]):
        got = actx.li_pixels(xs, ys, ss, depth, d["depth_arg"])
        assert np.array_equal(bits(got), bits(st.li_pixels(W, 56, xs, ys, ss, depth, d["depth_arg"])))
    actx.render_guides(2)
    for g, w in zip(actx.read_guides(), st.guides(W, 56, 2)):
        assert np.array_equal(bits(g), bits(w))


@pytest.mark.parametrize("h", [54, 56])
def test_cfg14_denoise_equals_the_statement(agpt, actx, cfg14, h):
    hs = cfg14[2]
    d = agpt.config_defaults(14)
    hs.upload(actx); actx.set_film(W, h); actx.set_moments(True); actx.clear()
    actx.render(0, 4, d["max_depth"], d["depth_arg"])
    actx.render_guides(3)
    alb, nd = actx.read_guides()
    walb, wnd = ab.AlphaScene(hs).guides(W, h, 3)
    assert np.array_equal(bits(alb), bits(walb)) and np.array_equal(bits(nd), bits(wnd))
    film, mom = actx.read_accum(), actx.read_moments()
    want_film = ab.AlphaScene(hs).render(W, h, 0, 4, d["max_depth"], d["depth_arg"])
    assert np.array_equal(bits(film[..., :3]), bits(want_film[..., :3]))
    for it in (0, 1, 5):
        p = agpt.denoise_params(iterations=it)
        out, _ = actx.denoise(p)
        want = dn.denoise(film, mom, alb, nd, it, p.sigma_luminance, p.sigma_depth, p.normal_power_log2)
        assert same_floats(out, want), it
    actx.set_moments(False)


def test_cfg14_adaptive_pixels_equal_plain_renders(agpt, actx, cfg14):
    hs = cfg14[1]
    d = agpt.config_defaults(14)
    hs.upload(actx); actx.set_film(48, 27); actx.set_moments(True)
    actx.render_adaptive(agpt.adaptive(2, 8, 2, 0.05), d["max_depth"])
    film, counts = actx.read_accum().copy(), actx.read_moments()[..., 3].copy()
    assert len(np.unique(counts)) > 1
    for k in np.unique(counts):
        actx.clear(); actx.render(0, int(k), d["max_depth"])
        plain = actx.read_accum()
        sel = counts == k
        assert np.array_equal(bits(film[sel]), bits(plain[sel]))
    actx.set_moments(False)


def test_cfg14_reprojection_follows_the_masked_guides(agpt, actx, cfg14):
    from oracle import reproject as rp
    hs = cfg14[1]
    d = agpt.config_defaults(14)
    st = ab.AlphaScene(hs)
    hs.upload(actx); actx.set_film(W, H); actx.set_moments(True); actx.clear()
    p = agpt.reproject_params()
    cam0 = hs.camera()
    actx.set_camera(cam0)
    actx.render_guides(2)
    alb0, nd0 = actx.read_guides()
    walb, wnd = st.guides(W, H, 2)
    assert np.array_equal(bits(alb0), bits(walb)) and np.array_equal(bits(nd0), bits(wnd))
    actx.reproject_film(p)                                             # saves the view
    _, _, G0 = rp.reproject(None, None, actx.read_accum().copy(), actx.read_moments().copy(), cam0, alb0, nd0, p.max_history, p.sigma_depth,
                            p.min_normal_dot)
    actx.render(0, 4, d["max_depth"])
    cam1 = rp.orbit(cam0, 2.5)
    actx.set_camera(cam1)
    actx.render_guides(2)
    film, mom = actx.read_accum().copy(), actx.read_moments().copy()
    alb, nd = actx.read_guides()
    actx.reproject_film(p)
    want_f, want_m, _ = rp.reproject(np.asarray(cam0, np.float32), G0, film, mom, cam1, alb, nd, p.max_history, p.sigma_depth, p.min_normal_dot)
    got_m = actx.read_moments()
    assert same_floats(actx.read_accum(), want_f) and same_floats(got_m, want_m)
    assert (got_m[..., 3] > 0).mean() > 0.3
    actx.set_moments(False)
    actx.set_camera(cam0)


def test_cfg14_two_gpus_equal_one(agpt, cfg14):
    if agpt.device_count() < 2:
        pytest.skip("one GPU visible")
    hs = cfg14[2]
    d = agpt.config_defaults(14)
    one, two = agpt.HostTracer(d["max_depth"], 0), agpt.HostTracer(d["max_depth"], devices=[0, 1])
    a = np.zeros((H, W, 4), np.float32); b = np.zeros((H, W, 4), np.float32)
    one.render(hs, W, H, a, 0, 4); two.render(hs, W, H, b, 0, 4)
    assert np.allclose(a, b, rtol=1e-5, atol=1e-6)
    one.close(); two.close()


def test_no_failed_device_checks(actx):
    """Meaningful under AGPT_LIB=libagpt_debug.so (test_debug_build_runs_this_file); a release build runs no checks."""
    s = actx.debug_status()
    print("MASKS_DEBUG_STATUS", s["failed"], s["first_code"], s["first_value"], s["checks"])
    assert s["failed"] == 0


def test_debug_build_runs_this_file():
    """The cfg 14 tests above under libagpt_debug.so (mask, texture and texel indices checked inside the masked kernels)."""
    lib = os.path.join(ROOT, "ag-pathtracer_b200", "libagpt_debug.so")
    assert os.path.exists(lib)
    env = dict(os.environ, AGPT_LIB=lib)
    out = subprocess.run([sys.executable, "-m", "pytest", "-q", "-s", "-p", "no:cacheprovider", os.path.abspath(__file__), "-k",
                          "(cfg14 and not two_gpus and not batches and not host_mirror) or all_zero or no_failed"], cwd=ROOT, env=env,
                         capture_output=True, text=True, timeout=1800)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if "MASKS_DEBUG_STATUS" in l][0]
    failed, checks = [int(v) for v in line.split("MASKS_DEBUG_STATUS")[1].split()[0:4:3]]
    assert checks > 100_000 and failed == 0
