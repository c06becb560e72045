"""GPU: textured and mapped shading in every k_shade_b instantiation a textured scene runs, against recoloured scenes and the
statements (include/agpt.h agpt_upload_textures, agpt_upload_material_textures).

A textured scene runs <false, false, false, T> or <true, true, true, T> (glass, the environment map and sampled shape lights),
T = 1 for base-colour textures, 2 for roughness-metallic or normal maps.  The checks here:
  * recoloured scenes (cfg 3, 5, 7, 10, 11): every Disney material bound to constant maps whose values differ from its own
    renders, bit for bit, what the untextured kernels render from a material table whose records already hold the derived
    values.  The TEX = 0 kernels are pinned to the reference, so every instantiation -- sampled shape lights included, which
    no statement covers together with textures -- is held to reference-pinned code: a use site that reads the material
    record instead of the hit's colours changes the film, the guides or the ray counts;
  * images that vary over the surface in <true, true, true, T> (cfg 10, cfg 7) against statements/maps_binding.py;
  * the device lookup per ray (agpt_probe_material_maps) against the statement's lookup and a float64 bilinear, at texel
    centres, texel edges, the seams and repeat-wrapped uvs, on images 1 texel wide or high and 4099 texels long;
  * renders and guides over several batches, and over two GPUs.
The construction of the recoloured scenes and its exactness are checked on the CPU in tests/test_textured_shading_cpu.py."""
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

from statements import maps_binding as mb  # noqa: E402
from statements import texture_binding as tb  # noqa: E402
from tests.test_gpu_textures import bits, materials, same_floats  # noqa: E402
from tests.test_textured_shading_cpu import FLAT, SCENES, floor_targets, recolouring, records, rewrite_metallic  # noqa: E402
from tests.test_textures_cpu import _Tables, bilinear64  # noqa: E402

# the ray counts that hold a render's path structure: traced + proven useless == what the statement issues
COUNTS = ("paths", "rays_closest", "rays_shadow", "rays_mis", "rays_mis_culled", "rays_tail_culled")


@pytest.fixture(scope="module")
def sctx(agpt):
    if agpt.device_count() == 0:
        pytest.fail("no CUDA device visible: -m gpu tests must run on the GPU box")
    ctx = agpt.Context(0)
    yield ctx
    ctx.close()


@pytest.fixture(scope="module")
def small_batch_ctx(agpt):
    """A context whose batches hold 2^10 paths (AGPT_BATCH_LOG2 is read when a context is created)."""
    old = os.environ.get("AGPT_BATCH_LOG2")
    os.environ["AGPT_BATCH_LOG2"] = "10"
    try:
        ctx = agpt.Context(0)
    finally:
        if old is None:
            os.environ.pop("AGPT_BATCH_LOG2", None)
        else:
            os.environ["AGPT_BATCH_LOG2"] = old
    yield ctx
    ctx.close()


def counted_render(agpt, ctx, n, max_depth, depth_arg, flags):
    """Film and COUNTS of samples [0, n) on the resident film, with exact ray accounting."""
    ctx.clear(); ctx.reset_stats()
    ctx.render(0, n, max_depth, depth_arg, flags | agpt.FLAG_COUNTERS)
    st = ctx.stats()
    return ctx.read_accum(), [getattr(st, k) for k in COUNTS]


def frame(agpt, ctx, d, flags):
    """96 x 54, 2 spp at the scene's own depth: the film, its ray counts, the guides of those samples and the denoised frame."""
    ctx.set_film(96, 54); ctx.set_moments(True)
    film, counts = counted_render(agpt, ctx, 2, d["max_depth"], d["depth_arg"], flags)
    ctx.render_guides(2)
    albedo, normal_depth = ctx.read_guides()
    denoised, _ = ctx.denoise(agpt.denoise_params())
    ctx.set_moments(False)
    return dict(film=film, albedo=albedo, normal_depth=normal_depth, denoised=denoised), counts


# ---- A. recoloured scenes: every instantiation against the untextured kernels ------------------------------------------------

@pytest.mark.parametrize("level", [1, 2])
@pytest.mark.parametrize("cfg,scene_level", SCENES)
def test_recoloured_scene_equals_the_untextured_render_of_its_records(agpt, sctx, cfg, scene_level, level):
    """Textured arm: the records after rewrite_metallic, bound to recolouring(level)'s maps (k_shade_b<..., level>,
    k_guides_tex / k_guides_maps).  Untextured arm: no textures, the expected records (k_shade_b<..., 0>, k_guides).  Film, ray
    counts, guides and denoised frame are equal bit for bit, and the film is not the scene's own."""
    d = agpt.config_defaults(cfg)
    flags = agpt.FLAG_RR_BY_BOUNCE if cfg == 10 else 0
    hs = agpt.HostScene(cfg, scene_level)
    hs.upload(sctx); sctx.set_film(96, 54); sctx.clear()
    sctx.render(0, 2, d["max_depth"], d["depth_arg"], flags)
    original = sctx.read_accum()
    base = rewrite_metallic(materials(hs))
    images, bind, want = recolouring(agpt, base, level)
    sctx.upload_table("materials", records(agpt, base))
    (sctx.upload_textures if level == 1 else sctx.upload_material_textures)(images, bind)
    got, got_counts = frame(agpt, sctx, d, flags)
    sctx.upload_textures([], [])
    sctx.upload_table("materials", records(agpt, want))
    ref, ref_counts = frame(agpt, sctx, d, flags)
    for k in ref:
        assert same_floats(got[k], ref[k]), k
    assert got_counts == ref_counts
    lit = np.any(original[..., :3] > 0, -1)
    changed = np.any(bits(got["film"][..., :3]) != bits(original[..., :3]), -1)
    assert lit.mean() > .5 and changed[lit].mean() > .5, (lit.mean(), changed[lit].mean())


# ---- B. varying maps in <true, true, true, T> against the statement ----------------------------------------------------------

def _image(W, H, seed):
    return np.random.default_rng(seed).uniform(.05, 1, (H, W, 3)).astype(np.float32)


def _roughness_metallic_checker(W, H):
    """G in {1/4, .6, 1}, B in {0, 1} over cells of 3 x 2 texels: the lobe set changes from texel to texel."""
    x, y = np.meshgrid(np.arange(W) // 3, np.arange(H) // 2)
    g = np.choose((x + 2 * y) % 3, [.25, .6, 1.0])
    return np.stack([np.full(g.shape, .5), g, ((x + y) & 1).astype(float)], -1).astype(np.float32)


def _height_field_normals(W, H, amplitude=.03, waves=3):
    """Tangent-space normals of h = amplitude sin(k u) sin(k v), stored as n / 2 + 1/2."""
    u, v = np.meshgrid((np.arange(W) + .5) / W, (np.arange(H) + .5) / H)
    k = 2 * np.pi * waves
    du, dv = amplitude * k * np.cos(k * u) * np.sin(k * v), amplitude * k * np.sin(k * u) * np.cos(k * v)
    n = np.stack([-du, -dv, np.ones_like(du)], -1)
    return (n / np.linalg.norm(n, axis=-1, keepdims=True) * .5 + .5).astype(np.float32)


def varying_maps(agpt, mats, level):
    """Disney material j: base image j % 3 of a 37 x 23, a 1 x 29 and a 31 x 1 image; level 2 adds a 13 x 9 roughness-metallic
    checker and a 48 x 40 height-field normal map.  Level 1 binds base images only, so the library selects T = 1."""
    images = [_image(37, 23, 1), _image(1, 29, 2), _image(31, 1, 3), _roughness_metallic_checker(13, 9), _height_field_normals(48, 40)]
    bind, j = [], 0
    for m in mats:
        if m["type"] != 1:
            bind.append(agpt.material_textures())
            continue
        bind.append(agpt.material_textures(j % 3) if level == 1 else agpt.material_textures(j % 3, 3, 4, .8))
        j += 1
    return images, bind


@pytest.mark.parametrize("level", [1, 2])
@pytest.mark.parametrize("cfg,scene_level", [(10, 2), (7, 0)])
def test_varying_maps_in_the_full_instantiation_equal_the_statement(agpt, sctx, cfg, scene_level, level):
    """cfg 10's rough glass and cfg 7's InfiniteAreaLight make RunWaves launch k_shade_b<true, true, true, level>; film
    (row-major 96 x 54, tiled 96 x 56; depth 1 and the scene's), li_pixels and the guides equal the statement bit for bit."""
    d = agpt.config_defaults(cfg)
    flags = agpt.FLAG_RR_BY_BOUNCE if cfg == 10 else 0
    hs = agpt.HostScene(cfg, scene_level)
    images, bind = varying_maps(agpt, materials(hs), level)
    ms = mb.MapsScene(hs, rr_by_bounce=cfg == 10)
    ms.set_textures(images, bind)
    hs.upload(sctx)
    sctx.upload_material_textures(images, bind)
    for w, h in ((96, 54), (96, 56)):
        sctx.set_film(w, h)
        for depth in (1, d["max_depth"]):
            sctx.clear()
            sctx.render(0, 2, depth, d["depth_arg"], flags)
            want = ms.render(w, h, 0, 2, depth, d["depth_arg"])
            assert np.array_equal(bits(sctx.read_accum()[..., :3]), bits(want[..., :3])), (w, h, depth)
    sctx.set_film(96, 54)
    rng = np.random.default_rng(cfg)
    xs, ys, ss = rng.integers(0, 96, 400), rng.integers(0, 54, 400), rng.integers(0, 50, 400)
    got = sctx.li_pixels(xs, ys, ss, d["max_depth"], d["depth_arg"], flags)
    assert np.array_equal(bits(got), bits(ms.li_pixels(96, 54, xs, ys, ss, d["max_depth"], d["depth_arg"])))
    sctx.set_film(96, 56)
    sctx.render_guides(3)
    alb, nd = sctx.read_guides()
    walb, wnd = ms.guides(96, 56, 3)
    assert np.array_equal(bits(alb), bits(walb)) and np.array_equal(bits(nd), bits(wnd))
    assert len(np.unique(alb[..., :3].reshape(-1, 3), axis=0)) > 500          # the albedo guide carries the images' detail
    sctx.upload_textures([], [])


# ---- C. the device lookup per ray -----------------------------------------------------------------------------------------

def _tables(agpt, hs):
    t = _Tables.from_buffer_copy(hs.tables().raw[:ctypes.sizeof(_Tables)])
    table = lambda p, n, dt: np.frombuffer(ctypes.string_at(p, dt.itemsize * n), dt)
    B = agpt.binding
    return table(t.prims, t.n_prims, B.PRIM_DTYPE), table(t.planes, t.n_planes, B.PLANE_DTYPE), table(t.spheres, t.n_spheres, B.SPHERE_DTYPE)


@pytest.mark.parametrize("W,H", [(1, 1), (1, 7), (7, 1), (2, 2), (5, 3), (37, 23), (4099, 3), (3, 4099)])
def test_lookup_per_ray_equals_the_statement_and_float64(agpt, sctx, W, H):
    """cfg 12's floor and plain quad grid carry a W x H base image (and a flat normal map, so the probe runs).  Rays from just
    above the floor straight down at texel centres, texel edges and one ulp inside its four edges, and rays at the grid where
    its uvs lie in [1, 2] (repeat wrap): the colour is the statement's lookup at the probe's uv bit for bit and a float64
    bilinear to 1e-6, and the floor's uv is the float64 (P - o) / half within 1e-6."""
    hs = agpt.HostScene(12, 0)
    prims, planes, spheres = _tables(agpt, hs)
    floor, grid = 0, 4                                             # the floor plane and the plain quad grid of cfg 12
    assert prims["type"][floor] == agpt.binding.PRIM_PLANE and prims["type"][grid] == agpt.binding.PRIM_MESH
    fm, gm = prims["material"][floor], prims["material"][grid]
    mats = materials(hs)
    mats["metallic"][[fm, gm]] = 0                                 # metallic 0: diffuse_r is the looked-up colour itself
    assert np.all(mats["lobes"][[fm, gm]] == 7)
    hs.upload(sctx)
    sctx.upload_table("materials", records(agpt, mats))
    # texels in [.5, 1]: at a seam fx is 1 - 2^-24 and a + fx * (b - a) rounds to within an ulp of the larger texel, so with a
    # wider range the relative 1e-6 would measure the stated lerp form's cancellation rather than the lookup
    img = np.random.default_rng(W * 7919 + H).uniform(.5, 1, (H, W, 3)).astype(np.float32)
    bind = [agpt.material_textures() for _ in mats]
    bind[fm] = bind[gm] = agpt.material_textures(1, -1, 0)
    sctx.upload_material_textures([FLAT, img], bind)
    # floor: straight down from 0.01 above it, away from the spheres that rest on it
    pl = planes[prims["payload"][floor]]
    o, half = pl["o"].astype(np.float64), np.array([pl["half_x"], pl["half_z"]], np.float64)
    xz = floor_targets(W, H, o[[0, 2]], half)
    y0 = np.float32(o[1] + .01)
    clear = np.ones(len(xz), bool)
    for s in spheres:
        rho2 = (xz[:, 0] - s["center"][0]) ** 2 + (xz[:, 1] - s["center"][2]) ** 2
        clear &= ~((rho2 < s["r"] ** 2) & (s["center"][1] - np.sqrt(np.maximum(s["r"] ** 2 - rho2, 0)) < y0 + .05))
    xz = xz[clear]
    n = len(xz)
    floor_rays = np.concatenate([xz[:, :1], np.full((n, 1), y0), xz[:, 1:], np.tile(np.float32([0, -1, 0, 1e30]), (n, 1))], 1)
    # grid: along +z at points of its upper-right quarter (uv = 2 (u, v) in [1, 2])
    u, v = [a.ravel() for a in np.meshgrid(np.linspace(.52, .98, 12), np.linspace(.52, .98, 12))]
    grid_rays = np.stack([-1.2 + (u - .5) * 2, 1.8 + (v - .5) * 2, np.full(len(u), 2.5), 0 * u, 0 * u, 0 * u + 1, np.full(len(u), 1e30)], 1)
    rows = sctx.probe_material_maps(np.concatenate([floor_rays, grid_rays]).astype(np.float32))
    sctx.upload_textures([], [])
    assert np.all(rows[:n, 0] == floor) and np.all(rows[n:, 0] == grid)          # every ray hits the surface it aims at
    assert np.all(rows[n:, 1:3] > 1)
    uv, colour = rows[:, 1:3], rows[:, 24:27]
    assert np.array_equal(bits(colour), bits(tb.lookup(img, uv)))
    want = bilinear64(img, uv)
    assert np.max(np.abs(colour - want) / np.maximum(np.abs(want), 1e-6)) < 1e-6
    closed = ((xz.astype(np.float64) - o[[0, 2]]) / half + 1) / 2
    assert np.max(np.abs(uv[:n] - closed)) <= 1e-6


# ---- D. split batches and two GPUs ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("w,h,n,batches", [(96, 54, 3, 3), (24, 16, 5, 3)])
@pytest.mark.parametrize("cfg,scene_level", [(12, 0), (13, 1), (13, 2)])
def test_split_batches_equal_one_batch_and_the_statement(agpt, sctx, small_batch_ctx, cfg, scene_level, w, h, n, batches):
    """cfg 12 (base-colour textures), cfg 13 (maps; level 2 adds glass) with 2^10-path batches: 96 x 54 holds one sample per
    batch, 24 x 16 (tiled) batches of 2, 2 and 1.  Film, ray counts and guides equal the one-batch context bit for bit, and
    the guides equal the statement."""
    hs = agpt.HostScene(cfg, scene_level)
    outs = []
    for ctx in (sctx, small_batch_ctx):
        hs.upload(ctx); ctx.set_film(w, h)
        film, counts = counted_render(agpt, ctx, n, 8, 0, 0)
        ctx.reset_stats()
        ctx.render_guides(n)
        outs.append((ctx.stats().launches_closest, film, counts, *ctx.read_guides()))
    (b1, f1, c1, a1, n1), (b2, f2, c2, a2, n2) = outs
    assert (b1, b2) == (1, batches)
    assert same_floats(f1, f2) and c1 == c2
    assert np.array_equal(bits(a1), bits(a2)) and np.array_equal(bits(n1), bits(n2))
    walb, wnd = (tb.TextureScene(hs) if cfg == 12 else mb.MapsScene(hs)).guides(w, h, n)
    assert np.array_equal(bits(a2), bits(walb)) and np.array_equal(bits(n2), bits(wnd))


def test_two_gpus_equal_one_with_maps(agpt):
    if agpt.device_count() < 2:
        pytest.skip("one GPU visible")
    hs = agpt.HostScene(13, 1)
    one, two = agpt.HostTracer(8, 0), agpt.HostTracer(8, devices=[0, 1])
    a = np.zeros((54, 96, 4), np.float32); b = np.zeros((54, 96, 4), np.float32)
    one.render(hs, 96, 54, a, 0, 4); two.render(hs, 96, 54, b, 0, 4)
    assert np.allclose(a, b, rtol=1e-5, atol=1e-6)
    one.close(); two.close()


def test_two_gpus_equal_one_with_recoloured_shape_lights(agpt):
    """cfg 11 with the level-1 recolouring: <true, true, true, 1> with sampled shape lights on every GPU.  HostTracer uploads
    the host scene's own tables, so the recoloured scene goes to each GPU's context and the two render as a Group."""
    if agpt.device_count() < 2:
        pytest.skip("one GPU visible")
    d = agpt.config_defaults(11)
    hs = agpt.HostScene(11, 2)
    base = rewrite_metallic(materials(hs))
    images, bind, _ = recolouring(agpt, base, 1)
    ctxs = [agpt.Context(g) for g in (0, 1, 0)]
    for c in ctxs:
        hs.upload(c); c.upload_table("materials", records(agpt, base)); c.upload_textures(images, bind)
        c.set_film(96, 54); c.clear()
    group = agpt.Group(ctxs[:2])
    group.render(0, 4, d["max_depth"], d["depth_arg"])
    group.reduce()
    ctxs[2].render(0, 4, d["max_depth"], d["depth_arg"])
    assert np.allclose(ctxs[0].read_accum(), ctxs[2].read_accum(), rtol=1e-5, atol=1e-6)
    for c in ctxs:
        c.close()


# ---- E. the debug build ---------------------------------------------------------------------------------------------------

def test_no_failed_device_checks(sctx):
    """Meaningful under AGPT_LIB=libagpt_debug.so (test_debug_build_runs_this_file); a release build runs no checks."""
    s = sctx.debug_status()
    print("SHADING_DEBUG_STATUS", s["failed"], s["first_code"], s["first_value"], s["checks"])
    assert s["failed"] == 0


def test_debug_build_runs_this_file():
    """The tests above under libagpt_debug.so (texture, texel and binding indices checked inside the kernels): none may fail."""
    lib = os.path.join(ROOT, "ag-pathtracer_b200", "libagpt_debug.so")
    assert os.path.exists(lib)
    env = dict(os.environ, AGPT_LIB=lib)
    out = subprocess.run([sys.executable, "-m", "pytest", "-q", "-s", "-p", "no:cacheprovider", os.path.abspath(__file__), "-k",
                          "not debug_build and not two_gpus"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if "SHADING_DEBUG_STATUS" in l][0]
    failed, checks = [int(v) for v in line.split("SHADING_DEBUG_STATUS")[1].split()[0:4:3]]
    assert checks > 100_000 and failed == 0
