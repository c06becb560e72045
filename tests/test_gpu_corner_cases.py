"""GPU: the branches the BASELINE configurations never reach (VERDICT r1 "untriggered branches").

* cfg 8 (host/scenes/config_scenes.h): degenerate triangles, a 29-deep chain-shaped SAH tree with
  exact-t ties, a plain TriangleMesh inside a run of BVH meshes, inf and NaN samples, live RR --
  against the golden fixture the reference produced and against the reference itself;
* hand-built node tables through the raw C ABI: a 100-deep tree (local-memory part of the traversal
  stack) against the CPU restatement; trees deeper than the stack, cyclic or shared links refused;
* Accumulator::CopyToSurface byte for byte against the reference's own lin2rgb / rgb2uint;
* a scene without any material; the -DAGPT_DEBUG build's in-kernel checks.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def same_floats(a, b):
    """Bit-equal, or NaN on both sides (x86 and the GPU produce different NaN payloads)."""
    a = np.ascontiguousarray(a, np.float32); b = np.ascontiguousarray(b, np.float32)
    return (bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))


def test_cfg8_against_golden(agpt, gpu_ctx):
    g = np.load(os.path.join(GOLDEN, "scene_cfg8.npz"))
    _, level, W, H, spp, md, da = [int(v) for v in g["case"]]
    hs = agpt.HostScene(8, level)
    hs.upload(gpu_ctx); gpu_ctx.set_film(W, H); gpu_ctx.clear(); gpu_ctx.reset_stats()
    hits = gpu_ctx.trace_primary(0, agpt.FLAG_COUNTERS)
    for f in ("found", "prim", "tri"):
        assert np.array_equal(hits[f], g["hits"][f]), f"primary {f}"
    assert np.array_equal(bits(hits["t"]), bits(g["hits"]["t"]))
    st = gpu_ctx.stats()
    assert (st.node_visits[0], st.box_tests[0], st.tri_tests[0]) == tuple(int(v) for v in g["walk_stats"])
    # the film: samples with NaN or inf luminance are zeroed (myapp.cpp:169-172), sums may overflow to inf
    gpu_ctx.render(0, spp, md, da)
    acc = gpu_ctx.read_accum()
    assert same_floats(acc[..., :3], g["accum"][..., :3]).all(), "accumulator differs from the reference's"
    assert np.isinf(g["accum"]).any(), "fixture lost its overflowing pixels"
    # hand-aimed rays: through all 30 chain triangles (ties, 29 pending far children), through the
    # triangle TriangleIntersect drops and TriangleIntersectP keeps
    got = gpu_ctx.trace_rays(g["probe_rays"], any_hit=False)
    want = g["probe_closest"]
    for f in ("found", "prim", "tri"):
        assert np.array_equal(got[f], want[f]), f
    assert np.array_equal(bits(got["t"]), bits(want["t"]))
    got_any = gpu_ctx.trace_rays(g["probe_rays"], any_hit=True)
    assert np.array_equal(got_any["found"], g["probe_any"]["found"])
    assert got["found"][5] == 0 and got_any["found"][5] == 1, "the underflowing triangle occludes but is never the closest hit"
    # single paths incl. the inf / NaN ones, unfiltered
    li = gpu_ctx.li_pixels(g["li_xs"], g["li_ys"], g["li_ss"], md, da)
    want = g["li"]
    assert np.isnan(want).any() and np.isinf(want).any()
    assert np.array_equal(np.isnan(li), np.isnan(want)) and np.array_equal(np.isinf(li), np.isinf(want))
    assert same_floats(li, want).all(axis=1).mean() >= 0.97


def test_cfg8_live_against_reference(agpt, ref_live, ref_golden, gpu_ctx):
    W, H, spp, level = 320, 180, 8, 3
    d = agpt.config_defaults(8)
    hs = agpt.HostScene(8, level)
    hs.upload(gpu_ctx); gpu_ctx.set_film(W, H); gpu_ctx.clear()
    gpu_ctx.render(0, spp, d["max_depth"], d["depth_arg"])
    got = gpu_ctx.read_accum()
    if ref_live:
        want, _ = ref_live.RefScene(8, level).render(W, H, 0, spp, d["max_depth"], d["depth_arg"])
    else:
        want = ref_golden("ref_cfg8_live.npz")["rgb"]
    exact = same_floats(got[..., :3], want[..., :3]).all(axis=-1).mean()
    print(f"cfg8 live: bit-identical pixels {exact:.5f}")
    assert exact >= 0.999
    # filtered slab test == strict, incl. the flat boxes of the chain mesh (0/0 slabs)
    gpu_ctx.clear(); gpu_ctx.render(0, spp, d["max_depth"], d["depth_arg"], agpt.FLAG_STRICT_BOXES)
    assert np.array_equal(bits(gpu_ctx.read_accum()), bits(got))


def chain_mesh(agpt, n, spacing=0.125):
    """n triangles perpendicular to x at x = i * spacing under a chain-shaped node table: interior I_j
    = { leaf j, I_(j+1) }, depth n - 1 (layout of bvhtrimesh.h:312-330: root 0, slot 1 unused, sibling pairs)."""
    verts = np.zeros((n, 3, 4), np.float32)
    for i in range(n):
        x = np.float32(i * spacing)
        verts[i, 0, :3] = (x, -1, -1); verts[i, 1, :3] = (x, 1, -1); verts[i, 2, :3] = (x, 0, 1)
    nodes = np.zeros(2 * n, agpt.NODE_DTYPE)
    lo = lambda a, b: (np.float32(a * spacing), -1, -1)
    hi = lambda a, b: (np.float32(b * spacing), 1, 1)
    def interior(k, j, child):
        nodes[k] = (lo(j, n - 1), hi(j, n - 1), child, 0)
    def leaf(k, j):
        nodes[k] = (lo(j, j), hi(j, j), j, 1)
    interior(0, 0, 2)
    for j in range(n - 1):
        leaf(2 + 2 * j, j)
        if j < n - 2:
            interior(3 + 2 * j, j + 1, 4 + 2 * j)
        else:
            leaf(3 + 2 * j, n - 1)
    return agpt.RawMesh(verts, nodes=nodes)


def upload_single_mesh(agpt, ctx, mesh):
    mat = agpt.make_material(agpt.MAT_DISNEY, (.7, .7, .7), .5, 0.)
    prims = np.zeros(1, agpt.PRIM_DTYPE)
    prims[0] = (agpt.PRIM_BVH_MESH, 0, 0, -1)
    ctx.upload_meshes([mesh])
    ctx.upload_table("spheres", np.zeros(0, agpt.SPHERE_DTYPE)); ctx.upload_table("planes", np.zeros(0, agpt.PLANE_DTYPE))
    ctx.upload_table("materials", [mat]); ctx.upload_table("lights", np.zeros(0, agpt.LIGHT_DTYPE))
    ctx.upload_table("primitives", prims)
    return prims, [mat]


def test_deep_chain_tree_matches_restatement(agpt):
    """A 100-level tree: rays against the chain keep up to 100 far children pending -- 24 in shared
    memory, the rest in the local-memory part of the stack.  Same hits, t bits and visit counts as
    the recursive CPU restatement on the same tables."""
    from oracle import port_binding as port
    n = 101
    mesh = chain_mesh(agpt, n)
    ctx = agpt.Context(0)
    prims, mats = upload_single_mesh(agpt, ctx, mesh)
    ps = port.PortScene.from_tables(prims, [mesh], materials=mats)
    rng = np.random.default_rng(5)
    m = 4096
    o = np.stack([np.full(m, 40.0), rng.uniform(-.9, .9, m), rng.uniform(-.9, .9, m)], 1)
    d = np.stack([np.full(m, -1.0), rng.normal(0, .02, m), rng.normal(0, .02, m)], 1)
    back = rng.random(m) < .3                      # from the near end too
    o[back, 0] = -3.0; d[back, 0] = 1.0
    tmax = np.where(rng.random(m) < .5, 3.0e38, rng.uniform(20, 45, m))
    rays = np.concatenate([o, d, tmax[:, None]], 1).astype(np.float32)
    for any_hit in (False, True):
        ctx.reset_stats()
        got = ctx.trace_rays(rays, any_hit=any_hit, flags=agpt.FLAG_COUNTERS)
        want, cnt = ps.trace_rays(rays, any_hit=any_hit)
        assert np.array_equal(got["found"], want["found"])
        if not any_hit:
            assert np.array_equal(got["tri"], want["tri"]) and np.array_equal(bits(got["t"]), bits(want["t"]))
            st = ctx.stats()
            assert (st.node_visits[0], st.box_tests[0], st.tri_tests[0]) == (cnt["interior"], cnt["boxes"], cnt["tris"])
            assert cnt["interior"] / m > 40, "rays must really descend the chain"
    ctx.close()


def test_bad_node_tables_are_refused(agpt):
    ctx = agpt.Context(0)
    good = chain_mesh(agpt, 40)
    upload_single_mesh(agpt, ctx, good)
    ray = np.array([[5.0, 0, 0, -1, 0, 0, 3e38]], np.float32)
    before = ctx.trace_rays(ray)
    # deeper than the traversal stack (128 levels)
    with pytest.raises(agpt.AgptError, match="deeper"):
        ctx.upload_meshes([chain_mesh(agpt, 140)])
    # a link back to an ancestor (the walk would never end), a child linked twice, links and leaf ranges outside the tables
    for edit, what in ((lambda nd: nd.__setitem__(5, (nd[5]["bmin"], nd[5]["bmax"], 2, 0)), "not a tree"),
                       (lambda nd: nd.__setitem__(7, (nd[7]["bmin"], nd[7]["bmax"], 4, 0)), "not a tree"),
                       (lambda nd: nd.__setitem__(3, (nd[3]["bmin"], nd[3]["bmax"], 79, 0)), "outside"),
                       (lambda nd: nd.__setitem__(2, (nd[2]["bmin"], nd[2]["bmax"], 39, 2)), "outside"),
                       (lambda nd: nd.__setitem__(3, (nd[3]["bmin"], nd[3]["bmax"], 1, 0)), "outside")):
        bad = chain_mesh(agpt, 40)
        edit(bad.nodes)
        with pytest.raises(agpt.AgptError, match=what):
            ctx.upload_meshes([bad])
    # a refused upload leaves the resident scene as it was
    after = ctx.trace_rays(ray)
    assert np.array_equal(before.view(np.uint32), after.view(np.uint32)) and after["found"][0] == 1
    ctx.close()


def test_resolve_is_byte_exact(agpt, ref, gpu_ctx):
    """Accumulator::CopyToSurface (myapp.h:34-41): the packed 0x00RRGGBB words equal the reference's own
    lin2rgb / rgb2uint (compiled from /root/reference) on a rendered film and on a sweep of float bit
    patterns: every channel value around each of the 255 byte thresholds, subnormals, huge values,
    negative, inf and NaN inputs."""
    cfg, W, H, spp = 1, 256, 144, 5
    d = agpt.config_defaults(cfg)
    hs = agpt.HostScene(cfg, 0)
    hs.upload(gpu_ctx); gpu_ctx.set_film(W, H); gpu_ctx.clear()
    gpu_ctx.render(0, spp, d["max_depth"], d["depth_arg"])
    acc = gpu_ctx.read_accum()
    assert np.array_equal(gpu_ctx.resolve(spp), ref.resolve(acc, spp))
    # synthetic film
    rng = np.random.default_rng(11)
    n = W * H * 3
    vals = np.empty(n, np.float32)
    k = np.arange(1, 256)
    thr = ((k / 256.0) ** 2.2).astype(np.float32)                       # pow(x, 1/2.2) crosses k/256 near here
    around = (bits(thr)[:, None].astype(np.int64) + np.arange(-40, 41)[None, :]).astype(np.uint32).view(np.float32).ravel()
    special = np.array([0.0, -0.0, 1e-45, 1e-40, 1.17549435e-38, 1.0, 0.999, 0.9990001, 2.0, 1e30, 3.4028235e38, np.inf, -np.inf, np.nan, -1.0, -1e-30], np.float32)
    fill = rng.integers(0, 0x7f800000, n - len(around) - len(special), dtype=np.uint32).view(np.float32)
    vals[:] = np.concatenate([around, special, fill])
    film = np.zeros((H, W, 4), np.float32)
    film[..., :3] = vals.reshape(H, W, 3)
    for samples in (1, 3, 256):
        gpu_ctx.write_accum(film)
        got = gpu_ctx.resolve(samples)
        want = ref.resolve(film, samples)
        assert np.array_equal(got, want), f"samples={samples}: {np.count_nonzero(got != want)} pixels differ"


def test_scene_without_materials(agpt):
    """Only null-material (emissive) shapes: legal upstream (integrator.h:152-161), the material table is empty."""
    from oracle import port_binding as port
    ctx = agpt.Context(0)
    prims = np.zeros(2, agpt.PRIM_DTYPE); spheres = np.zeros(2, agpt.SPHERE_DTYPE); lights = np.zeros(3, agpt.LIGHT_DTYPE)
    spheres[0] = ((0, 0, 0), 1.0, 1.0, (0, 0, 0)); spheres[1] = ((2.5, .5, 1), .75, .75 * .75, (0, 0, 0))
    prims[0] = (agpt.PRIM_SPHERE, 0, -1, 0); prims[1] = (agpt.PRIM_SPHERE, 1, -1, 1)
    lights[0] = (agpt.LIGHT_AREA, 0, (0, 0), (3, 2, 1), 0); lights[1] = (agpt.LIGHT_AREA, 1, (0, 0), (.5, 1, 2), 0)
    lights[2] = (agpt.LIGHT_UNIFORM_INFINITE, -1, (0, 0), (.1, .2, .3), 0)
    cam = agpt.HostScene(1, 0).camera()
    ctx.upload_meshes([]); ctx.upload_table("spheres", spheres); ctx.upload_table("planes", np.zeros(0, agpt.PLANE_DTYPE))
    ctx.upload_table("materials", []); ctx.upload_table("lights", lights); ctx.upload_table("primitives", prims)
    ctx.set_camera(cam)
    W, H = 96, 54
    ctx.set_film(W, H); ctx.clear()
    ctx.render(0, 3, 5)
    got = ctx.read_accum()
    ps = port.PortScene.from_tables(prims, spheres=spheres, lights=lights, camera=cam)
    want, _ = ps.render(W, H, 0, 3, 5)
    assert np.array_equal(bits(got), bits(want))
    assert got[..., :3].max() > 1.0
    ctx.close()


def test_debug_build_checks_pass():
    """libagpt_debug.so (-DAGPT_DEBUG): stack depth, node / triangle / primitive indices and queue slots are
    checked inside the kernels.  Renders the two corner-case scenes, the deepest accepted chain and a
    multi-mesh scene; no check may fail.  Own process: the library is chosen at load time (AGPT_LIB)."""
    lib = os.path.join(ROOT, "ag-pathtracer_b200", "libagpt_debug.so")
    assert os.path.exists(lib), "libagpt_debug.so not built (make -C ag-pathtracer_b200 debug)"
    code = r"""
import sys, numpy as np
sys.path.insert(0, %r)
from tests.conftest import load_agpt
from tests.test_gpu_corner_cases import chain_mesh, upload_single_mesh
agpt = load_agpt()
ctx = agpt.Context(0)
for cfg, level in ((6, 2), (8, 3), (4, 3), (5, 3)):
    d = agpt.config_defaults(cfg)
    hs = agpt.HostScene(cfg, level); hs.upload(ctx); ctx.set_film(160, 90); ctx.clear()
    ctx.render(0, 4, d["max_depth"], d["depth_arg"])
    ctx.trace_primary(0)
upload_single_mesh(agpt, ctx, chain_mesh(agpt, 129))
rays = np.array([[40.0, .1, .1, -1, 0, 0, 3e38]] * 64, np.float32)
ctx.trace_rays(rays); ctx.trace_rays(rays, any_hit=True)
s = ctx.debug_status()
print("DEBUG_STATUS", s["failed"], s["first_code"], s["first_value"], s["checks"])
""" % ROOT
    env = dict(os.environ, AGPT_LIB=lib)
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("DEBUG_STATUS")][0].split()
    failed, code_, value, checks = [int(v) for v in line[1:]]
    assert checks > 1_000_000, "the debug build ran no checks"
    assert failed == 0, f"in-kernel check failed: code {code_}, value {value}"
