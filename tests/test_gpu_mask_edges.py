"""GPU: the alpha-masked trace kernels (include/agpt.h agpt_upload_alpha_masks) on hand-built scenes, in every instantiation.

NOT REFERENCE BEHAVIOUR: the reference has no masks.  Every scene goes through the raw C ABI and is traced with flags 0,
FLAG_COUNTERS, FLAG_STRICT_BOXES and both, which runs each masked closest-hit and any-hit table kernel.  Hits, t bits and the
closest-hit walk's counters must equal the CPU statement (statements/agpt_alpha_oracle.cpp) on the same tables; where the
expectation is closed-form or float64 it is asserted too.  A rejected hit makes the walk go on, so the scenes aim at what then
matters: far children pending in the local-memory part of the stack, exact-t ties, degenerate triangles, runs longer than 32
mesh primitives and the root prepass after a rejected hit, and the edges of the lookup itself."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from statements import alpha_binding as ab  # noqa: E402
from tests.test_gpu_alpha_masks import ONES, bind_ones, scene_textures  # noqa: E402
from tests.test_gpu_corner_cases import bits, chain_mesh  # noqa: E402

ZERO = np.zeros((1, 1, 3), np.float32)
HALF = np.array([[[0, 0, 0], [1, 1, 1]]], np.float32)         # 2 x 1: (0 | 1)


@pytest.fixture(scope="module")
def mctx(agpt):
    if agpt.device_count() == 0:
        pytest.fail("no CUDA device visible: -m gpu tests must run on the GPU box")
    ctx = agpt.Context(0)
    yield ctx
    ctx.close()


def flag_sets(agpt):
    return (0, agpt.FLAG_COUNTERS, agpt.FLAG_STRICT_BOXES, agpt.FLAG_COUNTERS | agpt.FLAG_STRICT_BOXES)


def grey(agpt):
    return agpt.make_material(agpt.MAT_DISNEY, (.7, .7, .7), .5, 0.)


def image(texels):
    """A 1-row image whose texels are the given alphas, in all three channels."""
    return np.repeat(np.float32(texels)[None, :, None], 3, 2)


class Scene:
    """Hand-built tables, uploaded through the raw C ABI and stated by AlphaScene.from_tables on the same arrays."""

    def __init__(self, agpt, prims, meshes=(), spheres=None, planes=None, instances=None, n_materials=1, images=(), masks=()):
        self.agpt = agpt
        self.prims = np.asarray(prims, agpt.PRIM_DTYPE)
        self.meshes = list(meshes)
        self.spheres = np.zeros(0, agpt.SPHERE_DTYPE) if spheres is None else spheres
        self.planes = np.zeros(0, agpt.PLANE_DTYPE) if planes is None else planes
        self.instances = instances
        self.materials = [grey(agpt) for _ in range(n_materials)]
        self.images = list(images)
        self.masks = list(masks)

    def upload(self, ctx):
        a = self.agpt
        ctx.upload_meshes(self.meshes)
        ctx.upload_table("spheres", self.spheres); ctx.upload_table("planes", self.planes)
        ctx.upload_table("materials", self.materials); ctx.upload_table("lights", np.zeros(0, a.LIGHT_DTYPE))
        if self.instances is not None:
            ctx.upload_instances(self.instances)
        ctx.upload_table("primitives", self.prims)
        ctx.upload_material_textures(self.images, [a.material_textures() for _ in self.materials])
        ctx.upload_alpha_masks(self.masks)

    def statement(self):
        a = self.agpt
        return ab.AlphaScene.from_tables(self.prims, self.meshes, spheres=self.spheres, planes=self.planes, materials=self.materials,
                                         instances=self.instances, images=self.images,
                                         bindings=[a.material_textures() for _ in self.materials], masks=self.masks)


def same_hits(got, want, what=""):
    for f in ("found", "prim", "tri"):
        assert np.array_equal(got[f], want[f]), (what, f, np.count_nonzero(got[f] != want[f]))
    assert np.array_equal(bits(got["t"]), bits(want["t"])), what


def check(ctx, sc, rays7):
    """The scene's closest and any hits under every flag set equal the statement's, and so do the closest-hit walk's node
    visits, box tests and triangle tests.  Returns the statement's closest hits, any hits and counters."""
    agpt = sc.agpt
    sc.upload(ctx)
    st = sc.statement()
    want, cnt = st.trace_rays(rays7, counters=True)
    want_any = st.trace_rays(rays7, any_hit=True)
    for flags in flag_sets(agpt):
        ctx.reset_stats()
        got = ctx.trace_rays(rays7, False, flags)
        same_hits(got, want, flags)
        if flags & agpt.FLAG_COUNTERS:
            s = ctx.stats()
            assert (s.node_visits[0], s.box_tests[0], s.tri_tests[0]) == (cnt["interior"], cnt["boxes"], cnt["tris"]), flags
        got_any = ctx.trace_rays(rays7, True, flags)
        assert np.array_equal(got_any["found"], want_any["found"]), flags
    return want, want_any, cnt


def any_counters_keep_their_values_under_ones(ctx, sc, rays7):
    """The any-hit kernels count two boxes per visit, unlike the statement; with every mask replaced by a constant 1 the masked
    kernels must count what the unmasked ones count, field for field (table launches keep the ray order fixed)."""
    agpt = sc.agpt
    ones = Scene(agpt, sc.prims, sc.meshes, sc.spheres, sc.planes, sc.instances, len(sc.materials),
                 sc.images + [ONES], [agpt.alpha_mask(len(sc.images), 0, .5) if m.texture >= 0 else m for m in sc.masks])
    bare = Scene(agpt, sc.prims, sc.meshes, sc.spheres, sc.planes, sc.instances, len(sc.materials))
    fields = ("node_visits", "box_tests", "tri_tests", "analytic_tests", "warp_steps", "lane_steps")
    for flags in (agpt.FLAG_COUNTERS, agpt.FLAG_COUNTERS | agpt.FLAG_STRICT_BOXES):
        rows = []
        for s in (ones, bare):
            s.upload(ctx); ctx.reset_stats()
            hits = ctx.trace_rays(rays7, True, flags)
            st = ctx.stats()
            rows.append((hits["found"].copy(), [getattr(st, f)[1] for f in fields]))
        assert np.array_equal(rows[0][0], rows[1][0])
        assert rows[0][1] == rows[1][1], (flags, rows)
        assert rows[0][1][2] > 0


def rays(o, d, tmax=1e30):
    o = np.asarray(o, np.float64); d = np.asarray(d, np.float64)
    d = np.broadcast_to(d, o.shape); tmax = np.broadcast_to(np.asarray(tmax, np.float64), (len(o),))
    return np.concatenate([o, d, tmax[:, None]], 1).astype(np.float32)


def down(xz, y=5.0, tmax=1e30):
    """Axis-aligned rays straight down (-y) from height y over the given (x, z) points."""
    xz = np.asarray(xz, np.float64).reshape(-1, 2)
    return rays(np.stack([xz[:, 0], np.full(len(xz), y), xz[:, 1]], 1), [0, -1, 0], tmax)


def tree_mesh(agpt, verts, uvs, leaves):
    """A BVH mesh over triangles verts (n, 3, 3) whose node table is a chain of the given leaves (lists of consecutive triangle
    counts): interior I_j = { leaf j, I_(j+1) }, the last interior { leaf k-2, leaf k-1 }; boxes are the exact bounds."""
    verts = np.asarray(verts, np.float32)
    v4 = np.zeros((len(verts), 3, 4), np.float32)
    v4[..., :3] = verts
    starts = np.concatenate([[0], np.cumsum(leaves)]).astype(int)
    k = len(leaves)
    assert k >= 2 and starts[-1] == len(verts)
    box = lambda a, b: (verts[a:b].reshape(-1, 3).min(0), verts[a:b].reshape(-1, 3).max(0))
    nodes = np.zeros(2 * k, agpt.NODE_DTYPE)
    nodes[0] = (*box(0, len(verts)), 2, 0)
    for j in range(k - 1):
        nodes[2 + 2 * j] = (*box(starts[j], starts[j + 1]), starts[j], leaves[j])
        if j < k - 2:
            nodes[3 + 2 * j] = (*box(starts[j + 1], len(verts)), 4 + 2 * j, 0)
        else:
            nodes[3 + 2 * j] = (*box(starts[k - 1], starts[k]), starts[k - 1], leaves[k - 1])
    return agpt.RawMesh(v4, nodes=nodes, uvs=np.asarray(uvs, np.float32))


def plain_mesh(agpt, verts, uvs):
    v4 = np.zeros((len(verts), 3, 4), np.float32)
    v4[..., :3] = np.asarray(verts, np.float32)
    return agpt.RawMesh(v4, uvs=np.asarray(uvs, np.float32))


def key_uvs(keys, n_keys):
    """Constant uvs per triangle at the centre of texel `key` of an n_keys x 1 image: the triangle's alpha is that texel's."""
    u = (np.asarray(keys, np.float64) + .5) / n_keys
    uv = np.zeros((len(u), 3, 2), np.float32)
    uv[..., 0] = u[:, None]; uv[..., 1] = .5
    return uv


# ---- deep chains ------------------------------------------------------------------------------------------------------------------

def chain_rays(n_rays, length, seed):
    rng = np.random.default_rng(seed)
    o = np.stack([np.full(n_rays, length + 20.0), rng.uniform(-.9, .9, n_rays), rng.uniform(-.9, .9, n_rays)], 1)
    d = np.stack([np.full(n_rays, -1.0), rng.normal(0, .02, n_rays), rng.normal(0, .02, n_rays)], 1)
    back = rng.random(n_rays) < .3                                  # from the near end too
    o[back, 0] = -3.0; d[back, 0] = 1.0
    tmax = np.where(rng.random(n_rays) < .5, 3.0e38, rng.uniform(1, length + 25, n_rays))
    return rays(o, d, tmax)


def test_deep_chain_with_holes(agpt, mctx):
    """101 triangles under a 100-level chain (triangle i at x = i / 4) and a (0 | 1) mask: triangles 51-100 sit on texel 0, the
    rest alternate, odd ones kept.  A ray from +x descends to triangle 100 with 100 far children pending, then is rejected 51
    times in a row while the stack unwinds through its local-memory part (entries 24 and up) before triangle 49 stands.  Then the
    deepest chain the upload accepts (129 triangles, depth 128) with only triangle 0 kept: rays from +x are rejected up to 128
    times and pop the whole stack."""
    n = 101
    mesh = chain_mesh(agpt, n, spacing=.25)
    i = np.arange(n)
    mesh.uvs = key_uvs((i <= 50) & (i % 2 == 1), 2)
    prims = np.zeros(1, agpt.PRIM_DTYPE)
    prims[0] = (agpt.PRIM_BVH_MESH, 0, 0, -1)
    sc = Scene(agpt, prims, [mesh], images=[HALF], masks=[agpt.alpha_mask(0, 0, .5)])
    r = chain_rays(4096, n * .25, 5)
    want, want_any, cnt = check(mctx, sc, r)
    assert cnt["interior"] / len(r) > 30, "rays must really descend the chain"
    kept = want["tri"][want["found"] == 1]
    assert want["found"].mean() > .3 and np.all(kept % 2 == 1) and np.all(kept <= 49)
    bare = Scene(agpt, prims, [mesh]).statement().trace_rays(r)
    assert np.count_nonzero((bare["tri"] == 100) & (want["tri"] == 49)) > 400, "many rays must pass the 51 masked triangles"
    any_counters_keep_their_values_under_ones(mctx, sc, r)

    n = 129
    mesh = chain_mesh(agpt, n)
    mesh.uvs = key_uvs(np.arange(n) == 0, 2)
    sc = Scene(agpt, prims, [mesh], images=[HALF], masks=[agpt.alpha_mask(0, 0, .5)])
    r = chain_rays(2048, n * .125, 6)
    want, want_any, cnt = check(mctx, sc, r)
    assert set(np.unique(want["tri"])) <= {-1, 0} and want["found"].sum() > 500
    bare = Scene(agpt, prims, [mesh]).statement().trace_rays(r)
    assert np.count_nonzero((bare["tri"] == n - 1) & (want["tri"] == 0)) > 150, "rays rejected all along the chain"
    assert cnt["interior"] / len(r) > 60


# ---- exact-t ties -----------------------------------------------------------------------------------------------------------------

TRI = np.array([[-8, 0, -8], [8, 0, -8], [0, 0, 8]], np.float32)      # det = -256: t is exact for axis-aligned rays at integers


def aside(k):
    """A triangle off every tie ray (k: which)."""
    return TRI + np.float32([40 + 20 * k, 0, 0])


def tie_rays():
    """Straight down at integer (x, z) inside TRI and inside the plane of tie_scene, to t = 5 exactly."""
    xz = [(x, z) for z in range(-7, 8) for x in range(-7, 8) if abs(x) <= (8 - z) / 2 - .5]
    return down(xz)


def tie_scenes(agpt):
    """(name, scene maker, members): each member is a (prim, tri) pair that the tie rays hit at t = 5, in walk order.  The maker
    takes the set of members to mask out.  A triangle member has constant uvs on its own texel of one 8 x 1 image (material 0);
    a plane member has material 1, masked with a constant 0 when it is to be rejected."""
    def scene(prims, meshes, members, keys, planes=None):
        def make(rejected):
            texels = np.ones(8, np.float32)
            for m in rejected:
                if keys[members.index(m)] is not None:
                    texels[keys[members.index(m)]] = 0
            masks = [agpt.alpha_mask(0, 0, .5)]
            if planes is not None:
                masks.append(agpt.alpha_mask(1, 0, .5) if any(m[1] < 0 for m in rejected) else agpt.alpha_mask())
            return Scene(agpt, prims, meshes, planes=planes, n_materials=len(masks), images=[image(texels), ZERO], masks=masks)
        return make, members

    P = lambda *rows: np.array(list(rows), agpt.PRIM_DTYPE)
    out = []
    # one leaf: T0 == T1 in the leaf { T0, T1 }, T2 and T3 aside in a second leaf
    m = tree_mesh(agpt, [TRI, TRI, aside(0), aside(1)], key_uvs([0, 1, 7, 7], 8), [2, 2])
    out.append(("one leaf", *scene(P((agpt.PRIM_BVH_MESH, 0, 0, -1)), [m], [(0, 0), (0, 1)], [0, 1])))
    # sibling leaves: T0 in the left leaf, T2 == T0 in the right one; equal boxes, so the left leaf goes first
    m = tree_mesh(agpt, [TRI, aside(0), TRI, aside(1)], key_uvs([0, 7, 1, 7], 8), [2, 2])
    out.append(("sibling leaves", *scene(P((agpt.PRIM_BVH_MESH, 0, 0, -1)), [m], [(0, 0), (0, 2)], [0, 1])))
    # sibling leaves, the right box reaching nearer to the rays' origin: the right leaf goes first
    m = tree_mesh(agpt, [TRI, aside(0), TRI, aside(1) + np.float32([0, 3, 0])], key_uvs([0, 7, 1, 7], 8), [2, 2])
    out.append(("right leaf nearer", *scene(P((agpt.PRIM_BVH_MESH, 0, 0, -1)), [m], [(0, 2), (0, 0)], [1, 0])))
    # two BVH meshes of one run, a plain TriangleMesh between them
    a = tree_mesh(agpt, [TRI, aside(0)], key_uvs([0, 7], 8), [1, 1])
    b = plain_mesh(agpt, [aside(1), TRI], key_uvs([7, 1], 8))
    c = tree_mesh(agpt, [aside(2), TRI, aside(3)], key_uvs([7, 2, 7], 8), [1, 2])
    prims = P((agpt.PRIM_BVH_MESH, 0, 0, -1), (agpt.PRIM_MESH, 1, 0, -1), (agpt.PRIM_BVH_MESH, 2, 0, -1))
    out.append(("run of meshes", *scene(prims, [a, b, c], [(0, 0), (1, 1), (2, 1)], [0, 1, 2])))
    # a plane coincident with the triangles, between them in the list
    pl = np.zeros(1, agpt.PLANE_DTYPE)
    pl[0] = ((0, 0, 0), 9, 9, (0, 0, 0))
    prims = P((agpt.PRIM_BVH_MESH, 0, 0, -1), (agpt.PRIM_PLANE, 0, 1, -1), (agpt.PRIM_MESH, 1, 0, -1))
    out.append(("plane", *scene(prims, [a, b], [(0, 0), (1, -1), (2, 1)], [0, None, 1], planes=pl)))
    return out


def test_exact_t_ties_under_masks(agpt, mctx):
    """Coincident members hit at t = 5 exactly: the first in walk order wins.  Masking it out hands the hit to the next member,
    masking any other member changes nothing, masking all leaves a miss (any hit too)."""
    r = tie_rays()
    for name, make, members in tie_scenes(agpt):
        # the tie exists: each member alone is hit at the same t bits
        alone = []
        for m in members:
            want, _, _ = check(mctx, make([x for x in members if x != m]), r)
            assert want["found"].all() and (want["prim"] == m[0]).all(), (name, m)
            alone.append(want)
        t5 = bits(np.float32(5))
        for w in alone:
            assert (bits(w["t"]) == t5).all(), name
        for k in range(len(members)):
            for j in range(len(members)):
                rejected = [members[i] for i in range(len(members)) if i < k or i == j]     # the first k, and member j
                kept = [m for m in members if m not in rejected]
                want, want_any, _ = check(mctx, make(rejected), r)
                if not kept:
                    assert not want["found"].any() and not want_any["found"].any(), name
                else:
                    w = alone[members.index(kept[0])]
                    same_hits(want, w, (name, k, j))
        any_counters_keep_their_values_under_ones(mctx, make([]), r)


# ---- degenerate triangles ---------------------------------------------------------------------------------------------------------

def test_degenerate_triangles(agpt, mctx):
    """cfg 8's triangle whose |ng|^2 underflows (dropped by the closest-hit test, kept by the any-hit test) under a keep mask and
    a reject mask, and a sound triangle with collinear uvs."""
    tiny = np.array([[0, 0, 0], [1e-12, 0, 0], [0, 1e-12, 0]], np.float32)
    collinear = np.array([[4, -1, 2], [6, -1, 2], [5, 1, 2]], np.float32)
    uv = np.array([[[.5, .5]] * 3, [[0, .5], [1, .5], [.5, .5]]], np.float32)
    mesh = plain_mesh(agpt, [tiny, collinear], uv)
    prims = np.array([(agpt.PRIM_MESH, 0, 0, -1)], agpt.PRIM_DTYPE)
    o = np.array([[2.5e-13, 2.5e-13, -1]] * 3 + [[x, 0, -1] for x in np.linspace(4.55, 5.45, 61)])
    r = rays(o, [0, 0, 1], [3e38, 1.05, .9999] + [3e38] * 61)
    for img, cutoff in ((ONES, .5), (ZERO, .5), (HALF, .5)):
        sc = Scene(agpt, prims, [mesh], images=[img], masks=[agpt.alpha_mask(0, 0, cutoff)])
        want, want_any, _ = check(mctx, sc, r)
        assert not want["found"][:3].any(), "the underflowing triangle is never the closest hit"
        hit = want["found"][3:] == 1
        if img is HALF:                                          # u = (x - 4) / 2 along the collinear uvs: the cut at x = 5
            assert hit.any() and not hit.all()
        else:
            keep = img is ONES
            assert list(want_any["found"][:3]) == [keep, keep, 0]
            assert hit.all() == keep and hit.any() == keep


# ---- runs of more than 32 mesh primitives -----------------------------------------------------------------------------------------

def run_scene(agpt, rejected):
    """Spheres, 40 mesh primitives (BVH meshes, plain meshes and sheared or scaled instances of a chain) stacked along x, spheres.
    Primitive i's triangles lie near x = 44 - i, nearest first, so an accepted hit early in the list shrinks t and the roots
    of the later meshes are tested again; a rejected one leaves t as it was.  Each mesh primitive has its own material, masked
    with one channel of a 4 x 4 image (a checker, its inverse or stripes), a constant 1 or 0 per `rejected` (a set of primitive
    indices masked with 0), or not at all."""
    rng = np.random.default_rng(40)
    spheres = np.zeros(10, agpt.SPHERE_DTYPE)
    for k in range(10):
        c = (60 + 3 * k, rng.uniform(-2, 2), rng.uniform(-2, 2)) if k < 5 else (-30 - 3 * k, rng.uniform(-2, 2), rng.uniform(-2, 2))
        r = rng.uniform(.3, .8)
        spheres[k] = (c, r, r * r, (0, 0, 0))
    chain = chain_mesh(agpt, 5)
    chain.uvs = rng.uniform(-1, 2, (5, 3, 2)).astype(np.float32)
    meshes, rows, inst = [chain], [], []
    for k in range(5):
        rows.append((agpt.PRIM_SPHERE, k, -1, -1))
    for i in range(40):
        x = 44.0 - i
        kind = i % 4
        if kind == 3:                                           # an instance of the chain, scaled and sheared, at x
            s = np.array([[1, 0, 0], [.3 * rng.uniform(-1, 1), 1.5, 0], [.2, 0, 2.0]], np.float64) * rng.uniform(.8, 1.2)
            t = np.array([x, rng.uniform(-1, 1), rng.uniform(-1, 1)])
            inv = np.linalg.inv(s)
            inst.append((0, (0, 0, 0), np.concatenate([s, t[:, None]], 1).astype(np.float32).ravel(),
                         np.concatenate([inv, (-inv @ t)[:, None]], 1).astype(np.float32).ravel()))
            rows.append((agpt.PRIM_INSTANCE, len(inst) - 1, i, -1))
            continue
        n = rng.integers(1, 4) if kind == 1 else rng.integers(3, 7)
        c = rng.uniform(-2, 2, (n, 1, 3)) * np.array([.05, 1, 1])
        v = (c + rng.uniform(-1.5, 1.5, (n, 3, 3)) * np.array([.1, 1, 1]) + np.array([x, 0, 0])).astype(np.float32)
        uv = rng.uniform(-1, 2, (n, 3, 2)).astype(np.float32)
        if kind == 1:
            meshes.append(plain_mesh(agpt, v, uv))
            rows.append((agpt.PRIM_MESH, len(meshes) - 1, i, -1))
        else:
            leaves = [1] * n if kind == 0 else [2] + [1] * (n - 2)
            meshes.append(tree_mesh(agpt, v, uv, leaves))
            rows.append((agpt.PRIM_BVH_MESH, len(meshes) - 1, i, -1))
    for k in range(5, 10):
        rows.append((agpt.PRIM_SPHERE, k, -1, -1))
    inst = np.array(inst, np.dtype([("mesh", np.int32), ("pad", np.int32, 3), ("o2w", np.float32, 12), ("w2o", np.float32, 12)]))
    cells = np.kron(np.indices((2, 2)).sum(0) % 2, np.ones((2, 2)))
    checker = np.stack([cells, 1 - cells, np.tile([0, 0, 1, 1], (4, 1))], -1).astype(np.float32)   # per channel: checker, its inverse, stripes
    images = [checker, ONES, ZERO]
    masks = []
    for i in range(40):
        if i in rejected:
            masks.append(agpt.alpha_mask(2, 0, .5))
        else:
            masks.append([agpt.alpha_mask(0, (i // 3) % 3, .5), agpt.alpha_mask(1, 0, .5), agpt.alpha_mask()][i % 3])
    return Scene(agpt, np.array(rows, agpt.PRIM_DTYPE), meshes, spheres=spheres, instances=inst, n_materials=40, images=images,
                 masks=masks)


def test_runs_longer_than_32_mesh_primitives(agpt, mctx):
    rng = np.random.default_rng(41)
    n = 6000
    tgt = np.stack([rng.uniform(0, 50, n), rng.uniform(-2.5, 2.5, n), rng.uniform(-2.5, 2.5, n)], 1)
    o = np.where(rng.random((n, 1)) < .7, np.array([90.0, 0, 0]), np.array([-70.0, 0, 0])) + rng.uniform(-1, 1, (n, 3))
    r = rays(o, tgt - o, np.where(rng.random(n) < .7, 3e38, rng.uniform(30, 120, n)))
    for rejected in (set(), {0, 1, 2, 3, 5, 8, 33, 34, 35}):
        sc = run_scene(agpt, rejected)
        want, want_any, cnt = check(mctx, sc, r)
        prims = want["prim"][want["found"] == 1]
        assert np.any((prims >= 5) & (prims < 5 + 32)) and np.any(prims >= 5 + 32), "hits on both sides of the run split"
        assert np.any(prims < 5) and np.any(prims >= 45), "and on the spheres around the run"
        bare = Scene(agpt, sc.prims, sc.meshes, sc.spheres, sc.planes, sc.instances, 40).statement().trace_rays(r)
        assert np.count_nonzero(bare["prim"] != want["prim"]) > 200, "the masks must move many hits"
    any_counters_keep_their_values_under_ones(mctx, run_scene(agpt, set()), r)


# ---- the lookup's edges, with closed-form expectations ----------------------------------------------------------------------------

def edge_scene(agpt, img, channel, cutoff, tri_uvs):
    """A plane (material 0) at y = 0 over x, z in [-1, 1], and beside it at x = 10 one plain-mesh triangle (material 1) per uv
    in tri_uvs, all three vertices carrying that uv; both under the mask (img, channel, cutoff)."""
    pl = np.zeros(1, agpt.PLANE_DTYPE)
    pl[0] = ((0, 0, 0), 1, 1, (0, 0, 0))
    verts = [TRI + np.float32([20 + 20 * k, 0, 0]) for k in range(len(tri_uvs))]
    uv = np.zeros((len(tri_uvs), 3, 2), np.float32)
    uv[..., 0] = np.asarray(tri_uvs, np.float32)[:, None]; uv[..., 1] = .5
    prims = np.array([(agpt.PRIM_PLANE, 0, 0, -1), (agpt.PRIM_MESH, 0, 1, -1)], agpt.PRIM_DTYPE)
    m = agpt.alpha_mask(0, channel, cutoff)
    return Scene(agpt, prims, [plain_mesh(agpt, verts, uv)], planes=pl, n_materials=2, images=[img], masks=[m, m])


def edge_rays(plane_x, n_tris):
    """Straight down onto the plane at x in plane_x (z = 0.25), and onto vertex 0 of each triangle (barycentrics 0, 0: the uv
    is the vertex's bit for bit)."""
    xz = [(x, .25) for x in plane_x] + [(20 + 20 * k - 8, -8) for k in range(n_tris)]
    return down(np.array(xz, np.float64))


def test_lookup_edges_have_exact_outcomes(agpt, mctx):
    one_ulp_below_1 = np.nextafter(np.float32(1), np.float32(0))
    cases = []
    # alpha == cutoff is kept, the next float above it is not
    a = np.float32(.3)
    cases += [(image([a]), 0, a, True), (image([a]), 0, np.nextafter(a, np.float32(np.inf)), False)]
    # cutoff 0 keeps a 0 texel; a negative cutoff keeps everything; a cutoff above every texel rejects everything
    cases += [(ZERO, 0, 0., True), (ZERO, 0, -1e-30, True), (ONES, 0, np.nextafter(np.float32(1), np.float32(2)), False)]
    # channel selection: a (0.25, 0.5, 0.75) texel at cutoff 0.5
    c = np.float32([[[.25, .5, .75]]])
    cases += [(c, 0, .5, False), (c, 1, .5, True), (c, 2, .5, True)]
    xs = [-.5, 0, .75]
    tri_uvs = [.5, .25]
    for img, channel, cutoff, keep in cases:
        sc = edge_scene(agpt, img, channel, np.float32(cutoff), tri_uvs)
        r = edge_rays(xs, len(tri_uvs))
        want, want_any, _ = check(mctx, sc, r)
        assert (want["found"] == keep).all() and (want_any["found"] == keep).all(), (img.ravel(), channel, cutoff)
    # the (0 | 1) image where uv wraps: plane u = (x + 1) / 2 at 0, 1 - ulp, 1; triangle u at 1 - ulp, 1, -0, 1e30.  At u' = 0
    # the lookup blends the two texels half and half (alpha 0.5 exactly), at 1 - ulp it returns 0.5 + 2^-23
    plane_x = [-1, float(np.float32(1) - np.float32(2 ** -23)), 1]
    tri_uvs = [one_ulp_below_1, 1, -0., 1e30]
    want_alpha = np.float32([.5, .5 + 2 ** -23, .5, .5 + 2 ** -23, .5, .5, .5])
    uv = np.stack([np.concatenate([(np.float32(plane_x) + 1) * np.float32(.5), np.float32(tri_uvs)]), np.full(7, .5, np.float32)], 1)
    assert np.array_equal(bits(ab.lookup_channel(HALF, 0, uv)), bits(want_alpha))
    for cutoff in (np.float32(.5), np.nextafter(np.float32(.5), np.float32(1)), np.float32(.5 + 2 ** -23),
                   np.nextafter(np.float32(.5 + 2 ** -23), np.float32(1))):
        sc = edge_scene(agpt, HALF, 0, cutoff, tri_uvs)
        want, want_any, _ = check(mctx, sc, edge_rays(plane_x, len(tri_uvs)))
        assert np.array_equal(want["found"], (want_alpha >= cutoff).astype(np.uint32)), cutoff
        assert np.array_equal(want_any["found"], want["found"])


def test_the_cut_line_against_float64(agpt, mctx):
    """A plane and a triangle, each under a (0 | 1) mask at cutoff 0.5, where u = (x + 1) / 2 on both: 4097 rays each swept across
    the cut at x = 0, straight down onto both and slanted onto the plane (so that only the plane's own t gives the hit point).
    The device equals the statement bit for bit; against float64 the outcome may differ only where the float64 alpha lies
    within 1e-6 of the cutoff."""
    pl = np.zeros(1, agpt.PLANE_DTYPE)
    pl[0] = ((0, -1, 5), 1, 1, (0, 0, 0))
    tri = np.array([[-1, 0, -1], [1, 0, -1], [0, 0, 1]], np.float32)
    uv = np.array([[[0, .5], [1, .5], [.5, .5]]], np.float32)
    prims = np.array([(agpt.PRIM_BVH_MESH, 0, 0, -1), (agpt.PRIM_PLANE, 0, 1, -1)], agpt.PRIM_DTYPE)
    mesh = tree_mesh(agpt, [tri, tri + np.float32([5, 0, 0])], np.concatenate([uv, uv]), [1, 1])
    m = agpt.alpha_mask(0, 0, .5)
    sc = Scene(agpt, prims, [mesh], planes=pl, n_materials=2, images=[HALF], masks=[m, m])
    x = np.linspace(-.01, .01, 4097).astype(np.float32)
    slanted = rays(np.stack([x - .5, np.zeros_like(x), np.full_like(x, 5.3)], 1), [.5, -1, 0])
    r = np.concatenate([down(np.stack([x, np.full_like(x, -.5)], 1)), down(np.stack([x, np.full_like(x, 5.3)], 1)), slanted])
    want, want_any, _ = check(mctx, sc, r)
    o, d = slanted[:, :3].astype(np.float64), slanted[:, 3:6].astype(np.float64)
    x64 = np.concatenate([x, x, o[:, 0] + (-1 - o[:, 1]) / d[:, 1] * d[:, 0]]).astype(np.float64)
    s = (x64 + 1) / 2 * 2 - .5                                  # the lookup in float64: alpha = s - floor(s) between the centres
    alpha = s - np.floor(s)
    exact = alpha >= .5
    near = np.abs(alpha - .5) <= 1e-6
    got = want["found"] == 1
    assert not np.any((got != exact) & ~near)
    for part in np.split(got, 3):
        assert part.any() and not part.all()
    assert np.array_equal(want_any["found"], want["found"])


# ---- render-level counters --------------------------------------------------------------------------------------------------------

def counted_waves(agpt, ctx, d):
    """Per kernel kind, per bounce: rays, node visits, box and triangle tests, and the analytic records of the camera rays only.
    Later waves read sphere records where any lane of a warp may hit a sphere run's box, so their analytic count depends on which
    rays share a warp, i.e. on the order of queue appends, like the warp and lane steps."""
    ctx.set_film(96, 54); ctx.clear(); ctx.reset_stats()
    ctx.render(0, 2, d["max_depth"], d["depth_arg"], agpt.FLAG_COUNTERS)
    fields = ("rays", "node_visits", "box_tests", "tri_tests")
    waves = [[tuple(w[f] for f in fields) for w in ctx.wave_stats(kind)] for kind in (0, 1)]
    return waves, ctx.wave_stats(0)[0]["analytic_tests"], ctx.read_accum().copy()


@pytest.mark.parametrize("cfg,level", [(3, 2), (14, 1)])
def test_all_ones_masks_keep_the_per_bounce_counters(agpt, mctx, cfg, level):
    """A render with every mask a constant 1 counts, bounce by bounce and for both kernel kinds, what the render without masks
    counts (counted_waves leaves out what depends on the order of queue appends)."""
    hs = agpt.HostScene(cfg, level)
    d = agpt.config_defaults(cfg)
    hs.upload(mctx)
    if cfg == 3:
        want = counted_waves(agpt, mctx, d)
        assert bind_ones(agpt, mctx, hs) > 0
        got = counted_waves(agpt, mctx, d)
    else:
        images, binds, _, _ = scene_textures(agpt, hs)
        mctx.upload_material_textures(images + [ONES], binds)
        masks = [agpt.alpha_mask(len(images), 0, .5) if m.texture >= 0 else m for m in hs.alpha_masks()]
        mctx.upload_alpha_masks(masks)
        got = counted_waves(agpt, mctx, d)
        mctx.upload_alpha_masks([])
        want = counted_waves(agpt, mctx, d)
    assert got[0] == want[0] and len(want[0][0]) > 1 and len(want[0][1]) > 1
    assert got[1] == want[1]
    assert np.array_equal(bits(got[2]), bits(want[2]))


def test_no_failed_device_checks(mctx):
    """Meaningful under AGPT_LIB=libagpt_debug.so (test_debug_build_runs_this_file); a release build runs no checks."""
    s = mctx.debug_status()
    print("MASK_EDGES_DEBUG_STATUS", s["failed"], s["first_code"], s["first_value"], s["checks"])
    assert s["failed"] == 0


def test_debug_build_runs_this_file():
    """This module under libagpt_debug.so: stack depth, node, triangle, mask, texture and texel indices checked in the kernels."""
    lib = os.path.join(ROOT, "ag-pathtracer_b200", "libagpt_debug.so")
    assert os.path.exists(lib)
    env = dict(os.environ, AGPT_LIB=lib)
    out = subprocess.run([sys.executable, "-m", "pytest", "-q", "-s", "-p", "no:cacheprovider", os.path.abspath(__file__), "-k",
                          "not debug_build"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if "MASK_EDGES_DEBUG_STATUS" in l][0]
    failed, checks = [int(v) for v in line.split("MASK_EDGES_DEBUG_STATUS")[1].split()[0:4:3]]
    assert checks > 100_000 and failed == 0
