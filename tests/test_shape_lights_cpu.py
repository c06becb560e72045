"""CPU: the statement of sampled plane and mesh area lights (AGPT_LIGHT_SAMPLE_SHAPE, oracle/agpt_shape_oracle.cpp ShapeSample /
ShapePdf).  PARITY UNPINNED BY THE REFERENCE -- its Plane and TriangleMesh cannot be sampled -- so the statement is checked
for what makes it a correct light sampler: the pdf it reports is Pdf_Li of the direction it sampled, Pdf_Li integrates to 1
over the sphere, and the estimator reproduces Lambert's closed-form irradiance of a polygon."""
import numpy as np
import pytest


@pytest.fixture(scope="module")
def port():
    from oracle import shape_binding
    return shape_binding


def light_scene(agpt, port, shape, verts=None, plane=None):
    """One emissive shape, sampled: shape = 'plane' (plane = (o3, half_x, half_z)) or 'mesh' (verts [n, 3, 3])."""
    prims = np.zeros(1, agpt.PRIM_DTYPE)
    lights = np.zeros(1, agpt.LIGHT_DTYPE)
    lights[0] = (agpt.LIGHT_AREA, 0, (agpt.LIGHT_SAMPLE_SHAPE, 0), (1, 1, 1), 0)
    if shape == "plane":
        planes = np.zeros(1, agpt.PLANE_DTYPE)
        planes[0] = (plane[0], plane[1], plane[2], (0, 0, 0))
        prims[0] = (agpt.PRIM_PLANE, 0, -1, 0)
        return port.ShapeScene.from_tables(prims, planes=planes, lights=lights)
    v = np.zeros((len(verts), 3, 4), np.float32)
    v[..., :3] = verts
    prims[0] = (agpt.PRIM_MESH, 0, -1, 0)
    return port.ShapeScene.from_tables(prims, [agpt.RawMesh(v)], lights=lights)


def probe(ps, light, ref, u, wq):
    n = len(u)
    a = np.concatenate([np.broadcast_to(np.asarray(ref, np.float32), (n, 3)), u, np.broadcast_to(np.asarray(wq, np.float32), (n, 3))], 1)
    return ps.probe_light_sample(light, a)


QUAD = [[[-.5, 2, -.5], [.5, 2, -.5], [.5, 2, .5]], [[-.5, 2, -.5], [.5, 2, .5], [-.5, 2, .5]]]


def test_sampled_pdf_is_pdf_li_of_the_sampled_direction(agpt, port):
    """cfg 11's three lights (2-triangle panel, plane panel, level-2 BVH icosphere) from points all over the room: wherever the
    sampled point is the first hit along its direction, the pdf Sample_Li returns is Pdf_Li of that direction."""
    hs = agpt.HostScene(11, 1)
    ps = port.ShapeScene(hs)
    assert [hs.prim_info(p)["kind"] for p in (3, 4, 5)] == [agpt.PRIM_MESH, agpt.PRIM_PLANE, agpt.PRIM_BVH_MESH]
    rng = np.random.default_rng(11)
    n = 10000
    for light, prim in ((0, 3), (1, 4), (2, 5)):
        ref = rng.uniform([-3.8, -.8, -8.8], [3.8, 4.8, 3.8], (n, 3)).astype(np.float32)
        u = rng.random((n, 2), np.float32)
        a = np.concatenate([ref, u, np.zeros((n, 3), np.float32)], 1)
        s = ps.probe_light_sample(light, a)
        ok = s[:, 3] > 0
        assert ok.mean() > 0.9
        wi = s[:, :3] - ref
        dist = np.linalg.norm(wi.astype(np.float64), axis=1)
        wi = (wi / dist[:, None]).astype(np.float32)
        a[:, 5:8] = wi
        q = ps.probe_light_sample(light, a)
        hits, _ = ps.trace_rays(np.concatenate([ref, wi, np.full((n, 1), 3e38, np.float32)], 1))
        first = ok & (hits["prim"] == prim) & (np.abs(hits["t"] - dist) < 1e-4 * dist + 1e-5)
        if light != 1:
            # ... and on the sampled triangle (a grazing ray near an edge can meet the neighbour first)
            v = hs.mesh_verts(prim).reshape(-1, 3, 3).astype(np.float64)[np.where(hits["prim"] == prim, hits["tri"], 0)]
            tn = np.cross(v[:, 1] - v[:, 0], v[:, 2] - v[:, 0])
            tn /= np.linalg.norm(tn, axis=1, keepdims=True)
            first &= np.abs((tn * s[:, 5:8]).sum(1)) > 1 - 1e-6
        # (at grazing incidence the pdf's relative sensitivity to the last bits of the direction is 1 / cos: leave those out)
        first &= np.abs((wi * s[:, 5:8]).sum(1)) > 1e-2
        print(f"light {light}: {first.sum()} of {n} samples are first hits")
        assert first.sum() > 0.3 * n
        assert np.allclose(q[first, 4], s[first, 3], rtol=1e-4, atol=0)


@pytest.mark.parametrize("shape", ["quad", "plane"])
def test_pdf_li_integrates_to_one(agpt, port, shape):
    """Monte Carlo over uniform directions: the integral of Pdf_Li over the sphere is 1 (within 4 sigma)."""
    ps = light_scene(agpt, port, "mesh", verts=QUAD) if shape == "quad" else light_scene(agpt, port, "plane", plane=((0, 2, 0), .5, .5))
    rng = np.random.default_rng(3)
    for ref in ((0.1, 1.2, -0.2), (1.5, 0.3, 0.8)):
        n = 400000
        w = rng.normal(size=(n, 3))
        w /= np.linalg.norm(w, axis=1, keepdims=True)
        out = probe(ps, 0, ref, np.zeros((n, 2), np.float32), w.astype(np.float32))
        f = out[:, 4].astype(np.float64) * 4 * np.pi
        est, sigma = f.mean(), f.std() / np.sqrt(n)
        assert (f > 0).mean() > 0.005
        assert abs(est - 1) < 4 * sigma, (shape, ref, est, sigma)


def polygon_irradiance(x, n, poly):
    """Lambert's formula: E / L = 1/2 sum_i angle(v_i - x, v_i+1 - x) * (n . unit(cross(v_i - x, v_i+1 - x))), polygon above the horizon."""
    e = 0.0
    m = len(poly)
    for i in range(m):
        a, b = np.subtract(poly[i], x), np.subtract(poly[(i + 1) % m], x)
        c = np.cross(a, b)
        ang = np.arccos(np.clip(np.dot(a, b) / np.linalg.norm(a) / np.linalg.norm(b), -1, 1))
        e += ang * np.dot(n, c / np.linalg.norm(c))
    return abs(e) / 2


@pytest.mark.parametrize("shape", ["plane", "quad", "triangle"])
def test_estimator_matches_closed_form_irradiance(agpt, port, shape):
    tri = [[[-.6, 2, -.4], [.7, 2, -.2], [.1, 2, .9]]]
    if shape == "plane":
        ps, poly = light_scene(agpt, port, "plane", plane=((0, 2, 0), .5, .5)), [(-.5, 2, -.5), (.5, 2, -.5), (.5, 2, .5), (-.5, 2, .5)]
    elif shape == "quad":
        ps, poly = light_scene(agpt, port, "mesh", verts=QUAD), [(-.5, 2, -.5), (.5, 2, -.5), (.5, 2, .5), (-.5, 2, .5)]
    else:
        ps, poly = light_scene(agpt, port, "mesh", verts=tri), [tuple(v) for v in tri[0]]
    rng = np.random.default_rng(5)
    # straight below, off to the side, tilted, and near-grazing (the light a few degrees above the receiver's horizon)
    cases = [((0, 0, 0), (0, 1, 0)), ((1.2, .5, -.7), (0, 1, 0)), ((.3, 1., .4), (.6, .8, 0)), ((4., 1.85, .2), (0, 1, 0)), ((.2, 1.9, 3.), (0, 1, 0))]
    for x, nrm in cases:
        nrm = np.asarray(nrm, np.float64) / np.linalg.norm(nrm)
        n = 200000
        out = probe(ps, 0, x, rng.random((n, 2), np.float32), (0, 1, 0))
        ok = out[:, 3] > 0
        wi = out[:, :3].astype(np.float64) - np.asarray(x)
        wi /= np.linalg.norm(wi, axis=1, keepdims=True)
        f = np.zeros(n)
        f[ok] = np.maximum(0, wi[ok] @ nrm) / out[ok, 3]
        est, sigma = f.mean(), f.std() / np.sqrt(n)
        want = polygon_irradiance(np.asarray(x, np.float64), nrm, poly)
        assert abs(est - want) < 4 * sigma + 1e-6 * want, (shape, x, est, want, sigma)


def test_degenerate_triangles_are_never_sampled(agpt, port):
    """A triangle flagged degenerate (collinear vertices, far away at x = 100) is never picked -- not even by u.x = 1 or u.x on a
    cdf step; a mesh of degenerate triangles only gives pdf 0 and Pdf_Li 0."""
    deg = [[100, 2, 0], [101, 2, 0], [102, 2, 0]]
    verts = [deg, QUAD[0], deg, deg, QUAD[1], deg]
    ps = light_scene(agpt, port, "mesh", verts=verts)
    ux = np.concatenate([np.linspace(0, 1, 4001), [0.5, 1.0, np.nextafter(1, 0)]]).astype(np.float32)
    u = np.stack([ux, np.full_like(ux, .37)], 1)
    out = probe(ps, 0, (0, 0, 0), u, (0, 1, 0))
    ok = out[:, 3] > 0
    assert ok.mean() > 0.99
    assert np.all(np.abs(out[ok, 0]) <= .5) and np.all(out[ok, 1] == 2)
    both = np.unique(np.sign(out[ok, 0] - out[ok, 2]))           # both quad triangles are used
    assert len(both) >= 2
    none = light_scene(agpt, port, "mesh", verts=[deg, deg])
    rng = np.random.default_rng(2)
    w = rng.normal(size=(500, 3)).astype(np.float32)
    w[:, 1] = np.abs(w[:, 1])
    out = probe(none, 0, (101, 1, 0), rng.random((500, 2), np.float32), w)
    assert np.all(out[:, 3] == 0) and np.all(out[:, 4] == 0)


def test_without_flags_the_statement_is_the_oracle(agpt, port):
    """The statement restates EstimateDirect and Li with the extension added: with no light flagged (cfg 5, cfg 7's environment
    light) films and single paths are the oracle's bit for bit."""
    from oracle import port_binding
    for cfg, level in ((5, 2), (7, 0)):
        d = agpt.config_defaults(cfg)
        hs = agpt.HostScene(cfg, level)
        a, ca = port.ShapeScene(hs).render(64, 36, 0, 2, d["max_depth"], d["depth_arg"])
        b, cb = port_binding.PortScene(hs).render(64, 36, 0, 2, d["max_depth"], d["depth_arg"])
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)) and ca == cb
