"""GPU: scene-level parity against the golden fixtures (no oracle library needed on the box),
single-path radiance, arbitrary-ray traces, traversal counters, and the host C++ API."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def rel_rmse(gpu, cpu):
    g = gpu[..., :3].astype(np.float64); c = cpu[..., :3].astype(np.float64)
    return float(np.sqrt(np.mean((g - c) ** 2)) / max(np.mean(np.abs(c)), 1e-30))


@pytest.mark.parametrize("cfg", [1, 2, 3, 4, 5, 6, 7])
def test_against_golden(agpt, gpu_ctx, cfg):
    g = np.load(os.path.join(GOLDEN, f"scene_cfg{cfg}.npz"))
    _, level, W, H, spp, md, da = [int(v) for v in g["case"]]
    hs = agpt.HostScene(cfg, level)
    hs.upload(gpu_ctx); gpu_ctx.set_film(W, H); gpu_ctx.clear(); gpu_ctx.reset_stats()
    hits = gpu_ctx.trace_primary(0, agpt.FLAG_COUNTERS)
    for f in ("found", "prim", "tri"):
        assert np.array_equal(hits[f], g["hits"][f]), f"primary {f}"
    assert np.array_equal(bits(hits["t"]), bits(g["hits"]["t"])), "primary t bits"
    # traversal work counted on the device == the reference's instrumented walk
    st = gpu_ctx.stats()
    assert (st.node_visits[0], st.box_tests[0], st.tri_tests[0]) == tuple(int(v) for v in g["walk_stats"])
    gpu_ctx.render(0, spp, md, da)
    acc = gpu_ctx.read_accum()
    assert rel_rmse(acc, g["accum"]) <= 1e-3
    assert np.mean(np.all(bits(acc[..., :3]) == bits(g["accum"][..., :3]), axis=-1)) >= 0.999, "accumulator bit-identical to the reference's"
    # arbitrary rays: Scene::Intersect and Scene::IntersectP
    got = gpu_ctx.trace_rays(g["probe_rays"], any_hit=False)
    want = g["probe_closest"]
    for f in ("found", "prim", "tri"):
        assert np.array_equal(got[f], want[f])
    assert np.array_equal(bits(got["t"]), bits(want["t"]))
    got = gpu_ctx.trace_rays(g["probe_rays"], any_hit=True)
    assert np.array_equal(got["found"], g["probe_any"]["found"])
    # single paths (Integrator::Li): most are bit-identical, all are close
    li = gpu_ctx.li_pixels(g["li_xs"], g["li_ys"], g["li_ss"], md, da)
    want = g["li"]
    assert np.all(bits(li) == bits(want), axis=1).mean() >= 0.97, "single-path radiance bit-identical"
    assert np.isclose(li, want, rtol=1e-3, atol=1e-5).all(axis=1).mean() >= 0.97


def test_host_api_equals_c_abi(agpt, gpu_ctx):
    """CudaPathTracer::Render over host buffers == agpt_render + agpt_read_accum, bit for bit,
    and successive Render calls accumulate like successive Ticks."""
    cfg, level, W, H = 6, 2, 64, 36
    d = agpt.config_defaults(cfg)
    hs = agpt.HostScene(cfg, level)
    hs.upload(gpu_ctx); gpu_ctx.set_film(W, H); gpu_ctx.clear()
    gpu_ctx.render(0, 6, d["max_depth"], d["depth_arg"])
    direct = gpu_ctx.read_accum()
    tr = agpt.HostTracer(d["max_depth"], 0)
    acc = np.zeros((H, W, 4), np.float32)
    tr.render(hs, W, H, acc, 0, 2, d["depth_arg"])
    tr.render(hs, W, H, acc, 2, 4, d["depth_arg"])
    assert np.array_equal(bits(acc), bits(direct))
    # Li() single-ray entry point returns finite radiance and is deterministic per call index
    a = tr.li(hs, (-1.46, 1.16, -4.64), (1.46, -1.16, 4.64))
    assert np.isfinite(a).all()
    tr.close()


def test_resolve_matches_copy_to_surface(agpt, gpu_ctx):
    """Accumulator::CopyToSurface: /samples, pow(1/2.2), 8-bit pack (myapp.h:34-41)."""
    cfg, level, W, H, spp = 1, 0, 64, 36, 4
    d = agpt.config_defaults(cfg)
    hs = agpt.HostScene(cfg, level)
    hs.upload(gpu_ctx); gpu_ctx.set_film(W, H); gpu_ctx.clear()
    gpu_ctx.render(0, spp, d["max_depth"], d["depth_arg"])
    acc = gpu_ctx.read_accum()
    rgb = gpu_ctx.resolve(spp)
    c = np.power((acc[..., :3] / np.float32(spp)).astype(np.float32), np.float32(1 / 2.2))
    q = (256 * np.clip(c.astype(np.float64), 0.0, 0.999)).astype(np.int64)
    want = (q[..., 0] << 16) + (q[..., 1] << 8) + q[..., 2]
    diff = np.abs(((rgb[..., None] >> np.array([16, 8, 0])) & 255).astype(np.int64) - q)
    assert diff.max() <= 1, "8-bit channels within 1 LSB of the reference formula (powf ulp)"
    assert (rgb == want).mean() > 0.98


def test_error_paths(agpt):
    ctx = agpt.Context(0)
    with pytest.raises(agpt.AgptError):
        ctx.render(0, 1, 5)                      # nothing uploaded
    hs = agpt.HostScene(1, 0); hs.upload(ctx)
    with pytest.raises(agpt.AgptError):
        ctx.render(0, 1, 5)                      # film not set
    ctx.set_film(16, 9)
    with pytest.raises(agpt.AgptError):
        ctx.render(0, 1, -1)                     # bad depth
    ctx.render(0, 0, 5)                          # empty sample range is a no-op
    assert not ctx.read_accum().any()
    ctx.close()


@pytest.mark.parametrize("cfg,level", [(3, 4), (5, 4), (6, 2)])
def test_filtered_slab_test_equals_strict(agpt, gpu_ctx, cfg, level):
    """The exact-filtered slab test (reciprocal multiply + guard band) must take the same
    decisions as the reference's six-division test: identical hits, identical visit / box /
    triangle counts, identical radiance."""
    d = agpt.config_defaults(cfg)
    W, H = 192, 108
    hs = agpt.HostScene(cfg, level)
    hs.upload(gpu_ctx); gpu_ctx.set_film(W, H)
    out = {}
    for name, flag in (("filtered", 0), ("strict", agpt.FLAG_STRICT_BOXES)):
        gpu_ctx.clear(); gpu_ctx.reset_stats()
        hits = gpu_ctx.trace_primary(0, flag | agpt.FLAG_COUNTERS)
        gpu_ctx.render(0, 4, d["max_depth"], d["depth_arg"], flag | agpt.FLAG_COUNTERS)
        st = gpu_ctx.stats()
        out[name] = (hits.copy(), gpu_ctx.read_accum(), (list(st.node_visits), list(st.box_tests), list(st.tri_tests), st.rays))
    assert np.array_equal(out["filtered"][0].view(np.uint32), out["strict"][0].view(np.uint32))
    assert np.array_equal(bits(out["filtered"][1]), bits(out["strict"][1]))
    assert out["filtered"][2] == out["strict"][2]


def test_bucketing_does_not_change_results(agpt):
    """Queue order and batching are free: without the ray-bucket pass, without the side stream,
    with the run-ahead wave loop and with one sample per batch the film is bit-identical.  cfg 3, and
    cfg 14 level 1, whose alpha masks put the masked any-hit kernel on the side stream."""
    import os
    W, H = 160, 90
    for cfg, level in ((3, 3), (14, 1)):
        d = agpt.config_defaults(cfg)
        hs = agpt.HostScene(cfg, level)
        films = []
        for env in ({"AGPT_BUCKET_RAYS": "0"}, {"AGPT_BUCKET_RAYS": "1", "AGPT_OVERLAP_ANY": "0"}, {"AGPT_ASYNC_WAVES": "1"}, {"AGPT_BATCH_LOG2": "14"}):
            old = {k: os.environ.get(k) for k in env}
            os.environ.update(env)
            try:
                ctx = agpt.Context(0)
            finally:
                for k, v in old.items():
                    if v is None:
                        os.environ.pop(k, None)
                    else:
                        os.environ[k] = v
            hs.upload(ctx); ctx.set_film(W, H)
            ctx.render(0, 4, d["max_depth"], d["depth_arg"])
            films.append(ctx.read_accum())
            ctx.close()
        for f in films[1:]:
            assert np.array_equal(bits(films[0]), bits(f)), cfg
