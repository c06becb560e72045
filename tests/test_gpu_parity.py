"""GPU parity tests proper: CUDA path (through the C ABI) vs the reference oracle.

Gates (BASELINE.json north_star): primary-ray hit flags / primitive ids / triangle ids / t
bit-exact; radiance within a per-pixel relative RMSE of 1e-3 at matched spp and streams.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# (config, icosphere level, W, H) sized so the CPU oracle finishes in seconds
SMALL = [(1, 0, 160, 90), (2, 5, 160, 90), (3, 3, 160, 90), (4, 3, 160, 90), (5, 3, 160, 90), (6, 2, 160, 90), (7, 0, 120, 120)]


def rel_rmse(gpu, cpu):
    """sqrt(mean |gpu-cpu|^2) / mean |cpu| over rgb of all pixels (stated tolerance: 1e-3)."""
    g = gpu[..., :3].astype(np.float64); c = cpu[..., :3].astype(np.float64)
    return float(np.sqrt(np.mean((g - c) ** 2)) / max(np.mean(np.abs(c)), 1e-30))


@pytest.mark.parametrize("config,level,W,H", SMALL)
def test_primary_hits_bit_exact(agpt, ref_live, ref_golden, gpu_ctx, config, level, W, H):
    hs = agpt.HostScene(config, level)
    rs = ref_live.RefScene(config, level) if ref_live else None
    g = None if ref_live else ref_golden(f"ref_parity_cfg{config}.npz")
    hs.upload(gpu_ctx); gpu_ctx.set_film(W, H)
    for sample in (0, 3):
        if rs:
            want, st = rs.primary_hits(W, H, sample)
            assert st["walk_mismatches"] == 0
        else:
            want = g[f"hits{sample}"]
        got = gpu_ctx.trace_primary(sample)
        assert np.array_equal(got["found"], want["found"])
        assert np.array_equal(got["prim"], want["prim"])
        assert np.array_equal(got["tri"], want["tri"])
        assert np.array_equal(got["t"].view(np.uint32), want["t"].view(np.uint32))


@pytest.mark.parametrize("config,level,W,H", SMALL)
def test_radiance_rmse(agpt, ref_live, ref_golden, gpu_ctx, config, level, W, H):
    d = agpt.config_defaults(config)
    spp = 8
    hs = agpt.HostScene(config, level)
    hs.upload(gpu_ctx); gpu_ctx.set_film(W, H); gpu_ctx.clear()
    gpu_ctx.render(0, spp, d["max_depth"], d["depth_arg"])
    got = gpu_ctx.read_accum()
    if ref_live:
        want, _ = ref_live.RefScene(config, level).render(W, H, 0, spp, d["max_depth"], d["depth_arg"])
    else:
        want = ref_golden(f"ref_parity_cfg{config}.npz")["accum"]
    err = rel_rmse(got, want)
    exact = np.mean(np.all(got[..., :3].view(np.uint32) == want[..., :3].view(np.uint32), axis=-1))
    print(f"cfg{config}: rel-RMSE {err:.3e}, bit-identical pixels {exact:.4f}")
    assert err <= 1e-3                      # the north-star gate
    # stronger than the gate: sin/cos/acos follow glibc's algorithms on the device, so whole
    # paths -- and with the same summation order the accumulators -- come out bit-identical
    assert exact >= 0.999


@pytest.mark.parametrize("config,level,W,H", SMALL)
def test_ray_accounting_matches_reference(agpt, gpu_ctx, config, level, W, H):
    """Rays traced + rays proven useless and skipped == the rays the reference algorithm issues
    (counted by the restatement, which is itself checked against the reference's own counts)."""
    from oracle import port_binding as port
    d = agpt.config_defaults(config)
    hs = agpt.HostScene(config, level); ps = port.PortScene(hs)
    hs.upload(gpu_ctx); gpu_ctx.set_film(W, H); gpu_ctx.clear(); gpu_ctx.reset_stats()
    gpu_ctx.render(0, 2, d["max_depth"], d["depth_arg"], agpt.FLAG_COUNTERS)      # exact ray accounting needs the counting mode (agpt.h: rays_mis_culled)
    st = gpu_ctx.stats()
    _, cnt = ps.render(W, H, 0, 2, d["max_depth"], d["depth_arg"])
    assert st.rays_shadow == cnt["rays_any"]
    assert st.rays_closest + st.rays_mis + st.rays_mis_culled + st.rays_tail_culled == cnt["rays_closest"]
    assert st.rays_reference_equivalent == cnt["rays_closest"] + cnt["rays_any"]


def test_sphere_run_cull_is_exact(agpt, ref_live, ref_golden, gpu_ctx):
    """The trace kernels skip a whole run of sphere primitives when no ray of a warp can reach the
    run's (grown) bounding box.  Rays aimed at and around cfg 3's 5x5 sphere grid, from origins a
    few units to several hundred units away (beyond the distance the cull trusts itself), must
    give the reference's hits bit for bit, closest-hit and any-hit."""
    hs = agpt.HostScene(3, 2)
    hs.upload(gpu_ctx)
    rng = np.random.default_rng(20261018)          # tests/golden/make_golden_fullsize.py draws the same rays
    n = 120_000
    # targets: inside and just outside the slab the sphere grid occupies (centres -3..3 x -0.5 x -4..2, r = 0.5)
    tgt = np.stack([rng.uniform(-3.7, 3.7, n), rng.uniform(-1.15, 0.15, n), rng.uniform(-4.7, 2.7, n)], 1)
    dist = rng.choice([2.0, 8.0, 40.0, 150.0, 400.0], n)
    dirs = rng.normal(size=(n, 3)); dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    dirs[:, 1] = np.abs(dirs[:, 1]) * rng.choice([1.0, 0.02], n)          # from above, many at grazing angles
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    org = tgt + dirs * dist[:, None]
    rays = np.concatenate([org, -dirs, np.full((n, 1), 3.0e38)], 1).astype(np.float32)
    if ref_live:
        rs = ref_live.RefScene(3, 2)
        wants = [rs.trace_rays(rays, any_hit=a)[0] for a in (False, True)]
    else:
        g = ref_golden("ref_sphere_cull.npz")
        wants = [{"found": g["found"], "prim": g["prim"], "t": g["t"]}, {"found": g["found_any"]}]
    for any_hit, want in zip((False, True), wants):
        got = gpu_ctx.trace_rays(rays, any_hit=any_hit)
        assert np.array_equal(got["found"], want["found"])
        if not any_hit:
            assert np.array_equal(got["prim"], want["prim"])
            assert np.array_equal(got["t"].view(np.uint32), want["t"].view(np.uint32))
    assert 0.2 < want["found"].mean() < 1.0


def test_write_accum_begin_equals_write_accum(agpt, gpu_ctx):
    """agpt_write_accum_begin (the film upload that runs beside the render that follows) gives the frame agpt_write_accum
    gives, bit for bit; a film access without a render in between waits for the upload too."""
    d = agpt.config_defaults(1)
    W, H = 320, 180
    hs = agpt.HostScene(1, 0); hs.upload(gpu_ctx); gpu_ctx.set_film(W, H)
    film, owner = agpt.pinned_film(W, H)
    film[:] = np.random.default_rng(5).random((H, W, 4), dtype=np.float32)
    gpu_ctx.write_accum(film.copy()); gpu_ctx.render(0, 3, d["max_depth"], d["depth_arg"]); want = gpu_ctx.read_accum()
    gpu_ctx.clear()
    gpu_ctx.write_accum_begin(film); gpu_ctx.render(0, 3, d["max_depth"], d["depth_arg"]); got = gpu_ctx.read_accum()
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    gpu_ctx.clear()
    gpu_ctx.write_accum_begin(film)
    assert np.array_equal(gpu_ctx.read_accum().view(np.uint32), film.view(np.uint32))
    gpu_ctx.write_accum_begin(film); gpu_ctx.clear()
    assert not gpu_ctx.read_accum().any()
    del owner


@pytest.mark.parametrize("config,level,W,H,depth", [(1, 0, 157, 83, None), (6, 2, 157, 83, None), (1, 0, 1, 1, None), (6, 2, 9, 5, None),
                                                      (3, 2, 24, 11, 0), (3, 2, 40, 12, 1), (7, 0, 33, 17, None)])
def test_ragged_and_tiny_films(agpt, gpu_ctx, config, level, W, H, depth):
    """Films that are not a multiple of the 8x4 path-slot tile (row-major slot order), a 1x1 film, depth 0 (emission only)
    and depth 1: bit-identical to the restatement (itself pinned bit for bit to the reference), sample ranges that do not
    start at 0 included."""
    from oracle import port_binding as port
    d = agpt.config_defaults(config)
    depth = d["max_depth"] if depth is None else depth
    hs = agpt.HostScene(config, level); ps = port.PortScene(hs)
    hs.upload(gpu_ctx); gpu_ctx.set_film(W, H); gpu_ctx.clear()
    gpu_ctx.render(3, 5, depth, d["depth_arg"])
    got = gpu_ctx.read_accum()
    want, _ = ps.render(W, H, 3, 5, depth, d["depth_arg"])
    assert np.array_equal(got[..., :3].view(np.uint32), want[..., :3].view(np.uint32))


def test_batches_do_not_change_the_film(agpt):
    """A render split into many wavefront batches (the batch cap far below samples x pixels) and the same render in one
    batch give the same film: every path's arithmetic depends on its pixel and sample only."""
    import os
    d = agpt.config_defaults(3)
    hs = agpt.HostScene(3, 3)
    films = []
    for log2 in ("27", "16", "12"):           # 6, 3 and 1 samples per batch (the cap never cuts below one sample of the film)
        old = os.environ.get("AGPT_BATCH_LOG2")
        os.environ["AGPT_BATCH_LOG2"] = log2
        try:
            ctx = agpt.Context(0)
        finally:
            if old is None:
                os.environ.pop("AGPT_BATCH_LOG2", None)
            else:
                os.environ["AGPT_BATCH_LOG2"] = old
        hs.upload(ctx); ctx.set_film(200, 100)
        ctx.render(0, 6, d["max_depth"], d["depth_arg"])
        films.append(ctx.read_accum())
        ctx.close()
    assert np.array_equal(films[0].view(np.uint32), films[1].view(np.uint32))
    assert np.array_equal(films[0].view(np.uint32), films[2].view(np.uint32))
