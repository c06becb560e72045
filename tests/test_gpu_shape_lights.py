"""GPU: sampled plane and mesh area lights (AGPT_LIGHT_SAMPLE_SHAPE).

PARITY UNPINNED BY THE REFERENCE: upstream cannot sample a Plane or a TriangleMesh (pdf-0 stubs).  What sampling them means
is stated on the CPU in oracle/agpt_shape_oracle.cpp (ShapeSample / ShapePdf); these tests hold the CUDA path to that statement
bit for bit, check that scenes without the flag render exactly as before, and that two samplers of one rectangle agree."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


@pytest.fixture(scope="module")
def port():
    from oracle import shape_binding
    return shape_binding


def live_tables(agpt, port, hs):
    """Views into the host scene's flattened light and primitive rows (what hs.upload and PortScene(hs) read)."""
    t = port._Tables.from_buffer(hs.tables())
    lights = np.frombuffer((ctypes.c_char * (agpt.LIGHT_DTYPE.itemsize * t.n_lights)).from_address(t.lights), agpt.LIGHT_DTYPE)
    prims = np.frombuffer((ctypes.c_char * (agpt.PRIM_DTYPE.itemsize * t.n_prims)).from_address(t.prims), agpt.PRIM_DTYPE)
    return lights, prims


def render(ctx, d, spp, flags=0, first=0):
    ctx.clear()
    ctx.render(first, spp, d["max_depth"], d["depth_arg"], flags)
    return ctx.read_accum().copy()


def test_probe_matches_cpu_statement(agpt, port, gpu_ctx):
    """Sample_Li / Pdf_Li of cfg 11's 2-triangle panel, plane panel and level-2 BVH icosphere: rows bit-identical to the CPU
    statement (>= 99.9 %, the rest within rtol 2e-6, the glass probe's bar)."""
    hs = agpt.HostScene(11, 2); ps = port.ShapeScene(hs)
    hs.upload(gpu_ctx)
    rng = np.random.default_rng(7)
    n = 20000
    exact = total = 0
    for light in (0, 1, 2):
        ref = rng.uniform([-3.8, -.8, -8.8], [3.8, 4.8, 3.8], (n, 3)).astype(np.float32)
        u = rng.random((n, 2), np.float32)
        a = np.concatenate([ref, u, np.zeros((n, 3), np.float32)], 1)
        s = ps.probe_light_sample(light, a)
        # query directions: half towards the light's own samples (hits), half at random
        w = (s[:, :3] - ref).astype(np.float64)
        w /= np.linalg.norm(w, axis=1, keepdims=True)
        rnd = rng.normal(size=(n, 3)); rnd /= np.linalg.norm(rnd, axis=1, keepdims=True)
        a[:, 5:8] = np.where(np.arange(n)[:, None] % 2 == 0, w, rnd).astype(np.float32)
        want = ps.probe_light_sample(light, a)
        got = gpu_ctx.probe_light_sample(light, a)
        assert (want[:, 4] > 0).mean() > 0.4
        same = np.all(bits(got) == bits(want), axis=1)
        assert np.allclose(got, want, rtol=2e-6, atol=0), light
        exact += int(same.sum()); total += n
    print(f"shape-light probe rows bit-identical: {exact}/{total}")
    assert exact / total >= 0.999
    with pytest.raises(agpt.AgptError):
        gpu_ctx.probe_light_sample(3, a[:4])               # not a light of cfg 11


@pytest.mark.parametrize("level,W,H,spp", [(3, 160, 90, 4)])
def test_cfg11_matches_cpu_statement(agpt, port, gpu_ctx, level, W, H, spp):
    """cfg 11: film, ray accounting (the identity test_gpu_extensions.py uses) and single paths against the CPU statement."""
    d = agpt.config_defaults(11)
    hs = agpt.HostScene(11, level); ps = port.ShapeScene(hs)
    hs.upload(gpu_ctx); gpu_ctx.set_film(W, H); gpu_ctx.reset_stats()
    got = render(gpu_ctx, d, spp, agpt.FLAG_COUNTERS)
    st = gpu_ctx.stats()
    want, cnt = ps.render(W, H, 0, spp, d["max_depth"], d["depth_arg"])
    exact = np.all(bits(got[..., :3]) == bits(want[..., :3]), axis=-1).mean()
    print(f"cfg11: bit-identical pixels {exact:.5f}")
    assert exact >= 0.999
    assert st.rays_shadow == cnt["rays_any"]
    assert st.rays_closest + st.rays_mis + st.rays_mis_culled + st.rays_tail_culled == cnt["rays_closest"]
    # the MIS samples that cannot reach their light are dropped before their BSDF value is known: same film
    assert np.array_equal(bits(render(gpu_ctx, d, spp)), bits(got))
    xs = np.arange(0, W, 3, dtype=np.int32); ys = (xs * 7 % H).astype(np.int32); ss = (xs % 4).astype(np.int32)
    li = gpu_ctx.li_pixels(xs, ys, ss, d["max_depth"], d["depth_arg"])
    want_li, _ = ps.li_pixels(W, H, xs, ys, ss, d["max_depth"], d["depth_arg"])
    assert np.all(bits(li) == bits(want_li), axis=1).mean() >= 0.97
    # the walls are lit: far more light reaches the film than the panels seen directly carry
    assert got[..., :3].mean() > 0 and np.isfinite(got).all()


def test_without_the_flag_and_on_spheres_nothing_changes(agpt, port, gpu_ctx):
    """cfg 11 without the flag == the CPU statement with the flag off (walls lit only through specular chains, as upstream)
    and far darker; the flag on cfg 5's sphere light leaves its film bit-identical."""
    W, H, spp = 160, 90, 4
    d = agpt.config_defaults(11)
    hs = agpt.HostScene(11, 2)
    lights, _ = live_tables(agpt, port, hs)
    hs.upload(gpu_ctx); gpu_ctx.set_film(W, H)
    lit = render(gpu_ctx, d, spp)
    lights["ext"]["flags"] = 0
    ps = port.ShapeScene(hs)
    hs.upload(gpu_ctx)
    dark = render(gpu_ctx, d, spp)
    want, _ = ps.render(W, H, 0, spp, d["max_depth"], d["depth_arg"])
    assert np.all(bits(dark[..., :3]) == bits(want[..., :3]), axis=-1).mean() >= 0.999
    print(f"cfg11 mean radiance: sampled {lit[..., :3].mean():.4f}, unsampled {dark[..., :3].mean():.4f}")
    assert dark[..., :3].mean() < 0.5 * lit[..., :3].mean()

    d5 = agpt.config_defaults(5)
    hs5 = agpt.HostScene(5, 3)
    lights5, _ = live_tables(agpt, port, hs5)
    hs5.upload(gpu_ctx)
    before = render(gpu_ctx, d5, spp)
    lights5["ext"]["flags"] = agpt.LIGHT_SAMPLE_SHAPE
    hs5.upload(gpu_ctx)
    assert np.array_equal(bits(render(gpu_ctx, d5, spp)), bits(before))


def block_means(img, k=8):
    lum = img[..., :3].astype(np.float64) @ np.array([0.212671, 0.715160, 0.072169])
    H, W = lum.shape
    return lum.reshape(H // k, k, W // k, k).mean(axis=(1, 3))


def test_plane_and_two_triangles_sample_the_same_integral(agpt, port, gpu_ctx):
    """cfg 11's 2-triangle panel, replaced by a sampled Plane of the same rectangle: 8x8-block means of the two films agree
    within 5 sigma, sigma estimated from four independent sample ranges of each.  (Both films draw the same random numbers,
    which makes the difference far less noisy than sigma: a conservative test, still a few-percent bias fails the last line.)"""
    W, H, spp = 160, 96, 8
    d = agpt.config_defaults(11)
    hs = agpt.HostScene(11, 2)
    lights, prims = live_tables(agpt, port, hs)
    assert prims[3]["type"] == agpt.PRIM_MESH and lights[0]["prim"] == 3
    hs.upload(gpu_ctx); gpu_ctx.set_film(W, H)
    films = {}
    films["mesh"] = [render(gpu_ctx, d, spp, first=1000 * r) for r in range(4)]
    t = port._Tables.from_buffer(hs.tables())
    planes = np.zeros(2, agpt.PLANE_DTYPE)
    planes[0] = np.frombuffer((ctypes.c_char * 32).from_address(t.planes), agpt.PLANE_DTYPE)[0]
    planes[1] = ((0, 4.97, -1.6), .8, .6, (0, 0, 0))                   # the panel: x in [-.8, .8], z in [-2.2, -1], y = 4.97
    p2 = prims.copy()
    p2[3] = (agpt.PRIM_PLANE, 1, -1, 0)
    gpu_ctx.upload_table("planes", planes); gpu_ctx.upload_table("primitives", p2)
    films["plane"] = [render(gpu_ctx, d, spp, first=1000 * r) for r in range(4)]
    m = {k: np.stack([block_means(f) for f in v]) for k, v in films.items()}       # [range, by, bx]
    diff = m["mesh"].mean(0) - m["plane"].mean(0)
    sigma = np.sqrt(m["mesh"].var(0, ddof=1) / 4 + m["plane"].var(0, ddof=1) / 4)
    z = np.abs(diff) / np.maximum(sigma, 1e-30)
    print(f"block z: max {z.max():.2f}, mean z^2 {np.mean(z ** 2):.2f}, share > 5: {(z > 5).mean():.4f}")
    # (sigma comes from 3 + 3 degrees of freedom: its tails are Student's, so a few of 240 blocks may pass 5 by chance)
    assert (z > 5).mean() <= 0.02 and np.mean(z ** 2) < 4
    assert abs(m["mesh"].mean() / m["plane"].mean() - 1) < 0.02


def test_refused_flags_leave_the_scene_rendering(agpt, port, gpu_ctx):
    """Unknown flag bits and the flag on a sky light are refused at upload, the flag on an instanced shape when rendering;
    each is AGPT_ERR_INVALID and the scene renders the same film as before."""
    W, H, spp = 64, 36, 2
    d = agpt.config_defaults(11)
    hs = agpt.HostScene(11, 2)
    lights, _ = live_tables(agpt, port, hs)
    hs.upload(gpu_ctx); gpu_ctx.set_film(W, H)
    film = render(gpu_ctx, d, spp)
    bad = lights.copy(); bad[0]["ext"]["flags"] = 2
    with pytest.raises(agpt.AgptError, match="error -1"):
        gpu_ctx.upload_table("lights", bad)
    assert np.array_equal(bits(render(gpu_ctx, d, spp)), bits(film))
    sky = np.zeros(len(lights) + 1, agpt.LIGHT_DTYPE); sky[:-1] = lights
    sky[-1] = (agpt.LIGHT_UNIFORM_INFINITE, -1, (agpt.LIGHT_SAMPLE_SHAPE, 0), (1, 1, 1), 0)
    with pytest.raises(agpt.AgptError, match="error -1"):
        gpu_ctx.upload_table("lights", sky)
    assert np.array_equal(bits(render(gpu_ctx, d, spp)), bits(film))

    d9 = agpt.config_defaults(9)
    hs9 = agpt.HostScene(9, 1)
    lights9, prims9 = live_tables(agpt, port, hs9)
    hs9.upload(gpu_ctx)
    film9 = render(gpu_ctx, d9, spp)
    assert prims9[1]["type"] == agpt.PRIM_INSTANCE
    l2, p2 = lights9.copy(), prims9.copy()
    p2[l2[0]["prim"]]["area_light"] = -1; p2[1]["area_light"] = 0
    l2[0]["prim"] = 1; l2[0]["ext"]["flags"] = agpt.LIGHT_SAMPLE_SHAPE
    gpu_ctx.upload_table("lights", l2); gpu_ctx.upload_table("primitives", p2)
    with pytest.raises(agpt.AgptError, match="instanced"):
        render(gpu_ctx, d9, spp)
    gpu_ctx.upload_table("lights", lights9); gpu_ctx.upload_table("primitives", prims9)
    assert np.array_equal(bits(render(gpu_ctx, d9, spp)), bits(film9))


def test_scene_bytes_count_the_tables(agpt):
    ctx = agpt.Context(0)
    hs = agpt.HostScene(11, 2)
    hs.upload(ctx)
    before = ctx.scene_bytes()
    ctx.set_film(16, 16); ctx.render(0, 1, 2)                         # the tables are built on first use
    # 3 lights x 16 B + the cdfs of the panel (2 + 1 floats) and of the icosphere (320 + 1 floats)
    assert ctx.scene_bytes() - before == 3 * 16 + 4 * (3 + 321)
    ctx.close()


def test_no_failed_device_checks(gpu_ctx):
    """Meaningful under AGPT_LIB=libagpt_debug.so (test_debug_build_runs_this_file); a release build runs no checks."""
    s = gpu_ctx.debug_status()
    print("SHAPE_DEBUG_STATUS", s["failed"], s["first_code"], s["first_value"], s["checks"])
    assert s["failed"] == 0


def test_debug_build_runs_this_file():
    """The tests above under libagpt_debug.so (in-kernel stack / index / queue checks): none may fail.  Own process: the
    library is chosen at load time."""
    lib = os.path.join(ROOT, "ag-pathtracer_b200", "libagpt_debug.so")
    assert os.path.exists(lib)
    env = dict(os.environ, AGPT_LIB=lib)
    out = subprocess.run([sys.executable, "-m", "pytest", "-q", "-s", "-p", "no:cacheprovider", os.path.abspath(__file__), "-k", "not debug_build"],
                         cwd=ROOT, env=env, capture_output=True, text=True, timeout=1200)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if "SHAPE_DEBUG_STATUS" in l][0]      # (after pytest's progress dots)
    failed, checks = [int(v) for v in line.split("SHAPE_DEBUG_STATUS")[1].split()[0:4:3]]
    assert checks > 100_000 and failed == 0
