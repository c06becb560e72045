"""GPU: image textures on the base colour of Disney materials (include/agpt.h agpt_upload_textures).

NOT REFERENCE BEHAVIOUR except where a texture reduces to its material's own colour: the reference has one colour per material.
The extension is stated on the CPU in statements/agpt_texture_oracle.cpp; these tests hold the library to it bit for bit on
cfg 12 (every uv rule, every texture shape), and to the reference-pinned untextured films where each material's texture is a
1x1 image of its own colour."""
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
from statements import texture_binding as tb  # noqa: E402

MAT_DTYPE = np.dtype([("type", np.int32), ("lobes", np.uint32), ("roughness", np.float32), ("metallic", np.float32), ("diffuse_r", np.float32, 3),
                      ("eta", np.float32), ("spec_r0", np.float32, 3), ("alpha_x", np.float32), ("mirror_r", np.float32, 3), ("alpha_y", np.float32)])


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def same_floats(a, b):
    """Bit-equal, or NaN on both sides."""
    a = np.ascontiguousarray(a, np.float32); b = np.ascontiguousarray(b, np.float32)
    return bool(np.all((bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))))


@pytest.fixture(scope="module")
def tctx(agpt):
    if agpt.device_count() == 0:
        pytest.fail("no CUDA device visible: -m gpu tests must run on the GPU box")
    ctx = agpt.Context(0)
    yield ctx
    ctx.close()


@pytest.fixture(scope="module")
def cfg12(agpt):
    hs = agpt.HostScene(12, 0)
    return hs, tb.TextureScene(hs), tb.TextureScene(hs, rr_by_bounce=True)


def materials(hs):
    from tests.test_textures_cpu import _Tables
    t = _Tables.from_buffer_copy(hs.tables().raw[:ctypes.sizeof(_Tables)])
    return np.frombuffer(ctypes.string_at(t.materials, 64 * t.n_materials), MAT_DTYPE).copy()


def own_colour(m):
    """A colour c from which DisneyMaterial's arithmetic (agpt.h, textures step 3) gives back the record's diffuse_r and spec_r0
    bit for bit, or None."""
    f = np.float32
    dw = (f(1) - m["metallic"]) * (f(1) - f(0))
    eta = m["eta"]
    r0 = ((eta - f(1)) * (eta - f(1))) / ((eta + f(1)) * (eta + f(1)))
    seeds = [m["spec_r0"]] if not dw > 0 else [m["diffuse_r"] / dw, m["diffuse_r"]]
    c = np.zeros(3, np.float32)
    for k in range(3):
        found = None
        for s in seeds:
            for d in range(-4, 5):
                x = f(s[k])
                for _ in range(abs(d)):
                    x = np.nextafter(x, f(np.inf) if d > 0 else f(-np.inf))
                diff = dw * x if dw > 0 else f(0)
                spec = (f(1) - m["metallic"]) * r0 + m["metallic"] * x
                if bits(diff) == bits(m["diffuse_r"][k]) and bits(spec) == bits(m["spec_r0"][k]):
                    found = x
                    break
            if found is not None:
                break
        if found is None:
            return None
        c[k] = found
    return c


# cfg 3 (reduced level) and cfg 5 run the lean textured instantiation; cfg 10 (rough glass) and cfg 11 (sampled shape lights)
# the one that carries everything.
@pytest.mark.parametrize("cfg,level", [(3, 2), (5, 2), (10, 2), (11, 2)])
def test_own_colour_textures_leave_the_film_unchanged(agpt, tctx, cfg, level):
    d = agpt.config_defaults(cfg)
    hs = agpt.HostScene(cfg, level)
    hs.upload(tctx); tctx.set_film(96, 54); tctx.clear()
    flags = agpt.FLAG_RR_BY_BOUNCE if cfg == 10 else 0
    tctx.render(0, 2, d["max_depth"], d["depth_arg"], flags)
    want = tctx.read_accum().copy()
    mats = materials(hs)
    images, bind = [], []
    for m in mats:
        c = own_colour(m) if m["type"] == 1 else None
        bind.append(-1 if c is None else len(images))
        if c is not None:
            images.append(c.reshape(1, 1, 3))
    assert len(images) >= sum(mats["type"] == 1) - 1 and images
    tctx.upload_textures(images, bind)
    tctx.clear()
    tctx.render(0, 2, d["max_depth"], d["depth_arg"], flags)
    got = tctx.read_accum()
    tctx.upload_textures([], [])
    assert np.array_equal(bits(got), bits(want))


@pytest.mark.parametrize("w,h", [(96, 54), (96, 56)])
@pytest.mark.parametrize("depth,flags", [(1, 0), (8, 0), (8, 16)])
def test_cfg12_film_equals_the_statement(agpt, tctx, cfg12, w, h, depth, flags):
    """96x54: row-major slots, 96x56: tiled.  flags 16: roulette by bounce."""
    hs, ts, ts_rr = cfg12
    hs.upload(tctx); tctx.set_film(w, h); tctx.clear()
    tctx.render(0, 2, depth, 0, flags)
    got = tctx.read_accum()
    want = (ts_rr if flags else ts).render(w, h, 0, 2, depth, 0)
    assert np.array_equal(bits(got[..., :3]), bits(want[..., :3]))


def test_li_pixels_equal_the_statement(agpt, tctx, cfg12):
    hs, ts, _ = cfg12
    hs.upload(tctx); tctx.set_film(96, 54)
    rng = np.random.default_rng(3)
    xs = rng.integers(0, 96, 400); ys = rng.integers(0, 54, 400); ss = rng.integers(0, 50, 400)
    got = tctx.li_pixels(xs, ys, ss, 8)
    want = ts.li_pixels(96, 54, xs, ys, ss, 8, 0)
    assert np.array_equal(bits(got), bits(want))


def test_guides_and_denoise_equal_the_statement(agpt, tctx, cfg12):
    hs, ts, _ = cfg12
    hs.upload(tctx); tctx.set_film(96, 56); tctx.set_moments(True); tctx.clear()
    tctx.render(0, 4, 8)
    tctx.render_guides(3)
    alb, nd = tctx.read_guides()
    walb, wnd = ts.guides(96, 56, 3)
    assert np.array_equal(bits(alb), bits(walb)) and np.array_equal(bits(nd), bits(wnd))
    assert len(np.unique(alb[..., :3].reshape(-1, 3), axis=0)) > 500       # the albedo guide now carries texture detail
    film, mom = tctx.read_accum(), tctx.read_moments()
    for it in (0, 1, 5):
        p = agpt.denoise_params(iterations=it)
        out, _ = tctx.denoise(p)
        want = dn.denoise(film, mom, alb, nd, it, p.sigma_luminance, p.sigma_depth, p.normal_power_log2)
        assert same_floats(out, want), it
    tctx.set_moments(False)


def test_adaptive_pixels_equal_plain_renders(agpt, tctx, cfg12):
    hs, _, _ = cfg12
    hs.upload(tctx); tctx.set_film(48, 27); tctx.set_moments(True)
    tctx.render_adaptive(agpt.adaptive(2, 8, 2, 0.05), 8)
    film, counts = tctx.read_accum().copy(), tctx.read_moments()[..., 3].copy()
    for k in np.unique(counts):
        tctx.clear(); tctx.render(0, int(k), 8)
        plain = tctx.read_accum()
        sel = counts == k
        assert np.array_equal(bits(film[sel]), bits(plain[sel]))
    tctx.set_moments(False)


def test_host_mirror_equals_the_context(agpt, tctx, cfg12):
    hs, _, _ = cfg12
    tr = agpt.HostTracer(8, 0)
    acc = np.zeros((54, 96, 4), np.float32)
    tr.render(hs, 96, 54, acc, 0, 2)
    hs.upload(tctx); tctx.set_film(96, 54); tctx.clear(); tctx.render(0, 2, 8)
    assert np.array_equal(bits(acc), bits(tctx.read_accum()))
    tr.close()


def test_two_gpus_equal_one(agpt, cfg12):
    if agpt.device_count() < 2:
        pytest.skip("one GPU visible")
    hs, _, _ = cfg12
    one, two = agpt.HostTracer(8, 0), agpt.HostTracer(8, devices=[0, 1])
    a = np.zeros((54, 96, 4), np.float32); b = np.zeros((54, 96, 4), np.float32)
    one.render(hs, 96, 54, a, 0, 4); two.render(hs, 96, 54, b, 0, 4)
    assert np.allclose(a, b, rtol=1e-5, atol=1e-6)
    one.close(); two.close()


def test_refusals_and_state_rules(agpt, tctx, cfg12):
    hs, _, _ = cfg12
    hs.upload(tctx); tctx.set_film(32, 18); tctx.clear()
    n = len(materials(hs))
    good = [np.ones((2, 3, 3), np.float32)]
    before = tctx.scene_bytes()
    bad_calls = [
        ([np.ones((0, 3, 3), np.float32)], [0] * n),                       # height 0
        ([np.full((2, 2, 3), np.nan, np.float32)], [0] * n),               # NaN texel
        ([np.full((2, 2, 3), np.inf, np.float32)], [0] * n),               # inf texel
        (good, [1] * n),                                                   # index past the table
        (good, [-2] * n),                                                  # below -1
    ]
    for imgs, bind in bad_calls:
        with pytest.raises(agpt.AgptError):
            tctx.upload_textures(imgs, bind)
        assert tctx.scene_bytes() == before                                # refused: resident textures as they were
    with pytest.raises(agpt.AgptError):                                    # 2^28 + 1 texels (refused before any texel is read)
        T = agpt.binding.Texture
        rows = (T * 1)(T(16385, 16384, ctypes.cast(ctypes.c_void_p(8), ctypes.POINTER(ctypes.c_float))))
        agpt.binding._check(agpt.binding.core().agpt_upload_textures(tctx.handle, rows, 1, (ctypes.c_int * n)(*([0] * n)), n))
    with pytest.raises(agpt.AgptError):                                    # NULL texels
        T = agpt.binding.Texture
        rows = (T * 1)(T(2, 2, None))
        agpt.binding._check(agpt.binding.core().agpt_upload_textures(tctx.handle, rows, 1, (ctypes.c_int * n)(*([0] * n)), n))
    # wrong binding count, and a binding on a mirror material: refused at render time
    tctx.upload_textures(good, [0] * (n + 1))
    with pytest.raises(agpt.AgptError):
        tctx.render(0, 1, 2)
    hs1 = agpt.HostScene(1, 0)                                             # cfg 1: material 1 is a mirror
    hs1.upload(tctx)
    m1 = materials(hs1)
    bind = [-1] * len(m1); bind[int(np.nonzero(m1["type"] == 2)[0][0])] = 0
    tctx.upload_textures(good, bind)
    with pytest.raises(agpt.AgptError):
        tctx.render(0, 1, 2)
    # an upload makes the guides stale and drops the saved view
    hs.upload(tctx); tctx.set_moments(True); tctx.clear()
    tctx.render_guides(1)
    tctx.reproject_film(agpt.reproject_params())                           # saves the view
    tctx.upload_textures([], [])
    with pytest.raises(agpt.AgptError):
        tctx.denoise(agpt.denoise_params())
    tctx.render_guides(1)
    film = tctx.read_accum().copy()
    cam = hs.camera().copy(); cam[0] += 0.1
    tctx.set_camera(cam)
    tctx.render_guides(1)
    tctx.reproject_film(agpt.reproject_params())                           # no saved view after the upload: film left as it is
    assert np.array_equal(bits(tctx.read_accum()), bits(film))
    tctx.set_moments(False)


def test_scene_bytes_count_the_textures(agpt, tctx, cfg12):
    hs, _, _ = cfg12
    hs.upload(tctx)
    with_tex = tctx.scene_bytes()
    n = len(materials(hs))
    tctx.upload_textures([], [])
    texels = 2048 * 2048 + 37 * 23 + 64
    assert with_tex - tctx.scene_bytes() == 16 * texels + 16 * 3 + 4 * n


def test_no_failed_device_checks(tctx):
    """Meaningful under AGPT_LIB=libagpt_debug.so (test_debug_build_runs_this_file); a release build runs no checks."""
    s = tctx.debug_status()
    print("TEXTURE_DEBUG_STATUS", s["failed"], s["first_code"], s["first_value"], s["checks"])
    assert s["failed"] == 0


def test_debug_build_runs_this_file():
    """The tests above under libagpt_debug.so (texture and texel indices checked inside the kernels): none may fail."""
    lib = os.path.join(ROOT, "ag-pathtracer_b200", "libagpt_debug.so")
    assert os.path.exists(lib)
    env = dict(os.environ, AGPT_LIB=lib)
    out = subprocess.run([sys.executable, "-m", "pytest", "-q", "-s", "-p", "no:cacheprovider", os.path.abspath(__file__), "-k",
                          "not debug_build and not two_gpus and not host_mirror"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if "TEXTURE_DEBUG_STATUS" in l][0]
    failed, checks = [int(v) for v in line.split("TEXTURE_DEBUG_STATUS")[1].split()[0:4:3]]
    assert checks > 100_000 and failed == 0
