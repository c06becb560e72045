"""CPU: the plain-C++ restatement (oracle/agpt_oracle.cpp) against the golden fixtures that
the reference itself produced, and against oracle/_ref directly where it is built.
Bit-exact: same compiler, flags and libm => no tolerance."""
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = [1, 2, 3, 4, 5, 6, 7, 8]


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


@pytest.fixture(scope="module")
def port():
    from oracle import port_binding
    if not port_binding.available():
        pytest.fail("oracle/libagpt_oracle.so not built: run build() / make -C oracle port")
    return port_binding


def load(cfg):
    return np.load(os.path.join(GOLDEN, f"scene_cfg{cfg}.npz"))


@pytest.mark.parametrize("cfg", CASES)
def test_port_matches_golden(agpt, port, cfg):
    g = load(cfg)
    _, level, W, H, spp, md, da = [int(v) for v in g["case"]]
    hs = agpt.HostScene(cfg, level)
    ps = port.PortScene(hs)
    hits, walk = ps.primary_hits(W, H, 0, want_counts=True)
    for f in ("found", "prim", "tri"):
        assert np.array_equal(hits[f], g["hits"][f]), f
    assert np.array_equal(bits(hits["t"]), bits(g["hits"]["t"]))
    assert (walk["interior"], walk["boxes"], walk["tris"]) == tuple(int(v) for v in g["walk_stats"]), "walk counts differ from the reference's"
    acc, cnt = ps.render(W, H, 0, spp, md, da)
    assert np.array_equal(bits(acc), bits(g["accum"])), "accumulator differs from the reference's"
    li, draws = ps.li_pixels(W, H, g["li_xs"], g["li_ys"], g["li_ss"], md, da)
    assert np.array_equal(bits(li), bits(g["li"]))
    assert np.array_equal(draws, g["li_draws"]), "RNG draw count per path (draw-order contract)"
    assert cnt["paths"] == W * H * spp


@pytest.mark.parametrize("cfg", CASES)
def test_port_matches_reference_live(agpt, port, ref, cfg):
    """Fresh seeds / sizes against the compiled reference (skipped where oracle/_ref is absent)."""
    d = agpt.config_defaults(cfg)
    level = {1: 0, 2: 4, 3: 3, 4: 2, 5: 3, 6: 2, 7: 0, 8: 2}[cfg]
    W, H, spp = 96, 54, 3
    hs = agpt.HostScene(cfg, level); rs = ref.RefScene(cfg, level); ps = port.PortScene(hs)
    a, _ = rs.render(W, H, 5, spp, d["max_depth"], d["depth_arg"])
    b, cnt = ps.render(W, H, 5, spp, d["max_depth"], d["depth_arg"])
    assert np.array_equal(bits(a), bits(b))
    # ray counts: the reference counted through a do-nothing front primitive
    rc = ref.RefScene(cfg, level); rc.count_rays(); ref.ray_counts(reset=True)
    rc.render(W, H, 5, spp, d["max_depth"], d["depth_arg"])
    n = ref.ray_counts(reset=True)
    assert (n["closest"], n["any"]) == (cnt["rays_closest"], cnt["rays_any"])


def test_stream_definition(port):
    g = np.load(os.path.join(GOLDEN, "functions.npz"))
    for p, s, want in zip(g["stream_pixels"], g["stream_samples"], g["stream_floats"]):
        got = port.probe_stream(int(p), int(s), 16)
        assert np.array_equal(bits(got), bits(want))
    # float2 u(RandomFloat(), RandomFloat()): second argument is drawn first under g++
    ux, uy, first, second = g["draw_order"]
    assert (ux, uy) == (second, first)


def test_crop_and_stride_are_consistent(agpt, port):
    """Rendering a crop or a strided sample subset touches exactly those pixels / samples."""
    hs = agpt.HostScene(6, 2); ps = port.PortScene(hs)
    W, H = 48, 27
    full, _ = ps.render(W, H, 0, 4, 5, 0)
    crop, _ = ps.render(W, H, 0, 4, 5, 0, crop=(8, 4, 40, 20))
    view = crop[::-1]          # accumulator rows are stored flipped (myapp.h:17-19)
    fullv = full[::-1]
    assert np.array_equal(bits(view[4:20, 8:40]), bits(fullv[4:20, 8:40]))
    assert not view[:4].any() and not view[20:].any()
    even, _ = ps.render(W, H, 0, 2, 5, 0, sample_stride=2)
    odd, _ = ps.render(W, H, 1, 2, 5, 0, sample_stride=2)
    assert np.allclose(even + odd, full, rtol=1e-5, atol=1e-6)
