"""CPU: the statement of alpha-masked cutout geometry (include/agpt.h agpt_upload_alpha_masks, statements/agpt_alpha_oracle.cpp)
against the oracle and the texture statement, the host mirror's flattening of masks, and the binding's argument checks.

NOT REFERENCE BEHAVIOUR: the reference has no masks.  With no mask bound the statement must be the oracle."""
import ctypes
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from statements import alpha_binding as ab  # noqa: E402
from statements import maps_binding as mb  # noqa: E402
from statements import texture_binding as tb  # noqa: E402
from tests.test_gpu_textures import bits  # noqa: E402

pytestmark = pytest.mark.skipif(not ab.available(), reason="statements/libagpt_alpha_oracle.so not built (__graft_entry__.build())")
RNG = np.random.default_rng(14)


def _host(agpt):
    if not os.path.exists(agpt.lib_paths()[1]):
        pytest.skip("libagpt_host.so not built")


@pytest.mark.parametrize("cfg,level", [(1, 0), (5, 2), (7, 0), (9, 2), (10, 2), (12, 0), (13, 1)])
def test_without_masks_the_statement_is_the_oracle(agpt, cfg, level):
    """Film, counters, guides and hit tables.  cfg 7: environment map, 9: instances, 10: glass, 12 and 13: textures and maps (whose
    oracle is the maps statement)."""
    _host(agpt)
    from oracle import port_binding as port
    hs = agpt.HostScene(cfg, level)
    d = agpt.config_defaults(cfg)
    got, cnt = ab.AlphaScene(hs).render(32, 18, 0, 2, d["max_depth"], d["depth_arg"], counters=True)
    if cfg in (12, 13):       # bound images: the oracle with textures and maps is the maps statement
        want, wcnt = mb.MapsScene(hs).render(32, 18, 0, 2, d["max_depth"], d["depth_arg"], counters=True)
    else:
        want, wcnt = port.PortScene(hs).render(32, 18, 0, 2, d["max_depth"], d["depth_arg"])
    assert np.array_equal(bits(got), bits(want))
    for k in ("rays_closest", "rays_any", "interior", "boxes", "tris", "analytic"):
        assert cnt[k] == wcnt[k], k
    # the restated guide record and the any-hit and closest-hit tables, with the closest-hit walk's counters
    for g, w in zip(ab.AlphaScene(hs).guides(32, 18, 2), mb.MapsScene(hs).guides(32, 18, 2)):
        assert np.array_equal(bits(g), bits(w))
    ps = port.PortScene(hs)
    cam = hs.camera()
    rng = np.random.default_rng(cfg)
    D = rng.normal(size=(2000, 3)).astype(np.float32)
    O = np.broadcast_to(np.float32(cam[0:3]), D.shape)
    rays7 = np.concatenate([O, D, np.full((len(D), 1), 1e30, np.float32)], 1).astype(np.float32)
    for any_hit in (False, True):
        got_t, tcnt = ab.AlphaScene(hs).trace_rays(rays7, any_hit, counters=True)
        want_t, wtcnt = ps.trace_rays(rays7, any_hit)
        for f in ("found", "prim", "tri"):
            assert np.array_equal(got_t[f], want_t[f]), (any_hit, f)
        assert np.array_equal(bits(got_t["t"]), bits(want_t["t"]))
        assert tcnt["rays_any" if any_hit else "rays_closest"] == len(rays7)
        if not any_hit:
            assert (tcnt["interior"], tcnt["boxes"], tcnt["tris"]) == (wtcnt["interior"], wtcnt["boxes"], wtcnt["tris"])
            assert tcnt["tris"] + tcnt["analytic"] > 0
    hits, hcnt = ab.AlphaScene(hs).primary_hits(32, 18, 1, counters=True)
    want_hits, whcnt = ps.primary_hits(32, 18, 1, want_counts=True)
    for f in ("found", "prim", "tri"):
        assert np.array_equal(hits.reshape(-1)[f], want_hits[f])
    assert np.array_equal(bits(hits.reshape(-1)["t"]), bits(want_hits["t"]))
    assert hcnt["rays_closest"] == 32 * 18
    assert (hcnt["interior"], hcnt["boxes"], hcnt["tris"]) == (whcnt["interior"], whcnt["boxes"], whcnt["tris"])


def test_a_rejected_tie_goes_to_the_next_triangle(agpt):
    """Two coincident triangles of one plain TriangleMesh at the same t, in tables built by hand: the walk keeps the first it tests,
    so masking the first leaves the second's hit, masking the second changes nothing and masking both leaves a miss.  The first
    triangle's uvs sit on texel 0 of a 2 x 1 mask, the second's on texel 1."""
    verts = np.zeros((2, 3, 4), np.float32)
    verts[:, 0, :3] = (-1, 0, -1); verts[:, 1, :3] = (1, 0, -1); verts[:, 2, :3] = (0, 0, 1)
    uvs = np.zeros((2, 3, 2), np.float32)
    uvs[0] = (.25, .5); uvs[1] = (.75, .5)
    mesh = agpt.RawMesh(verts, tri_ids=[7, 9], uvs=uvs)
    prims = np.zeros(1, agpt.PRIM_DTYPE)
    prims[0] = (agpt.PRIM_MESH, 0, 0, -1)
    mat = agpt.make_material(agpt.MAT_DISNEY, (.7, .7, .7), .5, 0.)
    xz = np.array([[0, 0], [.25, -.5], [-.3, .1], [.5, -.9]], np.float32)
    rays7 = np.concatenate([xz[:, :1], np.full((len(xz), 1), 5), xz[:, 1:], np.tile([0, -1, 0, 1e30], (len(xz), 1))], 1).astype(np.float32)

    def trace(texels):
        img = np.repeat(np.float32([1, 1] if texels is None else texels)[None, :, None], 3, 2)
        st = ab.AlphaScene.from_tables(prims, [mesh], materials=[mat], images=[img], bindings=[agpt.material_textures()],
                                       masks=[agpt.alpha_mask(0, 0, .5)] if texels is not None else [])
        return st.trace_rays(rays7), st.trace_rays(rays7, any_hit=True)

    both, both_any = trace(None)
    first, _ = trace([1, 0])
    second, second_any = trace([0, 1])
    none, none_any = trace([0, 0])
    # the tie: each triangle alone is hit at the same t
    assert both["found"].all() and first["found"].all() and second["found"].all()
    assert np.array_equal(bits(first["t"]), bits(second["t"]))
    assert (first["tri"] == 7).all() and (second["tri"] == 9).all()
    for h in (first, trace([1, 1])[0]):
        for f in ("found", "prim", "tri"):
            assert np.array_equal(h[f], both[f]), f
        assert np.array_equal(bits(h["t"]), bits(both["t"]))
    assert (none["found"] == 0).all() and (none["prim"] == -1).all() and (none_any["found"] == 0).all()
    assert both_any["found"].all() and second_any["found"].all()


@pytest.mark.parametrize("channel", [0, 1, 2])
def test_mask_lookup_is_the_texture_lookup_of_one_channel(channel):
    img = RNG.random((5, 7, 3), dtype=np.float32)
    H, W = img.shape[:2]
    i, j = np.meshgrid(np.arange(W), np.arange(H))
    centres = np.stack([(i + .5) / W, (j + .5) / H], -1).reshape(-1, 2)
    edges = np.array([[0, 0], [1, 1], [0, .5], [1, .5], [.5, 0], [.5, 1], [1e-7, 1 - 1e-7]], np.float64)
    wrapped = np.concatenate([centres + 3, centres - 2, RNG.uniform(-4, 4, (200, 2))])
    uv = np.concatenate([centres, edges, wrapped]).astype(np.float32)
    got = ab.lookup_channel(img, channel, uv)
    want = tb.lookup(img, uv)[:, channel]
    assert np.array_equal(bits(got), bits(want))
    # at the centres the lookup returns the texels
    assert np.array_equal(bits(got[:W * H]), bits(img[..., channel].reshape(-1)))


def test_the_cut_line_of_a_half_mask_against_float64():
    """A 2 x 1 mask (0 | 1) at cutoff 0.5: the surface starts where the bilinear ramp between the texel centres reaches 0.5."""
    img = np.array([[[0, 0, 0], [1, 1, 1]]], np.float32)
    u = np.linspace(.2, .8, 4097).astype(np.float32)
    uv = np.stack([u, np.full_like(u, .5)], -1)
    got = ab.lookup_channel(img, 0, uv) >= np.float32(.5)
    s = u.astype(np.float64) * 2 - .5                          # the lookup's formula in float64: between the texel centres (s in
    fx = s - np.floor(s)                                        # [0, 1)) alpha rises 0 -> 1, outside them (wrapped) it falls 1 -> 0
    want = np.where(np.floor(s) == 0, fx, 1 - fx) >= .5
    # float32 rounding of u * W - 0.5 may only move the cut by the one sample nearest to u = 0.5
    assert np.count_nonzero(got != want) <= 1
    assert not got[u < .49].any() and got[u > .51].all()


def test_flattening_shares_images_between_slots_and_materials(agpt):
    _host(agpt)
    hs = agpt.HostScene(14, 1)
    masks = hs.alpha_masks()
    from tests.test_material_maps_cpu import _Tables
    t = _Tables.from_buffer_copy(hs.tables().raw[:ctypes.sizeof(_Tables)])
    assert len(masks) == t.n_materials == t.n_material_textures
    bound = [(m.texture, m.channel, m.cutoff) for m in masks if m.texture >= 0]
    assert len(bound) == 5                                       # leaves (one material for the mesh and an instance), second leaves, checker, grate, mirror
    # the leaves' mask is its base-colour image through the green channel: one texture, not two
    leaf = [i for i in range(t.n_materials) if t.material_textures[i].base >= 0][0]
    assert masks[leaf].texture == t.material_textures[leaf].base and masks[leaf].channel == 1
    # the disc image masks the second leaves and the mirror: flattened once
    discs = [m.texture for m in masks if m.texture >= 0 and m.channel == 0]
    assert len(discs) == 3 and len(set(discs)) == 2
    assert all(0 <= m.texture < t.n_textures for m in masks if m.texture >= 0)
    assert all(m.cutoff == np.float32(.5) for m in masks if m.texture >= 0)
    # scenes without a mask export none
    assert agpt.HostScene(12, 0).alpha_masks() == []


def test_binding_argument_checks(agpt):
    m = agpt.alpha_mask()
    assert (m.texture, m.channel, m.cutoff) == (-1, 0, .5) and ctypes.sizeof(m) == 16
    ctx = object.__new__(agpt.Context)
    ctx._h = ctypes.c_void_p()
    for bad in ([agpt.alpha_mask(-2)], [agpt.alpha_mask(0, 3)], [agpt.alpha_mask(0, -1)], [agpt.alpha_mask(0, 0, float("nan"))],
                [agpt.alpha_mask(0, 0, float("inf"))], [agpt.material_textures()]):
        with pytest.raises(agpt.AgptError):
            ctx.upload_alpha_masks(bad)
    # the C ABI refuses a null context and a missing table
    assert agpt.core().agpt_upload_alpha_masks(None, None, 0) < 0
