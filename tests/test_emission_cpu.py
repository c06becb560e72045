"""CPU: the statement of emissive materials (include/agpt.h agpt_upload_emission, statements/agpt_emission_oracle.cpp) against the
alpha-mask statement and the oracle, its closed-form cases, the host mirror's flattening of emission rows, and the binding's
argument checks.

NOT REFERENCE BEHAVIOUR: the reference has no emissive materials.  With no emitting row the statement must be the alpha
statement, itself the oracle when no image is bound."""
import ctypes
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from statements import alpha_binding as ab  # noqa: E402
from statements import emission_binding as eb  # noqa: E402
from tests.test_gpu_textures import bits  # noqa: E402

pytestmark = pytest.mark.skipif(not eb.available(), reason="statements/libagpt_emission_oracle.so not built (__graft_entry__.build())")


def _host(agpt):
    if not os.path.exists(agpt.lib_paths()[1]):
        pytest.skip("libagpt_host.so not built")


def closed_cube(agpt, r, e):
    """The camera of cfg 15 inside a closed cube of 12 triangles (cfg 15's room, one plain mesh) with MirrorMaterial r and
    emission factor e, no lights: every path ray hits a wall, and each wall hit adds beta * e with beta = r^k."""
    lo, hi = np.float32([-5, -1, -6]), np.float32([5, 5, 6])
    c = [np.float32([(hi if (k >> a) & 1 else lo)[a] for a in range(3)]) for k in range(8)]
    quads = [(0, 1, 5, 4), (2, 6, 7, 3), (0, 4, 6, 2), (1, 3, 7, 5), (4, 5, 7, 6), (0, 2, 3, 1)]
    tris = [(q[0], q[1], q[2]) for q in quads] + [(q[0], q[2], q[3]) for q in quads]
    verts = np.zeros((12, 3, 4), np.float32)
    for i, t in enumerate(tris):
        for k in range(3):
            verts[i, k, :3] = c[t[k]]
    mesh = agpt.RawMesh(verts, tri_ids=list(range(12)))
    prims = np.zeros(1, agpt.PRIM_DTYPE)
    prims[0] = (agpt.PRIM_MESH, 0, 0, -1)
    mat = agpt.make_material(agpt.MAT_MIRROR, (r, r, r), 0., 0.)
    cam = agpt.HostScene(15, 1).camera()
    return prims, mesh, mat, cam, agpt.emission(-1, (e, e, e))


def cube_statement(agpt, r, e):
    prims, mesh, mat, cam, row = closed_cube(agpt, r, e)
    keep = ab.AlphaScene.from_tables(prims, [mesh], materials=[mat], camera=cam)._keep
    return eb.EmissionScene(keep, masks=[], rows=[row])


@pytest.mark.parametrize("cfg,level", [(1, 0), (5, 2), (7, 0), (9, 2), (10, 2), (12, 0), (13, 1), (14, 1)])
def test_without_emitting_rows_the_statement_is_the_alpha_statement(agpt, cfg, level):
    """Film and every counter; cfg 1 and 5 also against the oracle itself.  All-zero rows are no emitting rows."""
    _host(agpt)
    hs = agpt.HostScene(cfg, level)
    d = agpt.config_defaults(cfg)
    want, wcnt = ab.AlphaScene(hs).render(32, 18, 0, 2, d["max_depth"], d["depth_arg"], counters=True)
    from tests.test_material_maps_cpu import _Tables
    n_mat = _Tables.from_buffer_copy(hs.tables().raw[:ctypes.sizeof(_Tables)]).n_materials
    for rows in ([], [agpt.emission(-1, (0, 0, 0))] * n_mat):
        got, cnt = eb.EmissionScene(hs, rows=rows).render(32, 18, 0, 2, d["max_depth"], d["depth_arg"], counters=True)
        assert np.array_equal(bits(got), bits(want))
        assert cnt == wcnt
    xs, ys, ss = np.arange(40) % 32, np.arange(40) % 18, np.arange(40)
    assert np.array_equal(bits(eb.EmissionScene(hs).li_pixels(32, 18, xs, ys, ss, d["max_depth"], d["depth_arg"])),
                          bits(ab.AlphaScene(hs).li_pixels(32, 18, xs, ys, ss, d["max_depth"], d["depth_arg"])))
    if cfg in (1, 5):
        from oracle import port_binding as port
        pwant, _ = port.PortScene(hs).render(32, 18, 0, 2, d["max_depth"], d["depth_arg"])
        assert np.array_equal(bits(got), bits(pwant))


def test_cfg15_emits_where_the_alpha_statement_is_dark(agpt):
    """cfg 15's emission rows change the film, and with no light (level 2) the film is emission only."""
    _host(agpt)
    for level in (1, 2):
        hs = agpt.HostScene(15, level)
        d = agpt.config_defaults(15)
        lit = eb.EmissionScene(hs).render(32, 18, 0, 2, d["max_depth"], d["depth_arg"])[..., :3]
        dark = eb.EmissionScene(hs, rows=[]).render(32, 18, 0, 2, d["max_depth"], d["depth_arg"])[..., :3]
        assert (lit >= dark).all() and np.count_nonzero(lit > dark) > 32 * 18 // 2
        if level == 2:
            assert not dark.any()


@pytest.mark.parametrize("depth", [0, 1, 2, 8])
def test_closed_mirror_cube_is_a_geometric_series(agpt, depth):
    """E * sum_{k <= depth} R^k per path (bit for bit at depth 0: one term, beta = 1)."""
    r, e, spp = .5, .75, 4
    st = cube_statement(agpt, r, e)
    film = st.render(48, 27, 0, spp, depth, 0)[..., :3].astype(np.float64)
    want = e * spp * sum(r ** k for k in range(depth + 1))
    if depth == 0:
        assert (film == e * spp).all()
    assert np.abs(film / want - 1).max() < 1e-5


def test_doubling_every_factor_doubles_the_film_without_lights(agpt):
    _host(agpt)
    hs = agpt.HostScene(15, 2)
    d = agpt.config_defaults(15)
    rows = hs.emission()
    twice = [agpt.emission(r.texture, tuple(2 * f for f in r.factor)) for r in rows]
    one = eb.EmissionScene(hs).render(32, 18, 0, 2, d["max_depth"], d["depth_arg"])
    two = eb.EmissionScene(hs, rows=twice).render(32, 18, 0, 2, d["max_depth"], d["depth_arg"])
    assert np.array_equal(bits(two), bits(2 * one))


def test_flattening_shares_images_and_rows_are_right(agpt):
    _host(agpt)
    from tests.test_material_maps_cpu import _Tables
    for level in (1, 2):
        hs = agpt.HostScene(15, level)
        rows = hs.emission()
        t = _Tables.from_buffer_copy(hs.tables().raw[:ctypes.sizeof(_Tables)])
        assert len(rows) == t.n_materials == t.n_material_textures
        emitting = [r for r in rows if max(r.factor) > 0]
        # screen, ball, strip, icosphere instances (one material); level 2 adds the sign
        assert len(emitting) == (4 if level == 1 else 5)
        assert all(0 <= r.texture < t.n_textures for r in rows if r.texture >= 0)
        assert sorted(tuple(np.float32(r.factor)) for r in emitting if r.texture < 0) == [(1.5, .6, .2), (4., 4., 4.5)]
        # the screen's emission image is its base-colour image: one texture, not two
        screen = [i for i in range(t.n_materials) if t.material_textures[i].base >= 0]
        assert len(screen) == 1 and rows[screen[0]].texture == t.material_textures[screen[0]].base
        assert tuple(rows[screen[0]].factor) == (2., 2., 2.)
        # images: colour bars, the icosphere's stripes (emission only), and at level 2 the letters (mask and emission: one texture)
        assert t.n_textures == (2 if level == 1 else 3)
        if level == 2:
            masks = hs.alpha_masks()
            sign = [i for i, m in enumerate(masks) if m.texture >= 0]
            assert len(sign) == 1 and rows[sign[0]].texture == masks[sign[0]].texture
    # scenes without emission export none
    assert agpt.HostScene(12, 0).emission() == [] and agpt.HostScene(14, 1).emission() == []


def test_binding_argument_checks(agpt):
    e = agpt.emission()
    assert (e.texture, tuple(e.factor)) == (-1, (0., 0., 0.)) and ctypes.sizeof(e) == 16
    ctx = object.__new__(agpt.Context)
    ctx._h = ctypes.c_void_p()
    for bad in ([agpt.emission(-2)], [agpt.emission(0, (-1, 0, 0))], [agpt.emission(0, (0, float("nan"), 0))],
                [agpt.emission(-1, (0, 0, float("inf")))], [agpt.alpha_mask()]):
        with pytest.raises(agpt.AgptError):
            ctx.upload_emission(bad)
    # the C ABI refuses a null context and a missing table
    assert agpt.core().agpt_upload_emission(None, None, 0) < 0
