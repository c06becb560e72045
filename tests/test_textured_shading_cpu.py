"""CPU: the recoloured scenes and the probe targets of tests/test_gpu_textured_shading.py, checked before any GPU runs them.

A recoloured scene binds every Disney material to constant images whose values differ from its own; its film must equal the
untextured film of a material table whose records already carry the derived values (include/agpt.h agpt_upload_textures
step 3, agpt_upload_material_textures step 1).  That holds bit for bit only if the float32 arithmetic behind the derived
records cannot round differently on the device: a compiler may contract (1 - t) * a + t * b into an FMA, the CPU statement
does not.  So every factor here is a power of two, every metallic outside {0, 1} is rewritten to 1/2 in both arms, and the
tests below check, record by record, that every product is exact and every sum is its float64 value rounded once."""
import ctypes
import itertools
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from statements import maps_binding as mb  # noqa: E402
from tests.test_gpu_textures import bits, materials  # noqa: E402
from tests.test_textures_cpu import _Tables  # noqa: E402

F32 = np.float32
MAT_DISNEY = 1
LOBE_DIFFUSE, LOBE_RETRO, LOBE_MICROFACET = 1, 2, 4
# (cfg, level) of the recoloured scenes and the shade instantiation each runs: cfg 3 and 5 <false, false, false, T>; cfg 7
# (InfiniteAreaLight), cfg 10 (rough glass) and cfg 11 (sampled shape lights) <true, true, true, T>
SCENES = [(3, 2), (5, 2), (7, 0), (10, 2), (11, 2)]
POW2 = F32([1 / 16, 1 / 8, 1 / 4, 1 / 2, 1])
# base colours: no two materials alike and no two channels of one colour alike, so a swapped material or channel shows
COLOURS = [F32(c) for c in itertools.permutations(POW2, 3)]
ROUGHNESS_FACTORS = F32([1 / 4, 1 / 2, 1])
METAL_FACTORS = F32([0, 1 / 2, 1])            # on a metal: 0 and 1/2 turn its diffuse and retro lobes on, 1 keeps it a metal
FLAT = np.array([[[.5, .5, 1.0]]], np.float32)     # a flat normal-map texel: the surface is left as it is


def rewrite_metallic(mats):
    """The records both arms start from: each Disney metallic outside {0, 1} becomes 1/2.  (1 - k) stays > 0, so the lobes
    the record holds are still the ones DisneyMaterial's constructor gives it."""
    out = mats.copy()
    k = out["metallic"]
    out["metallic"] = np.where((out["type"] == MAT_DISNEY) & (k != 0) & (k != 1), F32(.5), k)
    return out


def disney_colours(k, eta, c):
    """diffuse_r and spec_r0 of base colour c at metallic k, in the order agpt.h (agpt_upload_textures step 3) states."""
    k, eta, c = F32(k), F32(eta), np.asarray(c, np.float32)
    dw = (F32(1) - k) * (F32(1) - F32(0))
    diffuse = dw * c if dw > 0 else np.zeros(3, np.float32)
    r0 = ((eta - F32(1)) * (eta - F32(1))) / ((eta + F32(1)) * (eta + F32(1)))
    return diffuse, (F32(1) - k) * r0 + k * c


def recolouring(agpt, base, level):
    """Constant maps for every Disney material of `base` (records after rewrite_metallic) whose values differ from its own.

    level 1: a 1x1 base image c_m per material; returns (images, material_texture, expected records).
    level 2: a 1x1 roughness-metallic image (x, g, b), the base colour from the binding's `color` or from a 1x1 image (the
    materials alternate), a flat 1x1 normal map; returns (images, agpt.material_textures rows, expected records).
    The expected records are what DisneyMaterial's constructor makes of the derived values: the table the untextured arm
    uploads."""
    want = base.copy()
    images = [] if level == 1 else [FLAT]
    bind = []
    j = metals = 0
    for i, m in enumerate(base):
        if m["type"] != MAT_DISNEY:
            bind.append(-1 if level == 1 else agpt.material_textures())
            continue
        c = COLOURS[(7 * j + (0 if level == 1 else 3)) % len(COLOURS)]
        if level == 1:
            bind.append(len(images))
            images.append(c.reshape(1, 1, 3))
            want["diffuse_r"][i], want["spec_r0"][i] = disney_colours(m["metallic"], m["eta"], c)
        else:
            g = ROUGHNESS_FACTORS[j % 3]
            if m["metallic"] == 1:
                b = METAL_FACTORS[metals % 3]
                metals += 1
            elif m["metallic"] == .5:
                b = F32(j % 2)                       # k' stays in {0, 1/2}
            else:
                b = METAL_FACTORS[j % 3]
            rm = len(images)
            images.append(F32([[[.3, g, b]]]))
            if j % 2:
                images.append(c.reshape(1, 1, 3))
                bind.append(agpt.material_textures(len(images) - 1, rm, 0, 1.0))
            else:
                bind.append(agpt.material_textures(-1, rm, 0, 1.0, tuple(float(v) for v in c)))
            want[i] = mb.material(m, c, F32([.3, g, b]))
        j += 1
    return images, bind, want


def records(agpt, table):
    """MAT_DTYPE rows as the agpt_material rows Context.upload_table("materials", ...) takes."""
    return [agpt.binding.Material.from_buffer_copy(r.tobytes()) for r in table]


def arithmetic(k, eta, c, roughness=None, g=None, b=None):
    """Each float32 operation behind a derived record, as (what, float32 result, float64 value of the same operation on the
    float32 operands, is_sum).  With g, b: the roughness and metallic factors of agpt_upload_material_textures step 1 first.
    (alpha = max(.001, r' * r') is left out: a product that feeds no sum rounds the same under any contraction.)"""
    ops = []

    def mul(what, x, y):
        ops.append((what, F32(x) * F32(y), float(x) * float(y), False))
        return F32(x) * F32(y)

    def add(what, x, y):
        ops.append((what, F32(x) + F32(y), float(x) + float(y), True))
        return F32(x) + F32(y)

    if g is not None:
        mul("r * g", roughness, g)
        k = mul("k * b", k, b)
    one_k = add("1 - k", 1, -F32(k))
    dw = mul("dw", one_k, add("1 - 0", 1, -0.0))
    em, ep = add("eta - 1", eta, -1), add("eta + 1", eta, 1)
    r0 = mul("(eta - 1)^2", em, em) / mul("(eta + 1)^2", ep, ep)
    for ch in range(3):
        if dw > 0:
            mul("dw * c", dw, c[ch])
        add("spec_r0", mul("(1 - k) * r0", one_k, r0), mul("k * c", k, c[ch]))
    return ops


def _host(agpt):
    if not os.path.exists(agpt.lib_paths()[1]):
        pytest.skip("libagpt_host.so not built")


pytestmark = pytest.mark.skipif(not mb.available(), reason="statements/libagpt_material_maps_oracle.so not built (__graft_entry__.build())")


@pytest.mark.parametrize("level", [1, 2])
@pytest.mark.parametrize("cfg,scene_level", SCENES)
def test_every_derived_record_is_exact(agpt, cfg, scene_level, level):
    """Both arms' records: every product exact, every sum its float64 value rounded once, so an FMA anywhere in
    (1 - k) * r0 + k * c gives the same float.  The expected records equal the statement's DisneyMaterial arithmetic and the
    explicit float32 formula of agpt.h."""
    _host(agpt)
    base = rewrite_metallic(materials(agpt.HostScene(cfg, scene_level)))
    images, bind, want = recolouring(agpt, base, level)
    disney = np.nonzero(base["type"] == MAT_DISNEY)[0]
    assert len(disney) >= 2
    assert np.all(np.isin(base["metallic"][disney], F32([0, .5, 1])))
    for i in disney:
        m, w = base[i], want[i]
        assert mb.material(m, F32([.5, .5, .5]), F32([.3, 1, 1]))["lobes"] == m["lobes"]          # the rewrite keeps the lobes
        if level == 1:
            c = images[bind[i]][0, 0]
            ops = arithmetic(m["metallic"], m["eta"], c)
            assert mb.material(m, c, F32([.3, 1, 1])).tobytes() == w.tobytes()       # the statement's arithmetic agrees
        else:
            t = bind[i]
            rm = images[t.roughness_metallic][0, 0]
            c = images[t.base][0, 0] if t.base >= 0 else F32(list(t.color))
            ops = arithmetic(m["metallic"], m["eta"], c, m["roughness"], rm[1], rm[2])
            assert w["roughness"] == m["roughness"] * rm[1] and w["metallic"] == m["metallic"] * rm[2]
            assert w["metallic"] in (0, .5, 1)
        for what, got, exact, is_sum in ops:
            want64 = F32(exact) if is_sum else exact
            assert float(got) == float(want64), (cfg, i, what, got, exact)
        diffuse, spec = disney_colours(w["metallic"], w["eta"], c)
        assert np.array_equal(w["diffuse_r"], diffuse) and np.array_equal(w["spec_r0"], spec)
        assert np.any(w["diffuse_r"] != m["diffuse_r"]) or np.any(w["spec_r0"] != m["spec_r0"])        # the colours do change
    assert want[base["type"] != MAT_DISNEY].tobytes() == base[base["type"] != MAT_DISNEY].tobytes()


def test_recolourings_tell_materials_and_channels_apart_and_use_every_rule(agpt):
    """Distinct colours with distinct channels; at level 2 both sources of the base colour in every scene, every roughness
    factor, and on metals each metallic factor: 0 and 1/2 turn the diffuse and retro lobes on, 1 keeps a metal."""
    _host(agpt)
    assert len({c.tobytes() for c in COLOURS}) == len(COLOURS) and all(len(set(c.tolist())) == 3 for c in COLOURS)
    transitions, factors = set(), set()
    for cfg, scene_level in SCENES:
        base = rewrite_metallic(materials(agpt.HostScene(cfg, scene_level)))
        disney = base["type"] == MAT_DISNEY
        for level in (1, 2):
            images, bind, want = recolouring(agpt, base, level)
            assert len({want["diffuse_r"][i].tobytes() + want["spec_r0"][i].tobytes() for i in np.nonzero(disney)[0]}) == disney.sum()
            if level == 1:
                assert all((b >= 0) == d for b, d in zip(bind, disney))
                continue
            assert all((b.roughness_metallic >= 0 and b.normal == 0) == d for b, d in zip(bind, disney))
            assert {b.base >= 0 for b, d in zip(bind, disney) if d} == {True, False}
            for b, m, w in zip(bind, base, want):
                if b.roughness_metallic >= 0:
                    factors.add(float(images[b.roughness_metallic][0, 0, 1]))
                    transitions.add((int(m["lobes"]), int(w["lobes"]), float(w["metallic"])))
    assert factors == {.25, .5, 1.0}
    metal, all_lobes = LOBE_MICROFACET, LOBE_DIFFUSE | LOBE_RETRO | LOBE_MICROFACET
    assert {(metal, all_lobes, 0.0), (metal, all_lobes, .5), (metal, metal, 1.0), (all_lobes, all_lobes, .5)} <= transitions


class _WithMaterials:
    """A host scene's tables with another material table (MapsScene reads host_scene.tables())."""

    def __init__(self, hs, table):
        self._keep, self._table = hs, np.ascontiguousarray(table)
        raw = hs.tables().raw
        self._buf = ctypes.create_string_buffer(raw, len(raw))
        ctypes.c_void_p.from_buffer(self._buf, _Tables.materials.offset).value = self._table.ctypes.data

    def tables(self):
        return self._buf


@pytest.mark.parametrize("level", [1, 2])
@pytest.mark.parametrize("cfg,scene_level", [s for s in SCENES if s[0] != 11])
def test_statement_renders_the_recoloured_scene_as_its_records(agpt, cfg, scene_level, level):
    """The CPU twin of the device check, where the statement covers the scene (it has no sampled shape lights): textured arm
    and untextured records give the same film and guides, and the film is not the one the records had before."""
    _host(agpt)
    hs = agpt.HostScene(cfg, scene_level)
    d = agpt.config_defaults(cfg)
    base = rewrite_metallic(materials(hs))
    images, bind, want = recolouring(agpt, base, level)
    textured = mb.MapsScene(_WithMaterials(hs, base), rr_by_bounce=cfg == 10)
    textured.set_textures(images, [agpt.material_textures(b) for b in bind] if level == 1 else bind)
    plain, recorded = (mb.MapsScene(_WithMaterials(hs, t), rr_by_bounce=cfg == 10) for t in (base, want))
    film = [s.render(48, 27, 0, 2, d["max_depth"], d["depth_arg"]) for s in (textured, recorded, plain)]
    assert np.array_equal(bits(film[0]), bits(film[1]))
    for got, want_guide in zip(textured.guides(48, 27, 2), recorded.guides(48, 27, 2)):
        assert np.array_equal(bits(got), bits(want_guide))
    lit = np.any(film[2][..., :3] > 0, -1)
    assert lit.mean() > .5 and np.any(film[0][..., :3] != film[2][..., :3], -1)[lit].mean() > .9


# ---- probe targets on cfg 12's floor ----------------------------------------------------------------------------------------

def plane_uv(P, o, half):
    """agpt.h agpt_upload_textures step 1 for a plane, in float32 (u from x, v from z)."""
    return (((F32(P) - F32(o)) / F32(half) + F32(1)) * F32(.5)).astype(np.float32)


def floor_targets(W, H, o, half):
    """float32 (x, z) points on a plane of half-sizes `half` around o (x, z) aimed at texel centres, texel edges and one ulp
    inside the plane's four edges (the u = 0 / 1 and v = 0 / 1 seams) of a W x H image; at most 65 positions per axis."""
    def axis(n, offset):
        i = np.arange(n) if n <= 64 else np.unique(np.r_[np.linspace(0, n - 1, 62).round(), 0, 1, n - 2, n - 1])
        return (i + offset) / n
    centres_u, centres_v = axis(W, .5), axis(H, .5)
    edges_u, edges_v = axis(W, 0)[1:] if W > 1 else np.array([.5]), axis(H, 0)[1:] if H > 1 else np.array([.5])
    uv = [np.stack(np.meshgrid(a, b), -1).reshape(-1, 2) for a, b in ((centres_u, centres_v), (edges_u, edges_v), (centres_u, edges_v),
                                                                       (edges_u, centres_v))]
    xz = [np.asarray(o, np.float64) + (2 * np.concatenate(uv) - 1) * half]
    # seams: one ulp inside x = o.x -/+ half_x (along texel-centre rows of z) and z = o.z -/+ half_z (along centre columns of
    # x), and the four corners
    inside = [[np.nextafter(F32(o[k] + sign * half[k]), F32(o[k])) for sign in (-1, 1)] for k in (0, 1)]
    along = [o[1] + (2 * centres_v[:9] - 1) * half[1], o[0] + (2 * centres_u[:9] - 1) * half[0]]
    for k in (0, 1):
        for edge in inside[k]:
            pts = np.zeros((len(along[k]), 2))
            pts[:, k], pts[:, 1 - k] = edge, along[k]
            xz.append(pts)
    xz.append(np.array([[a, b] for a in inside[0] for b in inside[1]], np.float64))
    return np.concatenate(xz).astype(np.float32)


@pytest.mark.parametrize("W,H", [(1, 1), (1, 7), (7, 1), (2, 2), (5, 3), (37, 23), (4099, 3), (3, 4099)])
def test_floor_targets_aim_where_they_say(W, H):
    """The points the probe test aims at land, through the plane's float32 uv, on texel centres (s integral), on texel edges (s
    half-integral) and inside the first and last half texel (the seams) often enough to test each.  One ulp inside the far
    edge, u rounds to 1 itself, which the lookup wraps to 0."""
    o, half = (0.0, 0.0), (4.0, 4.0)
    xz = floor_targets(W, H, o, half)
    u, v = plane_uv(xz[:, 0], o[0], half[0]), plane_uv(xz[:, 1], o[1], half[1])
    assert np.all((u >= 0) & (u <= 1) & (v >= 0) & (v <= 1))
    for n, t in ((W, u), (H, v)):
        s = t * F32(n) - F32(.5)
        assert np.mean(s == np.floor(s)) > .2                                       # centres
        assert n == 1 or np.mean(s - np.floor(s) == .5) > .1                        # edges
        assert np.any(s < 0) and np.any(s > n - 1)                                  # both seams: a blend of the first and last texel
        assert np.any(t > 0) and np.min(t[t > 0]) <= 2 ** -24 and np.max(t) >= 1 - 2 ** -24
