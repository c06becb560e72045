"""Perf probe (not a test) of roughness-metallic and normal maps on Disney materials.  Prints JSON lines, at 1920 x 1080 and
16 spp: ms per 16-spp render (median of 5, host clock around calls that end in a device synchronise) and the shade kernels'
device time per render (AGPT_FLAG_TIMING, in a run of its own), for
  * cfg 13 (maps on every material: k_shade_b<false, false, false, 2>);
  * cfg 12 on the base-colour path (<..., 1>) and on the maps path (<..., 2>, forced by one 1x1 own-value roughness-metallic map
    on its untextured sphere: the film is bit-identical) -- the measurement that decides whether both paths stay;
  * cfg 3 untextured (<..., 0>) and with own-value maps on every Disney material (<..., 2>; bit-identical film);
and the card's name and power limit, read in the same run.

    python tests/perf_material_maps.py"""
import ctypes
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests.conftest import load_agpt  # noqa: E402
from tests.perf_denoise import card, timed  # noqa: E402
from tests.test_gpu_textures import materials, own_colour  # noqa: E402
from tests.test_gpu_material_maps import FLAT, ONES, own_value_bindings  # noqa: E402


def measure(agpt, ctx, d, label):
    render = lambda: (ctx.clear(), ctx.render(0, 16, d["max_depth"], d["depth_arg"]), ctx.read_accum())
    ms = timed(render, 5)
    ctx.reset_stats(); ctx.clear()
    ctx.render(0, 16, d["max_depth"], d["depth_arg"], agpt.FLAG_TIMING)
    st = ctx.stats()
    print(json.dumps({"workload": label, "ms_per_16spp": ms, "ms_shade": round(float(st.ms_shade), 3), "ms_render_timed": round(float(st.ms_render), 3)}),
          flush=True)


def cfg12_maps_bindings(agpt, hs):
    from tests.test_material_maps_cpu import _Tables
    t = _Tables.from_buffer_copy(hs.tables().raw[:ctypes.sizeof(_Tables)])
    imgs = [np.ctypeslib.as_array(ctypes.cast(t.textures[i].rgb, ctypes.POINTER(ctypes.c_float)), (t.textures[i].height, t.textures[i].width, 3)).copy()
            for i in range(t.n_textures)]
    mats = materials(hs)
    bind = []
    for i in range(t.n_material_textures):
        base = t.material_texture[i]
        C = own_colour(mats[i]) if base < 0 and mats[i]["type"] == 1 else None
        bind.append(agpt.material_textures(base) if C is None else agpt.material_textures(-1, len(imgs), -1, 1.0, tuple(float(v) for v in C)))
    return imgs + [ONES], bind


def main():
    agpt = load_agpt()
    print(json.dumps({"card": card()}), flush=True)
    ctx = agpt.Context(0)
    ctx.set_film(1920, 1080)
    for cfg in (13, 12, 3):
        d = agpt.config_defaults(cfg)
        hs = agpt.HostScene(cfg, 0)
        hs.upload(ctx); ctx.set_film(1920, 1080)
        if cfg == 13:
            measure(agpt, ctx, d, "cfg13 maps (TEX 2)")
        elif cfg == 12:
            measure(agpt, ctx, d, "cfg12 base colour (TEX 1)")
            ctx.upload_material_textures(*cfg12_maps_bindings(agpt, hs))
            measure(agpt, ctx, d, "cfg12 through the maps path (TEX 2)")
        else:
            measure(agpt, ctx, d, "cfg3 untextured (TEX 0)")
            ctx.upload_material_textures(*own_value_bindings(agpt, hs))
            measure(agpt, ctx, d, "cfg3 own-value maps (TEX 2)")
        ctx.upload_textures([], [])
    ctx.close()


if __name__ == "__main__":
    main()
