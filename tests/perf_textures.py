"""Perf probe (not a test) of image textures on the base colour of Disney materials.  Prints JSON lines:
  * cfg 3 at 1080p, 16 spp, in three forms: untextured; every Disney material bound to a 1x1 image of its own colour (the cost
    of the textured shade instantiation alone: the film is bit-identical); every Disney material bound to its own 2048 x 2048
    procedural image (texel traffic beyond the L2: 64 MB per image on the device).  ms per 16-spp render (median, host clock
    around calls that end in a device synchronise) and the device time of k_shade_b per render (torch.profiler, a run of its own);
  * cfg 12 at 480 x 270: relative MSE of the raw and the denoised 16-spp film against a 1024-spp film of the same frame;
  * the card's name and power limit, read in the same run.

relMSE = mean over pixels and channels of (x - r)^2 / (r^2 + 1e-2), x = pixel mean, r = the reference film's pixel mean.

    python tests/perf_textures.py"""
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests.conftest import load_agpt  # noqa: E402
from tests.perf_denoise import card, rel_mse, timed  # noqa: E402
from tests.test_gpu_textures import materials, own_colour  # noqa: E402


def shade_ms(ctx, d, spp):
    import torch
    from torch.profiler import ProfilerActivity, profile
    ctx.clear()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.render(0, spp, d["max_depth"], d["depth_arg"])
        torch.cuda.synchronize()
    us = sum(e.device_time_total for e in prof.key_averages() if "k_shade_b" in e.key)
    return round(us / 1e3, 3)


def big_image(k, n=2048):
    y, x = np.mgrid[0:n, 0:n].astype(np.float32) / n
    return np.stack([.2 + .6 * x, .2 + .6 * ((np.floor(x * 32) + np.floor(y * 32) + k) % 2), .2 + .6 * y], -1).astype(np.float32)


def main():
    agpt = load_agpt()
    print(json.dumps({"card": card()}), flush=True)
    ctx = agpt.Context(0)
    d = agpt.config_defaults(3)
    hs = agpt.HostScene(3, 0)
    hs.upload(ctx); ctx.set_film(1920, 1080)
    mats = materials(hs)
    disney = [i for i in range(len(mats)) if mats[i]["type"] == 1]
    forms = {"untextured": ([], []), "own_colour_1x1": None, "2048x2048_each": None}
    imgs, bind = [], [-1] * len(mats)
    for i in disney:
        c = own_colour(mats[i])
        if c is not None:
            bind[i] = len(imgs); imgs.append(c.reshape(1, 1, 3))
    forms["own_colour_1x1"] = (imgs, bind)
    forms["2048x2048_each"] = ([big_image(k) for k in range(len(disney))], [disney.index(i) if i in disney else -1 for i in range(len(mats))])
    for name, (im, b) in forms.items():
        ctx.upload_textures(im, b)
        render = lambda: (ctx.clear(), ctx.render(0, 16, d["max_depth"], d["depth_arg"]), ctx.read_accum())
        ms = timed(render, 5)
        print(json.dumps({"cfg": 3, "form": name, "textures": len(im), "scene_bytes": ctx.scene_bytes(), "ms_per_16spp": ms,
                          "k_shade_b_ms": shade_ms(ctx, d, 16)}), flush=True)
    ctx.upload_textures([], [])
    # quality on cfg 12
    d = agpt.config_defaults(12)
    hs = agpt.HostScene(12, 0)
    hs.upload(ctx); ctx.set_film(480, 270); ctx.set_moments(True); ctx.clear()
    ctx.render(1 << 20, 1024, d["max_depth"])
    ref = ctx.read_accum()[..., :3] / 1024.0
    ctx.clear(); ctx.render(0, 16, d["max_depth"])
    raw = ctx.read_accum()[..., :3] / 16.0
    ctx.render_guides(4)
    out, _ = ctx.denoise(agpt.denoise_params())
    print(json.dumps({"cfg": 12, "size": "480x270", "spp": 16, "rel_mse_raw": rel_mse(raw, ref), "rel_mse_denoised": rel_mse(out[..., :3], ref)}), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
