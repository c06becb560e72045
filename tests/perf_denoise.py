"""Perf probe (not a test) of the guide buffers and the a-trous denoiser at 1080p, cfg 3 and cfg 5.  Prints JSON lines:
  * ms per 16-spp render, per render_guides call at 1 and 4 samples, per denoise call at 5 iterations (host clock around calls
    that end in a device synchronise; the denoise call includes copying both outputs to the host), and the device time of each
    new kernel (torch.profiler, a run of its own);
  * relative MSE of the raw and the denoised 16-spp and 64-spp films against a 1024-spp film of the same frame (independent
    samples), for the defaults of agpt.denoise_params() and a small sweep around them at 16 spp;
  * the card's name and power limit, read in the same run.

relMSE = mean over pixels and channels of (x - r)^2 / (r^2 + 1e-2), x = pixel mean, r = the reference film's pixel mean.

    python tests/perf_denoise.py [reference_spp=1024]"""
import itertools
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests.conftest import load_agpt  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def rel_mse(mean, ref):
    return float(np.mean((mean - ref) ** 2 / (ref ** 2 + 1e-2)))


def timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t = time.perf_counter(); fn(); ts.append((time.perf_counter() - t) * 1e3)
    return round(float(np.median(ts)), 3)


def main():
    ref_spp = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
    agpt = load_agpt()
    print(json.dumps({"card": card()}), flush=True)
    ctx = agpt.Context(0)
    W, H = 1920, 1080
    defaults = agpt.denoise_params()
    for cfg in (3, 5):
        d = agpt.config_defaults(cfg)
        hs = agpt.HostScene(cfg, 0)
        hs.upload(ctx); ctx.set_film(W, H)
        ctx.set_moments(False)
        ctx.render(0, 16, d["max_depth"], d["depth_arg"])                       # warm-up: module load, bucket grid
        ctx.clear(); ctx.render(64, ref_spp, d["max_depth"], d["depth_arg"])     # samples no film below uses
        ref = ctx.read_accum()[..., :3].astype(np.float64) / ref_spp
        ctx.set_moments(True)
        ms_render = timed(lambda: (ctx.clear(), ctx.render(0, 16, d["max_depth"], d["depth_arg"])), 3)
        ms_g1 = timed(lambda: ctx.render_guides(1), 5)
        ms_g4 = timed(lambda: ctx.render_guides(4), 5)
        ms_dn = timed(lambda: ctx.denoise(defaults), 5)
        print(json.dumps(dict(cfg=cfg, width=W, height=H, ms_render_16spp=ms_render, ms_guides_1=ms_g1, ms_guides_4=ms_g4,
                              ms_denoise_5_iterations_with_copies=ms_dn)), flush=True)
        for spp in (16, 64):
            ctx.clear(); ctx.render(0, spp, d["max_depth"], d["depth_arg"])
            raw = ctx.read_accum()[..., :3].astype(np.float64) / spp
            out, _ = ctx.denoise(defaults)
            print(json.dumps(dict(cfg=cfg, spp=spp, guide_samples=4, rel_mse_raw=rel_mse(raw, ref), rel_mse_denoised=rel_mse(out[..., :3], ref),
                                  params=dict(iterations=defaults.iterations, sigma_luminance=defaults.sigma_luminance, sigma_depth=defaults.sigma_depth,
                                              normal_power_log2=defaults.normal_power_log2))), flush=True)
            if spp == 16:
                rows = []
                for it, sl, sz, npow in itertools.product((3, 5), (1.0, 2.0, 4.0, 8.0), (0.02, 0.1, 1.0), (3, 7)):
                    o, _ = ctx.denoise(agpt.denoise_params(it, sl, sz, npow))
                    rows.append((rel_mse(o[..., :3], ref), it, sl, sz, npow))
                rows.sort()
                print(json.dumps(dict(cfg=cfg, spp=16, sweep_best=[dict(rel_mse=r[0], iterations=r[1], sigma_luminance=r[2], sigma_depth=r[3],
                                                                        normal_power_log2=r[4]) for r in rows[:6]])), flush=True)
        ctx.set_moments(False)
    # device time of the new kernels (cfg 5 is resident), in a run of its own under torch.profiler
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.init()
        ctx.set_moments(True)
        d = agpt.config_defaults(5)
        ctx.clear(); ctx.render(0, 16, d["max_depth"], d["depth_arg"])
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ctx.render_guides(4)
            ctx.denoise(defaults)
            torch.cuda.synchronize()
        per = {}
        for e in prof.events():
            for key in ("k_guides", "k_denoise_prepare", "k_denoise_atrous<false>", "k_denoise_atrous<true>", "k_trace_closest", "k_generate"):
                if key in e.name:
                    per.setdefault(key, []).append(e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total)
        print(json.dumps(dict(cfg=5, kernel_us_per_launch={k: round(float(np.mean(v)), 2) for k, v in per.items()},
                              launches={k: len(v) for k, v in per.items()})), flush=True)
        ctx.set_moments(False)
    except Exception as e:                                                     # the timings above stand on their own
        print(json.dumps(dict(profiler_error=str(e)[:200])), flush=True)
    print(json.dumps({"card": card()}), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
