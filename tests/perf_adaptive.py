"""Perf probe (not a test) of adaptive sampling at 1080p: for cfg 3 and cfg 5, a uniform render and agpt_render_adaptive
against a converged uniform film.  Prints JSON lines: wall time, mean samples per pixel, rounds and relative MSE of each,
the device time of k_adaptive_select and of the list form of k_accumulate per round (torch.profiler),
and the card's name and power limit read in the same run.

relMSE = mean over pixels and channels of (x - r)^2 / (r^2 + 1e-2), x = pixel mean, r = the reference film's pixel mean.

    python tests/perf_adaptive.py [uniform_spp=256] [reference_spp=1024] [tolerances=0.05,0.1,0.2] [floor=0.01]"""
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


def adaptive_case(agpt, ctx, cfg, d, p, uni, ref, spp):
    """One agpt_render_adaptive of the uploaded scene, timed, against the reference and the uniform film."""
    t = time.perf_counter()
    rounds, paths = ctx.render_adaptive(p, d["max_depth"], d["depth_arg"])
    t_adaptive = time.perf_counter() - t
    film, mom = ctx.read_accum(), ctx.read_moments()
    n = mom[..., 3].astype(np.float64)
    ada = film[..., :3].astype(np.float64) / n[..., None]
    counts = np.unique(n, return_counts=True)
    print(json.dumps(dict(cfg=cfg, mode="adaptive", min_samples=p.min_samples, max_samples=p.max_samples, step=p.step, tolerance=round(p.tolerance, 4),
                          floor=round(p.floor, 4), wall_s=round(t_adaptive, 3), mean_spp=round(float(n.mean()), 2), rounds=rounds, paths=paths,
                          rel_mse=rel_mse(ada, ref), rel_mse_uniform_same_mean_spp_estimate=rel_mse(uni, ref) * spp / float(n.mean()),
                          counts={int(k): int(c) for k, c in zip(*counts)})), flush=True)
    # select alone on the final film (host clock around a call that ends in a device synchronise)
    reps = 20
    t = time.perf_counter()
    for _ in range(reps):
        ctx.adaptive_select(p, want_pixels=False)
    print(json.dumps(dict(cfg=cfg, select_call_ms=round((time.perf_counter() - t) * 1e3 / reps, 3))), flush=True)


def main():
    spp = int(sys.argv[1]) if len(sys.argv) > 1 else 256
    ref_spp = int(sys.argv[2]) if len(sys.argv) > 2 else 1024
    tols = [float(t) for t in (sys.argv[3] if len(sys.argv) > 3 else "0.05,0.1,0.2").split(",")]
    floor = float(sys.argv[4]) if len(sys.argv) > 4 else 0.01
    agpt = load_agpt()
    print(json.dumps({"card": card()}), flush=True)
    ctx = agpt.Context(0)
    for cfg in (3, 5):
        d = agpt.config_defaults(cfg)
        W, H = 1920, 1080
        hs = agpt.HostScene(cfg, 0)
        hs.upload(ctx); ctx.set_film(W, H)
        ctx.set_moments(False)
        ctx.render(0, 16, d["max_depth"], d["depth_arg"])                       # warm-up: module load, bucket grid
        ctx.clear(); ctx.render(0, ref_spp, d["max_depth"], d["depth_arg"])
        ref = ctx.read_accum()[..., :3].astype(np.float64) / ref_spp
        ctx.clear(); t = time.perf_counter()
        ctx.render(0, spp, d["max_depth"], d["depth_arg"])
        t_uniform = time.perf_counter() - t
        uni = ctx.read_accum()[..., :3].astype(np.float64) / spp
        print(json.dumps(dict(cfg=cfg, mode="uniform", width=W, height=H, spp=spp, wall_s=round(t_uniform, 3),
                              rel_mse=rel_mse(uni, ref), reference_spp=ref_spp)), flush=True)
        ctx.set_moments(True)
        ctx.render_adaptive(agpt.adaptive(16, 32, 16, tols[0], floor), d["max_depth"], d["depth_arg"])      # warm-up of the list kernels
        for tol in tols:
            adaptive_case(agpt, ctx, cfg, d, agpt.adaptive(16, spp, 16, tol, floor), uni, ref, spp)
    # device time of the new kernels per round, in a run of its own under torch.profiler (cfg 5 is the last scene uploaded)
    p = agpt.adaptive(16, spp, 16, tols[-1], floor)
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.init()
        d = agpt.config_defaults(5)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            rounds, _ = ctx.render_adaptive(p, d["max_depth"], d["depth_arg"])
            torch.cuda.synchronize()
        per = {}
        for e in prof.events():
            for key in ("k_adaptive_select", "k_accumulate<true, true>", "k_generate<true>"):
                if key in e.name:
                    per.setdefault(key, []).append(e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total)
        print(json.dumps(dict(cfg=5, profiled_rounds=rounds, kernel_us_per_launch={k: round(float(np.mean(v)), 2) for k, v in per.items()},
                              launches={k: len(v) for k, v in per.items()})), flush=True)
    except Exception as e:                                                     # the timings above stand on their own
        print(json.dumps(dict(profiler_error=str(e)[:200])), flush=True)
    print(json.dumps({"card": card()}), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
