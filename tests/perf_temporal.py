"""Perf probe (not a test) of the film reprojection (agpt_reproject_film) at 1080p, cfg 3 and cfg 5.  Prints JSON lines:
  * the card's name and power limit, read in the same run;
  * ms per reproject_film call (host clock around calls that end in a device synchronise), and the device time of
    k_reproject_film<true> and of the film copy after it (torch.profiler, a run of its own), against the least time the
    kernel's unique traffic could take: 128 B per pixel (current guides 32 B, history film + moments + G 48 B, writes 48 B) over
    the data-sheet HBM bandwidth (7.7 TB/s) and over the bandwidth agpt_probe_bandwidth reaches on this card;
  * per-frame relative MSE along a 16-frame orbit (0.5 degrees per frame, 4 spp per frame, 4 guide samples) against a
    1024-spp film of each frame's camera (independent samples), for denoising each frame's own 4 samples and for
    reproject + denoise, with the fraction of pixels that carried history into the frame;
  * a sweep of max_history, sigma_depth and min_normal_dot, ranked by the mean relative MSE of the last 8 frames.

relMSE = mean over pixels and channels of (x - r)^2 / (r^2 + 1e-2), x = pixel value, r = the reference film's pixel mean.

    python tests/perf_temporal.py [reference_spp=1024]"""
import itertools
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests.conftest import load_agpt  # noqa: E402
from oracle import reproject as rp  # noqa: E402

FRAMES, SPP, GUIDES, STEP_DEG = 16, 4, 4, 0.5
BYTES_PER_PIXEL = 128


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def rel_mse(x, ref):
    return float(np.mean((np.asarray(x, np.float64)[..., :3] - ref) ** 2 / (ref ** 2 + 1e-2)))


def orbit_run(ctx, d, cams, refs, p, dp, carried=None):
    """The viewer loop along the orbit: per-frame relMSE of reproject + denoise (p) or of denoise alone (p None)."""
    ctx.clear()
    out = []
    for i, c in enumerate(cams):
        ctx.set_camera(c)
        ctx.render_guides(GUIDES)
        if p is None:
            ctx.clear()
        else:
            ctx.reproject_film(p)
            if carried is not None:
                carried.append(round(float((ctx.read_moments()[..., 3] > 0).mean()), 4))
        ctx.render(i * SPP, SPP, d["max_depth"], d["depth_arg"])
        den, _ = ctx.denoise(dp)
        out.append(rel_mse(den, refs[i]))
    return out


def main():
    ref_spp = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
    agpt = load_agpt()
    print(json.dumps({"card": card()}), flush=True)
    ctx = agpt.Context(0)
    W, H = 1920, 1080
    hbm = ctx.probe_bandwidth(4 << 30, 4)
    dp, p0 = agpt.denoise_params(), agpt.reproject_params()
    for cfg in (3, 5):
        d = agpt.config_defaults(cfg)
        hs = agpt.HostScene(cfg, 0)
        hs.upload(ctx); ctx.set_film(W, H)
        cams = [rp.orbit(hs.camera(), STEP_DEG * i) for i in range(FRAMES)]
        ctx.set_moments(False)
        ctx.render(0, 16, d["max_depth"], d["depth_arg"])                       # warm-up: module load, bucket grid
        refs = []
        for c in cams:                                                          # samples no frame below uses
            ctx.set_camera(c); ctx.clear(); ctx.render(1 << 20, ref_spp, d["max_depth"], d["depth_arg"])
            refs.append(ctx.read_accum()[..., :3].astype(np.float64) / ref_spp)
        ctx.set_moments(True)
        # call time: alternate two cameras so that every call carries
        ts = []
        for i in range(12):
            ctx.set_camera(cams[i % 2]); ctx.render_guides(1)
            t = time.perf_counter(); ctx.reproject_film(p0); ts.append((time.perf_counter() - t) * 1e3)
        bound_us = BYTES_PER_PIXEL * W * H / 7.7e12 * 1e6
        print(json.dumps(dict(cfg=cfg, width=W, height=H, ms_reproject_call=round(float(np.median(ts[2:])), 4), unique_bytes=BYTES_PER_PIXEL * W * H,
                              bound_us_datasheet_7p7TBs=round(bound_us, 2), probe_hbm_gbs=round(hbm, 1),
                              bound_us_probe=round(BYTES_PER_PIXEL * W * H / (hbm * 1e9) * 1e6, 2))), flush=True)
        carried = []
        alone = orbit_run(ctx, d, cams, refs, None, dp)
        temporal = orbit_run(ctx, d, cams, refs, p0, dp, carried)
        print(json.dumps(dict(cfg=cfg, frames=FRAMES, spp_per_frame=SPP, orbit_deg_per_frame=STEP_DEG, guide_samples=GUIDES,
                              params=dict(max_history=p0.max_history, sigma_depth=p0.sigma_depth, min_normal_dot=p0.min_normal_dot),
                              rel_mse_denoise_alone=[round(v, 5) for v in alone], rel_mse_reproject_denoise=[round(v, 5) for v in temporal],
                              fraction_carried=carried, last_frame_ratio=round(alone[-1] / temporal[-1], 3))), flush=True)
        rows = []
        for mh, sz, mnd in itertools.product((4.0, 8.0, 16.0, 32.0), (0.02, 0.05, 0.2), (0.5, 0.9)):
            r = orbit_run(ctx, d, cams, refs, agpt.reproject_params(mh, sz, mnd), dp)
            rows.append((float(np.mean(r[FRAMES // 2:])), r[-1], mh, sz, mnd))
        rows.sort()
        print(json.dumps(dict(cfg=cfg, sweep_mean_last_8=[dict(rel_mse=round(r[0], 5), last=round(r[1], 5), max_history=r[2], sigma_depth=r[3],
                                                               min_normal_dot=r[4]) for r in rows])), flush=True)
        ctx.set_moments(False)
    # device time of the kernel (cfg 5 is resident), in a run of its own under torch.profiler
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.init()
        ctx.set_moments(True)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(10):
                ctx.set_camera(cams[i % 2]); ctx.render_guides(1); ctx.reproject_film(p0)
            torch.cuda.synchronize()
        per = {}
        for e in prof.events():
            for key in ("k_reproject_film<true>", "k_reproject_film<false>", "Memcpy DtoD"):
                if key in e.name:
                    per.setdefault(key, []).append(e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total)
        us = {k: round(float(np.median(v)), 2) for k, v in per.items()}
        k_us = us.get("k_reproject_film<true>")
        print(json.dumps(dict(cfg=5, width=W, height=H, kernel_us_median=us, launches={k: len(v) for k, v in per.items()},
                              kernel_gbs=None if not k_us else round(BYTES_PER_PIXEL * W * H / (k_us * 1e-6) / 1e9, 1))), flush=True)
        ctx.set_moments(False)
    except Exception as e:                                                     # the timings above stand on their own
        print(json.dumps(dict(profiler_error=str(e)[:200])), flush=True)
    print(json.dumps({"card": card()}), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
