"""Perf probe (not a test) of sampled plane / mesh area lights: cfg 11 (AGPT_LIGHT_SAMPLE_SHAPE on a 2-triangle panel, a
plane panel and a level-2 BVH icosphere) at 1080p.  Prints JSON lines: ms per 16 spp and Mrays/s of a 64-spp render, the
per-kernel split of the same render with AGPT_FLAG_TIMING, and the card's name and power limit read in the same run.

    python tests/perf_shape_lights.py [spp=64] [reps=3]"""
import json
import subprocess
import sys
import os

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests.conftest import load_agpt  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    spp = int(sys.argv[1]) if len(sys.argv) > 1 else 64
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    agpt = load_agpt()
    d = agpt.config_defaults(11)
    print(json.dumps({"card": card()}), flush=True)
    ctx = agpt.Context(0)
    hs = agpt.HostScene(11, 0)
    hs.upload(ctx)
    ctx.set_film(d["width"], d["height"])
    ctx.render(0, 16, d["max_depth"], d["depth_arg"])          # warm-up: module load, tables, bucket grid
    for flags in [0] * reps + [agpt.FLAG_TIMING]:
        ctx.clear(); ctx.reset_stats()
        ctx.render(0, spp, d["max_depth"], d["depth_arg"], flags)
        s = ctx.stats()
        out = dict(cfg=11, width=d["width"], height=d["height"], spp=spp, timing=bool(flags), ms=round(s.ms_render, 2),
                   ms_per_16spp=round(s.ms_render * 16 / spp, 2), Mrays_s=round(s.rays / s.ms_render / 1e3, 1),
                   rays_per_path=round(s.rays / s.paths, 3), closest=s.rays_closest, shadow=s.rays_shadow, mis=s.rays_mis, mis_culled=s.rays_mis_culled)
        if flags:
            out.update(ms_trace_closest=round(s.ms_trace_closest, 2), ms_trace_any=round(s.ms_trace_any, 2), ms_shade=round(s.ms_shade, 2),
                       ms_other=round(s.ms_other, 2))
        print(json.dumps(out), flush=True)
    # the same scene without the flag (the reference's behaviour: the lights are not sampled) for scale
    t = __import__("oracle.port_binding", fromlist=["_Tables"])._Tables.from_buffer(hs.tables())
    import ctypes
    import numpy as np
    lights = np.frombuffer((ctypes.c_char * (agpt.LIGHT_DTYPE.itemsize * t.n_lights)).from_address(t.lights), agpt.LIGHT_DTYPE)
    lights["ext"]["flags"] = 0
    hs.upload(ctx)
    ctx.render(0, 16, d["max_depth"], d["depth_arg"])
    for flags in [0, agpt.FLAG_TIMING]:
        ctx.clear(); ctx.reset_stats()
        ctx.render(0, spp, d["max_depth"], d["depth_arg"], flags)
        s = ctx.stats()
        out = dict(cfg=11, unsampled=True, timing=bool(flags), ms=round(s.ms_render, 2), ms_per_16spp=round(s.ms_render * 16 / spp, 2),
                   Mrays_s=round(s.rays / s.ms_render / 1e3, 1))
        if flags:
            out.update(ms_trace_closest=round(s.ms_trace_closest, 2), ms_trace_any=round(s.ms_trace_any, 2), ms_shade=round(s.ms_shade, 2))
        print(json.dumps(out), flush=True)
    print(json.dumps({"card": card()}), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
