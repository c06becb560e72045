"""Perf probe (not a test) of emissive materials.  Prints JSON lines, at 1920 x 1080 and 16 spp: ms per 16-spp render (median of
5, host clock around calls that end in a device synchronise), Mrays/s, the closest-hit trace and shade device time per render
(AGPT_FLAG_TIMING, a run of its own) and the device time of k_shade_a / k_shade_a_emit per render (torch.profiler, a run of its
own), for
  * cfg 3 and cfg 5, plain and with "an emitter nobody sees" (one extra material with factor (1, 1, 1) that no primitive uses):
    the film is bit-identical, but k_shade_a_emit runs and the tail rays are traced -- the whole cost of the feature on content
    without emission.  The two arms alternate three times in one run;
  * cfg 15 levels 1 and 2 (the emissive scene, with a light and without);
and the card's name, power limit and max SM clock, read in the same run.

    python tests/perf_emission.py"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests.conftest import load_agpt  # noqa: E402
from tests.perf_denoise import card, timed  # noqa: E402
from tests.test_gpu_emission import unseen_emitter  # noqa: E402


def shade_a_ms(ctx, d):
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.init()
        ctx.clear()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ctx.render(0, 16, d["max_depth"], d["depth_arg"])
            torch.cuda.synchronize()
        us = sum(e.device_time_total for e in prof.key_averages() if "k_shade_a" in e.key)
        return round(us / 1e3, 3)
    except Exception as e:          # the rest of the row stands without it
        return "profiler error: " + str(e)[:120]


def measure(agpt, ctx, d, label, extra=None):
    render = lambda: (ctx.clear(), ctx.render(0, 16, d["max_depth"], d["depth_arg"]), ctx.read_accum())
    ms = timed(render, 5)
    ctx.reset_stats(); ctx.clear()
    ctx.render(0, 16, d["max_depth"], d["depth_arg"], agpt.FLAG_TIMING)
    st = ctx.stats()
    row = {"workload": label, "ms_per_16spp": ms, "mrays_per_s": round(st.rays / (ms * 1e3), 1),
           "ms_trace_closest": round(float(st.ms_trace_closest), 3), "ms_shade": round(float(st.ms_shade), 3),
           "rays_closest": st.rays_closest, "rays_tail_culled": st.rays_tail_culled, "ms_k_shade_a": shade_a_ms(ctx, d)}
    row.update(extra or {})
    print(json.dumps(row), flush=True)


def main():
    agpt = load_agpt()
    print(json.dumps({"card": card()}), flush=True)
    ctx = agpt.Context(0)
    for cfg in (3, 5):
        d = agpt.config_defaults(cfg)
        hs = agpt.HostScene(cfg, 0)
        for rep in range(3):
            hs.upload(ctx); ctx.set_film(1920, 1080)
            measure(agpt, ctx, d, f"cfg{cfg} plain", {"rep": rep})
            unseen_emitter(agpt, ctx, hs)
            measure(agpt, ctx, d, f"cfg{cfg} emitter nobody sees (k_shade_a_emit, tails traced)", {"rep": rep})
    d = agpt.config_defaults(15)
    for level in (1, 2):
        hs = agpt.HostScene(15, level)
        hs.upload(ctx); ctx.set_film(1920, 1080)
        measure(agpt, ctx, d, f"cfg15 level {level}")
    print(json.dumps({"card": card()}), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
