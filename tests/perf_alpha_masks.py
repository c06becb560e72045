"""Perf probe (not a test) of alpha-masked cutout geometry.  Prints JSON lines, at 1920 x 1080 and 16 spp: ms per 16-spp render
(median of 5, host clock around calls that end in a device synchronise) and the trace kernels' device time per render
(AGPT_FLAG_TIMING, in a run of its own), for
  * cfg 3 and cfg 5 without masks and with an all-ones mask (a constant 1 at cutoff 0.5) on every material that may carry one:
    the film is bit-identical, the trace kernels are the MASK instantiations -- their overhead on unmasked content.  The two
    arms alternate three times in one run;
  * cfg 14 (the cutout scene): ms per 16 spp, Mrays/s, and the triangle tests of the closest-hit waves (agpt_get_wave_stats);
  * the same all-ones arms with the masked kernels built with a looser bound, AGPT_MASK_MIN_BLOCKS=8 (they spill under the trace
    kernels' (64, 16)): a copy of libagpt.so compiled into a temporary directory and run in a subprocess (AGPT_LIB);
and the card's name and power limit, read in the same run.

    python tests/perf_alpha_masks.py"""
import json
import os
import subprocess
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests.conftest import load_agpt  # noqa: E402
from tests.perf_denoise import card, timed  # noqa: E402
from tests.test_gpu_alpha_masks import bind_ones  # noqa: E402


def measure(agpt, ctx, d, label, extra=None):
    render = lambda: (ctx.clear(), ctx.render(0, 16, d["max_depth"], d["depth_arg"]), ctx.read_accum())
    ms = timed(render, 5)
    ctx.reset_stats(); ctx.clear()
    ctx.render(0, 16, d["max_depth"], d["depth_arg"], agpt.FLAG_TIMING)
    st = ctx.stats()
    row = {"workload": label, "ms_per_16spp": ms, "ms_trace_closest": round(float(st.ms_trace_closest), 3),
           "ms_trace_any": round(float(st.ms_trace_any), 3), "mrays_per_s": round(st.rays / (ms * 1e3), 1)}
    row.update(extra or {})
    print(json.dumps(row), flush=True)


def bound_arm():
    """The all-ones arms of cfg 3 and cfg 5 under this process's library (AGPT_LIB), labelled by AGPT_MASK_MIN_BLOCKS."""
    agpt = load_agpt()
    ctx = agpt.Context(0)
    for cfg in (3, 5):
        d = agpt.config_defaults(cfg)
        hs = agpt.HostScene(cfg, 0)
        for rep in range(3):
            hs.upload(ctx); ctx.set_film(1920, 1080)
            bind_ones(agpt, ctx, hs)
            measure(agpt, ctx, d, f"cfg{cfg} all-ones masks, AGPT_MASK_MIN_BLOCKS={os.environ['AGPT_MASK_MIN_BLOCKS']}", {"rep": rep})
    ctx.close()


def main():
    if len(sys.argv) > 1 and sys.argv[1] == "--bound-arm":
        return bound_arm()
    agpt = load_agpt()
    print(json.dumps({"card": card()}), flush=True)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with tempfile.TemporaryDirectory() as tmp:
        lib = os.path.join(tmp, "libagpt_mask8.so")
        pkg = os.path.join(root, "ag-pathtracer_b200")
        subprocess.check_call(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "--fmad=false", "-Xcompiler",
                               "-fPIC", "-I" + os.path.join(root, "include"), "-I" + os.path.join(pkg, "csrc"), "-DAGPT_MASK_MIN_BLOCKS=8", "-shared",
                               "-cudart", "static", "-o", lib, os.path.join(pkg, "csrc", "agpt_api.cu")])
        subprocess.check_call([sys.executable, os.path.abspath(__file__), "--bound-arm"],
                              env=dict(os.environ, AGPT_LIB=lib, AGPT_MASK_MIN_BLOCKS="8"))
    os.environ["AGPT_MASK_MIN_BLOCKS"] = "16"
    ctx = agpt.Context(0)
    for cfg in (3, 5):
        d = agpt.config_defaults(cfg)
        hs = agpt.HostScene(cfg, 0)
        for rep in range(3):
            hs.upload(ctx); ctx.set_film(1920, 1080)
            measure(agpt, ctx, d, f"cfg{cfg} no masks", {"rep": rep})
            bind_ones(agpt, ctx, hs)
            measure(agpt, ctx, d, f"cfg{cfg} all-ones masks (MASK kernels)", {"rep": rep})
    d = agpt.config_defaults(14)
    hs = agpt.HostScene(14, 1)
    hs.upload(ctx); ctx.set_film(1920, 1080)
    ctx.reset_stats(); ctx.clear()
    ctx.render(0, 16, d["max_depth"], d["depth_arg"], agpt.FLAG_COUNTERS)
    tri = sum(w["tri_tests"] for w in ctx.wave_stats(0))
    rays = sum(w["rays"] for w in ctx.wave_stats(0))
    measure(agpt, ctx, d, "cfg14 cutouts", {"closest_tri_tests_per_ray": round(tri / max(rays, 1), 2)})
    ctx.close()


if __name__ == "__main__":
    main()
