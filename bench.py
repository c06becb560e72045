#!/usr/bin/env python
"""bench.py -- throughput of the path-tracing hot path on N B200s of one node.

Contract (driver): `python bench.py --gpus N --steps K --warmup W` (N>1 under torchrun, one
rank per GPU) prints ONE JSON line from rank 0.

* workload  = BASELINE.json configs[2] -- the configuration the metric is quoted on ("1080p,
  8 bounces"): Disney multi-material scene, 1.31 M triangles in BVHTriMesh objects + 25
  analytic spheres + backdrop + floor, three sphere area lights + uniform sky, NEE + MIS,
  PathTracer(8), 1920x1080, 256 spp.  A STEP is one batch of `--spp-per-step` samples per
  pixel per GPU (default 64 = one full wavefront batch of 2^27 path slots at 1080p: four steps make the
  configuration's 256 spp on one GPU; bigger batches are fuller waves and more coherent ray buckets --
  16 / 32 / 64 spp per batch take 57.9 / 55.8 / 54.4 ms per 16 spp; `ms_per_16spp` keeps the figure of
  the earlier rounds comparable).  `--config
  {2,3,4,5}` times another BASELINE configuration instead; the default run also carries a
  short measurement of cfg 2, 4 and 5 in `other_configs` (cfg 4 = the multi-GPU configuration:
  at N > 1 a FIXED total of samples is split over the ranks -- strong scaling -- with the
  accumulator exchange and the resolve inside its timed region).
* value     = Mrays/s: rays actually traced by the GPU kernels (closest-hit path rays incl.
  skip-through, any-hit shadow rays, closest-hit MIS rays; counted by device atomics) summed
  over all ranks / device time of the timed region (CUDA events, max over ranks), scene and
  wavefront state resident in HBM.  At N > 1 the timed region ends with the exchange of the
  float4 accumulators (this library's peer-memory kernel over CUDA-IPC-mapped accumulators;
  `--reduce nccl` uses torch.distributed's NCCL all-reduce instead).
* e2e       = the same metric through the reference-facing API with HOST buffers: at N = 1
  CudaPathTracer::Render (ag-pathtracer_b200/host/integrator.h) -- film host->device, render,
  film device->host every step; at N > 1 the C-ABI calls a multi-process user makes: every rank
  uploads its host film and renders its share, the root sums and resolves all accumulators in
  one fused kernel and reads the final float film and the packed pixels back.
* roofline  = dominant kernel k_trace_closest: algorithmic bytes (64 B per interior visit +
  48 B per triangle test + 32 B per analytic record + 64 B per ray; SURVEY 8d, DESIGN.md)
  / its device time, against the measured HBM copy bandwidth in MEASURED_PEAKS.json; next to
  it the issue-side and L2-side figures that name the real limiter (per-ray instruction and
  sector counts come from the committed ncu capture of this same step, profiles/ncu_r2_step.json;
  rays, times, clocks and the L2 / HBM bandwidth probes are measured live).
* cpu_baseline = the reference's own CPU integrator (oracle/_ref, compiled from
  /root/reference) on all host cores and on one thread, on a bounded sample of the workload.

`--impl reference` times that CPU reference instead (rank 0 only); it does not load the product.
Inputs are larger than L2 (scene 215 MB + GBs of wavefront state vs 126 MB), so no L2 flush is
needed between timed iterations.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "Mrays/s (path+shadow+MIS rays traced, 1080p, 8 bounces)"

# BASELINE.json configurations as host/scenes/config_scenes.h defines them (the b200 arm checks this table
# against the library; the reference arm must not load the product, so it reads the table).
CONFIGS = {
    2: dict(name="cfg2_icosphere1p31M_direct_1080p_16spp", width=1920, height=1080, spp=16, max_depth=1, depth_arg=0, triangles=1310720),
    3: dict(name="cfg3_disney_multimaterial_1p31M_1080p_256spp_depth8", width=1920, height=1080, spp=256, max_depth=8, depth_arg=0, triangles=1310792),
    4: dict(name="cfg4_8xicosphere_10p5M_4k_1024spp_depth8", width=3840, height=2160, spp=1024, max_depth=8, depth_arg=0, triangles=10485760),
    5: dict(name="cfg5_closed_box_incoherent_1080p_depth16_rr", width=1920, height=1080, spp=64, max_depth=16, depth_arg=4, triangles=655372),
}


def bench_config(cfg, world, spp_step, level=0, width=0, height=0):
    """The `config` object of the JSON line -- identical in the b200 and the reference arm."""
    c = CONFIGS[cfg]
    return {"workload": c["name"], "width": width or c["width"], "height": height or c["height"], "max_depth": c["max_depth"],
            "rr_depth_arg": c["depth_arg"], "triangles": c["triangles"] if level == 0 else None, "spp_per_step_per_gpu": spp_step,
            "parallelism": f"sample-index split x{world}, one exchange of the float4 accumulators",
            "l2": "inputs larger than L2 (scene + wavefront state >> 126 MB); no flush needed"}


def load_pkg():
    import __graft_entry__ as ge
    return ge._load_pkg()


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(self.device)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for k, n in enumerate(names):
                if f[5 + k].lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_step_profile():
    """Per-ray instruction / sector / DRAM figures of the kernels of one bench step, from the committed ncu
    capture (profiles/ncu_r2_step.json, written by profiles/ncu_step_summary.py; capture command inside)."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_r2_step.json")) as f:
            return json.load(f)
    except Exception:
        return None


_REF_SCENES = {}


def cpu_reference_run(cfg, level, target_seconds, threads):
    """Time the reference's own CPU integrator (oracle/_ref) on a bounded sample of the
    workload: a centred crop of the film at 1 spp, grown until it costs ~target_seconds."""
    from oracle import ref_binding as ref
    if not ref.available():
        return None
    c = CONFIGS[cfg]
    W, H = c["width"], c["height"]
    key = (cfg, level)
    rs = _REF_SCENES.get(key)
    if rs is None:
        rs = _REF_SCENES[key] = ref.RefScene(cfg, level)      # BVH build excluded from the timing, as on the GPU side
        rs.count_rays()
    threads = threads or os.cpu_count() or 1

    def crop_run(cw, ch, spp):
        x0, y0 = (W - cw) // 2, (H - ch) // 2
        ref.ray_counts(reset=True)
        t0 = time.perf_counter()
        _, paths = rs.render(W, H, 0, spp, c["max_depth"], c["depth_arg"], threads=threads, crop=(x0, y0, x0 + cw, y0 + ch))
        dt = time.perf_counter() - t0
        rc = ref.ray_counts(reset=True)
        return paths, rc["closest"] + rc["any"], dt

    pw, ph = (320, 180) if threads > 1 else (96, 54)
    paths, rays, dt = crop_run(pw, ph, 1)                       # probe
    rate = paths / max(dt, 1e-6)
    want = max(int(rate * target_seconds), pw * ph)
    spp = 1
    frac = min(1.0, (want / (W * H)) ** 0.5)
    cw, ch = max(64, int(W * frac) // 16 * 16), max(36, int(H * frac) // 9 * 9)
    if want > W * H:
        spp = max(1, want // (W * H)); cw, ch = W, H
    paths, rays, dt = crop_run(cw, ch, spp)
    return dict(paths=paths, rays=rays, seconds=dt, cores=threads, sample=f"centred {cw}x{ch} crop of the {W}x{H} film, {spp} spp, all bounces")


def run_reference(args, rank, world, emit):
    if rank != 0:
        return
    cfg = args.config
    c = CONFIGS[cfg]
    W, H = c["width"], c["height"]
    steps, warm = args.steps, args.warmup
    # each step = a bounded sample; the whole run should end within a few minutes
    per_step = max(2.0, min(20.0, 150.0 / max(steps + warm, 1)))
    out = None
    try:
        runs = []
        for i in range(warm + steps):
            r = cpu_reference_run(cfg, args.level, per_step, args.cpu_threads)
            if r is None:
                break
            if i >= warm:
                runs.append(r)
        if runs:
            rays = sum(r["rays"] for r in runs); paths = sum(r["paths"] for r in runs); secs = sum(r["seconds"] for r in runs)
            value = rays / secs / 1e6
            out = {"impl": "reference", "metric": METRIC, "value": value, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": steps, "warmup": warm,
                   "ms_per_step": secs / len(runs) * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                   "data": "synthetic", "config": bench_config(cfg, args.gpus, args.spp_per_step, args.level),
                   "step_sample": runs[-1]["sample"],
                   "spp_per_s": paths / secs / (W * H), "Mpaths_per_s": paths / secs / 1e6,
                   "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": runs[-1]["cores"], "kind": "reference", "sample": runs[-1]["sample"]},
                   "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    except Exception as e:  # the oracle always exists in a built tree; say why if not
        out = {"impl": "reference", "unavailable": f"{type(e).__name__}: {e}"}
    if out is None:
        out = {"impl": "reference", "unavailable": "oracle/_ref/libagpt_ref.so not built (needs /root/reference at build time)"}
    emit(out)


class _DevMem:
    """A device allocation of the library as a __cuda_array_interface__ object (torch.as_tensor aliases it)."""

    def __init__(self, ptr, shape):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<f4", "data": (int(ptr), False), "version": 3, "strides": None}


def per_bounce_table(ctx, kind=0, limit=20):
    rows = []
    for w, r in enumerate(ctx.wave_stats(kind)[:limit]):
        if r["rays"] == 0:
            continue
        rows.append({"wave": w, "rays": r["rays"], "N_int": round(r["node_visits"] / r["rays"], 2), "N_tri": round(r["tri_tests"] / r["rays"], 2),
                     "N_analytic": round(r["analytic_tests"] / r["rays"], 2),
                     "rays_alive_per_walk_step_of_32": round(r["lane_steps"] / max(r["warp_steps"], 1), 2)})
    return rows


DUMP_BYTES = 63 << 20          # the dump stays under 64 MB, .npy headers included


def dump_outputs(dirname, film):
    """The float4 film [H, W, 4] the timed steps summed into, as the caller reads it back, as accum.npy.  A film larger
    than DUMP_BYTES (cfg 4 at 4K) is cut to a fixed, seeded sample of its pixels: accum.npy [n, 4] holds them in
    ascending order and accum_pixel_index.npy [n] their row-major indices into the film (float64, exact)."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    if film.nbytes > DUMP_BYTES:
        flat = film.reshape(-1, 4)
        n = DUMP_BYTES // (flat[0].nbytes + 8)
        keep = np.sort(np.random.default_rng(0).choice(len(flat), n, replace=False))
        film = flat[keep]
        np.save(os.path.join(dirname, "accum_pixel_index.npy"), keep.astype(np.float64))
    np.save(os.path.join(dirname, "accum.npy"), np.ascontiguousarray(film, np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=3, choices=[2, 3, 4, 5], help="BASELINE.json configuration to time (default 3: the one the metric is quoted on)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: every GPU renders --spp-per-step samples per step; strong: --spp-per-step samples per step in TOTAL, split over the GPUs")
    ap.add_argument("--reduce", default="peer", choices=["peer", "nccl"], help="accumulator exchange at N > 1: this library's peer-memory kernel, or torch.distributed NCCL")
    ap.add_argument("--spp-per-step", type=int, default=64)
    ap.add_argument("--level", type=int, default=0, help="icosphere subdivision override (tests); 0 = the configuration's own")
    ap.add_argument("--width", type=int, default=0)
    ap.add_argument("--height", type=int, default=0)
    ap.add_argument("--cpu-seconds", type=float, default=20.0)
    ap.add_argument("--cpu-threads", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the film they accumulated (rank 0, after the exchange) as DIR/accum.npy")
    args = ap.parse_args()

    # stdout carries exactly one JSON line: park fd 1 on stderr until then (NCCL / libraries may print)
    saved_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(obj), flush=True)
        os.dup2(2, 1)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world, emit)
        return

    import torch
    import torch.distributed as dist
    import numpy as np

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 path has no CPU fallback (use --impl reference for the CPU reference)")
    torch.cuda.set_device(local_rank)
    dev = f"cuda:{local_rank}"
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"          # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    pkg = load_pkg()
    CFG = args.config
    defaults = pkg.config_defaults(CFG)
    tab = CONFIGS[CFG]
    assert (defaults["name"], defaults["width"], defaults["height"], defaults["max_depth"], defaults["depth_arg"]) == \
        (tab["name"], tab["width"], tab["height"], tab["max_depth"], tab["depth_arg"]), "bench.py CONFIGS is out of step with config_scenes.h"
    W = args.width or defaults["width"]; H = args.height or defaults["height"]
    depth, depth_arg = defaults["max_depth"], defaults["depth_arg"]
    spp_step = args.spp_per_step
    strong = args.scaling == "strong"
    spp_all = spp_step if strong else spp_step * world        # samples per step over all ranks

    stream = torch.cuda.Stream(device=local_rank)     # kernels, events and NCCL all on this one stream
    torch.cuda.set_stream(stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def gather_handles(ctx):
        h = torch.tensor(list(ctx.accum_ipc_handle()), dtype=torch.uint8, device=dev)
        allh = [torch.empty_like(h) for _ in range(world)]
        dist.all_gather(allh, h)
        return [bytes(t.cpu().tolist()) for t in allh]

    def make_context(scene, w, h):
        """Context of this rank with the scene resident, the film set and (N > 1) the peers' accumulators mapped."""
        ctx = pkg.Context(local_rank)
        ctx.set_stream(stream.cuda_stream)
        scene.upload(ctx)
        ctx.set_film(w, h)
        ctx.clear()
        torch.cuda.synchronize()
        route = "single GPU"
        accum_t = None
        if world > 1:
            accum_t = torch.as_tensor(_DevMem(ctx.accum_ptr(), (h, w, 4)), device=dev)     # the same memory, for the NCCL route
            route = "nccl (torch.distributed all_reduce)"
            if args.reduce == "peer":
                ok = torch.ones(1, device=dev)
                try:
                    ctx.open_peer_accums(rank, gather_handles(ctx))
                except Exception as e:
                    print(f"[bench] rank {rank}: CUDA IPC peer mapping failed ({e}); using NCCL", file=sys.stderr)
                    ok.zero_()
                dist.all_reduce(ok, op=dist.ReduceOp.MIN)
                if ok.item() > 0:
                    route = "peer-memory kernel over CUDA-IPC-mapped accumulators (rank-order sums)"
        return ctx, accum_t, route

    _token = torch.zeros(1, device=dev) if world > 1 else None

    def light_barrier(sync=True):
        """One 4-byte NCCL all-reduce on the bench stream: kernels enqueued behind it start only after every rank has
        reached it (dist.barrier() costs ~2 ms per call at N = 8 here; this costs a small-message all-reduce)."""
        dist.all_reduce(_token)
        if sync:
            stream.synchronize()

    def exchange(ctx, accum_t, route):
        """Sum of all ranks' accumulators into every rank's (inside timed regions)."""
        if world == 1:
            return
        if route.startswith("peer"):
            light_barrier(sync=False)           # every rank has rendered (agpt_render returns synchronised): the kernel below queues behind it
            ctx.allreduce_accum_peers()
            light_barrier()                     # every slice has landed everywhere
        else:
            dist.all_reduce(accum_t, op=dist.ReduceOp.SUM)

    def close_context(ctx):
        if world > 1:
            barrier()
            try:
                ctx.close_peer_accums()
            except Exception:
                pass
            barrier()
        ctx.close()

    # ------------------------------------------------------------------------------------------
    # main workload
    # ------------------------------------------------------------------------------------------
    scene = pkg.HostScene(CFG, args.level)
    counts = scene.counts()
    if args.level == 0:
        assert counts["tris"] == tab["triangles"], f"bench.py CONFIGS triangles {tab['triangles']} != scene {counts['tris']}"
    ctx, accum_t, route = make_context(scene, W, H)

    def step(k, flags=0):
        # samples are split by index across ranks: rank g renders s = g (mod world)
        pkg.multigpu.render_sharded(ctx, k * spp_all, spp_all, depth, depth_arg, rank, world, flags)

    for k in range(args.warmup):
        step(k)
    exchange(ctx, accum_t, route)                         # warm-up of the collective too
    ctx.clear()
    ctx.reset_stats()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    ev0, ev1, ev2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    ev0.record(stream)
    for k in range(args.steps):
        step(args.warmup + k)
    ev1.record(stream)
    exchange(ctx, accum_t, route)                         # float4[W*H] accumulators -> final framebuffer (NVLink)
    ev2.record(stream)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms = ev0.elapsed_time(ev2)
    ms_exchange = ev1.elapsed_time(ev2)
    st = ctx.stats()
    t = torch.tensor([ms, ms_exchange], dtype=torch.float64, device=dev)
    tot = torch.tensor([float(st.rays), float(st.paths), float(st.kernel_launches), float(st.rays_reference_equivalent),
                        float(st.rays_closest), float(st.rays_shadow), float(st.rays_mis), float(st.rays_mis_culled), float(st.rays_tail_culled)],
                       dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms_max, ms_exchange = [float(v) for v in t.tolist()]
    rays, paths, launches, rays_ref_eq, r_closest, r_shadow, r_mis, r_mis_culled, r_tail_culled = [float(v) for v in tot.tolist()]
    value = rays / ms_max / 1e3
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ctx.read_accum())

    # ---- N > 1: is the N-GPU frame the 1-GPU frame?  (outside the timed region; SURVEY 8e: max rel diff <= 1e-5)
    multi_gpu_check = None
    collective = None
    if world > 1:
        check_spp = max(world, 8)
        ctx.clear()
        pkg.multigpu.render_sharded(ctx, 0, check_spp, depth, depth_arg, rank, world)
        exchange(ctx, accum_t, route)
        barrier()
        film_n = ctx.read_accum() if rank == 0 else None
        barrier()
        if rank == 0:
            ctx.clear()
            ctx.render(0, check_spp, depth, depth_arg)
            film_1 = ctx.read_accum()
            rel = float(np.max(np.abs(film_n - film_1) / np.maximum(np.abs(film_1), 1e-3)))
            multi_gpu_check = {"max_rel_diff": rel, "ok": bool(rel <= 1e-5), "tolerance": 1e-5, "samples": check_spp,
                               "what": f"{world}-rank sharded render + accumulator exchange vs rank 0 rendering the same samples alone, whole {W}x{H} film"}
        barrier()
        # both routes of the exchange, timed alone (3 repetitions after one warm-up; film contents are irrelevant)
        collective = {"bytes": W * H * 16, "used_in_timed_region": route}
        for name, r in (("peer_kernel_ms", "peer"), ("nccl_ms", "nccl")):
            if r == "peer" and not route.startswith("peer"):
                continue
            times = []
            for rep in range(4):
                barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                exchange(ctx, accum_t, "peer" if r == "peer" else "nccl")
                e1.record(stream)
                barrier()
                tt = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                if rep > 0:
                    times.append(float(tt.item()))
            collective[name] = min(times)
        collective["ms_in_timed_region"] = ms_exchange

    # ---- end-to-end through the reference-facing API (host buffers in and out) -------
    host_acc, _film_owner = pkg.pinned_film(W, H)          # page-locked host film, as the host mirror's Accumulator allocates it
    e2e_steps = max(1, min(args.steps, 3))
    if world == 1:
        tracer = pkg.HostTracer(depth, local_rank)
        tracer.render(scene, W, H, host_acc, 0, spp_step, depth_arg)      # uploads the scene, sizes the wavefront state, warms up
        tracer.stats(reset=True)
        barrier()
        t0 = time.perf_counter()
        for k in range(e2e_steps):
            tracer.render(scene, W, H, host_acc, (1 + k) * spp_step, spp_step, depth_arg)
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        e2e_rays = float(tracer.stats().rays)
        tracer.close()
        e2e_api = "CudaPathTracer::Render over host Accumulator buffers"
        h2d, d2h = W * H * 16 + 76, W * H * 16
    else:
        rgb = None
        ctx.reset_stats()
        barrier()
        t0 = time.perf_counter()
        for k in range(e2e_steps):
            ctx.write_accum_begin(host_acc)                             # every rank: its host film -> device, beside the render below
            pkg.multigpu.render_sharded(ctx, (1 + k) * spp_all, spp_all, depth, depth_arg, rank, world)
            if route.startswith("peer"):
                light_barrier(sync=False)
                if rank == 0:
                    rgb = ctx.reduce_resolve_peers((1 + k) * spp_all, keep_sum=True)      # fused sum + CopyToSurface -> host pixels
                    ctx.read_accum(host_acc)                            # the summed float film -> host
                light_barrier()
            else:
                dist.all_reduce(accum_t, op=dist.ReduceOp.SUM)
                if rank == 0:
                    rgb = ctx.resolve((1 + k) * spp_all)
                    ctx.read_accum(host_acc)
        torch.cuda.synchronize()
        barrier()
        e2e_s = time.perf_counter() - t0
        e2e_rays = float(ctx.stats().rays)
        e2e_api = "C ABI, one process per GPU: agpt_write_accum_begin + agpt_render(stride N) on every rank, agpt_reduce_resolve_peers + agpt_read_accum on the root"
        h2d, d2h = world * W * H * 16, W * H * 16 + W * H * 4
    e2e_t = torch.tensor([e2e_s, e2e_rays], dtype=torch.float64, device=dev)
    if world > 1:
        tmax = e2e_t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(e2e_t, op=dist.ReduceOp.SUM)
        e2e_s, e2e_rays = float(tmax[0].item()), float(e2e_t[1].item())
    e2e_value = e2e_rays / e2e_s / 1e6

    # ---- roofline of the dominant kernel + counters (rank 0, extra untimed steps) --------
    roofline = roofline_issue = l2_side = breakdown = per_bounce = counting_step = None
    ref_eq_ratio = rays_ref_eq / max(rays, 1.0)
    if rank == 0:
        ctx.clear()
        ctx.reset_stats()
        step(args.warmup + args.steps, pkg.FLAG_TIMING)
        tm = ctx.stats()
        ctx.reset_stats()
        step(args.warmup + args.steps, pkg.FLAG_COUNTERS)
        cn = ctx.stats()
        ref_eq_ratio = cn.rays_reference_equivalent / max(cn.rays, 1)
        counting_step = {"traced": float(cn.rays), "mis_culled_exactly": float(cn.rays_mis_culled), "tail_culled_exactly": float(cn.rays_tail_culled),
                         "reference_equivalent": float(cn.rays_reference_equivalent)}
        per_bounce = per_bounce_table(ctx, 0)
        peak, peak_src = measured_peak_gbs()
        l2_gbs = ctx.probe_bandwidth(32 << 20, 200)            # 32 MB, L2-resident: what a streaming read gets out of L2
        hbm_read_gbs = ctx.probe_bandwidth(8 << 30, 2)         # 8 GB: HBM read side
        bytes_closest = cn.algorithmic_bytes(0)
        secs_closest = tm.ms_trace_closest * 1e-3
        achieved = bytes_closest / secs_closest / 1e9
        rays_closest = cn.rays_closest + cn.rays_mis
        prof = ncu_step_profile()
        pk = (prof or {}).get("kernels", {}).get("k_trace_closest")
        sm_clock_hz = (clocks.get("sm_mhz") or 1965.0) * 1e6
        sms = torch.cuda.get_device_properties(local_rank).multi_processor_count
        roofline = {"bound": "hbm", "kernel": "k_trace_closest", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": (pk["dram_bytes_per_ray"] * rays_closest / max(cn.launches_closest, 1)) if pk else None,
                    "traffic_source": (prof or {}).get("source"),
                    "limiter": "instruction issue at a fraction of 32 threads per instruction + dependent-load latency (see roofline_issue, l2); "
                               "the HBM figure is the contractual algorithmic-bytes roofline -- L1/L2 absorb most of those bytes",
                    "peak_source": peak_src, "launches_per_step": tm.launches_closest,
                    "avg_launch_ms": tm.ms_trace_closest / max(tm.launches_closest, 1),
                    "algorithmic_bytes_per_launch": bytes_closest / max(cn.launches_closest, 1),
                    "bytes_per_ray": bytes_closest / max(rays_closest, 1),
                    "interior_visits_per_ray": cn.node_visits[0] / max(rays_closest, 1),
                    "tri_tests_per_ray": cn.tri_tests[0] / max(rays_closest, 1),
                    "analytic_tests_per_ray": cn.analytic_tests[0] / max(rays_closest, 1),
                    "rays_alive_per_walk_step_of_32": cn.lane_steps[0] / max(cn.warp_steps[0], 1),
                    "hbm_read_probe_gbs": hbm_read_gbs}
        if pk:
            inst_s = pk["warp_inst_per_ray"] * rays_closest / secs_closest
            issue_peak = sms * 4 * sm_clock_hz
            roofline_issue = {"kernel": "k_trace_closest", "warp_inst_per_ray": pk["warp_inst_per_ray"], "threads_per_inst": pk["threads_per_inst"],
                              "achieved_warp_inst_per_s": inst_s, "peak_warp_inst_per_s": issue_peak, "frac": inst_s / issue_peak,
                              "lane_frac": inst_s / issue_peak * pk["threads_per_inst"] / 32.0,
                              "peak": f"{sms} SMs x 4 schedulers x 1 warp instruction / clock at the SM clock sampled in the timed region ({sm_clock_hz / 1e6:.0f} MHz)",
                              "source": "instruction counts per ray: " + str((prof or {}).get("source")) + "; rays, kernel time and clock: this run"}
            l2_bytes_s = pk["l2_bytes_per_ray"] * rays_closest / secs_closest
            l2_side = {"kernel": "k_trace_closest", "l2_bytes_per_ray": pk["l2_bytes_per_ray"], "achieved_gbs": l2_bytes_s / 1e9, "peak_gbs": l2_gbs,
                       "frac": l2_bytes_s / 1e9 / l2_gbs if l2_gbs else None, "l1_hit_pct": pk.get("l1_hit_pct"), "l2_hit_pct": pk.get("l2_hit_pct"),
                       "peak_source": "agpt_probe_bandwidth: 32 MB read 200 times by a persistent grid with 128-bit ld.global.cg (this run)"}
        breakdown = {"ms_step": tm.ms_render, "ms_trace_closest": tm.ms_trace_closest, "ms_trace_any": tm.ms_trace_any, "ms_shade": tm.ms_shade,
                     "ms_other": tm.ms_other, "waves": tm.waves, "rays_per_path": cn.rays / max(cn.paths, 1)}
    barrier()
    close_context(ctx)
    del scene

    # ---- the other BASELINE configurations, briefly (driver-visible) ---------------------------
    other = None
    if not args.no_other_configs and CFG == 3 and args.level == 0:
        other = {}
        for oc in (2, 5, 4):
            multi = oc == 4 and world > 1
            if rank != 0 and not multi:
                barrier(); barrier()
                continue
            od = CONFIGS[oc]
            t0 = time.perf_counter()
            osc = pkg.HostScene(oc, 0)
            build_s = time.perf_counter() - t0
            barrier()
            if multi:
                octx, oacc, oroute = make_context(osc, od["width"], od["height"])
            else:
                octx = pkg.Context(local_rank); octx.set_stream(stream.cuda_stream); osc.upload(octx); octx.set_film(od["width"], od["height"]); octx.clear()
                oroute = "single GPU"
            # one frame = a FIXED number of samples per pixel in total (strong scaling at N > 1).  cfg 4 (4K): 128 = 16 per rank at
            # N = 8, i.e. one full wavefront batch of 2^27 paths per GPU and an eighth of the configuration's 1024 spp; cfg 2 / 5: 64
            total_spp = 128 if oc == 4 else 64
            nranks = world if multi else 1
            me = rank if multi else 0

            def orender(first, flags=0):
                pkg.multigpu.render_sharded(octx, first, total_spp, od["max_depth"], od["depth_arg"], me, nranks, flags)

            def end_of_frame(samples):
                # sum of the accumulators (N > 1) + CopyToSurface, pixels on the root's host
                if multi:
                    if oroute.startswith("peer"):
                        light_barrier(sync=False)
                        out = octx.reduce_resolve_peers(samples) if rank == 0 else None
                        light_barrier()
                        return out
                    dist.all_reduce(oacc, op=dist.ReduceOp.SUM)
                    return octx.resolve(samples) if rank == 0 else None
                return octx.resolve(samples)

            orender(0)                                          # warm-up of the render and of the end of frame
            end_of_frame(total_spp)
            octx.clear(); octx.reset_stats()
            torch.cuda.synchronize()
            if multi:
                dist.barrier()
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            reps = 2
            e0.record(stream)
            for k in range(reps):
                orender((1 + k) * total_spp)
            e1.record(stream)
            rgb = end_of_frame(reps * total_spp)
            e2.record(stream)
            torch.cuda.synchronize()
            ost = octx.stats()
            v = torch.tensor([e0.elapsed_time(e2), e1.elapsed_time(e2)], dtype=torch.float64, device=dev)
            s = torch.tensor([float(ost.rays), float(ost.paths)], dtype=torch.float64, device=dev)
            if multi:
                dist.all_reduce(v, op=dist.ReduceOp.MAX); dist.all_reduce(s, op=dist.ReduceOp.SUM)
            oms, oms_end = [float(x) for x in v.tolist()]
            orays, opaths = [float(x) for x in s.tolist()]
            entry = {"workload": od["name"], "width": od["width"], "height": od["height"], "max_depth": od["max_depth"], "triangles": osc.counts()["tris"],
                     "scaling": "strong" if multi else "single GPU", "n_gpus": nranks, "total_spp_per_frame": total_spp, "frames": reps,
                     "ms_render_per_frame": (oms - oms_end) / reps, "end_of_frame_ms": oms_end, "ms_timed_region": oms,
                     "Mrays_per_s": orays / oms / 1e3, "spp_per_s": opaths / (od["width"] * od["height"]) / (oms * 1e-3),
                     "rays_per_path": orays / max(opaths, 1),
                     "end_of_frame": ("accumulator sum + resolve over " + oroute) if multi else "resolve",
                     "host_bvh_build_s": build_s, "scene_bytes": osc.counts()["bytes"]}
            if rank == 0 and oc == 5:
                octx.reset_stats()
                pkg.multigpu.render_sharded(octx, 0, 4, od["max_depth"], od["depth_arg"], 0, 1, pkg.FLAG_COUNTERS)
                c5 = octx.stats()
                entry["per_bounce_closest_hit"] = per_bounce_table(octx, 0)
                entry["per_bounce_any_hit"] = per_bounce_table(octx, 1)
                entry["rays_alive_per_walk_step_of_32"] = c5.lane_steps[0] / max(c5.warp_steps[0], 1)
            if rank == 0:
                other[f"cfg{oc}"] = entry
            if multi:
                close_context(octx)
            else:
                octx.close()
            del osc
            barrier()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            r = cpu_reference_run(CFG, args.level, args.cpu_seconds, args.cpu_threads)
            if r:
                cpu = {"value": r["rays"] / r["seconds"] / 1e6, "unit": "Mrays/s", "cores": r["cores"], "kind": "reference", "sample": r["sample"],
                       "Mpaths_per_s": r["paths"] / r["seconds"] / 1e6, "seconds": r["seconds"]}
                r1 = cpu_reference_run(CFG, args.level, max(4.0, args.cpu_seconds / 2), 1)          # the reference's actual mode: one thread
                cpu["single_thread"] = {"value": r1["rays"] / r1["seconds"] / 1e6, "unit": "Mrays/s", "cores": 1, "sample": r1["sample"],
                                        "Mpaths_per_s": r1["paths"] / r1["seconds"] / 1e6, "seconds": r1["seconds"]}
        except Exception as e:
            cpu = {"value": None, "unit": "Mrays/s", "cores": 0, "kind": "reference", "sample": f"failed: {e}"}

    if rank == 0:
        cfg_obj = bench_config(CFG, world, spp_step, args.level, args.width, args.height)
        out = {"metric": METRIC, "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": ms_max / args.steps, "ms_per_16spp": ms_max / args.steps * 16.0 / spp_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32",
               "data": "synthetic", "config": cfg_obj,
               "scene": {"bvh_nodes": counts["nodes"], "primitives": counts["prims"], "lights": counts["lights"], "scene_bytes": counts["bytes"]},
               "spp_per_s": paths / (W * H) / (ms_max * 1e-3), "Mpaths_per_s": paths / ms_max / 1e3,
               # value counts rays actually traced through the scene.  The reference also traces rays whose
               # outcome cannot matter (MIS rays that miss their light's sphere, the discarded ray at MaxDepth);
               # the B200 path proves them useless and skips them, so spp/s is the like-for-like speed and
               # ref_equivalent_Mrays_per_s is the throughput in the reference's own ray accounting.
               # (The culled counts are exact only in a counting render -- agpt.h, rays_mis_culled -- so the ratio reference rays /
               # traced rays comes from the untimed AGPT_FLAG_COUNTERS step of this same workload and scales the measured value.)
               "ref_equivalent_Mrays_per_s": value * ref_eq_ratio,
               "rays": {"closest_path": r_closest, "shadow": r_shadow, "mis_traced": r_mis, "mis_not_traced_upper_bound": r_mis_culled,
                        "tail_culled_exactly": r_tail_culled, "counting_step": counting_step},
               "clocks": clocks,
               "e2e": {"value": e2e_value, "unit": "Mrays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                       "api": e2e_api, "steps": e2e_steps, "rays_counted": e2e_rays, "seconds": e2e_s},
               "gpu_launches": int(launches),
               "roofline": roofline, "roofline_issue": roofline_issue, "l2": l2_side, "breakdown": breakdown, "per_bounce_closest_hit": per_bounce,
               "multi_gpu_check": multi_gpu_check, "collective": collective, "other_configs": other, "cpu_baseline": cpu}
        emit(out)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
