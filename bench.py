#!/usr/bin/env python
"""bench.py — path segments/sec of the B200-native ray_color bounce loop (see BASELINE.json / BASELINE.md).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload C1|C2|C3|C4|C5] [--impl reference] [--dump-outputs DIR]

One "step" = one full render of the workload (every pixel, `spp` samples) on each rank.  N > 1 is launched by
torchrun (one process per GPU): rank r renders global samples [r*spp, (r+1)*spp) of every pixel (WEAK scaling: per-GPU
work fixed), the float4 accumulation buffers are summed onto rank 0 by the LIBRARY (rtb_render_device with
RTB_RENDER_REDUCE: one ncclReduce per frame on a communicator the ranks join through rtb_context_comm_init; torch only
carries the 128-byte id), rank 0 finalises.
`value` = segments traced by all ranks / max-over-ranks device time of the K steps, scene resident in HBM.
`strong_scaling` (sub-record, every N): BASELINE.json's scaling config C5 — the book-2 final scene at 3840x2160, a FIXED
total spp (--strong-spp, stated) SPLIT across the ranks, 133 MB reduce — so the per-N lines give a strong-scaling curve.
`e2e`   = the same through the host-facing C ABI: scene records handed over from host memory (flatten + BVH build +
          H2D), render, reduce, D2H of the accumulation buffer — every step.
`--impl reference` times the reference's CPU algorithm (the f64 oracle port: the Rust reference cannot be compiled in
this image) on all host cores, on a bounded sample (1 spp at full resolution per step) of the same workload.
`--dump-outputs DIR` writes what the last timed step computed (rank 0's accumulation buffer and its path counters) as
.npy files, so that two builds can be compared output for output on the same seeded workload.
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

# SURVEY §8d constants: algorithmic bytes / FP32 flops per BVH8 node visit and per primitive test
B_NODE, F_NODE = 80, 280
B_PRIM = {"sphere": 16, "moving": 32, "quad": 48, "tri": 48}
F_PRIM = {"sphere": 30, "moving": 38, "quad": 60, "tri": 48}


def get_config(name, spp=None):
    from ray_tracer_archive_b200 import scenes
    mk = {"C1": scenes.config_random_spheres, "C2": scenes.config_cornell, "C3": scenes.config_final_scene,
          "C4": scenes.config_mesh, "C5": scenes.config_scaling}[name]
    cfg = mk()
    if spp:
        cfg.spp = spp
    return cfg


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        import statistics
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows), "window": "warm-up + timed + e2e steps"}


def measure_bandwidths(ctx, F):
    """Physical denominators, measured in this run by the library's own microbenchmark (rtb_measure_bandwidth): read-only
    128-bit ld.global.nc streams over a 48 MB L2-resident buffer and a 2 GB HBM-resident one, and 128-bit shared-memory
    loads on all SMs.  MEASURED_PEAKS.json has no L2 / shared-memory figure (SURVEY §8d asks the builder to measure one)."""
    return {"l2_read_gbs": ctx.measure_bandwidth(F.BW_L2_READ), "hbm_read_gbs": ctx.measure_bandwidth(F.BW_HBM_READ),
            "shared_read_gbs": ctx.measure_bandwidth(F.BW_SHARED_READ)}


def bounded_cpu_sample(osc, rtb, cfg, cores, budget_s=12.0):
    """Times the oracle (the reference's CPU algorithm) on a bounded sample of the workload: a probe render at 1/16
    resolution calibrates the rate, then full resolution with as many spp as fit the budget, or a reduced resolution at
    1 spp when even that does not fit (the 1M-triangle linear scan).  Rate in segments/s is spp- and
    resolution-independent to first order; the sample is stated in the JSON."""
    pw, ph = max(cfg.width // 16, 8), max(cfg.height // 16, 8)
    prm = rtb.make_params(pw, ph, 1, cfg.max_depth, cfg.background, seed=1)
    t0 = time.perf_counter()
    osc.render(cfg.camera, prm, threads=cores)
    dt = max(time.perf_counter() - t0, 1e-4)
    paths_budget = pw * ph / dt * budget_s
    npix = cfg.width * cfg.height
    if paths_budget >= npix:
        w, h, spp = cfg.width, cfg.height, int(min(max(paths_budget // npix, 1), 64))
    else:
        k = (paths_budget / npix) ** 0.5
        w, h, spp = max(int(cfg.width * k), 8), max(int(cfg.height * k), 8), 1
    prm = rtb.make_params(w, h, spp, cfg.max_depth, cfg.background, seed=1)
    t0 = time.perf_counter()
    _, segs, _ = osc.render(cfg.camera, prm, threads=cores)
    dt = time.perf_counter() - t0
    sample = (f"{spp} spp at {w}x{h} (full size {cfg.width}x{cfg.height}); {segs} segments in {dt:.1f} s; f64 oracle, "
              "linear HittableList scan as the reference executes")
    return segs, dt, sample


def ncu_traffic(workload):
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture (profiles/traffic.json), or None."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(p) as f:
            t = json.load(f).get(workload)
        return t["dram_bytes_per_launch"] if t else None
    except Exception:
        return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback"


DUMP_BYTES = 64 << 20
DUMP_SAMPLE_PIXELS = 1 << 21


def dump_outputs(out_dir, accum, st):
    """Writes the last timed step's outputs: accum.npy, the (H, W, 4) float32 sums of R, G, B, Y^2 per pixel, and
    counters.npy, float64 [paths, segments, rejected].  A buffer over DUMP_BYTES is cut to a fixed seeded sample of
    DUMP_SAMPLE_PIXELS pixels, (n, 4) float32, whose row-major pixel indices go to accum_pixel_index.npy (float64)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    if accum.nbytes > DUMP_BYTES:
        h, w, _ = accum.shape
        idx = np.sort(np.random.default_rng(0).choice(h * w, DUMP_SAMPLE_PIXELS, replace=False))
        np.save(os.path.join(out_dir, "accum_pixel_index.npy"), idx.astype(np.float64))
        accum = accum.reshape(-1, 4)[idx]
    np.save(os.path.join(out_dir, "accum.npy"), accum)
    np.save(os.path.join(out_dir, "counters.npy"), np.array([st["paths"], st["segments"], st["rejected"]], dtype=np.float64))


def run_reference(args, rank):
    """The reference's CPU implementation of the path (oracle port, all host threads), bounded sample per step."""
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import orc
    import ray_tracer_archive_b200 as rtb
    orc.build()
    cfg = get_config(args.workload)
    cs = rtb.compile_scene(cfg.world, cfg.lights)
    osc = orc.OracleScene(cs)
    cores = os.cpu_count() or 1
    segs, dt, sample = 0, 0.0, ""
    budget = 12.0 if args.steps <= 3 else max(40.0 / args.steps, 3.0)
    for k in range(args.steps):
        s_, d_, sample = bounded_cpu_sample(osc, rtb, cfg, cores, budget_s=budget)
        segs += s_
        dt += d_
    val = segs / dt / 1e6
    print(json.dumps({
        "impl": "reference", "metric": "path segments/sec", "value": val, "unit": "Mrays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": cfg.name, "width": cfg.width, "height": cfg.height, "spp": cfg.spp,
                   "max_depth": cfg.max_depth, "sample": sample},
        "cpu_baseline": {"value": val, "unit": "Mrays/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="C1")
    ap.add_argument("--spp", type=int, default=0, help="override samples per pixel (changes the workload; for experiments)")
    ap.add_argument("--impl", default="rtb200")
    ap.add_argument("--pool", type=int, default=0)
    ap.add_argument("--rr", type=int, default=0, help="Russian-roulette start depth (0 = reference behaviour, off)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--strong", action="store_true",
                    help="strong scaling: the workload's spp is SPLIT across the ranks (BASELINE config C5) instead of "
                         "rendered by every rank (weak, default)")
    ap.add_argument("--strong-spp", type=int, default=2048,
                    help="total spp of the C5 strong-scaling sub-record (split across the ranks); 0 = skip it")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's accumulation buffer and path counters to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    # exactly ONE line may reach stdout (the JSON): libraries that print there (NCCL's version banner) go to stderr
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    import numpy as np
    import torch
    import torch.distributed as dist
    import ray_tracer_archive_b200 as rtb
    from ray_tracer_archive_b200 import parallel

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the CUDA library is the only implementation (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    W = max(args.warmup, 3)
    F = rtb._ffi

    cfg = get_config(args.workload, args.spp or None)
    cs = rtb.compile_scene(cfg.world, cfg.lights)
    ctx = rtb.Context(local_rank)
    if world > 1:  # the library's own communicator: torch.distributed only carries the 128-byte id to the other ranks
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(rtb.Context.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, src=0)
        ctx.comm_init(bytes(idt.cpu().numpy().tobytes()), rank, world)
    reduce_flag = F.RENDER_REDUCE if world > 1 else 0
    scene = rtb.Scene(ctx, cs)
    info = scene.info()
    npix = cfg.width * cfg.height
    spp = cfg.spp
    if args.strong:  # rank r renders its share of the workload's samples
        spp = parallel.rank_sample_range(cfg.spp, rank, world)[1]
    first_sample = parallel.rank_sample_range(cfg.spp, rank, world)[0] if args.strong else rank * spp
    total_spp = cfg.spp if args.strong else world * spp
    accum = torch.zeros((cfg.height, cfg.width, 4), dtype=torch.float32, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    stream = torch.cuda.current_stream()

    def params(flags=0):
        return rtb.make_params(cfg.width, cfg.height, spp, cfg.max_depth, cfg.background, seed=1,
                               sample_offset=first_sample, total_spp=total_spp, rr_start_depth=args.rr,
                               pool_paths=args.pool, flags=flags)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    reduce_ms_list, wait_ms_list = [], []

    def step(flags=0):
        flush.zero_()  # flush L2 between steps
        # render + (N > 1) the library's ncclReduce of the float4 accumulation buffer onto rank 0, on this stream
        st = scene.render_device(cfg.camera, params(flags | reduce_flag), accum.data_ptr(), stream.cuda_stream)
        reduce_ms_list.append(st["ms_nccl"])
        wait_ms_list.append(st["ms_nccl_wait"])
        return st

    # clocks / throttle reasons are sampled from the first warm-up step to the last e2e step (everything under load)
    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(W):
        step()
    # ---- timed region: exactly K steps, device time, max over ranks ---------------------------------------------
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reduce_ms_list.clear()
    wait_ms_list.clear()
    e0.record(stream)
    segs = launches = 0
    for _ in range(args.steps):
        st = step()
        segs += st["segments"]
        launches += st["launches"]
    e1.record(stream)
    barrier()
    if args.dump_outputs and rank == 0:  # before the e2e and roofline renders below overwrite the buffer
        dump_outputs(args.dump_outputs, accum.cpu().numpy(), st)
    ms = e0.elapsed_time(e1)
    reduce_ms = sum(reduce_ms_list) / max(len(reduce_ms_list), 1)
    wait_ms = sum(wait_ms_list) / max(len(wait_ms_list), 1)
    tot = torch.tensor([ms, float(segs), float(launches)], dtype=torch.float64, device="cuda")
    if world > 1:
        mx = tot.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        ms = mx[0].item()
    all_segs, all_launches = tot[1].item(), tot[2].item()
    value = all_segs / (ms * 1e-3) / 1e6

    # ---- e2e: host buffers in, host buffer out, every step ----------------------------------------------------------
    host_out = torch.empty((cfg.height, cfg.width, 4), dtype=torch.float32).pin_memory()
    h2d = int(info["bvh_bytes"] + info["prim_bytes"] + cs.materials.nbytes + cs.textures.nbytes + cs.lights.nbytes
              + sum(i.nbytes for i in cs.images) + 4 * npix)
    d2h = npix * 16

    sc2 = rtb.Scene(ctx)  # device buffers are reused across steps (a per-frame scene update, no malloc/free churn)

    def step_e2e():
        t0 = time.perf_counter()
        flush.zero_()
        sc2.set_compiled(cs)  # scene records from host memory: tables + flatten ...
        sc2.commit()          # ... + BVH build + H2D
        t1 = time.perf_counter()
        st = sc2.render_device(cfg.camera, params(reduce_flag), accum.data_ptr(), stream.cuda_stream)
        t2 = time.perf_counter()
        if rank == 0:
            host_out.copy_(accum, non_blocking=True)
        torch.cuda.synchronize()
        if os.environ.get("RTB_BENCH_DEBUG"):
            print(f"e2e step: scene {t1 - t0:.4f}s render {t2 - t1:.4f}s (device {st['ms_total'] / 1e3:.4f}s) "
                  f"reduce+d2h {time.perf_counter() - t2:.4f}s", file=sys.stderr)
        return st

    step_e2e()
    barrier()
    t0 = time.perf_counter()
    e_segs = 0
    for _ in range(args.steps):
        e_segs += step_e2e()["segments"]
    barrier()
    dt = time.perf_counter() - t0
    et = torch.tensor([dt, float(e_segs)], dtype=torch.float64, device="cuda")
    if world > 1:
        emx = et.clone()
        dist.all_reduce(emx, op=dist.ReduceOp.MAX)
        dist.all_reduce(et, op=dist.ReduceOp.SUM)
        dt = emx[0].item()
    e2e_value = et[1].item() / dt / 1e6
    sampler.stop_flag = True

    # ---- strong scaling on BASELINE.json's scaling config (C5): fixed total spp split across the ranks ---------------
    strong = None
    if args.strong_spp > 0 and not args.strong and args.workload == "C1":
        c5 = get_config("C5", args.strong_spp)
        first5, cnt5 = parallel.rank_sample_range(c5.spp, rank, world)
        cs5 = rtb.compile_scene(c5.world, c5.lights)
        sc5 = rtb.Scene(ctx, cs5)
        acc5 = torch.zeros((c5.height, c5.width, 4), dtype=torch.float32, device="cuda")

        def step5(spp_override=None):
            flush.zero_()
            n_s = cnt5 if spp_override is None else spp_override
            p5 = rtb.make_params(c5.width, c5.height, max(n_s, 1), c5.max_depth, c5.background, seed=1, sample_offset=first5,
                                 total_spp=c5.spp, flags=reduce_flag)
            return sc5.render_device(c5.camera, p5, acc5.data_ptr(), stream.cuda_stream)

        step5(min(cnt5, 8))  # warm-up (pool allocation, caches) at a few spp
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record(stream)
        st5 = step5()
        s1.record(stream)
        barrier()
        t5 = torch.tensor([s0.elapsed_time(s1), float(st5["segments"]), st5["ms_render"]], dtype=torch.float64, device="cuda")
        if world > 1:
            m5 = t5.clone()
            dist.all_reduce(m5, op=dist.ReduceOp.MAX)
            mn5 = t5.clone()
            dist.all_reduce(mn5, op=dist.ReduceOp.MIN)
            dist.all_reduce(t5, op=dist.ReduceOp.SUM)
        else:
            m5 = mn5 = t5
        strong = {"workload": c5.name, "width": c5.width, "height": c5.height, "total_spp": c5.spp, "spp_per_gpu": cnt5,
                  "scaling": "strong", "value": t5[1].item() / (m5[0].item() * 1e-3) / 1e6, "unit": "Mrays/s",
                  "ms_per_step": m5[0].item(), "ms_render_slowest_rank": m5[2].item(), "ms_render_fastest_rank": mn5[2].item(),
                  "reduce_bytes": c5.width * c5.height * 16, "reduce_ms_rank0": st5["ms_nccl"], "ms_rank0_waited_for_the_slowest_rank": st5["ms_nccl_wait"],
                  "reduce_frac_of_step": st5["ms_nccl"] / m5[0].item(), "segments": t5[1].item(),
                  "note": "efficiency = value(N) / (N x value(1)) across the per-N lines; what limits it is the wavefront drain "
                          "tail of each rank's shorter render (fewer samples per pixel to refill the path pool from), not the collective"}
        sc5.close()
        del acc5

    # ---- roofline of the dominant kernel (extend), measured live on rank 0 ------------------------------------------
    roofline = None
    cpu_baseline = None
    cpu_fair = None
    if rank == 0:
        stc = scene.render_device(cfg.camera, params(F.RENDER_COUNT), accum.data_ptr(), stream.cuda_stream)
        stt = scene.render_device(cfg.camera, params(F.RENDER_TIME_EXTEND), accum.data_ptr(), stream.cuda_stream)
        n_seg = stc["segments"]
        nodes_per_seg = stc["nodes_visited"] / n_seg
        prims_per_seg = stc["prims_tested"] / n_seg
        # primitive mix: the instrumented kernel counts the tests it EXECUTES per type (not the scene's primitive counts)
        per_type = dict(zip(("sphere", "moving", "quad", "tri"), (x / n_seg for x in stc["prims_tested_type"])))
        flops_seg = nodes_per_seg * F_NODE + sum(F_PRIM[k] * v for k, v in per_type.items())
        bytes_seg = nodes_per_seg * B_NODE + sum(B_PRIM[k] * v for k, v in per_type.items())
        ext_ms, n_ext = stt["ms_extend"], stt["extend_launches"]
        seg_per_launch = stt["segments"] / n_ext
        avg_launch_ms = ext_ms / n_ext
        peaks, which = measured_peaks()
        dev = ctx.device_info()
        clk = sampler.summary()
        sm_mhz = clk["sm_mhz"] or peaks.get("sm_max_mhz", 1965.0)
        fp32_peak = dev["sm_count"] * 128 * 2 * sm_mhz * 1e6 / 1e12  # TFLOP/s at the clock seen during the run
        ach_tflops = flops_seg * seg_per_launch / (avg_launch_ms * 1e-3) / 1e12
        ach_gbs = bytes_seg * seg_per_launch / (avg_launch_ms * 1e-3) / 1e9
        scene_bytes = info["bvh_bytes"] + info["prim_bytes"]
        in_l2 = scene_bytes <= dev["l2_bytes"]
        # where the scene's bytes physically come from decides the memory side of the roofline:
        #   all nodes staged in shared memory / primitives in the constant bank  -> shared-memory read bandwidth
        #   scene <= L2 (every other config)                                      -> L2 read bandwidth (read-only 128-bit stream)
        #   scene >  L2                                                           -> HBM (MEASURED_PEAKS.json)
        bw = measure_bandwidths(ctx, F)
        on_chip = bool(scene_bytes <= 56 * 1024)
        if on_chip:
            mem_gbs, mem_name = bw["shared_read_gbs"], "shared"
        elif in_l2:
            mem_gbs, mem_name = bw["l2_read_gbs"], "l2"
        else:
            mem_gbs, mem_name = peaks["hbm_gbs"], "hbm"
        t_flops, t_bytes = flops_seg / (fp32_peak * 1e12), bytes_seg / (mem_gbs * 1e9)
        fp_bound = t_flops >= t_bytes
        roofline = {
            "kernel": "k_extend", "bound": "fp32" if fp_bound else mem_name,
            "achieved": ach_tflops if fp_bound else ach_gbs,
            "peak": fp32_peak if fp_bound else mem_gbs,
            "unit": "TFLOP/s" if fp_bound else "GB/s",
            "frac": (ach_tflops / fp32_peak) if fp_bound else (ach_gbs / mem_gbs),
            "traffic": ncu_traffic(args.workload),
            "peak_source": f"FP32 = SMs*128*2*f_SM at the median SM clock seen in this run ({sm_mhz:.0f} MHz) = {fp32_peak:.1f} TFLOP/s; "
                           f"measured in this run by rtb_measure_bandwidth (read-only 128-bit streams): L2 {bw['l2_read_gbs']:.0f} GB/s (48 MB resident), "
                           f"HBM {bw['hbm_read_gbs']:.0f} GB/s (2 GB), shared memory {bw['shared_read_gbs']:.0f} GB/s; HBM copy {which} {peaks['hbm_gbs']} GB/s (MEASURED_PEAKS.json)",
            "bandwidths": bw,
            "fp32": {"achieved_tflops": ach_tflops, "peak_tflops": fp32_peak, "frac": ach_tflops / fp32_peak},
            "hbm": {"achieved_gbs": ach_gbs, "peak_gbs": peaks["hbm_gbs"], "frac": ach_gbs / peaks["hbm_gbs"],
                    "scene_bytes": scene_bytes, "scene_fits_l2": bool(in_l2)},
            "l2": {"achieved_gbs": ach_gbs, "peak_gbs": bw["l2_read_gbs"], "frac": ach_gbs / bw["l2_read_gbs"]},
            "shared": {"achieved_gbs": ach_gbs, "peak_gbs": bw["shared_read_gbs"], "frac": ach_gbs / bw["shared_read_gbs"]},
            "algorithmic": {"nodes_per_segment": nodes_per_seg, "prims_per_segment": prims_per_seg,
                            "prim_tests_per_segment_by_type": per_type,
                            "flops_per_segment": flops_seg, "bytes_per_segment": bytes_seg,
                            "segments_per_launch": seg_per_launch},
            # the whole scene sits in the kernel's shared-memory stage / the constant bank: its bytes never reach L2
            "on_chip_scene": on_chip,
            "extend_ms_per_launch": avg_launch_ms, "extend_launches_per_step": n_ext,
            "extend_share_of_step": ext_ms / stt["ms_total"],
            "exact_pass": {"rays_retraced_per_segment": stc["exact_rays"] / n_seg, "hits_refined_per_segment": stc["refined_rays"] / n_seg},
            "roofline_mrays_s": 1.0 / max(t_flops, t_bytes) / 1e6,
        }
        if not args.no_cpu_baseline:
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            import orc
            orc.build()
            osc = orc.OracleScene(cs)
            cores = os.cpu_count() or 1
            csegs, cdt, csample = bounded_cpu_sample(osc, rtb, cfg, cores)
            cpu_baseline = {"value": csegs / cdt / 1e6, "unit": "Mrays/s", "cores": cores, "kind": "port", "sample": csample}
            # CPU-fair (BASELINE.md §2): the same oracle culling candidates with the SAME wide BVH the GPU traverses
            osc.attach_bvh(scene)
            fsegs, fdt, fsample = bounded_cpu_sample(osc, rtb, cfg, cores, budget_s=6.0)
            cpu_fair = {"value": fsegs / fdt / 1e6, "unit": "Mrays/s", "cores": cores, "kind": "port",
                        "sample": fsample.replace("linear HittableList scan as the reference executes",
                                                  "reference per-primitive tests, candidates culled by the shipped BVH8")}
        line = {
            "metric": "path segments/sec", "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
            "warmup": W, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong" if args.strong else "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg.name, "width": cfg.width, "height": cfg.height, "spp_per_gpu": spp,
                       "total_spp": total_spp, "max_depth": cfg.max_depth, "rr_start_depth": args.rr,
                       "prims": info["n_prims"], "bvh_nodes": info["n_bvh_nodes"], "parallelism": f"spp-split x{world} + NCCL reduce",
                       "l2": "L2 flushed (256 MB write) between steps; path-state pool exceeds the 126 MB L2; the scene is cache-resident by design"},
            "e2e": {"value": e2e_value, "unit": "Mrays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(all_launches),
            "reduce": {"collective": "ncclReduce(sum) of W*H float4 onto rank 0, issued by librtb200 (RTB_RENDER_REDUCE)" if world > 1 else "none (1 GPU)",
                       "bytes": npix * 16, "ms_per_step_rank0": reduce_ms, "frac_of_step": reduce_ms / (ms / args.steps),
                       "ms_rank0_waited_for_the_slowest_rank": wait_ms},
            "strong_scaling": strong,
            "clocks": clk,
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "cpu_baseline_fair": cpu_fair,
            "segments_per_step": all_segs / args.steps,
            "paths_per_step": npix * total_spp,
        }
        print(json.dumps(line), file=real_stdout, flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    sc2.close()
    scene.close()
    ctx.close()


if __name__ == "__main__":
    main()
