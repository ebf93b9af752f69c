#!/usr/bin/env python
"""Cost of the denoiser guide pass (rtb_render_aov) next to the render it guides (GPU box).

  python tools/bench_aov.py [--spp 64] [--reps 3] [--out profiles/r7/bench_aov.json]

For C1 (1200x675), C3 (800x800) and C4 (1920x1080) at the same spp and params: one warm-up call of each, then `reps` AOV
passes alternated with `reps` renders, each into a device buffer on the current torch stream.  Times are the calls' own
CUDA-event times (rtb_stats::ms_total).  Reports the AOV time and its primary rays/s, the render's time and segments/s,
and AOV / render.  The AOV pass traces only the first segment of each sample the render traces, so it must take less
time than the render.  The GPU's name, power limit and SM clock are read with an nvidia-smi query."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKLOADS = ("C1", "C3", "C4")


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                         timeout=60).stdout.strip().splitlines()
    return dict(zip(q.split(","), (s.strip() for s in out[0].split(",")))) if out else {}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--spp", type=int, default=64)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r7", "bench_aov.json"))
    args = ap.parse_args()
    sys.path.insert(0, ROOT)
    import torch
    import ray_tracer_archive_b200 as rtb
    from bench import get_config

    ctx = rtb.Context(0)
    stream = torch.cuda.current_stream()
    res = {"gpu": gpu_info(), "spp": args.spp, "workloads": {}}
    print(res["gpu"])
    for w in WORKLOADS:
        cfg = get_config(w, args.spp)
        sc = rtb.Scene(ctx, rtb.compile_scene(cfg.world, cfg.lights))
        prm = rtb.make_params(cfg.width, cfg.height, cfg.spp, cfg.max_depth, cfg.background, seed=1)
        accum = torch.zeros((cfg.height, cfg.width, 4), dtype=torch.float32, device="cuda")
        aov = torch.zeros((cfg.height, cfg.width, 8), dtype=torch.float32, device="cuda")
        sc.render_aov_device(cfg.camera, prm, aov.data_ptr(), stream.cuda_stream)
        sc.render_device(cfg.camera, prm, accum.data_ptr(), stream.cuda_stream)
        aov_ms, ren_ms, segs = [], [], []
        for _ in range(args.reps):
            st = sc.render_aov_device(cfg.camera, prm, aov.data_ptr(), stream.cuda_stream)
            assert st["paths"] == cfg.width * cfg.height * cfg.spp and st["rejected"] == 0
            aov_ms.append(st["ms_total"])
            st = sc.render_device(cfg.camera, prm, accum.data_ptr(), stream.cuda_stream)
            ren_ms.append(st["ms_total"])
            segs.append(st["segments"])
        rays = cfg.width * cfg.height * cfg.spp
        a, r = statistics.median(aov_ms), statistics.median(ren_ms)
        rec = {"width": cfg.width, "height": cfg.height, "spp": cfg.spp, "aov_ms": aov_ms, "render_ms": ren_ms,
               "aov_mrays_per_s": rays / (a * 1e-3) / 1e6, "render_segments": segs[-1],
               "render_mseg_per_s": segs[-1] / (r * 1e-3) / 1e6, "aov_over_render": a / r}
        res["workloads"][w] = rec
        print(f"{w} {cfg.width}x{cfg.height} {cfg.spp} spp: AOV {a:.2f} ms ({rec['aov_mrays_per_s']:.0f} Mrays/s), "
              f"render {r:.2f} ms ({rec['render_mseg_per_s']:.0f} Mseg/s, {segs[-1] / rays:.2f} segments/path), "
              f"AOV / render {rec['aov_over_render']:.3f}")
        sc.close()
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    ok = all(v["aov_over_render"] < 1.0 for v in res["workloads"].values())
    print("AOV pass faster than the render on every workload:", ok)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
