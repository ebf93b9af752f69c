#!/usr/bin/env python
"""Cost of smooth shading on C4 (GPU box): the 1 M-triangle height field rendered flat and with vertex normals
(scenes.config_mesh(smooth=True)) at the full 1920x1080.

  python tools/bench_mesh_attrs.py [--spp 1024] [--reps 3] [--base BASE.so] [--out profiles/r8/bench_mesh_attrs.json]

One warm-up render of each, then `reps` flat renders alternated with `reps` smooth renders into device buffers; each time is
the call's own CUDA-event time (rtb_stats::ms_total) and the medians are reported.  With --base, another build of
librtb200.so (e.g. the parent commit's) times the flat scene the same way in a child process before and after, so the flat
time of this build can be read against the spread of that one.  The GPU's name, power limit and SM clock are read with an
nvidia-smi query in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                         timeout=60).stdout.strip().splitlines()
    return dict(zip(q.split(","), (s.strip() for s in out[0].split(",")))) if out else {}


def run(variants, spp, reps):
    """-> {variant: {"ms": [...], "segments": n}} for variants in ("flat", "smooth"), alternated."""
    sys.path.insert(0, ROOT)
    import torch
    import ray_tracer_archive_b200 as rtb
    from ray_tracer_archive_b200 import scenes

    ctx = rtb.Context(0)
    stream = torch.cuda.current_stream()
    cfg = scenes.config_mesh(spp=spp)
    cs = rtb.compile_scene(cfg.world, cfg.lights)
    if "smooth" in variants:
        cs_smooth = rtb.compile_scene(*(lambda c: (c.world, c.lights))(scenes.config_mesh(spp=spp, smooth=True)))
    prm = rtb.make_params(cfg.width, cfg.height, cfg.spp, cfg.max_depth, cfg.background, seed=1)
    accum = torch.zeros((cfg.height, cfg.width, 4), dtype=torch.float32, device="cuda")
    sc = {"flat": rtb.Scene(ctx, cs)}
    if "smooth" in variants:
        sc["smooth"] = rtb.Scene(ctx, cs_smooth)
    res = {v: {"ms": [], "segments": 0} for v in variants}
    for v in variants:  # warm-up
        sc[v].render_device(cfg.camera, prm, accum.data_ptr(), stream.cuda_stream)
    for _ in range(reps):
        for v in variants:
            st = sc[v].render_device(cfg.camera, prm, accum.data_ptr(), stream.cuda_stream)
            assert st["paths"] == cfg.width * cfg.height * cfg.spp
            res[v]["ms"].append(st["ms_total"])
            res[v]["segments"] = st["segments"]
    for s in sc.values():
        s.close()
    ctx.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--spp", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--base", help="another librtb200.so whose flat C4 time is measured before and after")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r8", "bench_mesh_attrs.json"))
    ap.add_argument("--child", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.child:  # flat only, in a process whose RTB200_LIB names the base build
        print(json.dumps(run(("flat",), args.spp, args.reps)))
        return 0

    def base_run():
        env = dict(os.environ, RTB200_LIB=os.path.abspath(args.base))
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "--spp", str(args.spp), "--reps",
                              str(args.reps)], env=env, capture_output=True, text=True, check=True, cwd=ROOT)
        return json.loads(out.stdout.strip().splitlines()[-1])["flat"]

    res = {"gpu": gpu_info(), "width": 1920, "height": 1080, "spp": args.spp, "reps": args.reps}
    print(res["gpu"])
    if args.base:
        res["base_flat_before"] = base_run()
    res.update(run(("flat", "smooth"), args.spp, args.reps))
    if args.base:
        res["base_flat_after"] = base_run()
    rays = 1920 * 1080 * args.spp
    for k in ("base_flat_before", "flat", "smooth", "base_flat_after"):
        if k in res:
            m = statistics.median(res[k]["ms"])
            res[k]["median_ms"] = m
            print(f"{k:>16}: median {m:.2f} ms of {[round(x, 2) for x in res[k]['ms']]} "
                  f"({rays / (m * 1e-3) / 1e6:.0f} Mpaths/s, {res[k]['segments'] / (m * 1e-3) / 1e6:.0f} Mseg/s)")
    res["smooth_over_flat"] = res["smooth"]["median_ms"] / res["flat"]["median_ms"]
    print(f"smooth / flat: {res['smooth_over_flat']:.4f}")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    return 0


if __name__ == "__main__":
    sys.exit(main())
