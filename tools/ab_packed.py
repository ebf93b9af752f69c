#!/usr/bin/env python
"""Same-result check of two builds of librtb200.so (GPU box): each build runs in its own process (RTB200_LIB), on C1-C4 at
reduced spp, and the two are compared.

  python tools/ab_packed.py BASE.so NEW.so [--spp-scale 0.1] [--out DIR]

- Counters of an instrumented render (RTB_RENDER_COUNT): segments, node visits, primitive tests per type, exactly
  re-traced and refined rays.  They must be EQUAL: any difference means a node or primitive decision changed.
- P1 probe (rtb_primary_rays + the production kernels): primitive ids and t BITWISE equal on every pixel.
- bench.py --dump-outputs (C1 defaults without the C5 sub-record, 1 step): counters equal; accum may differ only by the order of the float
  atomics, bounded by the difference of two runs of the base build.
Exit code 0 iff everything holds."""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKLOADS = ("C1", "C2", "C3", "C4")


def child(out, spp_scale):
    """Runs in a process whose RTB200_LIB names one build; writes counters and probe arrays to `out`."""
    sys.path.insert(0, ROOT)
    import numpy as np
    import ray_tracer_archive_b200 as rtb
    from bench import get_config
    F = rtb._ffi
    ctx = rtb.Context(0)
    res = {}
    for w in WORKLOADS:
        spp = max(1, int(round(get_config(w).spp * spp_scale)))
        cfg = get_config(w, spp)
        sc = rtb.Scene(ctx, rtb.compile_scene(cfg.world, cfg.lights))
        prm = rtb.make_params(cfg.width, cfg.height, cfg.spp, cfg.max_depth, cfg.background, seed=1, flags=F.RENDER_COUNT)
        _, st = sc.render(cfg.camera, prm, readback=False)
        res[w] = {k: st[k] for k in ("paths", "segments", "rejected", "nodes_visited", "prims_tested", "prims_tested_type",
                                     "exact_rays", "refined_rays")}
        res[w]["spp"] = spp
        ids, ts, _ = sc.primary_hits(cfg.camera, cfg.width, cfg.height)
        np.save(os.path.join(out, f"{w}_ids.npy"), np.ascontiguousarray(ids).view(np.uint32))
        np.save(os.path.join(out, f"{w}_t.npy"), np.ascontiguousarray(ts, dtype=np.float32).view(np.uint32))
        sc.close()
    ctx.close()
    with open(os.path.join(out, "counters.json"), "w") as f:
        json.dump(res, f)


def run_build(lib, out, spp_scale):
    os.makedirs(out, exist_ok=True)
    env = dict(os.environ, RTB200_LIB=os.path.abspath(lib))
    subprocess.check_call([sys.executable, os.path.abspath(__file__), "--child", out, "--spp-scale", str(spp_scale)], env=env, cwd=ROOT)


def run_bench_dump(lib, out):
    env = dict(os.environ, RTB200_LIB=os.path.abspath(lib))
    subprocess.check_call([sys.executable, "bench.py", "--gpus", "1", "--steps", "1", "--warmup", "1", "--no-cpu-baseline",
                           "--strong-spp", "0", "--dump-outputs", out], env=env, cwd=ROOT, stdout=subprocess.DEVNULL)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("base", nargs="?")
    ap.add_argument("new", nargs="?")
    ap.add_argument("--spp-scale", type=float, default=0.1)
    ap.add_argument("--out", default=None, help="directory for the per-build outputs (default: a temporary one)")
    ap.add_argument("--child", metavar="DIR")
    args = ap.parse_args()
    if args.child:
        return child(args.child, args.spp_scale)
    import numpy as np
    out = args.out or tempfile.mkdtemp(prefix="ab_packed_")
    ok = True
    dirs = {k: os.path.join(out, k) for k in ("base", "new")}
    run_build(args.base, dirs["base"], args.spp_scale)
    run_build(args.new, dirs["new"], args.spp_scale)
    cnt = {k: json.load(open(os.path.join(d, "counters.json"))) for k, d in dirs.items()}
    for w in WORKLOADS:
        b, n = cnt["base"][w], cnt["new"][w]
        same = b == n
        ok &= same
        print(f"{w} spp={b['spp']}: counters {'EQUAL' if same else 'DIFFER'}  "
              f"segments={n['segments']} nodes={n['nodes_visited']} prims/type={n['prims_tested_type']} "
              f"exact={n['exact_rays']} refined={n['refined_rays']}")
        if not same:
            print("   base", json.dumps(b), "\n   new ", json.dumps(n))
        for a in ("ids", "t"):
            x, y = (np.load(os.path.join(dirs[k], f"{w}_{a}.npy")) for k in ("base", "new"))
            eq = x.shape == y.shape and np.array_equal(x, y)
            ok &= eq
            print(f"   P1 {a}: {'bitwise equal' if eq else 'DIFFER in %d of %d pixels' % (int((x != y).sum()), x.size)}")
    # bench.py --dump-outputs: two base runs give the spread of the float-atomic order, then the new build
    runs = {k: os.path.join(out, "bench_" + k) for k in ("base1", "base2", "new")}
    for k, d in runs.items():
        run_bench_dump(args.base if k.startswith("base") else args.new, d)
    acc = {k: np.load(os.path.join(d, "accum.npy")).astype(np.float64) for k, d in runs.items()}
    ctr = {k: np.load(os.path.join(d, "counters.npy")) for k, d in runs.items()}
    same = np.array_equal(ctr["base1"], ctr["new"]) and np.array_equal(ctr["base1"], ctr["base2"])
    ok &= same
    spread = float(np.max(np.abs(acc["base1"] - acc["base2"])))
    diff = float(np.max(np.abs(acc["base1"] - acc["new"])))
    within = diff <= spread
    ok &= within
    print(f"bench --dump-outputs C1: counters {'EQUAL' if same else 'DIFFER'} {ctr['new'].tolist()}; "
          f"max |accum base - new| = {diff:.3g}, base-vs-base spread = {spread:.3g} -> {'within' if within else 'OUTSIDE'}")
    print("AB_PACKED", "PASS" if ok else "FAIL")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
