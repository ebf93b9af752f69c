"""Traversal statistics of the device header compiled for the host (tests/emul, -DRTB_EMUL_STATS): per ray class, node
visits, visits that found no child to continue with, internal / leaf children hit.  python tools/emul_stats.py C3 C4"""
import ctypes as C, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import numpy as np
import helpers as H
import ray_tracer_archive_b200 as rtb
from ray_tracer_archive_b200 import scenes

src = os.path.join(ROOT, "tests", "emul", "emul_traverse.cpp")
out = "/tmp/libemul_stats.so"
subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-std=c++17", "-fPIC", "-shared", "-Wno-attributes", "-D__noinline__=",
                       "-DRTB_EMUL_STATS", "-I/usr/local/cuda/include", "-o", out, src])
lib = C.CDLL(out)
VP = C.c_void_p
lib.emul_trace.argtypes = ([VP, C.c_uint32] + [VP] * 8 + [VP] * 3 + [C.c_float, C.c_float, C.c_uint32] +
                           [VP, C.c_uint32, C.c_uint32, C.c_uint32, VP, VP, VP, C.c_uint32, VP, VP, VP, VP])
def stats(reset=True):
    a = (C.c_ulonglong * 8)()
    lib.emul_stats(a, int(reset))
    return list(a)
mk = {"C1": scenes.config_random_spheres, "C2": scenes.config_cornell, "C3": scenes.config_final_scene, "C4": scenes.config_mesh}
for w in sys.argv[1:] or ["C3", "C4"]:
    cfg = mk[w]()
    hs = rtb.Scene(None, rtb.compile_scene(cfg.world, cfg.lights))
    W, Hh = cfg.width // 4, cfg.height // 4
    o, d = H.primary_rays(cfg.camera, W, Hh)
    o32, d32 = o.astype(np.float32), d.astype(np.float32)
    tm = np.zeros(len(o), np.float32)
    rng = np.random.default_rng(7)
    for bounce in range(3):
        stats()
        ids, ts, nv, nt = H.emul_trace(lib, hs, o32, d32, tm)
        s = stats()
        n = len(o32)
        print(f"{w} bounce {bounce}: {n} rays, {s[0] / n:.2f} node visits/ray, {s[1] / max(s[0], 1):.3f} of them without a hit child, "
              f"{s[2] / n:.2f} internal + {s[3] / n:.2f} leaf children hit/ray, {nt / n:.2f} prim tests/ray")
        nl = max(s[4] + s[5] + s[6], 1)
        print(f"      visits with leaf hits: {(s[4] + s[5] + s[6]) / n:.2f}/ray, holding 1 / 2 / 3+ primitives: "
              f"{s[4] / nl:.3f} / {s[5] / nl:.3f} / {s[6] / nl:.3f}, {s[7] / nl:.2f} primitives per such visit")
        # the same rays again with t_max initialised to the hit distance found: what perfect culling of stale stack entries
        # (groups pushed before the hit was known) could save at most
        t0 = np.where(ids != H.NONE, ts * (1 + 3e-4), np.inf).astype(np.float32)
        lib.emul_set_tmax0(t0.ctypes.data_as(C.c_void_p))
        ids2, ts2, nv2, nt2 = H.emul_trace(lib, hs, o32, d32, tm)
        lib.emul_set_tmax0(None)
        s2 = stats()
        same = float(np.mean(ids == ids2))  # (a hit whose own error bound exceeds 1e-5 t gets culled by this t_max: estimate only)
        print(f"      with t_max known in advance: {s2[0] / n:.2f} node visits/ray ({s2[1] / max(s2[0], 1):.3f} without a hit child), {nt2 / n:.2f} prim tests/ray, same hit {same:.4f}")
        hit = ids != H.NONE
        p = (o32[hit] + ts[hit, None] * d32[hit]).astype(np.float32)
        nd = rng.normal(0, 1, p.shape).astype(np.float32)
        nd /= np.linalg.norm(nd, axis=1, keepdims=True)
        o32, d32, tm = p, nd, rng.random(len(p)).astype(np.float32)
