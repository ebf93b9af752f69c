"""Thin object wrappers over the C ABI (include/rtb200.h).  The CUDA library is the only implementation."""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import _ffi as F
from .scene import CompiledScene


class Context:
    """One GPU — or, with a list of device ids, several GPUs driven by this process (rtb_context_create_multi: the
    library splits every render's samples across them and sums the accumulation buffers with one NCCL reduce).
    With one process per GPU use comm_unique_id() / comm_init() and the RENDER_REDUCE flag instead."""

    def __init__(self, device_id=0):
        self.lib = F.load()
        h = C.c_void_p()
        if isinstance(device_id, (list, tuple)):
            ids = (C.c_int * len(device_id))(*device_id)
            F.check(self.lib.rtb_context_create_multi(ids, len(device_id), C.byref(h)))
            self.device_id = int(device_id[0])
        else:
            F.check(self.lib.rtb_context_create(device_id, C.byref(h)))
            self.device_id = device_id
        self.h = h

    @property
    def device_count(self) -> int:
        return self.lib.rtb_context_device_count(self.h)

    @staticmethod
    def comm_unique_id() -> bytes:
        """128 bytes (ncclGetUniqueId) that rank 0 hands to the other ranks."""
        buf = (C.c_uint8 * 128)()
        F.check(F.load().rtb_comm_unique_id(buf))
        return bytes(buf)

    def comm_init(self, unique_id: bytes, rank: int, n_ranks: int):
        """Join the communicator (ncclCommInitRank); collective: every rank must call it."""
        buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        F.check(self.lib.rtb_context_comm_init(self.h, buf, rank, n_ranks))

    def close(self):
        if getattr(self, "h", None):
            self.lib.rtb_context_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def primary_rays(self, cam: F.Camera, width: int, height: int):
        """The f32 pixel-centre rays rtb_primary_hits traces: (origin (n,3), direction (n,3), time (n,)) float32."""
        n = width * height
        o, d, t = np.empty((n, 3), np.float32), np.empty((n, 3), np.float32), np.empty(n, np.float32)
        F.check(self.lib.rtb_primary_rays(self.h, C.byref(cam), width, height, F.ptr(o), F.ptr(d), F.ptr(t)))
        return o, d, t

    def kat(self, op: int, words, out_stride: int, scene=None, cam=None, params=None):
        """Tier-U2 hook (rtb_device_kat): `words` (n, in_stride) uint32 -> (n, out_stride) uint32."""
        w = np.ascontiguousarray(words, dtype=np.uint32)
        out = np.zeros((w.shape[0], out_stride), dtype=np.uint32)
        F.check(self.lib.rtb_device_kat(self.h, scene.h if scene is not None else None,
                                        C.byref(cam) if cam is not None else None,
                                        C.byref(params) if params is not None else None, op, F.ptr(w), w.shape[0],
                                        w.shape[1], F.ptr(out), out_stride))
        return out

    def check_failures(self):
        """RTB_CHECKED build: failed device-side bounds assertions by kind (all 0xFFFFFFFF in a normal build)."""
        out = np.zeros(8, dtype=np.uint32)
        F.check(self.lib.rtb_debug_check_failures(self.h, F.ptr(out)))
        return out

    def measure_bandwidth(self, kind: int, repeats: int = 5) -> float:
        """GB/s of a read-only stream: F.BW_L2_READ (48 MB, L2-resident), F.BW_HBM_READ (2 GB), F.BW_SHARED_READ."""
        v = C.c_double()
        F.check(self.lib.rtb_measure_bandwidth(self.h, kind, repeats, C.byref(v)))
        return v.value

    def device_info(self):
        sm, l2, khz = C.c_int(), C.c_int(), C.c_int()
        name = C.create_string_buffer(128)
        F.check(self.lib.rtb_context_device_info(self.h, C.byref(sm), C.byref(l2), C.byref(khz), name, 128))
        return {"sm_count": sm.value, "l2_bytes": l2.value, "clock_khz": khz.value, "name": name.value.decode()}


class Scene:
    def __init__(self, ctx: Optional[Context], cs: Optional[CompiledScene] = None):
        """ctx=None gives a host-only scene (flatten + BVH build + export; no device needed, cannot render)."""
        self.ctx = ctx
        self.lib = ctx.lib if ctx is not None else F.load()
        h = C.c_void_p()
        F.check(self.lib.rtb_scene_create(ctx.h if ctx is not None else None, C.byref(h)))
        self.h = h
        self.cs = cs
        if cs is not None:
            self.set_compiled(cs)
            if ctx is not None:
                self.commit()
            else:
                self.build_bvh()

    def close(self):
        if getattr(self, "h", None):
            self.lib.rtb_scene_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_tables(self, cs: CompiledScene):
        lib = self.lib
        F.check(lib.rtb_scene_set_materials(self.h, F.ptr(cs.materials), len(cs.materials)))
        F.check(lib.rtb_scene_set_textures(self.h, F.ptr(cs.textures), len(cs.textures)))
        for i, img in enumerate(cs.images):
            a = np.ascontiguousarray(img, dtype=np.uint8)
            F.check(lib.rtb_scene_set_image(self.h, i, F.ptr(a), a.shape[1], a.shape[0]))
        for i, p in enumerate(cs.perlins):
            rv = np.ascontiguousarray(p.ranvec, dtype=np.float64)
            px, py, pz = (np.ascontiguousarray(x, dtype=np.uint32) for x in (p.perm_x, p.perm_y, p.perm_z))
            F.check(lib.rtb_scene_set_perlin(self.h, i, F.ptr(rv), F.ptr(px), F.ptr(py), F.ptr(pz)))
        for i, (v, idx) in enumerate(cs.meshes):
            F.check(lib.rtb_scene_set_mesh(self.h, i, F.ptr(v), len(v), F.ptr(idx), len(idx)))
        F.check(lib.rtb_scene_set_lights(self.h, F.ptr(cs.lights) if len(cs.lights) else None, len(cs.lights)))

    def set_compiled(self, cs: CompiledScene):
        self.set_tables(cs)
        F.check(self.lib.rtb_scene_set_graph(self.h, F.ptr(cs.nodes), len(cs.nodes), F.ptr(cs.child_index),
                                              len(cs.child_index), cs.root))

    def set_build_options(self, max_leaf_triangles=2, keep_huge_primitives_out=True, open_min_extent=0.125):
        """BVH builder quality knobs (rtb_scene_set_build_options); call before build_bvh() / commit()."""
        o = F.BuildOptions(max_leaf_triangles, 1 if keep_huge_primitives_out else 0, open_min_extent, 0)
        F.check(self.lib.rtb_scene_set_build_options(self.h, C.byref(o)))

    def build_bvh(self):
        F.check(self.lib.rtb_scene_build_bvh(self.h))

    def commit(self):
        F.check(self.lib.rtb_scene_commit(self.h))

    def info(self):
        i = F.SceneInfo()
        F.check(self.lib.rtb_scene_get_info(self.h, C.byref(i)))
        return i.as_dict()

    def export_bvh(self):
        info = self.info()
        nodes = np.zeros(info["n_bvh_nodes"] * 80, dtype=np.uint8)
        F.check(self.lib.rtb_scene_export_bvh(self.h, F.ptr(nodes), nodes.nbytes))
        prims = []
        counts = [info["n_spheres"], info["n_moving"], info["n_quads"], info["n_triangles"]]
        words = [4, 8, 12, 12]
        for t in range(4):
            g = np.zeros(counts[t] * words[t], dtype=np.float32)
            inf = np.zeros(counts[t] * 2, dtype=np.uint32)
            if counts[t]:
                F.check(self.lib.rtb_scene_export_prims(self.h, t, F.ptr(g), g.nbytes, F.ptr(inf), inf.nbytes))
            prims.append((g, inf))
        return nodes, prims

    def export_exact(self):
        """([records of spheres, moving spheres, quads] as float64 arrays of 16 per primitive, coord_max, eps_ab)"""
        info = self.info()
        counts = [info["n_spheres"], info["n_moving"], info["n_quads"]]
        cm, ea = C.c_float(), C.c_float()
        out = []
        for t in range(3):
            a = np.zeros(counts[t] * 16, dtype=np.float64)
            F.check(self.lib.rtb_scene_export_exact(self.h, t, F.ptr(a) if counts[t] else None, a.nbytes, C.byref(cm),
                                                    C.byref(ea)))
            out.append(a)
        return out, cm.value, ea.value

    def export_globals(self):
        """refs (type << 29 | index) of the primitives that are tested for every ray instead of living in the tree"""
        refs = np.zeros(64, dtype=np.uint32)
        n = C.c_uint32()
        F.check(self.lib.rtb_scene_export_globals(self.h, F.ptr(refs), 64, C.byref(n)))
        return refs[:n.value].copy()

    # ---- hot path -------------------------------------------------------------------------------------------
    def render(self, cam: F.Camera, params: F.Params, readback: bool = True):
        """rtb_render: returns (accum (H,W,4) float32 or None, stats dict)."""
        st = F.Stats()
        out = np.empty((params.height, params.width, 4), dtype=np.float32) if readback else None
        F.check(self.lib.rtb_render(self.ctx.h, self.h, C.byref(cam), C.byref(params), F.ptr(out), C.byref(st)))
        return out, st.as_dict()

    def render_device(self, cam: F.Camera, params: F.Params, d_accum_ptr: int, stream_ptr: int = 0):
        """rtb_render_device: accumulate into a caller-owned device buffer (e.g. a torch tensor's data_ptr())."""
        st = F.Stats()
        F.check(self.lib.rtb_render_device(self.ctx.h, self.h, C.byref(cam), C.byref(params), C.c_void_p(d_accum_ptr),
                                           C.c_void_p(stream_ptr), C.byref(st)))
        return st.as_dict()

    def render_aov(self, cam: F.Camera, params: F.Params, readback: bool = True):
        """rtb_render_aov: denoiser guide sums of the render's first segments -> ((H,W,8) float32 or None, stats dict).
        Per pixel: albedo rgb, coverage, shading normal xyz, depth, each summed over samples (io.aov_images divides)."""
        st = F.Stats()
        out = np.empty((params.height, params.width, 8), dtype=np.float32) if readback else None
        F.check(self.lib.rtb_render_aov(self.ctx.h, self.h, C.byref(cam), C.byref(params), F.ptr(out), C.byref(st)))
        return out, st.as_dict()

    def render_aov_device(self, cam: F.Camera, params: F.Params, d_ptr: int, stream_ptr: int = 0):
        """rtb_render_aov_device: sum the guide values into a caller-owned device buffer of W*H*8 floats."""
        st = F.Stats()
        F.check(self.lib.rtb_render_aov_device(self.ctx.h, self.h, C.byref(cam), C.byref(params), C.c_void_p(d_ptr),
                                               C.c_void_p(stream_ptr), C.byref(st)))
        return st.as_dict()

    def finalize_rgb8(self, width, height, total_spp, d_accum_ptr: int = 0):
        out = np.empty((height, width, 3), dtype=np.uint8)
        F.check(self.lib.rtb_finalize_rgb8(self.ctx.h, C.c_void_p(d_accum_ptr) if d_accum_ptr else None, width, height,
                                           total_spp, F.ptr(out)))
        return out

    def primary_hits(self, cam: F.Camera, width: int, height: int):
        ids = np.empty((height, width), dtype=np.uint32)
        ts = np.empty((height, width), dtype=np.float32)
        st = F.Stats()
        F.check(self.lib.rtb_primary_hits(self.ctx.h, self.h, C.byref(cam), width, height, F.ptr(ids), F.ptr(ts),
                                          C.byref(st)))
        return ids, ts, st.as_dict()

    def trace_rays(self, origin, direction, time=None):
        o = np.ascontiguousarray(origin, dtype=np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(direction, dtype=np.float32).reshape(-1, 3)
        tm = None if time is None else np.ascontiguousarray(time, dtype=np.float32)
        ids = np.empty(len(o), dtype=np.uint32)
        ts = np.empty(len(o), dtype=np.float32)
        st = F.Stats()
        F.check(self.lib.rtb_trace_rays(self.ctx.h, self.h, F.ptr(o), F.ptr(d), F.ptr(tm), len(o), F.ptr(ids), F.ptr(ts),
                                        C.byref(st)))
        return ids, ts, st.as_dict()


def make_params(width, height, spp, max_depth=50, background=(0.0, 0.0, 0.0), seed=1, sample_offset=0, total_spp=None,
                rr_start_depth=0, pool_paths=0, flags=0) -> F.Params:
    p = F.Params()
    p.width, p.height, p.spp, p.sample_offset = width, height, spp, sample_offset
    p.total_spp = total_spp if total_spp is not None else spp
    p.max_depth, p.rr_start_depth, p.seed = max_depth, rr_start_depth, seed
    p.background[:] = background
    p.pool_paths, p.flags = pool_paths, flags
    return p
