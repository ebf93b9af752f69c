"""ctypes binding of include/rtb200.h (librtb200.so).  Loading fails loudly: there is no CPU fallback."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RTB200_LIB", os.path.join(_HERE, "librtb200.so"))  # RTB200_LIB: A/B builds only

RTB_NONE = 0xFFFFFFFF

# node / material / texture / light enums (include/rtb200.h)
NODE_SPHERE, NODE_MOVING_SPHERE, NODE_XY_RECT, NODE_XZ_RECT, NODE_YZ_RECT, NODE_BOX = 1, 2, 3, 4, 5, 6
NODE_TRIANGLE, NODE_QUAD, NODE_MESH = 7, 8, 9
NODE_TRANSLATE, NODE_ROTATE_Y, NODE_FLIP_FACE, NODE_CONSTANT_MEDIUM = 16, 17, 18, 19
NODE_LIST, NODE_BVH = 32, 33
MAT_LAMBERTIAN, MAT_METAL, MAT_DIELECTRIC, MAT_DIFFUSE_LIGHT, MAT_ISOTROPIC = 0, 1, 2, 3, 4
TEX_SOLID, TEX_CHECKER, TEX_NOISE, TEX_IMAGE = 0, 1, 2, 3
LIGHT_XZ_RECT, LIGHT_SPHERE = 0, 1
RENDER_ACCUMULATE, RENDER_COUNT, RENDER_TIME_EXTEND, RENDER_REDUCE = 1, 2, 4, 8
BW_L2_READ, BW_HBM_READ, BW_SHARED_READ = 0, 1, 2
(KAT_PHILOX, KAT_SPHERE, KAT_SPHERE_F64, KAT_LIGHTS_PDF, KAT_LIGHTS_RANDOM, KAT_PERLIN_NOISE, KAT_PERLIN_TURB, KAT_Q2F, KAT_ONB,
 KAT_REFLECT, KAT_REFRACT, KAT_CAMERA_RAY, KAT_MEDIA, KAT_TEXTURE, KAT_EXACT) = range(15)

NODE_DTYPE = np.dtype([("type", "<u4"), ("material", "<u4"), ("first_child", "<u4"), ("n_children", "<u4"),
                       ("p", "<f8", (12,))])
MATERIAL_DTYPE = np.dtype([("type", "<u4"), ("texture", "<u4"), ("param", "<f8")])
TEXTURE_DTYPE = np.dtype([("type", "<u4"), ("even", "<u4"), ("odd", "<u4"), ("table", "<u4"),
                          ("rgb", "<f8", (3,)), ("scale", "<f8")])
LIGHT_DTYPE = np.dtype([("type", "<u4"), ("_pad", "<u4"), ("p", "<f8", (5,))])
assert NODE_DTYPE.itemsize == 112 and MATERIAL_DTYPE.itemsize == 16 and TEXTURE_DTYPE.itemsize == 48
assert LIGHT_DTYPE.itemsize == 48


class Camera(C.Structure):
    """Camera::new arguments (raytracer/src/camera.rs:21-28)."""
    _fields_ = [("lookfrom", C.c_double * 3), ("lookat", C.c_double * 3), ("vup", C.c_double * 3),
                ("vfov_deg", C.c_double), ("aspect_ratio", C.c_double), ("aperture", C.c_double),
                ("focus_dist", C.c_double), ("time0", C.c_double), ("time1", C.c_double)]

    @classmethod
    def new(cls, lookfrom, lookat, vup, vfov, aspect_ratio, aperture, focus_dist, time0=0.0, time1=1.0):
        c = cls()
        c.lookfrom[:] = lookfrom
        c.lookat[:] = lookat
        c.vup[:] = vup
        c.vfov_deg, c.aspect_ratio, c.aperture, c.focus_dist = vfov, aspect_ratio, aperture, focus_dist
        c.time0, c.time1 = time0, time1
        return c


class Params(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("spp", C.c_uint32), ("sample_offset", C.c_uint32),
                ("total_spp", C.c_uint32), ("max_depth", C.c_int32), ("rr_start_depth", C.c_uint32),
                ("seed", C.c_uint32), ("background", C.c_float * 3), ("pool_paths", C.c_uint32),
                ("flags", C.c_uint32)]


class Stats(C.Structure):
    _fields_ = [("paths", C.c_uint64), ("segments", C.c_uint64), ("rejected", C.c_uint64),
                ("iterations", C.c_uint64), ("launches", C.c_uint64), ("extend_launches", C.c_uint64),
                ("ms_total", C.c_double), ("ms_extend", C.c_double), ("nodes_visited", C.c_uint64),
                ("prims_tested", C.c_uint64), ("exact_rays", C.c_uint64), ("refined_rays", C.c_uint64),
                ("ms_nccl", C.c_double), ("ms_render", C.c_double), ("n_devices", C.c_uint32), ("_pad", C.c_uint32),
                ("prims_tested_type", C.c_uint64 * 4), ("ms_nccl_wait", C.c_double)]

    def as_dict(self):
        return {k: (list(getattr(self, k)) if k == "prims_tested_type" else getattr(self, k)) for k, _ in self._fields_}


class BuildOptions(C.Structure):
    _fields_ = [("max_leaf_triangles", C.c_uint32), ("keep_huge_primitives_out", C.c_uint32),
                ("open_min_extent", C.c_float), ("_reserved", C.c_uint32)]


class SceneInfo(C.Structure):
    _fields_ = [("n_spheres", C.c_uint32), ("n_moving", C.c_uint32), ("n_quads", C.c_uint32),
                ("n_triangles", C.c_uint32), ("n_media", C.c_uint32), ("n_lights", C.c_uint32),
                ("n_materials", C.c_uint32), ("n_textures", C.c_uint32), ("n_prims", C.c_uint32),
                ("n_bvh_nodes", C.c_uint32), ("bvh_width", C.c_uint32), ("bvh_max_depth", C.c_uint32),
                ("bvh_bytes", C.c_uint64), ("prim_bytes", C.c_uint64), ("global_f64_mask", C.c_uint32),
                ("_pad", C.c_uint32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


# every symbol include/rtb200.h declares: name -> (restype, argtypes)
_VP, _U32, _I, _SZ = C.c_void_p, C.c_uint32, C.c_int, C.c_size_t
SIGNATURES = {
    "rtb_abi_version": (C.c_uint32, []),
    "rtb_last_error": (C.c_char_p, []),
    "rtb_context_create": (_I, [_I, C.POINTER(_VP)]),
    "rtb_context_destroy": (None, [_VP]),
    "rtb_context_create_multi": (_I, [C.POINTER(C.c_int), _I, C.POINTER(_VP)]),
    "rtb_context_device_count": (_I, [_VP]),
    "rtb_comm_unique_id": (_I, [_VP]),
    "rtb_context_comm_init": (_I, [_VP, _VP, _I, _I]),
    "rtb_context_device_info": (_I, [_VP, C.POINTER(_I), C.POINTER(_I), C.POINTER(_I), C.c_char_p, _SZ]),
    "rtb_scene_create": (_I, [_VP, C.POINTER(_VP)]),
    "rtb_scene_destroy": (None, [_VP]),
    "rtb_scene_set_materials": (_I, [_VP, _VP, _U32]),
    "rtb_scene_set_textures": (_I, [_VP, _VP, _U32]),
    "rtb_scene_set_image": (_I, [_VP, _U32, _VP, _U32, _U32]),
    "rtb_scene_set_perlin": (_I, [_VP, _U32, _VP, _VP, _VP, _VP]),
    "rtb_scene_set_mesh": (_I, [_VP, _U32, _VP, _U32, _VP, _U32]),
    "rtb_scene_set_mesh_attributes": (_I, [_VP, _U32, _VP, _U32, _VP, _VP, _U32, _VP]),
    "rtb_scene_set_lights": (_I, [_VP, _VP, _U32]),
    "rtb_scene_set_graph": (_I, [_VP, _VP, _U32, _VP, _U32, _U32]),
    "rtb_scene_set_spheres": (_I, [_VP, _VP, _VP, _VP, _VP, _U32]),
    "rtb_scene_set_moving_spheres": (_I, [_VP, _VP, _VP, _VP, _VP, _VP, _VP, _U32]),
    "rtb_scene_set_quads": (_I, [_VP, _VP, _VP, _VP, _VP, _VP, _VP, _U32]),
    "rtb_scene_set_triangles": (_I, [_VP, _VP, _VP, _VP, _VP, _VP, _VP, _U32]),
    "rtb_scene_set_media": (_I, [_VP, _VP, _U32]),
    "rtb_scene_set_build_options": (_I, [_VP, _VP]),
    "rtb_scene_build_bvh": (_I, [_VP]),
    "rtb_scene_commit": (_I, [_VP]),
    "rtb_scene_get_info": (_I, [_VP, C.POINTER(SceneInfo)]),
    "rtb_scene_export_bvh": (_I, [_VP, _VP, _SZ]),
    "rtb_scene_export_globals": (_I, [_VP, _VP, _U32, C.POINTER(C.c_uint32)]),
    "rtb_scene_export_prims": (_I, [_VP, _U32, _VP, _SZ, _VP, _SZ]),
    "rtb_scene_export_exact": (_I, [_VP, _U32, _VP, _SZ, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "rtb_scene_export_triangle_attributes": (_I, [_VP, _VP, _SZ]),
    "rtb_render": (_I, [_VP, _VP, C.POINTER(Camera), C.POINTER(Params), _VP, C.POINTER(Stats)]),
    "rtb_render_device": (_I, [_VP, _VP, C.POINTER(Camera), C.POINTER(Params), _VP, _VP, C.POINTER(Stats)]),
    "rtb_render_aov": (_I, [_VP, _VP, C.POINTER(Camera), C.POINTER(Params), _VP, C.POINTER(Stats)]),
    "rtb_render_aov_device": (_I, [_VP, _VP, C.POINTER(Camera), C.POINTER(Params), _VP, _VP, C.POINTER(Stats)]),
    "rtb_finalize_rgb8": (_I, [_VP, _VP, _U32, _U32, _U32, _VP]),
    "rtb_primary_hits": (_I, [_VP, _VP, C.POINTER(Camera), _U32, _U32, _VP, _VP, C.POINTER(Stats)]),
    "rtb_trace_rays": (_I, [_VP, _VP, _VP, _VP, _VP, _U32, _VP, _VP, C.POINTER(Stats)]),
    "rtb_debug_check_failures": (_I, [_VP, _VP]),
    "rtb_measure_bandwidth": (_I, [_VP, _U32, _U32, C.POINTER(C.c_double)]),
    "rtb_primary_rays": (_I, [_VP, C.POINTER(Camera), _U32, _U32, _VP, _VP, _VP]),
    "rtb_device_kat": (_I, [_VP, _VP, C.POINTER(Camera), C.POINTER(Params), _U32, _VP, _U32, _U32, _VP, _U32]),
}

_lib = None


class RtbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"rtb200 error {code}: {msg}")
        self.code = code


def load():
    """Load librtb200.so and bind every declared symbol.  Raises if the CUDA extension was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(the CUDA library is the only implementation; there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        if "RTB200_LIB" in os.environ and not hasattr(lib, name):
            continue  # A/B build of an older ABI (tools only)
        fn = getattr(lib, name)  # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise RtbError(rc, load().rtb_last_error().decode("utf-8", "replace"))


def ptr(a):
    """void* of a contiguous numpy array (or None)."""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.c_void_p)
