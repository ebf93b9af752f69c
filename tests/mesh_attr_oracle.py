"""f64 reference of smooth-shaded, UV-mapped meshes (TEST INFRASTRUCTURE ONLY): tests/oracle_mesh_attributes.cpp, compiled
with the CPU oracle and tests/oracle_aov.cpp into one library, bound with the oracle's own ctypes signatures
(oracle/orc.py) plus the attribute entry points."""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

import aov_oracle
import orc

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def load():
    """Compile into a temporary directory (the tree may be read-only), load, and remove the file again."""
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="rtb_attr_oracle_")
        try:
            so = os.path.join(tmp, "liboracle_attr.so")
            subprocess.check_call([os.environ.get("CXX", "g++"), *aov_oracle.CXXFLAGS, "-o", so,
                                   os.path.join(_HERE, "oracle_mesh_attributes.cpp")])
            saved = orc._lib, orc.LIB_PATH
            try:
                orc._lib, orc.LIB_PATH = None, so
                lib = orc.load()
            finally:
                orc._lib, orc.LIB_PATH = saved
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        _VP, _U32 = C.c_void_p, C.c_uint32
        lib.orc_aov_rays.argtypes = [_VP, _VP, _VP, _VP, _VP, _VP, _U32, _U32, _VP, _VP, _VP]
        lib.orc_aov_rays_attr.argtypes = [_VP, _VP, _VP, _VP, _VP, _VP, _U32, _U32, _VP, _VP, _VP]
        lib.orc_scene_set_mesh_attributes.argtypes = [_VP, _U32, _VP, _U32, _VP, _VP, _U32, _VP]
        lib.orc_attr_reset.argtypes = [_VP]
        lib.orc_render_attr.argtypes = [_VP, _VP, _VP, _VP, _VP, _VP, C.c_int]
        _lib = lib
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class OracleScene(aov_oracle.OracleScene):
    """The oracle scene with the compiled scene's mesh attributes; render() and aov_rays() shade with them."""

    def __init__(self, cs):
        lib = load()
        saved = orc._lib, aov_oracle._lib
        orc._lib, aov_oracle._lib = lib, lib
        try:
            super().__init__(cs)
        finally:
            orc._lib, aov_oracle._lib = saved
        lib.orc_attr_reset(self.h)
        for i, attrs in enumerate(cs.mesh_attrs):
            if attrs is None:
                continue
            n, ni, uv, ui = attrs
            rc = lib.orc_scene_set_mesh_attributes(self.h, i, _p(n), 0 if n is None else len(n), _p(ni), _p(uv),
                                                   0 if uv is None else len(uv), _p(ui))
            assert rc == 0

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.orc_attr_reset(self.h)
        super().__del__()

    def render(self, cam, params, threads=0):
        acc = np.zeros((params.height, params.width, 4), dtype=np.float64)
        seg, rej = C.c_uint64(), C.c_uint64()
        rc = self.lib.orc_render_attr(self.h, C.byref(cam), C.byref(params), _p(acc), C.byref(seg), C.byref(rej), threads)
        assert rc == 0
        return acc, seg.value, rej.value

    def aov_rays(self, origin, direction, time, pixel, sample, seed, background=(0.0, 0.0, 0.0)):
        o = np.ascontiguousarray(origin, dtype=np.float64).reshape(-1, 3)
        d = np.ascontiguousarray(direction, dtype=np.float64).reshape(-1, 3)
        n = len(o)
        tm = np.ascontiguousarray(np.broadcast_to(np.asarray(time, dtype=np.float64), (n,)))
        px = np.ascontiguousarray(np.broadcast_to(np.asarray(pixel, dtype=np.uint32), (n,)))
        sm = np.ascontiguousarray(np.broadcast_to(np.asarray(sample, dtype=np.uint32), (n,)))
        ids = np.empty(n, dtype=np.uint32)
        vals = np.empty((n, 8), dtype=np.float64)
        kinds = np.empty(n, dtype=np.uint32)
        rc = self.lib.orc_aov_rays_attr(self.h, _p(o), _p(d), _p(tm), _p(px), _p(sm), seed, n, _p(ids), _p(vals), _p(kinds))
        assert rc == 0
        miss = ids == 0xFFFFFFFF
        vals[miss, 0:3] = np.clip(np.asarray(background, dtype=np.float64), 0.0, 1.0)
        return ids, vals, kinds
