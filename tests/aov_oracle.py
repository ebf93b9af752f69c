"""f64 reference of rtb_render_aov (TEST INFRASTRUCTURE ONLY): tests/oracle_aov.cpp, compiled together with the CPU oracle
into one library, bound with the oracle's own ctypes signatures (oracle/orc.py) plus `orc_aov_rays`."""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

import orc

_HERE = os.path.dirname(os.path.abspath(__file__))
# oracle/Makefile's flags: -ffp-contract=off keeps every f64 operation rounded on its own, as in the oracle library
CXXFLAGS = ["-O3", "-march=x86-64-v3", "-ffp-contract=off", "-std=c++17", "-fPIC", "-pthread", "-shared"]
_lib = None


def load():
    """Compile into a temporary directory (the tree may be read-only), load, and remove the file again."""
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="rtb_aov_oracle_")
        try:
            so = os.path.join(tmp, "liboracle_aov.so")
            subprocess.check_call([os.environ.get("CXX", "g++"), *CXXFLAGS, "-o", so, os.path.join(_HERE, "oracle_aov.cpp")])
            saved = orc._lib, orc.LIB_PATH
            try:
                orc._lib, orc.LIB_PATH = None, so
                lib = orc.load()
            finally:
                orc._lib, orc.LIB_PATH = saved
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        _VP = C.c_void_p
        lib.orc_aov_rays.argtypes = [_VP, _VP, _VP, _VP, _VP, _VP, C.c_uint32, C.c_uint32, _VP, _VP, _VP]
        _lib = lib
    return _lib


class OracleScene(orc.OracleScene):
    """orc.OracleScene on the library that also holds orc_aov_rays."""

    def __init__(self, cs):
        lib = load()
        saved = orc._lib
        orc._lib = lib
        try:
            super().__init__(cs)
        finally:
            orc._lib = saved

    def aov_rays(self, origin, direction, time, pixel, sample, seed, background=(0.0, 0.0, 0.0)):
        """-> (ids (n,) uint32, vals (n, 8) float64 per-sample guide values with `background` as the albedo of a miss,
        kinds (n,) uint32 texture type of the albedo, 0xFF if it is not a texture value)."""
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        o = np.ascontiguousarray(origin, dtype=np.float64).reshape(-1, 3)
        d = np.ascontiguousarray(direction, dtype=np.float64).reshape(-1, 3)
        n = len(o)
        tm = np.ascontiguousarray(np.broadcast_to(np.asarray(time, dtype=np.float64), (n,)))
        px = np.ascontiguousarray(np.broadcast_to(np.asarray(pixel, dtype=np.uint32), (n,)))
        sm = np.ascontiguousarray(np.broadcast_to(np.asarray(sample, dtype=np.uint32), (n,)))
        ids = np.empty(n, dtype=np.uint32)
        vals = np.empty((n, 8), dtype=np.float64)
        kinds = np.empty(n, dtype=np.uint32)
        rc = self.lib.orc_aov_rays(self.h, p(o), p(d), p(tm), p(px), p(sm), seed, n, p(ids), p(vals), p(kinds))
        assert rc == 0
        miss = ids == 0xFFFFFFFF
        vals[miss, 0:3] = np.clip(np.asarray(background, dtype=np.float64), 0.0, 1.0)
        return ids, vals, kinds
