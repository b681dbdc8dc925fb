"""TEST INFRASTRUCTURE: ctypes binding of tests/cpp/orc_normals_radius.cpp, the CPU reference of ope_normals_radius.

The library is compiled on first use with the oracle's flags into a temporary directory keyed by the source's hash, so nothing is
written into the tree."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_SRC = os.path.join(_ROOT, "tests", "cpp", "orc_normals_radius.cpp")
_ORACLE = os.path.join(_ROOT, "oracle")
_LIB = None
f32p = C.POINTER(C.c_float)


def lib():
    global _LIB
    if _LIB is None:
        h = hashlib.sha256()
        for p in (_SRC, os.path.join(_ORACLE, "orc_kdtree.h"), os.path.join(_ORACLE, "orc_linalg.h")):
            with open(p, "rb") as f:
                h.update(f.read())
        d = os.path.join(tempfile.gettempdir(), "ope_orc_radius_%d_%s" % (os.getuid(), h.hexdigest()[:16]))
        path = os.path.join(d, "liborc_radius.so")
        if not os.path.exists(path):
            os.makedirs(d, exist_ok=True)
            tmp = "%s.%d" % (path, os.getpid())
            subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-shared", "-I" + _ORACLE, "-o", tmp,
                            _SRC], check=True)
            os.replace(tmp, path)
        L = C.CDLL(path)
        L.orc_normals_radius.argtypes = [f32p, C.c_size_t, C.c_size_t, C.c_float, f32p, f32p]
        _LIB = L
    return _LIB


def normals_radius(pts, r, vp=(0, 0, 0)):
    """(n, 4) nx, ny, nz, curvature of NormalEstimation with setRadiusSearch(r), on the CPU"""
    p = np.ascontiguousarray(pts, np.float32)
    assert p.ndim == 2 and p.shape[1] >= 3
    out = np.empty((p.shape[0], 4), np.float32)
    v = (C.c_float * 3)(*vp)
    rc = lib().orc_normals_radius(p.ctypes.data_as(f32p), p.shape[0], p.shape[1], C.c_float(r), v, out.ctypes.data_as(f32p))
    if rc != 0:
        raise RuntimeError("orc_normals_radius failed: rc=%d" % rc)
    return out
