"""TEST INFRASTRUCTURE: ctypes binding of oracle/_ref/libope_ref_{mod,modcorr}.so — the reference's own vendored registration
sources (VP) compiled against the mock PCL of oracle/refstub (see oracle/ref_harness.cpp). Used by tests/test_ref.py to pin
the oracle's restatement of the VP-held half of the path. Never imported by the product.

The reference's sources are not part of this repository. Where oracle/_ref cannot be built, Recorded answers the same calls
from tests/golden/ref_registration.json (made by tests/golden/make_ref_golden.py)."""
import ctypes as C
import hashlib
import json
import os
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(_HERE), "object-pose-estimation_b200"))
import abi_types as T  # noqa: E402

_LIBS = {}
f32p = C.POINTER(C.c_float)


def available():
    return all(os.path.exists(os.path.join(_HERE, "_ref", "libope_ref_%s.so" % v)) for v in ("mod", "modcorr"))


def lib(variant="mod"):
    if variant not in _LIBS:
        # the oracle first (RTLD_GLOBAL): the harness resolves orc_point_to_plane from it
        C.CDLL(os.path.join(_HERE, "libope_oracle.so"), mode=C.RTLD_GLOBAL)
        L = C.CDLL(os.path.join(_HERE, "_ref", "libope_ref_%s.so" % variant), mode=os.RTLD_LOCAL | os.RTLD_NOW)
        L.ref_variant.restype = C.c_char_p
        _LIBS[variant] = L
    return _LIBS[variant]


def _xyz(a):
    return np.ascontiguousarray(np.asarray(a, np.float32)[:, :3])


def _corr_buf(fixed):
    n = 0 if fixed is None else len(fixed[0])
    buf = (T.Correspondence * max(n, 1))()
    for i in range(n):
        buf[i] = T.Correspondence(int(fixed[0][i]), int(fixed[1][i]), float(fixed[2][i]) if len(fixed) > 2 else 0.0)
    return buf, n


def icp(src, tgt, prm, guess=None, src_normals=None, tgt_normals=None, fixed=None, variant="mod", want_corr=False):
    """returns dict(res=RegResult, corr=(q, m, d), aligned=(n,3), fitness, align_strength)"""
    s, t = _xyz(src), _xyz(tgt)
    sn = None if src_normals is None else np.ascontiguousarray(src_normals, np.float32)
    tn = None if tgt_normals is None else np.ascontiguousarray(tgt_normals, np.float32)
    res = T.RegResult()
    cbuf = (T.Correspondence * (len(s) + (0 if fixed is None else 2 * len(fixed[0])) + 1))()
    aligned = np.zeros((len(s), 3), np.float32)
    fit, strength = C.c_double(0), C.c_double(0)
    fbuf, nf = _corr_buf(fixed)
    g = None if guess is None else T.mat4_to_c(guess)
    rc = lib(variant).ref_icp(s.ctypes.data_as(f32p), C.c_size_t(len(s)), None if sn is None else sn.ctypes.data_as(f32p),
                              t.ctypes.data_as(f32p), C.c_size_t(len(t)), None if tn is None else tn.ctypes.data_as(f32p),
                              C.byref(prm), g, fbuf, C.c_size_t(nf), C.byref(res), cbuf, aligned.ctypes.data_as(f32p),
                              C.byref(fit), C.byref(strength))
    if rc != 0:
        raise RuntimeError("ref_icp rc=%d" % rc)
    a = np.ctypeslib.as_array(cbuf)[:res.n_correspondences]
    return {"res": res, "corr": (a["index_query"].copy(), a["index_match"].copy(), a["distance"].copy()), "aligned": aligned,
            "fitness": fit.value, "align_strength": strength.value}


def correspondences(src, tgt, max_distance, reciprocal=False, fixed=None, variant="mod"):
    s, t = _xyz(src), _xyz(tgt)
    fbuf, nf = _corr_buf(fixed)
    out = (T.Correspondence * (len(s) + nf + 1))()
    n = C.c_size_t(0)
    rc = lib(variant).ref_correspondences(s.ctypes.data_as(f32p), C.c_size_t(len(s)), t.ctypes.data_as(f32p), C.c_size_t(len(t)),
                                          C.c_double(max_distance), int(bool(reciprocal)), fbuf, C.c_size_t(nf), out, C.byref(n))
    if rc != 0:
        raise RuntimeError("ref_correspondences rc=%d" % rc)
    a = np.ctypeslib.as_array(out)[:n.value]
    return a["index_query"].copy(), a["index_match"].copy(), a["distance"].copy()


# ---- the recorded reference: what oracle/_ref returned, keyed by the inputs of each call ----
GOLDEN = os.path.join(os.path.dirname(_HERE), "tests", "golden", "ref_registration.json")


def digest(a):
    """SHA-256 of an array's shape and values (integers widened to int64, floats to float64): equal digests, equal values"""
    a = np.asarray(a)
    a = np.ascontiguousarray(a, np.int64 if a.dtype.kind in "biu" else np.float64)
    h = hashlib.sha256(repr(a.shape).encode())
    h.update(a.tobytes())
    return h.hexdigest()


def same_values(a, b):
    """a equals b bit for bit, where b is an array or the digest() of one (a recorded result)"""
    return digest(a) == b if isinstance(b, str) else np.array_equal(a, b)


def _key(kind, arrays, scalars):
    h = hashlib.sha256(kind.encode())
    for a in arrays:
        h.update(b"-" if a is None else digest(a).encode())
    h.update(repr(scalars).encode())
    return h.hexdigest()[:32]


def _params(prm):
    return [(name, list(v) if isinstance(v, C.Array) else v) for name, v in ((f[0], getattr(prm, f[0])) for f in prm._fields_)]


def icp_key(src, tgt, prm, guess=None, src_normals=None, tgt_normals=None, fixed=None, variant="mod"):
    g = None if guess is None else np.asarray(guess, np.float32)
    return _key("icp", [_xyz(src), _xyz(tgt), src_normals, tgt_normals, g] + list(fixed or ()), [_params(prm), variant])


def correspondences_key(src, tgt, max_distance, reciprocal=False, fixed=None, variant="mod"):
    return _key("correspondences", [_xyz(src), _xyz(tgt)] + list(fixed or ()), [float(max_distance), bool(reciprocal), variant])


class Recorded:
    """icp() and correspondences() answered from GOLDEN: the scalars and transforms oracle/_ref returned, and digest()s of its
    arrays. Inputs that were not recorded raise KeyError; so does a field of a result that was not recorded."""
    T = T

    def __init__(self, path=GOLDEN):
        with open(path) as f:
            self.calls = json.load(f)["calls"]

    def _get(self, key):
        if key not in self.calls:
            raise KeyError("no recorded reference result for these inputs (tests/golden/make_ref_golden.py records them)")
        return self.calls[key]

    def icp(self, src, tgt, prm, guess=None, src_normals=None, tgt_normals=None, fixed=None, variant="mod", want_corr=False):
        r = dict(self._get(icp_key(src, tgt, prm, guess, src_normals, tgt_normals, fixed, variant)))
        r.pop("case", None)
        if "res" in r:
            res = T.RegResult()
            res.T[:] = r["res"]["T"]
            for name in ("converged", "state", "iterations", "n_correspondences"):
                setattr(res, name, r["res"][name])
            r["res"] = res
        if "corr" in r:
            r["corr"] = tuple(r["corr"])
        return r

    def correspondences(self, src, tgt, max_distance, reciprocal=False, fixed=None, variant="mod"):
        return tuple(self._get(correspondences_key(src, tgt, max_distance, reciprocal, fixed, variant))["corr"])
