"""ctypes front-end of tests/ransac_oracle.c, the CPU restatement of the RANSAC solve's hypothesis stage.  TEST INFRASTRUCTURE
ONLY.  The library is compiled on first use into a per-user directory under the system's temporary directory, named by the
hash of its source, so that a read-only checkout works and an edited source is rebuilt."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ransac_oracle.c")
_lib = None


def build():
    """compile ransac_oracle.c (once per source version) and return the path of the shared library"""
    src = open(_SRC, "rb").read()
    d = os.path.join(tempfile.gettempdir(), "pnpb200_tests_%d" % os.getuid())
    os.makedirs(d, exist_ok=True)
    path = os.path.join(d, "ransac_oracle_%s.so" % hashlib.sha1(src).hexdigest()[:16])
    if not os.path.exists(path):
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else os.environ.get("CC", "gcc")
        tmp = "%s.%d.tmp" % (path, os.getpid())
        subprocess.check_call([cc, "-O2", "-fPIC", "-fvisibility=hidden", "-std=c99", "-D_GNU_SOURCE", "-shared", "-o", tmp, _SRC, "-lm"])
        os.replace(tmp, path)                                  # atomic: parallel workers never load a half-written file
    return path


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        for name in ("ransac_oracle_p3p", "ransac_oracle_hypothesize_one"):
            getattr(_lib, name).restype = C.c_int
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def p3p(X, f):
    """Grunert's P3P (a quartic, Ferrari, Newton polish; pose by triads): X [3,3] pattern points, f [3,3] unit bearings.
    Returns (R [k,3,3], t [k,3]) for the k <= 4 roots with positive finite depths."""
    X, f = _f64(X).reshape(9), _f64(f).reshape(9)
    R, t = np.zeros(36), np.zeros(12)
    k = lib().ransac_oracle_p3p(_p(X), _p(f), _p(R), _p(t))
    return R[:9 * k].reshape(k, 3, 3), t[:3 * k].reshape(k, 3)


def draw4(c, g, s, seed=0):
    """the candidate positions (0 .. c-1, in draw order) of sample s of problem g in the hypothesis stage"""
    pos = np.zeros(4, np.int32)
    lib().ransac_oracle_draw4(C.c_int(c), C.c_uint64(int(g)), C.c_int(int(s)), C.c_uint64(int(seed)), _p(pos))
    return pos


def hypothesize_one(uv, patterns, K, cand, g, samples=128, consensus_px=4.0, confidence=0.999, seed=0):
    """The rule of pnpb200_hypothesize_batch for one problem: uv [n_total,2], patterns [P,n_total,3], cand = its candidates
    (landmark indices in candidate order), g = idx0 + b.  Returns dict(R, t, best_pattern, mask bool [n_total], consensus,
    sample (the winner's index, -1: none), drawn, near (some decision distance within 1e-9 relative of a threshold))."""
    uv, patterns, K = _f64(uv), _f64(patterns), _f64(K)
    if patterns.ndim == 2:
        patterns = patterns[None]
    n_total = uv.shape[0]
    cand = np.ascontiguousarray(cand, dtype=np.int32)
    R, t, mask = np.zeros(9), np.zeros(3), np.zeros(n_total, np.uint8)
    bp, cons, ws, near = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
    drawn = lib().ransac_oracle_hypothesize_one(
        C.c_int(len(cand)), _p(cand), C.c_int(n_total), _p(uv), C.c_int(patterns.shape[0]), _p(patterns), _p(K), C.c_int(int(samples)),
        C.c_double(consensus_px), C.c_double(confidence), C.c_uint64(int(seed)), C.c_uint64(int(g)), _p(R), _p(t), C.byref(bp),
        _p(mask), C.byref(cons), C.byref(ws), C.byref(near))
    return dict(R=R.reshape(3, 3), t=t, best_pattern=bp.value, mask=mask.astype(bool), consensus=cons.value, sample=ws.value,
                drawn=int(drawn), near=bool(near.value))
