"""The C parity oracle with per-landmark weights.  TEST INFRASTRUCTURE ONLY.

oracle/pnp_oracle.c is the pinned restatement of the reference and stays as it is.  This module compiles a weighted variant
of that same source: it applies the rule of include/pnpb200.h literally -- each landmark's two measurement rows of the
residual and the Jacobian multiplied by sqrt(w) (LM, LM+'s LM stage; QEIF and EIF2 through H^T Q^-1 H, which is Q^-1 times w
on the landmark's rows), the linear stages' least-squares rows multiplied by sqrt(w) -- at the three places where the rows
are made (the measurement model qekf_hx_H / ekf2_hx_H_ex, and the systems of F1 and F2).  Everything else is the oracle's
own code.  With sqrt(w) = 1 a row is left untouched, so all weights 1 give the unweighted oracle bit for bit.  The numerics
deliberately differ from the device's weighted moments.  Landmarks whose weight does not take part (not 0 < w < +Inf as
float32) are dropped before the solve, as the masked oracle tests compact their problems.  Fewer than 4 left: NaN pose and
res_norm, 0 iterations (the masked rule).  Compiled on first use into a per-user temporary directory named by the hash of
the generated source."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle as orc

_ORACLE_SRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "pnp_oracle.c")
_lib = None

_SQRTW = """
/* ---- weighted variant (tests/weighted_oracle.py): sqrt(w_i) of the problem being solved, or NULL ---- */
static __thread const double *g_sw = NULL;
"""

_QEKF_WRAP = """
/* the landmark's rows of z - hx and H times sqrt(w): hx' = z - s (z - hx), so that every z - hx the solver forms is s (z - hx) */
static void qekf_hx_H(int n, const double *x, const double *bx, const double *by, const double *P, double *hx, double *H)
{
    int i, c;
    qekf_hx_H_unweighted(n, x, bx, by, P, hx, H);
    if (!g_sw) return;
    for (i = 0; i < n; ++i) {
        const double s = g_sw[i];
        if (s == 1.0) continue;
        hx[i] = bx[i] - s * (bx[i] - hx[i]);
        hx[n + i] = by[i] - s * (by[i] - hx[n + i]);
        for (c = 0; c < 6; ++c) { H[i * 6 + c] *= s; H[(n + i) * 6 + c] *= s; }
    }
}

"""

_EKF2_WRAP = """
/* the landmark's two measurement rows of z - hx and J times sqrt(w); the nine constraint rows stay as they are */
static void ekf2_hx_H_ex(int n, const double *x, const double *bx, const double *by, const double *P, double *hx, double *J,
                         int true_jac)
{
    int i, c;
    ekf2_hx_H_ex_unweighted(n, x, bx, by, P, hx, J, true_jac);
    if (!g_sw) return;
    for (i = 0; i < n; ++i) {
        const double s = g_sw[i];
        if (s == 1.0) continue;
        hx[i] = bx[i] - s * (bx[i] - hx[i]);
        hx[n + i] = by[i] - s * (by[i] - hx[n + i]);
        for (c = 0; c < 12; ++c) { J[i * 12 + c] *= s; J[(n + i) * 12 + c] *= s; }
    }
}

"""

_ENTRY = """
/* one weighted problem: the landmarks with 0 < w < +Inf, each with its weight */
ORACLE_API int pnp_weighted_solve(int method, int n, const double *P, const double *uv, const double *K, const oracle_params_t *prm,
                                  const double *w, double *R, double *t, double *euler, double *res)
{
    double *buf = (double *)malloc(sizeof(double) * (size_t)(n > 0 ? n : 1) * 6);
    double *Pc = buf, *uvc = buf + 3 * n, *sw = buf + 5 * n;
    int i, m = 0, it = 0;
    for (i = 0; i < n; ++i) {
        const float wf = (float)w[i];
        if (!(wf > 0.0f && wf < (float)INFINITY)) continue;
        Pc[3 * m] = P[3 * i]; Pc[3 * m + 1] = P[3 * i + 1]; Pc[3 * m + 2] = P[3 * i + 2];
        uvc[2 * m] = uv[2 * i]; uvc[2 * m + 1] = uv[2 * i + 1];
        sw[m] = sqrt((double)wf);
        ++m;
    }
    if (m < 4) {
        for (i = 0; i < 9; ++i) R[i] = NAN;
        for (i = 0; i < 3; ++i) { t[i] = NAN; euler[i] = NAN; }
        *res = NAN;
        free(buf);
        return 0;
    }
    g_sw = sw;
    switch (method) {
    case 0: it = pnp_oracle_qeif(m, Pc, uvc, K, prm, R, t, euler, res, NULL); break;
    case 1: it = pnp_oracle_lm(m, Pc, uvc, K, prm, R, t, euler, res, NULL); break;
    case 2: it = pnp_oracle_linear_f2(m, Pc, uvc, K, prm, R, t, euler, res, NULL); break;
    case 3: it = pnp_oracle_linear_f1(m, Pc, uvc, K, prm, R, t, euler, res, NULL); break;
    case 4: it = pnp_oracle_lm_plus(m, Pc, uvc, K, prm, R, t, euler, res, NULL); break;
    default: it = pnp_oracle_eif2(m, Pc, uvc, K, prm, R, t, euler, res, NULL); break;
    }
    g_sw = NULL;
    free(buf);
    return it;
}

typedef struct { int method, n; const double *P, *uv, *K, *w; const oracle_params_t *prm; double *R, *t, *e, *res; int32_t *it; } wbatch_t;

static void wbatch_range(int64_t lo, int64_t hi, void *vctx)
{
    wbatch_t *c = (wbatch_t *)vctx;
    int64_t b;
    for (b = lo; b < hi; ++b)
        c->it[b] = pnp_weighted_solve(c->method, c->n, c->P, c->uv + (size_t)b * c->n * 2, c->K, c->prm, c->w + (size_t)b * c->n,
                                      c->R + b * 9, c->t + b * 3, c->e + b * 3, c->res + b);
}

ORACLE_API void pnp_weighted_solve_batch(int method, int64_t B, int n, const double *P, const double *uv, const double *K,
                                         const oracle_params_t *prm, const double *w, double *R, double *t, double *euler,
                                         double *res, int32_t *iters, int n_threads)
{
    wbatch_t c = { method, n, P, uv, K, w, prm, R, t, euler, res, iters };
    parallel_for(B, n_threads, 16, wbatch_range, &c);
}
"""


def _edit(s, old, new):
    assert s.count(old) == 1, old
    return s.replace(old, new)


def source():
    """the weighted variant of oracle/pnp_oracle.c"""
    s = open(_ORACLE_SRC).read()
    s = _edit(s, "#define ORACLE_API __attribute__((visibility(\"default\")))",
              "#define ORACLE_API __attribute__((visibility(\"default\")))\n" + _SQRTW)
    s = _edit(s, "static void qekf_hx_H(int n,", "static void qekf_hx_H_unweighted(int n,")
    s = _edit(s, "/* One QEIF solve.", _QEKF_WRAP + "/* One QEIF solve.")
    s = _edit(s, "static void ekf2_hx_H_ex(int n,", "static void ekf2_hx_H_ex_unweighted(int n,")
    s = _edit(s, "static void ekf2_hx_H(int n,", _EKF2_WRAP + "static void ekf2_hx_H(int n,")
    # linear F1: the rows of B and A times sqrt(w) (phi = pinv(A) B, res = ||B - A phi|| on the weighted rows)
    s = _edit(s, "    for (i = 0; i < n; ++i) { Ball[2 * i] = bx[i]; Ball[2 * i + 1] = by[i]; }   /* get_B_all :3094-3111 */",
              "    for (i = 0; i < n; ++i) { Ball[2 * i] = bx[i]; Ball[2 * i + 1] = by[i]; }   /* get_B_all :3094-3111 */\n"
              "    if (g_sw) for (i = 0; i < n; ++i) { Ball[2 * i] *= g_sw[i]; Ball[2 * i + 1] *= g_sw[i]; }")
    s = _edit(s, "        pinv_svd((int)m, 8, A, Ap, work);",
              "        if (g_sw) for (r = 0; r < m; ++r) for (k = 0; k < 8; ++k) A[r * 8 + k] *= g_sw[r / 2];\n"
              "        pinv_svd((int)m, 8, A, Ap, work);")
    # linear F2: the rows of D = [P | 1] and of B times sqrt(w) (D^+ is pinv of the weighted D; the residual rows follow)
    s = _edit(s, "    pinv_svd(n, 4, D, Dp, work);",
              "    if (g_sw) for (i = 0; i < n; ++i) for (k = 0; k < 4; ++k) D[i * 4 + k] *= g_sw[i];\n"
              "    pinv_svd(n, 4, D, Dp, work);\n"
              "    if (g_sw) for (i = 0; i < n; ++i) { bx[i] *= g_sw[i]; by[i] *= g_sw[i]; }")
    return s + _ENTRY


def build():
    src = source().encode()
    d = os.path.join(tempfile.gettempdir(), "pnpb200_tests_%d" % os.getuid())
    os.makedirs(d, exist_ok=True)
    h = hashlib.sha1(src).hexdigest()[:16]
    path = os.path.join(d, "weighted_oracle_%s.so" % h)
    if not os.path.exists(path):
        csrc = os.path.join(d, "weighted_oracle_%s.%d.c" % (h, os.getpid()))
        open(csrc, "wb").write(src)
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else os.environ.get("CC", "gcc")
        tmp = "%s.%d.tmp" % (path, os.getpid())
        subprocess.check_call([cc, "-O2", "-fPIC", "-pthread", "-fvisibility=hidden", "-std=c99", "-D_GNU_SOURCE", "-shared",
                               "-o", tmp, csrc, "-lm"])
        os.replace(tmp, path)
        os.remove(csrc)
    return path


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.pnp_weighted_solve.restype = C.c_int
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def solve_one(method, P, uv, K, w=None, params=None):
    """one problem; w=None is oracle.solve_one"""
    if w is None:
        return orc.solve_one(method, P, uv, K, params=params)
    m = orc.METHODS[method] if isinstance(method, str) else method
    P, uv, K, w = (np.ascontiguousarray(a, dtype=np.float64) for a in (P, uv, K, w))
    params = params or orc.default_params()
    R, t, e, res = np.zeros(9), np.zeros(3), np.zeros(3), C.c_double(0.0)
    it = lib().pnp_weighted_solve(m, P.shape[0], _p(P), _p(uv), _p(K), C.byref(params), _p(w), _p(R), _p(t), _p(e), C.byref(res))
    return dict(R=R.reshape(3, 3), t=t, euler=e, res_norm=res.value, iters=int(it))


def solve_batch(method, uv, P, K, w, params=None, n_threads=0):
    """uv [B, n, 2], P [n, 3], w [B, n] -> dict of arrays, each problem solved as solve_one does"""
    m = orc.METHODS[method] if isinstance(method, str) else method
    uv, P, K, w = (np.ascontiguousarray(a, dtype=np.float64) for a in (uv, P, K, w))
    B, n = uv.shape[0], uv.shape[1]
    params = params or orc.default_params()
    o = dict(R=np.zeros((B, 3, 3)), t=np.zeros((B, 3)), euler=np.zeros((B, 3)), res_norm=np.zeros(B), iters=np.zeros(B, np.int32))
    lib().pnp_weighted_solve_batch(C.c_int(m), C.c_int64(B), C.c_int(n), _p(P), _p(uv), _p(K), C.byref(params), _p(w), _p(o["R"]),
                                   _p(o["t"]), _p(o["euler"]), _p(o["res_norm"]), _p(o["iters"]), C.c_int(n_threads))
    return o
