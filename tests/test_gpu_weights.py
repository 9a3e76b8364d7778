"""Per-landmark weights (pnpb200_solve_batch_weighted, weights= in Python): weights in {0, 1} are the masked solve bit for bit,
integer weights are the problem with each landmark repeated that often, hidden values hide, and the filters' exit decisions in
the moment mapping stay certified or resolved under weights spanning six decades."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from pnp_solver_test_b200 import patterns as pt

from conftest import compare_solutions
from gpu_util import dev, oracle_stability
import weighted_oracle as wo
import weights_accuracy as wa

pytestmark = pytest.mark.gpu

MAP_AUTO, MAP_THREAD, MAP_MOMENT, MAP_WARP = 0, 1, 2, 32
FLAG_LM_TRUE_JACOBIAN = 4
KEYS = ("R", "t", "euler", "res_norm", "iters", "best_pattern")


def _workload(n, B, seed=42, quantized=True):
    pat = pt.get_golden_pattern() if n == 15 else pt.synthetic_pattern(n)
    P, K = pt.pattern_array(pat), pt.default_camera_matrix()
    w = orc.synth(0, B, P, K, cfg=orc.default_synth(seed=seed, is_quantized=quantized))
    return pat, P, K, w


def _solve(method, uv, pats, K, dtype=torch.float64, mapping=MAP_AUTO, flags=0, point_index=None, vis=None, weights=None):
    """the device solve; a refused call returns the exception instead of the outputs"""
    import pnp_solver_test_b200 as pnp
    try:
        out = pnp.solve_batch(method, dev(uv, dtype), dev(pats, dtype), K, point_index=point_index,
                              params=pnp.default_params(mapping=mapping, flags=flags),
                              visible=None if vis is None else torch.from_numpy(vis).cuda(),
                              weights=None if weights is None else torch.from_numpy(weights).cuda())
    except pnp.PnpB200Error as e:
        return e
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


def _assert_bits(a, b, what):
    for k in KEYS:
        x, y = np.ascontiguousarray(a[k]), np.ascontiguousarray(b[k])
        assert x.shape == y.shape and np.array_equal(x.view(np.uint8), y.view(np.uint8)), (what, k)


def _masks(B, sel, n_total, seed, lo=3):
    """per problem lo .. |sel| of the selected landmarks visible (row 0: all, row 1: exactly 3, so not solved)"""
    rng = np.random.default_rng(seed)
    vis = rng.random((B, n_total)) < 0.5                    # landmarks outside the selection: no effect either way
    for b in range(B):
        k = len(sel) if b == 0 else (3 if b == 1 else int(rng.integers(lo, len(sel) + 1)))
        vis[b, np.asarray(sel)] = False
        vis[b, np.asarray(sel)[rng.permutation(len(sel))[:k]]] = True
    return vis


# (n_total, selection, B, patterns): solve_pnp's 6 of 15, all 15, 68 (streaming chunks), 98, an unsorted selection of 40 of 68
# with two patterns (whole-row tiles), 300 (the per-warp streaming shape)
SHAPES = [(15, "six", 33, 1), (15, None, 31, 1), (68, None, 1037, 1), (98, None, 1, 1), (68, "unsorted", 33, 2), (300, None, 33, 1)]
METHODS = [("qeif", 0), ("lm", 0), ("lm_plus", 0), ("linear_f2", 0), ("linear_f1", 0), ("eif2", 0), ("lm", FLAG_LM_TRUE_JACOBIAN)]


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("method,flags", METHODS)
def test_binary_weights_are_the_masked_solve_bit_for_bit(method, flags, dtype):
    for n, subset, B, n_pat in SHAPES:
        pat, P, K, w = _workload(n, B, seed=n + B)
        rng = np.random.default_rng(n)
        sel = {None: None, "six": [list(pat).index(k) for k in pt.LM_KEY_LIST_6] if n == 15 else None,
               "unsorted": list(rng.permutation(68)[:40])}[subset]
        pats = P[None] if n_pat == 1 else np.stack([P, P * np.array([1.02, 0.97, 1.01])])
        vis = _masks(B, sel if sel is not None else list(range(n)), n, seed=B)
        wts = vis.astype(np.float32)
        for mapping in (MAP_AUTO, MAP_THREAD, MAP_WARP, MAP_MOMENT):
            m = _solve(method, w["uv"], pats, K, dtype, mapping, flags, sel, vis=vis)
            g = _solve(method, w["uv"], pats, K, dtype, mapping, flags, sel, weights=wts)
            what = (method, flags, dtype, n, subset, B, mapping)
            if isinstance(m, Exception):                    # a mapping the masked call refuses, the weighted one refuses too
                assert isinstance(g, Exception) and str(g).split(":")[1][:12] == str(m).split(":")[1][:12], (what, str(m), str(g))
                continue
            assert not isinstance(g, Exception), (what, str(g))
            if method == "eif2" and dtype == torch.float32 and mapping in (MAP_AUTO, MAP_THREAD, MAP_WARP):
                # FP32 EIF2 in the direct mappings: nvcc contracts the state's dot products (u_i . u_j) of eif2_loop differently
                # in the weighted instantiation, so the two agree to FP32 rounding, not bit for bit (DESIGN 9)
                assert np.array_equal(g["iters"], m["iters"]) and np.array_equal(g["best_pattern"], m["best_pattern"]), what
                ok = ~np.isnan(m["res_norm"])
                assert np.array_equal(np.isnan(g["res_norm"]), ~ok), what
                if ok.any():
                    assert np.abs(g["R"][ok] - m["R"][ok]).max() < 1e-3, what
                    assert (np.abs(g["t"][ok] - m["t"][ok]).max(axis=1) / np.abs(m["t"][ok][:, 2])).max() < 1e-3, what
                    assert np.abs(g["euler"][ok] - m["euler"][ok]).max() < 0.1, what
                    assert (np.abs(g["res_norm"][ok] - m["res_norm"][ok]) / m["res_norm"][ok]).max() < 1e-2, what
                continue
            _assert_bits(g, m, what)
            if B > 1:
                assert np.isnan(g["res_norm"][1]) and g["iters"][1] == 0, what      # 3 landmarks take part: not solved


@pytest.mark.parametrize("method,n,subset", [("qeif", 15, "six"), ("qeif", 68, None), ("lm", 68, None), ("eif2", 68, None),
                                             ("linear_f2", 68, None), ("linear_f1", 68, None), ("lm_plus", 68, None)])
def test_integer_weights_are_the_repeated_landmark_problem(method, n, subset):
    """weights in {0, 1, 2, 3} against the problem with landmark i repeated w_i times (point_index repeats indices): the device's
    unweighted solve of that problem and the oracle's, to the FP64 contract of DESIGN 4"""
    pat, P, K, w = _workload(n, 3 * 96, seed=11 + n)
    sel = [list(pat).index(k) for k in pt.LM_KEY_LIST_6] if subset == "six" else list(range(n))
    rng = np.random.default_rng(n)
    for g in range(3):                                    # three weight patterns, each shared by 96 problems (one point_index)
        rows = slice(96 * g, 96 * (g + 1))
        wi = rng.integers(1 if subset == "six" else 0, 4, size=n).astype(np.float32)
        wts = np.repeat(wi[None], 96, axis=0)
        rep = [j for j in sel for _ in range(int(wi[j]))]
        uv = w["uv"][rows]
        got = _solve(method, uv, P[None], K, point_index=sel if subset else None, weights=wts)
        dev_rep = _solve(method, uv, P[None], K, point_index=rep)
        ref, stable, it_stable = oracle_stability(method, uv[:, rep], P[rep], K)
        got["R"] = got["R"].reshape(-1, 3, 3)
        dev_rep["R"] = dev_rep["R"].reshape(-1, 3, 3)
        mask = stable if method in ("lm", "lm_plus") else None
        compare_solutions(got, ref, mask=mask, iters_mask=it_stable)
        compare_solutions(got, dev_rep, mask=mask, iters_mask=it_stable)


def _logw(rng, shape, lo=1e-3, hi=1e3):
    return np.exp(rng.uniform(np.log(lo), np.log(hi), size=shape)).astype(np.float32)


@pytest.mark.parametrize("quantized", [True, False])
@pytest.mark.parametrize("method", ["qeif", "eif2"])
def test_weighted_filter_exit_decisions_are_certified_or_resolved(method, quantized):
    """The moment mapping's exit decisions under weights from 1e-3 to 1e3 (an understated res2_error_bound certifies a decision
    the direct mapping takes the other way): iteration counts identical wherever the residual is above rounding noise"""
    B = 8192
    _, P, K, w = _workload(68, B, seed=5, quantized=quantized)
    wts = _logw(np.random.default_rng(3), (B, 68))
    a = _solve(method, w["uv"], P[None], K, mapping=MAP_MOMENT, weights=wts)
    d = _solve(method, w["uv"], P[None], K, mapping=MAP_THREAD, weights=wts)
    assert (a["iters"] > 0).all()                         # no mark survives the fix-up
    well = d["res_norm"] > 1e-10
    assert well.mean() > 0.9 or not quantized            # (noise-free: QEIF ends at rounding noise, no decision is well-posed)
    assert np.array_equal(a["iters"][well], d["iters"][well])
    R_a, R_d = a["R"].reshape(B, -1), d["R"].reshape(B, -1)
    assert np.abs(R_a - R_d).max() < 1e-9
    assert (np.abs(a["t"] - d["t"]).max(axis=1) / np.abs(d["t"][:, 2])).max() < 1e-9


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("method,n,subset", [("qeif", 15, "six"), ("lm", 68, None), ("eif2", 68, None), ("linear_f2", 68, None),
                                             ("qeif", 300, None)])
def test_hidden_weights_hide_and_too_few_is_not_solved(method, n, subset, dtype):
    """0, -0, -1, NaN, +Inf and -Inf hide a landmark: with NaN, +-Inf or garbage pixels under them every output is bit for bit
    that of weight 0 over finite pixels.  Fewer than 4 taking part: the masked rule's outputs, and the neighbours unaffected."""
    B = 67
    pat, P, K, w = _workload(n, B, seed=n)
    sel = [list(pat).index(k) for k in pt.LM_KEY_LIST_6] if subset == "six" else None
    rng = np.random.default_rng(1)
    base = _logw(rng, (B, n), 0.25, 4.0)
    hide = rng.random((B, n)) < 0.3
    cand = np.asarray(sel) if sel is not None else np.arange(n)
    hide[:, cand[:2]] = False
    few = [5, 40]                                         # these two keep only 3 landmarks
    for b in few:
        hide[b] = True
        hide[b, cand[:3]] = False
    ref_w = np.where(hide, np.float32(0), base)
    bad = np.array([0.0, -0.0, -1.0, np.nan, np.inf, -np.inf], np.float32)
    odd_w = np.where(hide, bad[rng.integers(0, 6, size=(B, n))], base)
    uv_bad = w["uv"].copy()
    junk = np.array([np.nan, np.inf, -np.inf, 1e300, -7.0])
    uv_bad[hide] = junk[rng.integers(0, 5, size=(int(hide.sum()), 2))]
    r = _solve(method, w["uv"], P[None], K, dtype, point_index=sel, weights=ref_w)
    g = _solve(method, uv_bad, P[None], K, dtype, point_index=sel, weights=odd_w)
    _assert_bits(g, r, (method, n, dtype))
    for b in few:
        assert np.isnan(g["R"][b]).all() and np.isnan(g["t"][b]).all() and np.isnan(g["res_norm"][b])
        assert g["iters"][b] == 0 and g["best_pattern"][b] == 0
    # the same batch with the two rows solvable: every other problem is bit for bit unchanged
    ok_w = ref_w.copy()
    ok_w[few] = base[few]
    o = _solve(method, w["uv"], P[None], K, dtype, point_index=sel, weights=ok_w)
    keep = np.setdiff1d(np.arange(B), few)
    _assert_bits({k: v[keep] for k, v in g.items()}, {k: v[keep] for k, v in o.items()}, "neighbours")


@pytest.mark.parametrize("method", ["lm", "qeif", "eif2", "linear_f1"])
def test_batch_independence_and_canary_rows(method):
    """a batch and its slices agree bit for bit (B stays below the filters' per-thread fix-up threshold, the header's one
    exception); rows past B of every output stay untouched"""
    import pnp_solver_test_b200 as pnp
    from pnp_solver_test_b200 import _lib
    B, n = 1037, 68
    _, P, K, w = _workload(n, B, seed=9)
    wts = _logw(np.random.default_rng(2), (B, n), 0.1, 10.0)
    full = _solve(method, w["uv"], P[None], K, weights=wts)
    for lo, hi in ((0, 1), (0, 31), (31, 64), (500, 1037)):
        part = _solve(method, w["uv"][lo:hi], P[None], K, weights=wts[lo:hi])
        _assert_bits({k: v[lo:hi] for k, v in full.items()}, part, (lo, hi))
    # canaries: outputs one row longer than B, filled with a pattern the solve must not touch
    Bs = 100
    uv, pat_t, w_t = dev(w["uv"][:Bs]), dev(P[None]), torch.from_numpy(wts[:Bs]).cuda()
    fill = -12345.0
    R = torch.full((Bs + 1, 9), fill, dtype=torch.float64, device="cuda")
    t, e = (torch.full((Bs + 1, 3), fill, dtype=torch.float64, device="cuda") for _ in range(2))
    res = torch.full((Bs + 1,), fill, dtype=torch.float64, device="cuda")
    it, best = (torch.full((Bs + 1,), -777, dtype=torch.int32, device="cuda") for _ in range(2))
    Kh = np.ascontiguousarray(K, dtype=np.float64)
    PI = C.POINTER(C.c_int32)
    rc = _lib.lib.pnpb200_solve_batch_weighted(
        _lib.METHODS[method], _lib.DTYPE_F64, Bs, n, n, C.c_void_p(uv.data_ptr()), C.c_void_p(pat_t.data_ptr()), 1, None,
        Kh.ctypes.data_as(C.POINTER(C.c_double)), None, C.c_void_p(R.data_ptr()), C.c_void_p(t.data_ptr()),
        C.c_void_p(e.data_ptr()), C.c_void_p(res.data_ptr()), C.cast(C.c_void_p(it.data_ptr()), PI),
        C.cast(C.c_void_p(best.data_ptr()), PI), C.cast(C.c_void_p(w_t.data_ptr()), C.POINTER(C.c_float)),
        C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0
    torch.cuda.synchronize()
    assert (R[Bs] == fill).all() and (t[Bs] == fill).all() and (e[Bs] == fill).all() and res[Bs] == fill
    assert it[Bs] == -777 and best[Bs] == -777
    assert np.array_equal(R[:Bs].cpu().numpy().reshape(-1), full["R"][:Bs].reshape(-1))
    # NULL / misaligned weights: EINVAL
    for wp in (None, C.c_void_p(w_t.data_ptr() + 2)):
        rc = _lib.lib.pnpb200_solve_batch_weighted(
            _lib.METHODS[method], _lib.DTYPE_F64, Bs, n, n, C.c_void_p(uv.data_ptr()), C.c_void_p(pat_t.data_ptr()), 1, None,
            Kh.ctypes.data_as(C.POINTER(C.c_double)), None, C.c_void_p(R.data_ptr()), None, None, None, None, None,
            None if wp is None else C.cast(wp, C.POINTER(C.c_float)), None)
        assert rc == -1


def test_solve_pnp_batch_weights_and_check():
    """the script-level entry: weights reach the weighted solve, and check= runs on the landmarks that take part"""
    import pnp_solver_test_b200 as pnp
    pat, P, K, w = _workload(68, 64, seed=3)
    s = pnp.PNP_SOLVER(K, [pat])
    wts = _logw(np.random.default_rng(4), (64, 68), 0.5, 2.0)
    wts[:, :5] = 0
    out = s.solve_pnp_batch(w["uv"], method="lm", weights=wts, check=2.0)
    ref = pnp.solve_batch("lm", dev(w["uv"]), dev(P[None]), K, weights=torch.from_numpy(wts).cuda())
    assert torch.equal(out["R"].cpu(), ref["R"].cpu())
    chk = pnp.check_batch(dev(w["uv"]), dev(P[None]), K, ref["R"], ref["t"], res_norm=ref["res_norm"], reproj_limit_px=2.0,
                          visible=torch.from_numpy(wts > 0).cuda())
    assert torch.equal(out["status"], chk["status"])


@pytest.mark.parametrize("method", ["qeif", "lm", "eif2", "linear_f2", "linear_f1", "lm_plus"])
def test_real_weights_match_the_weighted_oracle(method):
    """the float32 weights of the heteroscedastic accuracy workload, widened for the weighted oracle: FP64 to the contract of
    DESIGN 4 (LM on the oracle-stable subset, iteration counts wherever the decision is well-posed)"""
    P, K, uv, gt, wts = wa.workload("hetero")
    uv, wts = uv[:512], wts[:512]
    got = _solve(method, uv, P[None], K, weights=wts.astype(np.float32))
    got["R"] = got["R"].reshape(-1, 3, 3)
    ref = wo.solve_batch(method, uv, P, K, wts)
    stable, it_stable = np.ones(len(uv), bool), np.ones(len(uv), bool)
    for sgn in (1.0, -1.0):
        o = wo.solve_batch(method, uv * (1.0 + sgn * 1e-13), P, K, wts)
        d = np.maximum(np.abs(o["R"] - ref["R"]).reshape(len(uv), -1).max(axis=1),
                       np.abs(o["t"] - ref["t"]).max(axis=1) / np.abs(ref["t"][:, 2]))
        stable &= d < (1e-11 if method == "eif2" else 1e-10)   # (EIF2 under strong weights: the condition number amplifies rounding)
        it_stable &= o["iters"] == ref["iters"]
    compare_solutions(got, ref, mask=stable if method in ("lm", "lm_plus", "eif2") else None, iters_mask=it_stable)
