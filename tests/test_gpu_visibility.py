"""Per-problem landmark visibility (the *_masked entries, visible= in Python): every problem is solved, reported and checked
as the problem made of its visible landmarks alone, which the oracle pins problem by problem on the compacted inputs."""
import numpy as np
import pytest
import torch

from oracle import oracle as orc
from pnp_solver_test_b200 import patterns as pt

from conftest import compare_solutions
from gpu_util import dev, to_np

pytestmark = pytest.mark.gpu

METHODS = ("qeif", "lm", "linear_f2", "eif2", "linear_f1", "lm_plus")
NONFINITE, DEPTH, BEHIND, REPROJ = 1, 2, 4, 8


def _workload(n, B, seed=42):
    pat = pt.get_golden_pattern() if n == 15 else pt.synthetic_pattern(n)
    P, K = pt.pattern_array(pat), pt.default_camera_matrix()
    w = orc.synth(0, B, P, K, cfg=orc.default_synth(seed=seed))
    return pat, P, K, w


def _masks(B, n_sel, sel, n_total, seed, lo=6):
    """per problem 6 .. n_sel of the selected landmarks visible (row 0: all, row 1: exactly 6); [B, n_total] bool"""
    rng = np.random.default_rng(seed)
    vis = np.zeros((B, n_total), bool)
    for b in range(B):
        k = n_sel if b == 0 else (lo if b == 1 else int(rng.integers(lo, n_sel + 1)))
        vis[b, np.asarray(sel)[rng.permutation(n_sel)[:k]]] = True
    if n_sel < n_total:                                    # landmarks outside the selection may be visible or not: no effect
        vis[:, [j for j in range(n_total) if j not in set(sel)]] = rng.random((B, n_total - n_sel)) < 0.5
    return vis


def _compact(sel, vis_b):
    return [j for j in sel if vis_b[j]]


def _oracle(method, P, uv, K, vis, sel, patterns=None, stability=False):
    """each problem solved by the oracle on its visible selected landmarks (several patterns: the strict-< arg-min)"""
    patterns = P[None] if patterns is None else patterns
    B = uv.shape[0]
    ref = dict(R=np.full((B, 3, 3), np.nan), t=np.full((B, 3), np.nan), euler=np.full((B, 3), np.nan),
               res_norm=np.full(B, np.nan), iters=np.zeros(B, np.int64), best_pattern=np.zeros(B, np.int64))
    stable, it_stable = np.ones(B, bool), np.ones(B, bool)
    for b in range(B):
        c = _compact(sel, vis[b])
        if len(c) < 4:
            continue
        best = None
        for p in range(patterns.shape[0]):
            o = orc.solve_one(method, patterns[p][c], uv[b][c], K)
            if best is None or o["res_norm"] < best[0]["res_norm"]:
                best = (o, p)
        o, p = best
        ref["R"][b], ref["t"][b], ref["euler"][b] = o["R"], o["t"], o["euler"]
        ref["res_norm"][b], ref["iters"][b], ref["best_pattern"][b] = o["res_norm"], o["iters"], p
        if stability:
            for s in (1.0, -1.0):
                q = orc.solve_one(method, patterns[p][c], uv[b][c] * (1.0 + s * 1e-13), K)
                d = max(np.abs(q["R"] - o["R"]).max(), np.abs(q["t"] - o["t"]).max() / abs(o["t"][2]))
                stable[b] &= d < 1e-10
                it_stable[b] &= q["iters"] == o["iters"]
    return ref, stable, it_stable


def _solve(method, uv, P, K, vis=None, dtype=torch.float64, mapping=0, point_index=None, patterns=None, flags=0):
    import pnp_solver_test_b200 as pnp
    pats = (P[None] if patterns is None else patterns)
    out = pnp.solve_batch(method, dev(uv, dtype), dev(pats, dtype), K, point_index=point_index,
                          params=pnp.default_params(mapping=mapping, flags=flags),
                          visible=None if vis is None else torch.from_numpy(vis).cuda())
    torch.cuda.synchronize()
    return to_np(out)


def _full_rank(P, vis, sel):
    """the visible landmarks are not coplanar: D = [P | 1] has rank 4.  The linear stages need that -- the reference's pinv of a
    rank-deficient system has no counterpart in the device's LDL^T / SPD solves, which return NaN there (include/pnpb200.h)"""
    ok = np.ones(len(vis), bool)
    for b in range(len(vis)):
        c = _compact(sel, vis[b])
        ok[b] = len(c) >= 4 and np.linalg.matrix_rank(np.c_[P[c], np.ones(len(c))], tol=1e-9) == 4
    return ok


def _assert_parity(method, got, ref, stable, it_stable, full_rank=None):
    # (LM+ starts from linear F2: it needs a visible set that is not coplanar too)
    mask = stable if method == "lm" else (full_rank if method in ("linear_f1", "linear_f2") else None)
    if method == "lm_plus":
        mask = stable & full_rank
    compare_solutions(got, ref, mask=mask, iters_mask=it_stable)


# subset: None = all landmarks; "six" = solve_pnp's 6 keys (4 .. 6 of them visible); "forty" = 40 of 68 through point_index
# (the whole-row tile shape of the moment mapping)
CASES = [("qeif", 15, "six"), ("qeif", 15, None), ("qeif", 68, None), ("lm", 15, None), ("lm", 68, None), ("lm", 68, "forty"),
         ("linear_f2", 15, None), ("linear_f2", 68, None), ("linear_f2", 68, "forty"), ("eif2", 15, None), ("eif2", 68, None),
         ("eif2", 68, "forty"), ("linear_f1", 15, None), ("linear_f1", 68, None), ("lm_plus", 15, None), ("lm_plus", 68, None)]


@pytest.mark.parametrize("method,n,subset", CASES)
def test_masked_parity_with_oracle_on_compacted_problems(method, n, subset):
    pat, P, K, w = _workload(n, 256, seed=7)
    sel = {None: list(range(n)), "six": [list(pat).index(k) for k in pt.LM_KEY_LIST_6] if n == 15 else None,
           "forty": [j for j in range(68) if j % 5 in (1, 3, 4)][:40]}[subset]
    vis = _masks(256, len(sel), sel, n, seed=n + len(sel), lo=4 if subset == "six" else 6)
    ref, stable, it_stable = _oracle(method, P, w["uv"], K, vis, sel, stability=True)
    got = _solve(method, w["uv"], P, K, vis, point_index=sel if subset else None)
    full = _full_rank(P, vis, sel)
    assert method not in ("linear_f1", "linear_f2", "lm_plus") or full.mean() > 0.85
    _assert_parity(method, got, ref, stable, it_stable, full_rank=full)


def _solve_report_check(method, w, P, K, vis, dtype, mapping):
    """solve, then the masked report and check of the returned poses: every output as NumPy"""
    import pnp_solver_test_b200 as pnp
    from pnp_solver_test_b200 import workload as wl
    out = _solve(method, w["uv"], P, K, vis, dtype=dtype, mapping=mapping)
    uvd, visd = dev(w["uv"], dtype), torch.from_numpy(vis).cuda()
    R, t, e = dev(out["R"], dtype), dev(out["t"], dtype), dev(out["euler"], dtype)
    r = wl.report_batch(P, uvd, K, R, t, e, torch.from_numpy(w["gt"]).cuda(), visible=visd)
    c = pnp.check_batch(uvd, dev(P, dtype), K, R, t, res_norm=dev(out["res_norm"], dtype), reproj_limit_px=1.0, visible=visd)
    torch.cuda.synchronize()
    out.update({"report": r["report"].cpu().numpy(), "flags": r["flags"].cpu().numpy(), "max_idx": r["max_idx"].cpu().numpy(),
                "status": c["status"].cpu().numpy(), "reproj": c["reproj"].double().cpu().numpy()})
    return out


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("mapping", [0, 1, 32])
def test_hidden_pixels_are_never_read(method, dtype, mapping):
    pat, P, K, w = _workload(68, 200, seed=3)
    vis = _masks(200, 68, list(range(68)), 68, seed=11)
    vis[5, :] = False
    vis[5, :3] = True                                      # a degenerate problem among them
    if method == "lm_plus" and mapping != 0:
        return                                             # LM+ exists in the moment mapping only
    clean = _solve_report_check(method, w, P, K, vis, dtype, mapping)
    rng = np.random.default_rng(0)
    for fill in (np.nan, np.inf, -np.inf, 1e300, None):
        uv = w["uv"].copy()
        hid = ~vis
        uv[hid] = rng.normal(0, 1e4, size=(hid.sum(), 2)) if fill is None else fill
        dirty = _solve_report_check(method, dict(w, uv=uv), P, K, vis, dtype, mapping)
        for k in clean:
            np.testing.assert_array_equal(dirty[k], clean[k], err_msg="%s %s" % (k, fill))


def test_mask_equals_point_index():
    import pnp_solver_test_b200 as pnp
    pat, P, K, w = _workload(68, 512, seed=5)
    rng = np.random.default_rng(1)
    groups = [np.sort(rng.permutation(68)[:int(rng.integers(6, 69))]) for _ in range(8)]
    gid = rng.integers(0, 8, size=512)
    vis = np.zeros((512, 68), bool)
    for b in range(512):
        vis[b, groups[gid[b]]] = True
    for method in METHODS:
        got = _solve(method, w["uv"], P, K, vis)
        _, stable, it_stable = _oracle(method, P, w["uv"], K, vis, list(range(68)), stability=True)
        for g in range(8):
            m = gid == g
            ref = _solve(method, w["uv"][m], P, K, point_index=groups[g])
            sub = {k: v[m] for k, v in got.items()}
            compare_solutions(sub, ref, mask=stable[m] if method in ("lm", "lm_plus") else None, iters_mask=it_stable[m])
        # all visible agrees with the call without a mask (for LM, QEIF-68 and EIF2 that is the moment mapping)
        allv = _solve(method, w["uv"], P, K, np.ones((512, 68), bool))
        ref = _solve(method, w["uv"], P, K)
        _, stable, it_stable = _oracle(method, P, w["uv"][:64], K, np.ones((64, 68), bool), list(range(68)), stability=True)
        sl = {k: v[:64] for k, v in allv.items()}
        compare_solutions(sl, {k: v[:64] for k, v in ref.items()}, mask=stable if method in ("lm", "lm_plus") else None, iters_mask=it_stable)
    # the true-Jacobian LM (moment mapping only): masked groups = the same groups through point_index, bit for bit in the
    # iterations (one problem per thread, same order of the visible landmarks), to rounding in the constants
    got = _solve("lm", w["uv"], P, K, vis, flags=4)          # PNPB200_FLAG_LM_TRUE_JACOBIAN
    for g in range(8):
        m = gid == g
        ref = _solve("lm", w["uv"][m], P, K, point_index=groups[g], flags=4)
        fin = np.isfinite(ref["res_norm"]) & (np.abs(ref["t"][:, 2]) > 0)
        dR = np.abs(got["R"][m] - ref["R"]).reshape(m.sum(), -1).max(axis=1)
        assert np.median(dR[fin]) < 1e-9, g


@pytest.mark.parametrize("mapping", [0, 1, 32])
def test_fewer_than_four_visible(mapping):
    pat, P, K, w = _workload(68, 96, seed=9)
    vis = _masks(96, 68, list(range(68)), 68, seed=2)
    degenerate = np.array([3, 17, 40, 41, 64, 95])
    for b, k in zip(degenerate, (0, 1, 2, 3, 3, 0)):
        vis[b] = False
        vis[b, :k] = True
    keep = np.setdiff1d(np.arange(96), degenerate)
    for method in METHODS:
        if method == "lm_plus" and mapping != 0:
            continue                                       # LM+ exists in the moment mapping only
        got = _solve(method, w["uv"], P, K, vis, mapping=mapping)
        for k in ("R", "t", "euler", "res_norm"):
            assert np.isnan(got[k][degenerate]).all(), (method, k)
        assert (got["iters"][degenerate] == 0).all() and (got["best_pattern"][degenerate] == 0).all()
        # below 4 through the selection: 20 landmarks visible, 3 of them among the selected ones
        sel = list(range(0, 68, 2))
        v2 = vis.copy()
        v2[3] = False
        v2[3, 1:40:2] = True
        v2[3, [0, 2, 4]] = True
        g2 = _solve(method, w["uv"], P, K, v2, mapping=mapping, point_index=sel)
        assert np.isnan(g2["R"][3]).all() and np.isnan(g2["res_norm"][3]) and g2["iters"][3] == 0, method
        alone = _solve(method, w["uv"][keep], P, K, vis[keep], mapping=mapping)
        for k in got:
            np.testing.assert_array_equal(got[k][keep], alone[k], err_msg="%s %s" % (method, k))


def _report_check(method, n, B=256, seed=13, dtype=torch.float64):
    import pnp_solver_test_b200 as pnp
    from pnp_solver_test_b200 import workload as wl
    pat, P, K, w = _workload(n, B, seed=seed)
    vis = _masks(B, n, list(range(n)), n, seed=seed)
    vis[7] = False
    vis[7, :2] = True
    uvd, Pd, visd = dev(w["uv"], dtype), dev(P, dtype), torch.from_numpy(vis).cuda()
    gt = torch.from_numpy(w["gt"]).cuda()
    o = wl.solve_report_batch(method, uvd, Pd, K, gt, visible=visd)
    gt1 = gt.clone()
    gt1[:, 0] = 1.0
    r1 = wl.report_batch(P, uvd, K, o["R"], o["t"], o["euler"], gt1, visible=visd)
    c = pnp.check_batch(uvd, Pd, K, o["R"], o["t"], res_norm=o["res_norm"], reproj_limit_px=1.0, visible=visd)
    torch.cuda.synchronize()
    return P, K, w, vis, to_np(o), to_np(r1), to_np(c)


@pytest.mark.parametrize("n", [68, 300])
def test_masked_report_and_check(n):
    P, K, w, vis, o, r1, c = _report_check("lm", n)
    B = vis.shape[0]
    rep = o["report"]
    for b in range(B):
        cidx = np.flatnonzero(vis[b])
        if len(cidx) < 4:
            assert np.isnan(rep[b, 4:10]).all() and (o["max_idx"][b] == -1).all()
            assert c["status"][b] & NONFINITE and np.isnan(c["reproj"][b]).all()
            continue
        ref = orc.report_batch(P[cidx], w["uv"][b:b + 1, cidx], K, o["R"][b:b + 1], o["t"][b:b + 1], o["euler"][b:b + 1],
                               w["gt"][b:b + 1])
        np.testing.assert_allclose(rep[b], ref["report"][0], rtol=1e-9, atol=1e-12)
        np.testing.assert_array_equal(o["flags"][b], ref["flags"][0])
        np.testing.assert_array_equal(o["max_idx"][b], cidx[ref["max_idx"][0]])
    assert not o["flags"][7].any()
    # reproj = report columns 6, 7 at distance_GT = 1, bit for bit (both streaming kernels at n = 68)
    ok = np.array([vis[b].sum() >= 4 for b in range(B)])
    if n == 68:
        np.testing.assert_array_equal(c["reproj"][ok], r1["report"][ok][:, 6:8])
    else:
        np.testing.assert_allclose(c["reproj"][ok], r1["report"][ok][:, 6:8], rtol=1e-12)
    # status against a NumPy restatement over the visible landmarks
    for b in np.flatnonzero(ok):
        R, t = o["R"][b].reshape(3, 3), o["t"][b]
        z = (K @ (R @ P[vis[b]].T + t[:, None]))[2]
        s = 0
        if not (np.isfinite(R).all() and np.isfinite(t).all() and np.isfinite(o["res_norm"][b]) and np.isfinite(c["reproj"][b]).all()):
            s |= NONFINITE
        if t[2] <= 0:
            s |= DEPTH
        if (z < 0).any():
            s |= BEHIND
        if c["reproj"][b, 0] > 1.0:
            s |= REPROJ
        assert c["status"][b] == s, (b, c["status"][b], s)


@pytest.mark.parametrize("method", ["qeif", "lm", "eif2", "linear_f2"])
def test_shapes_the_bench_does_not_touch(method):
    # n = 98 in FP64 (the reference's 98-point detector) runs one problem per warp; n = 300 is above the ring threshold
    for n, B in ((98, 96), (300, 64)):
        pat, P, K, w = _workload(n, B, seed=n)
        vis = _masks(B, n, list(range(n)), n, seed=n, lo=n // 2)
        ref, stable, it_stable = _oracle(method, P, w["uv"], K, vis, list(range(n)), stability=method == "lm")
        for mapping in (0, 2):
            _assert_parity(method, _solve(method, w["uv"], P, K, vis, mapping=mapping), ref, stable, it_stable)
    # explicit mappings and two patterns (the arg-min on the masked res_norm)
    pat, P, K, w = _workload(68, 128, seed=4)
    vis = _masks(128, 68, list(range(68)), 68, seed=4)
    P2 = np.stack([P, P * np.array([1.02, 0.98, 1.01])])
    ref, stable, it_stable = _oracle(method, P, w["uv"], K, vis, list(range(68)), patterns=P2, stability=method == "lm")
    for mapping in (1, 32):
        got = _solve(method, w["uv"], P, K, vis, mapping=mapping, patterns=P2)
        _assert_parity(method, got, ref, stable, it_stable)
        m = stable if method == "lm" else np.isfinite(ref["res_norm"])
        np.testing.assert_array_equal(got["best_pattern"][m], ref["best_pattern"][m])


def test_fp32_qeif_within_fp32_bounds_of_masked_fp64():
    pat, P, K, w = _workload(68, 2048, seed=21)
    vis = _masks(2048, 68, list(range(68)), 68, seed=21)
    f64 = _solve("qeif", w["uv"], P, K, vis)
    f32 = _solve("qeif", w["uv"], P, K, vis, dtype=torch.float32)
    dR = np.abs(f32["R"] - f64["R"]).reshape(2048, -1).max(axis=1)
    dt = np.abs(f32["t"] - f64["t"]).max(axis=1) / np.abs(f64["t"][:, 2])
    assert np.quantile(dR, 0.999) <= 5e-4 and np.quantile(dt, 0.999) <= 2e-4, (dR.max(), dt.max())


@pytest.mark.parametrize("method", ["qeif", "lm", "eif2"])
@pytest.mark.parametrize("pix", ["float64", "int16", "float32"])
def test_host_entry_equals_device_entry(method, pix):
    import pnp_solver_test_b200 as pnp
    pat, P, K, w = _workload(68, 3000, seed=17)
    vis = _masks(3000, 68, list(range(68)), 68, seed=17)
    vis[11] = False
    solver = pnp.PNP_SOLVER(K, [pat], method=method)
    uv = w["uv"].copy()
    dref = solver.solve_pnp_batch(uv, key_list=None, visible=vis, check=1.0)
    dref = {k: (v.detach().cpu().numpy().reshape(3000, -1) if torch.is_tensor(v) else v) for k, v in dref.items()}
    uv_h = uv.astype({"float64": np.float64, "int16": np.int16, "float32": np.float32}[pix])
    for chunk in (256, 1000, 4096):
        for packing in ((0, 4) if pix == "float64" else (0,)):
            fills = (None, "random", 7) if pix == "int16" else (None, np.nan, np.inf, 1e300, "random", 7.0)
            for hidden in fills:
                u = uv_h.copy()
                if isinstance(hidden, str):
                    u[~vis] = np.random.default_rng(3).integers(-30000, 30000, size=((~vis).sum(), 2)).astype(u.dtype) * \
                        (1 if pix == "int16" else 1.37)
                elif hidden is not None:
                    u[~vis] = hidden                   # NaN / Inf in the hidden slots: such a chunk travels unpacked; 7: packed
                h = solver.solve_pnp_batch_host(u, key_list=None, chunk_problems=chunk, pack_threads=packing, visible=vis, check=1.0)
                for k, v in h.items():
                    np.testing.assert_array_equal(v.reshape(3000, -1), dref[k], err_msg="%s chunk %d packing %d" % (k, chunk, packing))
