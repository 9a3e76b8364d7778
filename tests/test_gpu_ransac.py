"""The RANSAC solve on the GPU: the P3P hook against ground truth and the Grunert P3P of tests/ransac_oracle.c, the
hypothesis stage (pnpb200_hypothesize_batch) against that file's restatement of its rule, and the RANSAC entry's contract: every output is the
masked solve's on the returned inliers, max_samples = 0 is the robust entry, hidden pixels change nothing, idx0 shards."""
import ctypes as C

import numpy as np
import pytest
import torch

import outlier_accuracy as oa
import ransac_accuracy as ra
import ransac_oracle as ro
from oracle import oracle as orc
from pnp_solver_test_b200 import patterns as pt

from gpu_util import dev, to_np

pytestmark = pytest.mark.gpu

KEYS = ("R", "t", "euler", "res_norm", "iters", "best_pattern")
ROBUST = KEYS + ("inliers", "rounds", "robust_status")


def _workload(n, B, seed=42, f=0.1, a=30.0, b=150.0):
    pat = pt.get_golden_pattern() if n == 15 else pt.synthetic_pattern(n)
    P, K = pt.pattern_array(pat), pt.default_camera_matrix()
    w = orc.synth(0, B, P, K, cfg=orc.default_synth(seed=seed))
    return P, K, w, oa.add_outliers(w["uv"], f, a, b, seed)


def _case(n, case, B, seed):
    rng = np.random.default_rng(seed)
    sel = rng.permutation(n)[: n - n // 5] if "idx" in case else None          # (not sorted: candidate order is its order)
    vis = (rng.random((B, n)) < 0.85) if "vis" in case else None
    return sel, vis


def _cand(n, B, sel, vis):
    order = np.arange(n) if sel is None else np.asarray(sel)
    return [[j for j in order if vis is None or vis[b, j]] for b in range(B)]


def _bits_equal(got, ref, keys=KEYS):
    for k in keys:
        a, b = np.ascontiguousarray(got[k]), np.ascontiguousarray(ref[k])
        assert a.shape == b.shape, k
        assert a.tobytes() == b.tobytes(), "%s differs on %d problems" % (k, int((a.reshape(len(a), -1) != b.reshape(len(b), -1)).any(1).sum()))


def _vis_dev(kw):
    if kw.get("visible") is not None:
        kw["visible"] = torch.from_numpy(kw["visible"]).cuda()
    return kw


def _hyp(uv, pats, K, dtype=torch.float64, **kw):
    import pnp_solver_test_b200 as pnp
    out = pnp.hypothesize_batch(dev(uv, dtype), dev(pats, dtype), K, **_vis_dev(kw))
    torch.cuda.synchronize()
    return to_np(out)


def _ransac(method, uv, pats, K, dtype=torch.float64, samples=128, **kw):
    import pnp_solver_test_b200 as pnp
    out = pnp.solve_robust_batch(method, dev(uv, dtype), dev(pats, dtype), K, samples=samples, **_vis_dev(kw))
    torch.cuda.synchronize()
    return to_np(out)


def _p3p_triples(m, seed):
    """noise-free triples of the synthetic workload's poses: X [m,3,3], f [m,3,3], R_gt, t_gt"""
    P, K = pt.pattern_array(pt.synthetic_pattern(68)), pt.default_camera_matrix()
    w = orc.synth(0, m, P, K, cfg=orc.default_synth(seed=seed, is_quantized=False))
    rng = np.random.default_rng(seed)
    tri = np.stack([rng.choice(68, 3, replace=False) for _ in range(m)])
    X = P[tri]
    px = np.concatenate([w["uv"][np.arange(m)[:, None], tri], np.ones((m, 3, 1))], axis=2) @ np.linalg.inv(K).T
    return X, px / np.linalg.norm(px, axis=2, keepdims=True), w["R_gt"], w["t_gt"]


def test_p3p_hook_recovers_the_pose_and_the_oracles_roots():
    from pnp_solver_test_b200 import _lib
    m = 4096
    X, f, Rg, tg = _p3p_triples(m, 7)
    Xd, fd = dev(X), dev(f)
    R = torch.empty((m, 4, 9), dtype=torch.float64, device="cuda")
    t = torch.empty((m, 4, 3), dtype=torch.float64, device="cuda")
    ns = torch.empty((m,), dtype=torch.int32, device="cuda")
    _lib.check(_lib.lib.pnpb200_selftest_p3p(m, Xd.data_ptr(), fd.data_ptr(), R.data_ptr(), t.data_ptr(), ns.data_ptr(), None),
               "pnpb200_selftest_p3p")
    torch.cuda.synchronize()
    R, t, ns = R.cpu().numpy().reshape(m, 4, 3, 3), t.cpu().numpy(), ns.cpu().numpy()
    assert ((ns >= 0) & (ns <= 4)).all()
    hit, same = np.zeros(m, bool), np.zeros(m, bool)
    for i in range(m):
        k = ns[i]
        e = [max(np.abs(R[i, r] - Rg[i]).max(), np.abs(t[i, r] - tg[i]).max() / tg[i, 2]) for r in range(k)]
        hit[i] = bool(e) and min(e) <= 1e-9
        assert np.isnan(R[i, k:]).all()
        oR, ot = ro.p3p(X[i], f[i])
        def match(A, At, Bm, Bt):
            return all(any(max(np.abs(A[a] - Bm[b]).max(), np.abs(At[a] - Bt[b]).max() / abs(Bt[b][2])) <= 1e-8 for b in range(len(Bm)))
                       for a in range(len(A)))
        same[i] = match(R[i, :k], t[i, :k], oR, ot) and match(oR, ot, R[i, :k], t[i, :k])
    print("P3P: ground truth among the roots on %.3f %%, root sets equal on %.3f %%" % (100 * hit.mean(), 100 * same.mean()))
    # the misses are nearly collinear triples (the face pattern's landmarks lie close together), and the differing root sets
    # near-double roots, which either solver may resolve as a pair or drop as complex
    assert hit.mean() >= 0.99
    assert same.mean() >= 0.98


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("n", [15, 68, 98, 300])
@pytest.mark.parametrize("case", ["all", "vis", "idx", "vis_idx"])
@pytest.mark.parametrize("f", [0.1, 0.3])
def test_hypotheses_match_the_oracle(n, dtype, case, f):
    B = 200
    P, K, w, uv = _workload(n, B, seed=n + int(100 * f), f=f)
    sel, vis = _case(n, case, B, seed=n + 3)
    pats = P[None] if n != 68 else np.stack([P, P * 1.04])       # two patterns at n = 68
    if dtype == torch.float32:                                    # the oracle sees what the kernel reads
        uv, pats = uv.astype(np.float32).astype(np.float64), pats.astype(np.float32).astype(np.float64)
    u = uv.copy()
    if vis is not None:
        u[~vis] = np.nan
    got = _hyp(u, pats, K, dtype=dtype, point_index=sel, visible=vis)
    cand = _cand(n, B, sel, vis)
    same, near = np.zeros(B, bool), np.zeros(B, bool)
    for b in range(B):
        h = ro.hypothesize_one(uv[b], pats, K, cand[b], b)
        near[b] = h["near"]
        same[b] = (got["drawn"][b] == h["drawn"] and got["consensus"][b] == h["consensus"] and got["best_pattern"][b] == h["best_pattern"]
                   and (got["consensus_mask"][b] == h["mask"]).all())
        assert not (got["consensus_mask"][b] & ~np.isin(np.arange(n), cand[b])).any()     # the consensus set lies in C
        if got["consensus"][b] == 0:
            assert np.isnan(got["t"][b]).all() and not got["consensus_mask"][b].any()
        else:
            assert got["consensus_mask"][b].sum() == got["consensus"][b]
    bad = ~same & ~near
    assert near.mean() <= 0.01, near.mean()
    assert bad.mean() <= 0.01, (np.flatnonzero(bad)[:10], got["drawn"][bad][:5], got["consensus"][bad][:5])
    assert (got["consensus"] > 0).mean() > 0.9


def test_clean_data_ends_after_the_first_good_sample():
    P, K, w, uv = _workload(68, 512, f=0.0)
    got = _hyp(uv, P[None], K)
    assert np.median(got["drawn"]) == 1 and (got["consensus"] >= 64).mean() > 0.95


def test_parameters_and_degenerate_problems():
    P, K, w, uv = _workload(68, 128, f=0.3)
    vis = np.ones((128, 68), bool)
    vis[3] = False
    vis[3, :3] = True                                             # c < 4: nothing drawn
    got = _hyp(uv, P[None], K, visible=vis, samples=5, confidence=1.0)
    assert got["drawn"][3] == 0 and got["consensus"][3] == 0 and np.isnan(got["R"][3]).all()
    others = np.arange(128) != 3
    assert (got["drawn"][others] == 5).all()                      # confidence 1 stops only at w = 1, which 30 % outliers exclude
    none = _hyp(uv, P[None], K, samples=0)
    assert (none["drawn"] == 0).all() and (none["consensus"] == 0).all() and np.isnan(none["t"]).all()
    seeded = _hyp(uv, P[None], K, seed=12345)                     # other samples: other winners (drawn depends on the count only)
    assert (seeded["R"] != _hyp(uv, P[None], K)["R"]).any()


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("n", [15, 68, 98, 300])
@pytest.mark.parametrize("method", ["lm", "lm_plus", "qeif", "eif2"])
@pytest.mark.parametrize("case", ["all", "vis", "idx", "vis_idx"])
def test_outputs_are_the_masked_solve_on_the_inliers(method, n, dtype, case):
    import pnp_solver_test_b200 as pnp
    B = 256
    P, K, w, uv = _workload(n, B, seed=n, f=0.3)
    sel, vis = _case(n, case, B, seed=n + 1)
    if vis is not None:
        uv[~vis] = np.nan
    got = _ransac(method, uv, P[None], K, dtype=dtype, point_index=sel, visible=vis)
    ref = to_np(pnp.solve_batch(method, dev(uv, dtype), dev(P[None], dtype), K, point_index=sel,
                                visible=torch.from_numpy(got["inliers"]).cuda()))
    _bits_equal(got, ref)
    cand = np.zeros((B, n), bool)
    for b, c in enumerate(_cand(n, B, sel, vis)):
        cand[b, c] = True
    assert not (got["inliers"] & ~cand).any()
    assert ((got["rounds"] >= 1) & (got["rounds"] <= 4)).all() and (got["consensus"] > 0).mean() > 0.9


def test_two_patterns():
    import pnp_solver_test_b200 as pnp
    P, K, w, uv = _workload(68, 512, seed=3, f=0.3)
    pats = np.stack([P, P * 1.04])
    for method in ("lm_plus", "eif2"):
        got = _ransac(method, uv, pats, K)
        ref = to_np(pnp.solve_batch(method, dev(uv), dev(pats), K, visible=torch.from_numpy(got["inliers"]).cuda()))
        _bits_equal(got, ref)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_no_samples_is_the_robust_entry(dtype):
    import pnp_solver_test_b200 as pnp
    P, K, w, uv = _workload(68, 512, seed=5, f=0.3)
    vis = np.random.default_rng(2).random((512, 68)) < 0.9
    for method in ("lm_plus", "qeif", "eif2", "lm"):
        got = _ransac(method, uv, P[None], K, dtype=dtype, samples=0, visible=vis)
        ref = to_np(pnp.solve_robust_batch(method, dev(uv, dtype), dev(P[None], dtype), K, visible=torch.from_numpy(vis).cuda()))
        _bits_equal(got, ref, ROBUST)
        assert (got["consensus"] == 0).all() and (got["drawn"] == 0).all()


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_hidden_pixels_change_no_bit(dtype):
    P, K, w, uv = _workload(68, 384, seed=9, f=0.3)
    vis = np.random.default_rng(4).random((384, 68)) < 0.8
    clean_h = _hyp(uv, P[None], K, dtype=dtype, visible=vis)
    clean = _ransac("lm_plus", uv, P[None], K, dtype=dtype, visible=vis)
    for fill in (np.nan, np.inf, 1e300):
        u = uv.copy()
        u[~vis] = fill
        _bits_equal(_hyp(u, P[None], K, dtype=dtype, visible=vis), clean_h, ("R", "t", "best_pattern", "consensus_mask", "consensus", "drawn"))
        _bits_equal(_ransac("lm_plus", u, P[None], K, dtype=dtype, visible=vis), clean, ROBUST + ("consensus", "drawn"))


def test_shards_with_idx0_are_the_unsharded_call():
    P, K, w, uv = _workload(68, 2048, seed=13, f=0.3)
    full_h = _hyp(uv, P[None], K)
    full = _ransac("lm_plus", uv, P[None], K)
    for b0, b1 in ((0, 37), (37, 1000), (1500, 2048), (777, 778)):
        part_h = _hyp(uv[b0:b1], P[None], K, idx0=b0)
        _bits_equal(part_h, {k: v[b0:b1] for k, v in full_h.items()}, ("R", "t", "best_pattern", "consensus_mask", "consensus", "drawn"))
        part = _ransac("lm_plus", uv[b0:b1], P[None], K, idx0=b0)
        _bits_equal(part, {k: v[b0:b1] for k, v in full.items()}, ROBUST + ("consensus", "drawn"))


def test_pass_rate_at_30_percent_far_outliers():
    """the header's RANSAC pass rates (tests/ransac_accuracy.py, the same 8 192 problems) within 1 point"""
    import re
    import os
    from pnp_solver_test_b200 import workload as wl
    hdr = open(os.path.join(ra.ROOT, "include", "pnpb200.h")).read()
    row = re.search(r" \*   30-150 px +30 % +(.*)\n", hdr[hdr.index("pnpb200_solve_ransac_batch"):]).group(1).split()
    table = {"lm_plus": float(row[2]), "eif2": float(row[8])}
    P, K = pt.pattern_array(pt.synthetic_pattern(68)), pt.default_camera_matrix()
    w = orc.synth(0, ra.B, P, K, cfg=orc.default_synth(seed=ra.SEED))
    uv = oa.add_outliers(w["uv"], 0.3, 30.0, 150.0, ra.SEED)
    for method, ref in table.items():
        import pnp_solver_test_b200 as pnp
        out = pnp.solve_robust_batch(method, dev(uv), dev(P[None]), K, samples=128)
        r = wl.report_batch(P, dev(w["uv"]), K, out["R"], out["t"], out["euler"], torch.from_numpy(w["gt"]).cuda())
        rate = 100.0 * r["flags"].all(dim=1).double().mean().item()
        print("%s RANSAC pass rate %.2f %% (header %.1f %%)" % (method, rate, ref))
        assert abs(rate - ref) <= 1.0, (method, rate, ref)


def test_solve_pnp_batch_ransac():
    import pnp_solver_test_b200 as pnp
    P, K, w, uv = _workload(68, 256, seed=17, f=0.3)
    s = pnp.PNP_SOLVER(K, [pt.synthetic_pattern(68)])
    out = to_np(s.solve_pnp_batch(uv, method="lm_plus", robust=dict(samples=64, consensus_px=4.0), check=1.0))
    ref = to_np(s.solve_pnp_batch(uv, method="lm_plus", visible=out["inliers"], check=1.0))
    _bits_equal(out, ref, KEYS + ("status", "reproj"))
    assert (out["drawn"] >= 1).all() and (out["drawn"] <= 64).all()
    with pytest.raises(ValueError):
        s.solve_pnp_batch(uv, method="lm_plus", robust=dict(samples=-1))
    with pytest.raises(ValueError):
        s.solve_pnp_batch(uv, method="lm_plus", robust=dict(samples=8, confidence=0.0))
