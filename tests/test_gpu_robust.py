"""The outlier-robust solve (pnpb200_solve_robust_batch, solve_robust_batch in Python): every output of a problem is bit for bit
the masked solve's on the returned inlier mask, and the masks, round counts and status words are those of the rule restated in
NumPy over the oracle (tests/outlier_accuracy.py)."""
import numpy as np
import pytest
import torch

import outlier_accuracy as oa
from oracle import oracle as orc
from pnp_solver_test_b200 import patterns as pt

from conftest import compare_solutions
from gpu_util import dev, to_np

pytestmark = pytest.mark.gpu

KEYS = ("R", "t", "euler", "res_norm", "iters", "best_pattern")


def _workload(n, B, seed=42, f=0.1, a=30.0, b=150.0):
    pat = pt.get_golden_pattern() if n == 15 else pt.synthetic_pattern(n)
    P, K = pt.pattern_array(pat), pt.default_camera_matrix()
    w = orc.synth(0, B, P, K, cfg=orc.default_synth(seed=seed))
    return P, K, w, oa.add_outliers(w["uv"], f, a, b, seed)


def _robust(method, uv, pats, K, dtype=torch.float64, **kw):
    import pnp_solver_test_b200 as pnp
    if "visible" in kw and kw["visible"] is not None:
        kw["visible"] = torch.from_numpy(kw["visible"]).cuda()
    out = pnp.solve_robust_batch(method, dev(uv, dtype), dev(pats, dtype), K, **kw)
    torch.cuda.synchronize()
    return to_np(out)


def _masked(method, uv, pats, K, inliers, dtype=torch.float64, point_index=None, params=None):
    import pnp_solver_test_b200 as pnp
    out = pnp.solve_batch(method, dev(uv, dtype), dev(pats, dtype), K, point_index=point_index, params=params,
                          visible=torch.from_numpy(inliers).cuda())
    torch.cuda.synchronize()
    return to_np(out)


def _bits_equal(got, ref, keys=KEYS):
    for k in keys:
        a, b = np.ascontiguousarray(got[k]), np.ascontiguousarray(ref[k])
        assert a.shape == b.shape, k
        assert a.tobytes() == b.tobytes(), "%s differs on %d problems" % (k, int((a.reshape(len(a), -1) != b.reshape(len(b), -1)).any(1).sum()))


def _case(n, case, B, seed):
    rng = np.random.default_rng(seed)
    sel = np.sort(rng.permutation(n)[: n - n // 5]) if "idx" in case else None
    vis = (rng.random((B, n)) < 0.85) if "vis" in case else None
    return sel, vis


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("n", [15, 68, 98, 300])
@pytest.mark.parametrize("method", ["lm", "lm_plus", "qeif", "eif2"])
@pytest.mark.parametrize("case", ["all", "vis", "idx", "vis_idx"])
def test_outputs_are_the_masked_solve_on_the_inliers(method, n, dtype, case):
    B = 256 if n == 300 else 512
    P, K, w, uv = _workload(n, B, seed=n)
    sel, vis = _case(n, case, B, seed=n + 1)
    if vis is not None:
        uv[~vis] = np.nan                                   # hidden pixels are never read
    got = _robust(method, uv, P[None], K, dtype=dtype, point_index=sel, visible=vis)
    ref = _masked(method, uv, P[None], K, got["inliers"], dtype=dtype, point_index=sel)
    _bits_equal(got, ref)
    cand = np.ones((B, n), bool) if vis is None else vis.copy()
    if sel is not None:
        cand[:, np.setdiff1d(np.arange(n), sel)] = False
    assert not (got["inliers"] & ~cand).any()              # inliers lie in C
    assert ((got["rounds"] >= 1) & (got["rounds"] <= 4)).all()
    assert (got["rounds"] > 1).any()                        # the outliers made it re-solve


def test_two_patterns():
    P, K, w, uv = _workload(68, 512, seed=3)
    pats = np.stack([P, P * 1.04])
    for method in ("lm", "qeif", "lm_plus"):
        got = _robust(method, uv, pats, K)
        _bits_equal(got, _masked(method, uv, pats, K, got["inliers"]))
        assert (got["best_pattern"] == 1).any() and (got["best_pattern"] == 0).any()


@pytest.mark.parametrize("method", ["lm_plus", "qeif", "eif2", "lm"])
def test_rule_matches_the_oracle_restatement(method):
    B = 192
    P, K, w, uv = _workload(68, B, seed=11, f=0.2, a=5.0, b=150.0)
    got = _robust(method, uv, P[None], K)
    ref = {k: [] for k in KEYS}
    masks, rounds, status, near = np.zeros((B, 68), bool), np.zeros(B, int), np.zeros(B, int), np.zeros(B, bool)
    stable = np.ones(B, bool)
    for b in range(B):
        o, p, m, r, s, nr = oa.robust_one(method, P[None], uv[b], K, list(range(68)))
        for k in KEYS[:5]:
            ref[k].append(o[k])
        ref["best_pattern"].append(p)
        masks[b, m], rounds[b], status[b], near[b] = True, r, s, nr
        # the oracle's own path under a 1e-13 relative change of the pixels (the stability tag of the parity tests): where it
        # takes other inlier sets or moves the pose by more than 1e-10, the rule's outcome is not a well-posed target
        for sg in (1.0, -1.0):
            q, _, qm, qr, qs, _ = oa.robust_one(method, P[None], uv[b] * (1.0 + sg * 1e-13), K, list(range(68)))
            with np.errstate(invalid="ignore"):
                moved = not np.abs(q["R"] - o["R"]).max() <= 1e-10
            stable[b] &= sorted(qm) == sorted(m) and qr == r and qs == s and (not moved or not np.isfinite(o["t"]).all())
    ref = {k: np.asarray(v) for k, v in ref.items()}
    same = (got["inliers"] == masks).all(1) & (got["rounds"] == rounds) & (got["robust_status"] == status)
    # distances within 1e-9 of a threshold may fall either way (the kernel fuses multiply-adds)
    exempt = near | ~stable
    bad = ~same & ~exempt
    assert bad.mean() <= 0.01, (method, np.flatnonzero(bad)[:10], exempt.mean())
    # (measured: no distance near a threshold; the oracle's own path is unstable on 15 - 16 % of these contaminated problems
    # for LM+ and EIF2 and on 73 % for LM, whose plain solve is chaotic)
    assert near.mean() < 0.02 and exempt.mean() < (0.85 if method == "lm" else 0.3), (near.mean(), exempt.mean())
    m = same & ~exempt & np.isfinite(ref["t"][:, 2])
    # the parity tolerances, doubled: on these solves over contaminated, trimmed landmark sets EIF2's Euler angles reach
    # 1.09e-7 deg from the oracle's with R within 1e-9 (measured)
    compare_solutions(got, ref, mask=m, check_iters=False, tol_scale=2.0)


def test_one_round_or_infinite_floor_is_the_plain_masked_solve():
    P, K, w, uv = _workload(68, 512, seed=5)
    rng = np.random.default_rng(2)
    vis = rng.random((512, 68)) < 0.9
    for method in ("lm_plus", "qeif"):
        plain = _masked(method, uv, P[None], K, vis)
        for kw in (dict(max_rounds=1), dict(floor_px=float("inf"))):
            got = _robust(method, uv, P[None], K, visible=vis, **kw)
            _bits_equal(got, plain)
            assert (got["rounds"] == 1).all()
            np.testing.assert_array_equal(got["inliers"], vis)
            if "max_rounds" in kw:
                assert set(np.unique(got["robust_status"])) <= {0, 1, 2}
            else:
                assert (got["robust_status"] == 0).all()


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_hidden_pixels_change_no_bit(dtype):
    P, K, w, uv = _workload(68, 384, seed=9)
    vis = np.random.default_rng(4).random((384, 68)) < 0.8
    clean = _robust("qeif", uv, P[None], K, dtype=dtype, visible=vis)
    for fill in (np.nan, np.inf, 1e300):
        u = uv.copy()
        u[~vis] = fill
        dirty = _robust("qeif", u, P[None], K, dtype=dtype, visible=vis)
        _bits_equal(dirty, clean, KEYS + ("inliers", "rounds", "robust_status"))


def test_results_do_not_depend_on_the_batch():
    P, K, w, uv = _workload(68, 2048, seed=13, f=0.2)
    for method in ("lm_plus", "qeif", "eif2", "lm"):
        full = _robust(method, uv, P[None], K)
        for b0, b1 in ((0, 37), (37, 1000), (1500, 2048), (777, 778)):
            part = _robust(method, uv[b0:b1], P[None], K)
            _bits_equal(part, {k: v[b0:b1] for k, v in full.items()}, KEYS + ("inliers", "rounds", "robust_status"))
        perm = np.random.default_rng(0).permutation(2048)
        sh = _robust(method, uv[perm], P[None], K)
        _bits_equal(sh, {k: v[perm] for k, v in full.items()}, KEYS + ("inliers", "rounds", "robust_status"))


def test_too_few_not_converged_and_empty_batch():
    import pnp_solver_test_b200 as pnp
    P, K, w, uv = _workload(68, 256, seed=21, f=0.3, a=30.0, b=150.0)
    vis = np.ones((256, 68), bool)
    vis[1] = False
    vis[1, :3] = True                                       # NaN pose from the start: every distance NaN -> TOO_FEW
    uv[2, 10] = np.nan                                      # a non-finite VISIBLE pixel: NaN round-0 pose, TOO_FEW
    got = _robust("lm_plus", uv, P[None], K, visible=vis)
    assert got["robust_status"][1] == pnp.ROBUST_TOO_FEW and np.isnan(got["t"][1]).all() and got["rounds"][1] == 1
    assert got["robust_status"][2] == pnp.ROBUST_TOO_FEW and np.isnan(got["t"][2]).all() and got["inliers"][2].all()
    # min_inliers = all 68: every problem whose mask would change keeps its round-0 pose and mask
    strict = _robust("lm_plus", uv, P[None], K, visible=vis, min_inliers=68)
    tf = strict["robust_status"] == pnp.ROBUST_TOO_FEW
    assert tf.mean() > 0.5 and (strict["rounds"] == 1).all() and (strict["inliers"] == vis).all()
    _bits_equal(strict, _masked("lm_plus", uv, P[None], K, vis))
    two = _robust("lm_plus", uv, P[None], K, visible=vis, max_rounds=2)
    nc = two["robust_status"] == pnp.ROBUST_NOT_CONVERGED
    assert nc.any() and (two["rounds"][nc] == 2).all()
    _bits_equal(two, _masked("lm_plus", uv, P[None], K, two["inliers"]))
    empty = pnp.solve_robust_batch("qeif", dev(uv[:0]), dev(P[None]), K)
    assert empty["inliers"].shape == (0, 68) and empty["R"].shape == (0, 3, 3)


def test_pass_rate_at_scale():
    """65 536 problems at 10 % far outliers: the oracle table's robust pass rates (include/pnpb200.h), within 1.5 points"""
    import pnp_solver_test_b200 as pnp
    from pnp_solver_test_b200 import workload as wl
    P, K = pt.pattern_array(pt.synthetic_pattern(68)), pt.default_camera_matrix()
    B = 65536
    w = orc.synth(0, B, P, K, cfg=orc.default_synth(seed=42), n_threads=0)
    uv = oa.add_outliers(w["uv"], 0.1, 30.0, 150.0, 42)
    table = {"lm_plus": 87.2, "qeif": 100.0}                # the 8 192-problem oracle table
    for method, floor in table.items():
        out = pnp.solve_robust_batch(method, dev(uv), dev(P[None]), K)
        r = wl.report_batch(P, dev(w["uv"]), K, out["R"], out["t"], out["euler"], torch.from_numpy(w["gt"]).cuda())
        rate = 100.0 * r["flags"].all(dim=1).double().mean().item()
        print("%s robust pass rate %.2f %%" % (method, rate))
        assert rate >= floor - 1.5, (method, rate)


def test_solve_pnp_batch_robust():
    import pnp_solver_test_b200 as pnp
    P, K, w, uv = _workload(68, 256, seed=17)
    s = pnp.PNP_SOLVER(K, [pt.synthetic_pattern(68)])
    out = to_np(s.solve_pnp_batch(uv, method="lm_plus", robust=dict(k=3.0), check=1.0))
    ref = to_np(s.solve_pnp_batch(uv, method="lm_plus", visible=out["inliers"], check=1.0))
    _bits_equal(out, ref, KEYS + ("status", "reproj"))
    assert (out["rounds"] > 1).any()
    with pytest.raises(ValueError):
        s.solve_pnp_batch(uv, method="lm_plus", robust=dict(kk=3.0))
    with pytest.raises(ValueError):
        s.solve_pnp_batch(uv, method="lm_plus", robust=dict(min_inliers=3))
