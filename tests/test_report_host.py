"""The extended-precision report reference (tests/report_ref.py) against the C oracle and the reference's golden report, and
its bound against the mistakes it must catch.  CPU only."""
import numpy as np

import report_ref as rr
from conftest import load_golden
from oracle import oracle as orc
from pnp_solver_test_b200 import patterns as pt


def _stress(B=4096, n=68, seed=3):
    """the stress workload with perturbed, medium, diverged and behind-camera estimated poses"""
    P, K = pt.pattern_array(pt.synthetic_pattern(n)), pt.default_camera_matrix()
    w = orc.synth(0, B, P, K, orc.default_synth(seed=seed))
    rng = np.random.default_rng(seed)
    kind = rng.integers(0, 4, B)
    scale = np.array([1e-4, 3e-2, 1.0, 0.2])[kind]
    d = rng.normal(0, 1, (B, 3)) * scale[:, None]
    R = np.array([orc.R_from_euler(*a) for a in d]) @ w["R_gt"]
    t = w["t_gt"] * (1 + rng.normal(0, 1, (B, 3)) * scale[:, None] * 0.3)
    t[kind == 3, 2] *= -1
    euler = np.array([orc.euler_from_R(r, True) for r in R])
    return P, w["uv"], K, R, t, euler, w["gt"]


def _agree(got, ref):
    assert rr.columns_ok(got["report"], ref).all()
    assert np.array_equal(got["flags"], ref["flags"])
    assert rr.max_idx_ok(got["max_idx"], ref).all()


def test_reference_matches_the_c_oracle_on_the_stress_workload():
    args = _stress()
    ref = rr.report(*args)
    got = orc.report_batch(*args)
    _agree(got, ref)
    assert (got["max_idx"] == ref["max_idx"]).mean() > 0.999
    assert (ref["flags"].all(1) == 0).mean() > 0.2 and (args[4][:, 2] < 0).any()       # failures and t3 < 0 are in the batch
    assert np.isfinite(ref["report"]).all()


def test_reference_matches_the_golden_report():
    g = load_golden("stress_report")
    gt = g["gt"].copy()
    gt[:, 0] = (gt[:, 0] * 100.0) * 0.01          # the reference's distance_GT is dist_cm * 0.01 (its flags use dist_cm)
    ref = rr.report(g["pattern"], g["uv"], g["K"], g["R"], g["t"], g["euler"], gt)
    assert rr.columns_ok(g["report"], ref).all()
    assert np.array_equal(g["flags"][:, 1:], ref["flags"][:, 1:])
    assert np.array_equal(g["flags"][:, 0], rr.depth_flag(g["t"][:, 2], g["gt"][:, 0], 10.0).astype(np.int32))
    assert rr.max_idx_ok(g["max_idx"], ref).all()


def test_bound_is_tight_and_catches_wrong_kernels():
    args = _stress(B=1024)
    ref = rr.report(*args)
    good = ref["kappa"] <= 1e3
    assert good.mean() > 0.9
    lb = np.nan_to_num(ref["lm_bound"], nan=0.0).max((1, 2))
    assert (lb[good] <= 1e-12 * ref["px"][good]).all()
    e = ref["e"].astype(np.float64)
    n = e.shape[-1]
    dist = args[6][:, 0:1]
    cols, b = ref["report"][:, [4, 6, 8]], ref["bound"][:, [4, 6, 8]]
    pos = cols > 0
    # a division by n - 1 or n + 1, a landmark dropped or counted twice
    for wrong in (cols * n / (n - 1), cols * n / (n + 1), cols - e[..., 7] / n * dist, cols + e[..., 7] / n * dist):
        assert (np.abs(wrong - cols) > b)[pos & (e[..., 7] > 1e-3)].all()
    # one landmark's pixel rounded to FP32
    P, uv, K, R, t, euler, gt = args
    uv32 = uv.copy()
    uv32[:, 5] = uv32[:, 5] + 0.3                      # off the integer grid, so the FP32 rounding is visible
    r64 = rr.report(P, uv32, K, R, t, euler, gt)
    uv32[:, 5] = uv32[:, 5].astype(np.float32)
    r32 = rr.report(P, uv32, K, R, t, euler, gt)
    d = np.abs(r32["report"][:, 6] - r64["report"][:, 6])
    assert (d > r64["bound"][:, 6]).mean() > 0.99


def test_reference_rules_at_the_edges():
    """hand-worked: NaN never wins, strict > with the first landmark winning, -1 without a positive distance, fewer than 4
    visible, and depth 0 gives NaN"""
    P = np.array([[0.0, 0.0, 0.0], [0.1, 0.0, 0.0], [0.0, 0.1, 0.0], [0.1, 0.1, 0.0], [0.0, 0.0, -1.0]])
    K = np.array([[100.0, 0.0, 50.0], [0.0, 100.0, 50.0], [0.0, 0.0, 1.0]])
    R, t = np.eye(3)[None], np.array([[0.0, 0.0, 1.0]])
    p = (P[:4] + t) @ K.T
    uv = np.zeros((1, 5, 2))
    uv[0, :4] = p[:, :2] / p[:, 2:]
    uv[0, 1] += [3.0, 4.0]
    uv[0, 3] += [4.0, 3.0]
    gt = np.array([[1.0, 0.0, 0.0, 0.0]])
    r = rr.report(P, uv, K, R, t, np.zeros((1, 3)), gt)
    assert np.isnan(r["e"][0, 1, 4]) and np.isnan(r["report"][0, 6])       # landmark 4 is at depth 0
    assert r["max_idx"][0, 1] == 1 and r["report"][0, 7] == 5.0            # the tie of 1 and 3: the first wins
    assert r["max_idx"][0, 2] == -1 and r["report"][0, 9] == 0.0           # prediction = GT everywhere
    vis = np.array([[True, True, True, False, False]])
    r = rr.report(P, uv, K, R, t, np.zeros((1, 3)), gt, visible=vis)
    assert np.isnan(r["report"][0, 4:10]).all() and (r["max_idx"] == -1).all()
    vis[0, 3] = True
    r = rr.report(P, uv, K, R, t, np.zeros((1, 3)), gt, visible=vis)
    assert r["report"][0, 6] == 2.5 and r["max_idx"][0, 1] == 1
