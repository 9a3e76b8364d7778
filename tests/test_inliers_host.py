"""The extended-precision restatement of the inlier rule (tests/test_gpu_inliers.py) against the classification step of
outlier_accuracy.robust_one and against hand-worked cases, and the argument checks of pnpb200_selftest_inliers (CPU only)."""
import ctypes as C

import numpy as np
import pytest

import outlier_accuracy as oa
from test_gpu_inliers import TOO_FEW, NOT_CONVERGED, decide, rule

NAN = np.nan


def _robust_one_step(d, k, floor_px, monkeypatch):
    """M' of robust_one for the distances d of one problem: with min_inliers = 0 and two rounds it adopts M' and, the distances
    being the same, stops there"""
    monkeypatch.setattr(oa, "distances", lambda P, uv, K, R, t: d)
    monkeypatch.setattr(oa, "solve_on", lambda method, patterns, uv, K, land: (dict(R=np.eye(3), t=np.zeros(3)), 0))
    cand = list(range(len(d)))
    _, _, mask, _, _, _ = oa.robust_one("lm", np.zeros((1, len(d), 3)), np.zeros((len(d), 2)), np.eye(3), cand, max_rounds=2,
                                        k=k, floor_px=floor_px, min_inliers=0)
    out = np.zeros(len(d), bool)
    out[mask] = True
    return out


@pytest.mark.parametrize("k,floor_px", [(3.0, 2.0), (1.0, 0.0), (0.0, 1.0), (2.0, float("inf")), (1e308, 0.5)])
def test_rule_matches_robust_one(k, floor_px, monkeypatch):
    rng = np.random.default_rng(int(min(k, 100.0) * 7) + int(floor_px < 1.0))
    for trial in range(200):
        c = int(rng.integers(1, 40))
        d = np.round(rng.exponential(1.0, c) * 8) / 4 if trial % 2 else rng.exponential(1.0, c) * 3   # ties on even trials
        d[rng.random(c) < 0.1 * (trial % 4)] = NAN
        d[rng.random(c) < 0.05] = 1e308 * (trial % 3 == 0)
        tau, new = rule(d[None], np.ones((1, c), bool), k, floor_px)
        np.testing.assert_array_equal(new[0], _robust_one_step(d, k, floor_px, monkeypatch), err_msg=str(d))


@pytest.mark.parametrize("d,k,floor_px,tau_want,new_want", [
    ([], 3.0, 2.0, 2.0, []),                                           # c = 0: tau = floor_px
    ([5.0], 3.0, 2.0, 15.0, [1]),                                      # c = 1: rank 0
    ([1.0, 4.0], 1.0, 0.0, 1.0, [1, 0]),                               # c = 2: the LOWER median, rank 0
    ([4.0, 1.0, 2.0], 1.0, 0.0, 2.0, [0, 1, 1]),                       # c = 3: rank 1; d = tau is kept
    ([NAN, 1.0, NAN], 1.0, 0.0, NAN, [0, 0, 0]),                       # NaN last: rank 1 is NaN -> tau = floor_px = 0 ...
    ([NAN, 1.0, 3.0], 1.0, 0.5, 3.0, [0, 1, 1]),                       # ... and with one NaN, rank 1 is the larger finite one
    ([2.0, 2.0, 2.0, 7.0], 1.5, 0.0, 3.0, [1, 1, 1, 0]),               # ties at the median
    ([1.0, 2.0, 3.0], 0.0, 2.5, 2.5, [1, 1, 0]),                       # k = 0: tau = floor_px
    ([1.0, 2.0, 3.0], 1.0, 2.0, 2.0, [1, 1, 0]),                       # k med = floor_px
    ([1.0, 2.0, 3.0], 1e308, 1.0, 1.0, [1, 0, 0]),                     # k med overflows: floor_px
    ([1.0, NAN, 1e300], 1.0, float("inf"), float("inf"), [1, 0, 1]),   # +Inf floor keeps every finite distance
])
def test_rule_hand_worked(d, k, floor_px, tau_want, new_want):
    d = np.array(d, float).reshape(1, -1)
    tau, new = rule(d, np.ones(d.shape, bool), k, floor_px)
    want = floor_px if np.isnan(tau_want) else tau_want
    assert float(tau[0]) == want
    np.testing.assert_array_equal(new[0], np.array(new_want, bool))


def test_decision_hand_worked():
    new = np.array([[1, 1, 0], [1, 1, 1], [1, 0, 0], [1, 1, 0]], bool)
    mask = np.array([[1, 1, 1], [1, 1, 1], [1, 1, 1], [1, 1, 0]], bool)
    rounds, status = np.array([1, 2, 3, 1]), np.zeros(4, int)
    flag, m, r, s = decide(new, mask, rounds, status, 2, 0)
    np.testing.assert_array_equal(flag, [1, 0, 0, 0])                  # changed; same; too few; same
    np.testing.assert_array_equal(s, [0, 0, TOO_FEW, 0])
    np.testing.assert_array_equal(r, [2, 2, 3, 1])
    np.testing.assert_array_equal(m, np.where(np.array([1, 0, 0, 0], bool)[:, None], new, mask))
    flag, m, r, s = decide(new, mask, rounds, status, 2, 1)
    np.testing.assert_array_equal(s, [NOT_CONVERGED, 0, TOO_FEW, 0])   # last round: M kept
    np.testing.assert_array_equal(flag, 0)
    np.testing.assert_array_equal(m, mask)
    flag, m, r, s = decide(new, mask, rounds, status, 3, 0)            # |M'| = min_inliers - 1
    np.testing.assert_array_equal(s, [TOO_FEW, 0, TOO_FEW, 0])


def test_hook_arguments_need_no_gpu():
    from pnp_solver_test_b200 import _lib
    f = _lib.lib.pnpb200_selftest_inliers
    K = (C.c_double * 9)(225.7, 0, 160, 0, 225.7, 120, 0, 0, 1)
    p = C.c_void_p(0x10000)

    def call(dtype=0, B=4, n_total=6, n=6, uv=p, pattern=p, n_patterns=1, K=K, robust=None, R=p, t=p, inliers=p, rounds=p,
             status=p, flag=p, shape=0):
        U32, I32 = C.POINTER(C.c_uint32), C.POINTER(C.c_int32)
        return f(dtype, B, n_total, n, uv, pattern, n_patterns, None, K, None, None if robust is None else C.byref(robust), R, t,
                 None, None, 0, C.cast(inliers, U32), C.cast(rounds, I32), C.cast(status, I32), flag, None, shape, None)

    for bad in (dict(shape=3), dict(shape=-1), dict(n_total=0, n=0), dict(dtype=2), dict(uv=None), dict(uv=C.c_void_p(0x10008)),
                dict(R=None), dict(t=None), dict(inliers=None), dict(rounds=None), dict(status=None), dict(flag=None),
                dict(n=5), dict(n_patterns=0), dict(n_patterns=9), dict(B=-1),
                dict(robust=_lib.RobustParams(max_rounds=4, k_median=-1.0, floor_px=2.0, min_inliers=6)),
                dict(robust=_lib.RobustParams(max_rounds=4, k_median=float("inf"), floor_px=2.0, min_inliers=6)),
                dict(robust=_lib.RobustParams(max_rounds=4, k_median=3.0, floor_px=float("nan"), min_inliers=6)),
                dict(robust=_lib.RobustParams(max_rounds=4, k_median=3.0, floor_px=2.0, min_inliers=3)),
                dict(robust=_lib.RobustParams(max_rounds=0, k_median=3.0, floor_px=2.0, min_inliers=6))):
        assert call(**bad) == -1, bad
    assert call(B=0) == 0                                             # nothing to do: no CUDA call
    import torch
    if not torch.cuda.is_available():
        assert call() in (-2, -3)                                     # valid arguments reach the device
