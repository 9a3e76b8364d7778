"""The RANSAC solve without a GPU: argument checks of pnpb200_hypothesize_batch and pnpb200_solve_ransac_batch (EINVAL before
any launch), the ValueErrors of the Python layer, defaults, the workspace query, the P3P and draw rule of
tests/ransac_oracle.c, and the accuracy tables of include/pnpb200.h against tests/ransac_accuracy.py."""
import ctypes as C

import numpy as np
import pytest
import torch

EINVAL = -1
FAKE = C.c_void_p(1 << 20)                                 # 16-byte aligned, never dereferenced: every call below fails its checks first
PI = C.POINTER(C.c_int32)
U32 = C.POINTER(C.c_uint32)


@pytest.fixture(scope="module")
def lib():
    from pnp_solver_test_b200 import _lib
    return _lib


def _K():
    return (C.c_double * 9)(800.0, 0.0, 320.0, 0.0, 800.0, 240.0, 0.0, 0.0, 1.0)


def _hp(lib, **kw):
    p = lib.HypothesisParams(max_samples=128, consensus_px=4.0, confidence=0.999, seed=0, idx0=0)
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def _hyp_call(lib, hyp=None, **kw):
    a = dict(dtype=0, B=64, n_total=68, n=68, uv=FAKE, pattern=FAKE, n_patterns=1, point_index=None, K=_K(), visible=None, R=FAKE,
             t=FAKE, best=C.cast(FAKE, PI), mask=C.cast(FAKE, U32), consensus=C.cast(FAKE, PI), drawn=None)
    a.update(kw)
    return lib.lib.pnpb200_hypothesize_batch(a["dtype"], a["B"], a["n_total"], a["n"], a["uv"], a["pattern"], a["n_patterns"],
                                             a["point_index"], a["K"], a["visible"], None if hyp is None else C.byref(hyp), a["R"],
                                             a["t"], a["best"], a["mask"], a["consensus"], a["drawn"], None)


def _ransac_call(lib, hyp=None, **kw):
    a = dict(method=4, dtype=0, B=64, n_total=68, n=68, uv=FAKE, pattern=FAKE, n_patterns=1, point_index=None, K=_K(), R=FAKE,
             t=FAKE, best=C.cast(FAKE, PI), visible=None, inliers=C.cast(FAKE, U32), rounds=C.cast(FAKE, PI), status=C.cast(FAKE, PI),
             consensus=C.cast(FAKE, PI))
    a.update(kw)
    return lib.lib.pnpb200_solve_ransac_batch(a["method"], a["dtype"], a["B"], a["n_total"], a["n"], a["uv"], a["pattern"],
                                              a["n_patterns"], a["point_index"], a["K"], None, a["R"], a["t"], None, None, None,
                                              a["best"], a["visible"], None, a["inliers"], a["rounds"], a["status"],
                                              None if hyp is None else C.byref(hyp), a["consensus"], None, None)


def test_default_hypothesis_params(lib):
    p = lib.HypothesisParams()
    assert lib.lib.pnpb200_default_hypothesis_params(C.byref(p)) == 0
    assert (p.max_samples, p.consensus_px, p.confidence, p.seed, p.idx0) == (128, 4.0, 0.999, 0, 0)
    assert lib.lib.pnpb200_default_hypothesis_params(None) == EINVAL
    assert C.sizeof(lib.HypothesisParams) == 40


@pytest.mark.parametrize("field,value", [("max_samples", -1), ("consensus_px", -0.5), ("consensus_px", float("nan")),
                                         ("confidence", 0.0), ("confidence", -0.1), ("confidence", 1.5),
                                         ("confidence", float("nan"))])
def test_bad_hypothesis_params_are_einval(lib, field, value):
    assert _hyp_call(lib, _hp(lib, **{field: value})) == EINVAL
    assert _ransac_call(lib, _hp(lib, **{field: value})) == EINVAL


@pytest.mark.parametrize("bad", ["R", "t", "mask", "consensus", "best_two_patterns", "misaligned_visible", "misaligned_mask",
                                 "point_index", "dtype", "n_patterns", "uv", "pattern", "n_without_index"])
def test_bad_hypothesis_arguments_are_einval(lib, bad):
    kw = {"R": dict(R=None), "t": dict(t=None), "mask": dict(mask=None), "consensus": dict(consensus=None),
          "best_two_patterns": dict(n_patterns=2, best=None), "misaligned_visible": dict(visible=C.cast(C.c_void_p((1 << 20) | 2), U32)),
          "misaligned_mask": dict(mask=C.cast(C.c_void_p((1 << 20) | 1), U32)),
          "point_index": dict(n=2, point_index=(C.c_int32 * 2)(0, 68)), "dtype": dict(dtype=2), "n_patterns": dict(n_patterns=9),
          "uv": dict(uv=None), "pattern": dict(pattern=None), "n_without_index": dict(n=60)}[bad]
    assert _hyp_call(lib, **kw) == EINVAL


def test_too_many_candidates_is_etoolarge(lib):
    assert _hyp_call(lib, n_total=1025, n=1025) == -4
    assert _hyp_call(lib, B=0) == 0


@pytest.mark.parametrize("bad", ["consensus", "R", "inliers", "method"])
def test_bad_ransac_arguments_are_einval(lib, bad):
    kw = {"consensus": dict(consensus=None), "R": dict(R=None), "inliers": dict(inliers=None), "method": dict(method=6)}[bad]
    assert _ransac_call(lib, _hp(lib), **kw) == EINVAL
    assert _ransac_call(lib, _hp(lib), B=0) == 0


def test_workspace_query(lib):
    # the robust scratch plus the hypothesis stage's pose, pattern, mask and sample count
    for dtype, esz in ((0, 8), (1, 4)):
        for method in range(6):
            ws = lib.lib.pnpb200_ransac_workspace_bytes(method, dtype, 1 << 20, 68, 1, 0)
            robust = lib.lib.pnpb200_robust_workspace_bytes(method, dtype, 1 << 20, 68, 1, 0)
            assert ws >= robust + (1 << 20) * (12 * esz + 4 + 3 * 4 + 4)
    assert lib.lib.pnpb200_ransac_workspace_bytes(4, 0, 0, 68, 1, 0) == 0


@pytest.mark.parametrize("kw", [dict(samples=-1), dict(consensus_px=-1.0), dict(consensus_px=float("nan")), dict(confidence=0.0),
                                dict(confidence=1.01), dict(seed=-1), dict(idx0=-1)])
def test_python_value_errors(kw):
    from pnp_solver_test_b200 import solver
    with pytest.raises(ValueError):
        solver.hypothesis_params(**kw)
    uv, pat = torch.zeros((8, 68, 2), dtype=torch.float64), torch.zeros((68, 3), dtype=torch.float64)
    with pytest.raises(ValueError):                        # before any launch: these tensors are not even on a device
        solver.hypothesize_batch(uv, pat, np.eye(3), **kw)
    with pytest.raises(ValueError):
        solver.solve_robust_batch("lm_plus", uv, pat, np.eye(3), **dict(dict(samples=8), **kw))
    solver.hypothesis_params(samples=0, consensus_px=float("inf"), confidence=1.0)


def test_oracle_p3p_recovers_the_pose():
    """noise-free triples of random poses: some root of Grunert's P3P is the ground truth to 1e-9"""
    import ransac_oracle as ro
    rng = np.random.default_rng(1)
    errs = []
    for _ in range(500):
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        a, b, c, d = q
        R = np.array([[a * a + b * b - c * c - d * d, 2 * (b * c - a * d), 2 * (b * d + a * c)],
                      [2 * (b * c + a * d), a * a - b * b + c * c - d * d, 2 * (c * d - a * b)],
                      [2 * (b * d - a * c), 2 * (c * d + a * b), a * a - b * b - c * c + d * d]])
        t = np.array([rng.uniform(-0.3, 0.3), rng.uniform(-0.3, 0.3), rng.uniform(0.5, 2.0)])
        X = rng.normal(size=(3, 3)) * 0.1
        Y = X @ R.T + t
        Rs, ts = ro.p3p(X, Y / np.linalg.norm(Y, axis=1, keepdims=True))
        assert len(Rs) <= 4 and (ts[:, 2] > 0).all()
        errs.append(min(max(np.abs(Rs[k] - R).max(), np.abs(ts[k] - t).max() / t[2]) for k in range(len(Rs))))
    assert max(errs) <= 1e-9, max(errs)


def test_draw_rule_gives_distinct_uniform_candidates():
    import ransac_oracle as ro
    c, S = 20, 20000
    counts = np.zeros((4, c))
    for s in range(S):
        pos = ro.draw4(c, s // 200, s % 200, seed=7)
        assert len(set(pos.tolist())) == 4 and ((pos >= 0) & (pos < c)).all()
        counts[np.arange(4), pos] += 1
    chi2 = (((counts - S / c) ** 2) / (S / c)).sum(axis=1)
    assert (chi2 < 60.0).all(), chi2                      # 19 degrees of freedom: P(chi2 > 60) ~ 4e-6
    assert (ro.draw4(4, 3, 5) == ro.draw4(4, 3, 5)).all() and sorted(ro.draw4(4, 3, 5).tolist()) == [0, 1, 2, 3]


def test_ransac_accuracy_tables_in_the_header():
    """the pass rates beside pnpb200_solve_ransac_batch in include/pnpb200.h are what tests/ransac_accuracy.py measures, and
    the sweep picks the default consensus_px"""
    import os
    import ransac_accuracy as ra
    from pnp_solver_test_b200 import _lib
    hdr = open(os.path.join(ra.ROOT, "include", "pnpb200.h")).read()
    tab, sw = ra.run()
    for line in ra.header_lines(tab, sw):
        assert line + "\n" in hdr, line
    p = _lib.HypothesisParams()
    _lib.lib.pnpb200_default_hypothesis_params(C.byref(p))
    assert ra.best_px(sw) == p.consensus_px == ra.DEFAULT_PX
