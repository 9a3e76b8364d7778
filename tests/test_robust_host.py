"""The outlier-robust solve without a GPU: argument checks of pnpb200_solve_robust_batch (EINVAL before any launch), the
ValueErrors of the Python layer, the workspace query, and the accuracy table of include/pnpb200.h against its script."""
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


def _call(lib, robust=None, **kw):
    a = dict(method=4, dtype=0, B=64, n_total=68, n=68, uv=FAKE, pattern=FAKE, n_patterns=1, point_index=None, K=_K(), R=FAKE,
             t=FAKE, best=C.cast(FAKE, PI), visible=None, inliers=C.cast(FAKE, U32), rounds=C.cast(FAKE, PI), status=C.cast(FAKE, PI))
    a.update(kw)
    return lib.lib.pnpb200_solve_robust_batch(a["method"], a["dtype"], a["B"], a["n_total"], a["n"], a["uv"], a["pattern"],
                                              a["n_patterns"], a["point_index"], a["K"], None, a["R"], a["t"], None, None, None,
                                              a["best"], a["visible"], None if robust is None else C.byref(robust), a["inliers"],
                                              a["rounds"], a["status"], None)


def test_default_robust_params(lib):
    p = lib.RobustParams()
    assert lib.lib.pnpb200_default_robust_params(C.byref(p)) == 0
    assert (p.max_rounds, p.k_median, p.floor_px, p.min_inliers) == (4, 3.0, 2.0, 6)
    assert lib.lib.pnpb200_default_robust_params(None) == EINVAL


@pytest.mark.parametrize("field,value", [("max_rounds", 0), ("min_inliers", 3), ("k_median", -1.0), ("k_median", float("nan")),
                                         ("k_median", float("inf")), ("floor_px", -0.5), ("floor_px", float("nan"))])
def test_bad_robust_params_are_einval(lib, field, value):
    p = lib.RobustParams(max_rounds=4, k_median=3.0, floor_px=2.0, min_inliers=6)
    setattr(p, field, value)
    assert _call(lib, p) == EINVAL


@pytest.mark.parametrize("bad", ["R", "t", "inliers", "rounds", "status", "best_two_patterns", "misaligned_visible",
                                 "misaligned_inliers", "point_index", "method", "dtype", "n_patterns"])
def test_bad_arguments_are_einval(lib, bad):
    kw = {"R": dict(R=None), "t": dict(t=None), "inliers": dict(inliers=None), "rounds": dict(rounds=None),
          "status": dict(status=None), "best_two_patterns": dict(n_patterns=2, best=None),
          "misaligned_visible": dict(visible=C.cast(C.c_void_p((1 << 20) | 2), U32)),
          "misaligned_inliers": dict(inliers=C.cast(C.c_void_p((1 << 20) | 1), U32)),
          "point_index": dict(n=2, point_index=(C.c_int32 * 2)(0, 68)), "method": dict(method=6), "dtype": dict(dtype=2),
          "n_patterns": dict(n_patterns=9)}[bad]
    assert _call(lib, **kw) == EINVAL


def test_empty_batch_is_ok(lib):
    assert _call(lib, B=0) == 0


def test_workspace_query(lib):
    # the masked solve's scratch plus the compacted batch: at least the pixel rows of every problem
    for dtype, esz in ((0, 8), (1, 4)):
        for method in range(6):
            ws = lib.lib.pnpb200_robust_workspace_bytes(method, dtype, 1 << 20, 68, 1, 0)
            masked = lib.lib.pnpb200_workspace_bytes_masked(method, dtype, 1 << 20, 1, 0)
            assert ws >= masked + esz * (1 << 20) * 68 * 2
    assert lib.lib.pnpb200_robust_workspace_bytes(4, 0, 0, 68, 1, 0) == 0


@pytest.mark.parametrize("kw", [dict(max_rounds=0), dict(min_inliers=3), dict(k=-1.0), dict(k=float("inf")), dict(floor_px=-1.0),
                                dict(floor_px=float("nan"))])
def test_python_value_errors(kw):
    from pnp_solver_test_b200 import solver
    with pytest.raises(ValueError):
        solver.robust_params(**kw)
    uv, pat = torch.zeros((8, 68, 2), dtype=torch.float64), torch.zeros((68, 3), dtype=torch.float64)
    with pytest.raises(ValueError):                        # before any launch: these tensors are not even on a device
        solver.solve_robust_batch("qeif", uv, pat, np.eye(3), **kw)
    solver.robust_params(floor_px=float("inf"), k=0.0, min_inliers=4, max_rounds=1)


def test_word_unpacking_inverts_packing():
    from pnp_solver_test_b200.solver import unpack_words, visible_words
    for n_total in (1, 15, 32, 33, 68, 300):
        vis = torch.from_numpy(np.random.default_rng(n_total).random((19, n_total)) < 0.5)
        assert torch.equal(unpack_words(visible_words(vis, "cpu"), n_total), vis)


def test_outlier_accuracy_table_in_the_header():
    """the pass rates beside pnpb200_solve_robust_batch in include/pnpb200.h are what tests/outlier_accuracy.py measures"""
    import os
    import outlier_accuracy as oa
    hdr = open(os.path.join(oa.ROOT, "include", "pnpb200.h")).read()
    for line in oa.header_lines(oa.table()):
        assert line + "\n" in hdr, line
