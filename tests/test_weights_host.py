"""Per-landmark weights without a GPU: argument checks of the weighted C entry (EINVAL before any CUDA call), its workspace
query, and the ValueErrors of the Python layer."""
import ctypes as C

import numpy as np
import pytest
import torch

EINVAL = -1
FAKE = C.c_void_p(1 << 20)                                 # 16-byte aligned, never dereferenced: every call below fails its checks first
PI = C.POINTER(C.c_int32)
PF = C.POINTER(C.c_float)


@pytest.fixture(scope="module")
def lib():
    from pnp_solver_test_b200 import _lib
    return _lib.lib


@pytest.mark.parametrize("wts", [None, 2, 1 << 20 | 1])
def test_weighted_entry_rejects_null_or_misaligned_weights(lib, wts):
    w = None if wts is None else C.cast(C.c_void_p(wts), PF)
    K = (C.c_double * 9)(800.0, 0.0, 320.0, 0.0, 800.0, 240.0, 0.0, 0.0, 1.0)
    for method in range(6):
        for dtype in (0, 1):
            assert lib.pnpb200_solve_batch_weighted(method, dtype, 64, 68, 68, FAKE, FAKE, 1, None, K, None, FAKE, FAKE, FAKE,
                                                    FAKE, C.cast(FAKE, PI), C.cast(FAKE, PI), w, None) == EINVAL


def test_weighted_entry_checks_the_rest_before_any_cuda_call(lib):
    # aligned weights: the remaining argument checks of pnpb200_solve_batch still come first (null uv, misaligned uv, bad method)
    K = (C.c_double * 9)(800.0, 0.0, 320.0, 0.0, 800.0, 240.0, 0.0, 0.0, 1.0)
    w = C.cast(FAKE, PF)
    assert lib.pnpb200_solve_batch_weighted(1, 0, 64, 68, 68, None, FAKE, 1, None, K, None, FAKE, None, None, None, None, None,
                                            w, None) == EINVAL
    assert lib.pnpb200_solve_batch_weighted(1, 0, 64, 68, 68, C.c_void_p((1 << 20) + 8), FAKE, 1, None, K, None, FAKE, None,
                                            None, None, None, None, w, None) == EINVAL
    assert lib.pnpb200_solve_batch_weighted(9, 0, 64, 68, 68, FAKE, FAKE, 1, None, K, None, FAKE, None, None, None, None, None,
                                            w, None) == EINVAL


def test_weighted_workspace_query(lib):
    # the weighted moment mapping keeps 10 weighted pattern moments and the count of landmarks taking part per problem
    for dtype, esz in ((0, 8), (1, 4)):
        for method in range(6):
            for mapping in (0, 1, 2, 32):
                plain = lib.pnpb200_workspace_bytes(method, dtype, 1 << 20, 1, mapping)
                assert lib.pnpb200_workspace_bytes_weighted(method, dtype, 1 << 20, 1, mapping) == (plain + 11 * esz * (1 << 20) if plain else 0)


@pytest.mark.parametrize("bad", ["shape", "int", "bool", "complex", "list", "with_visible"])
def test_python_value_errors(bad):
    from pnp_solver_test_b200 import solver
    B, n = 8, 68
    w = {"shape": np.ones((B, n + 1), np.float32), "int": np.ones((B, n), np.int32), "bool": torch.ones((B, n), dtype=torch.bool),
         "complex": torch.ones((B, n), dtype=torch.complex64), "list": [[1.0] * n] * B,
         "with_visible": np.ones((B, n), np.float64)}[bad]
    vis = np.ones((B, n), bool) if bad == "with_visible" else None
    with pytest.raises(ValueError):
        solver._check_weights(w, B, n, vis)
    solver._check_weights(np.ones((B, n), np.float16), B, n)
    solver._check_weights(torch.ones((B, n), dtype=torch.float64), B, n)


def test_solve_pnp_batch_refuses_weights_with_robust_or_visible_before_any_launch():
    from pnp_solver_test_b200 import solver
    s = object.__new__(solver.PNP_SOLVER)                 # no device needed: the checks come before anything touches one
    s.method = "lm"
    s.np_point_3d_pretransfer_dict_list = [{k: np.zeros(3) for k in range(68)}]
    uv = np.zeros((4, 68, 2))
    w = np.ones((4, 68), np.float32)
    with pytest.raises(ValueError):
        s.solve_pnp_batch(uv, weights=w, robust={"max_rounds": 2})
    with pytest.raises(ValueError):
        s.solve_pnp_batch(uv, weights=w, visible=np.ones((4, 68), bool))
    with pytest.raises(ValueError):
        s.solve_pnp_batch(uv, weights=np.ones((4, 67), np.float32))


def test_weights_that_take_part():
    from pnp_solver_test_b200.solver import weights_take_part
    w = np.array([[1.0, 0.0, -0.0, -1.0, np.nan, np.inf, -np.inf, 1e-30, 3e38, 1e39]])
    # float32: 1e-30 is a positive normal, 3e38 is finite, 1e39 rounds to +Inf
    assert weights_take_part(w).numpy().tolist() == [[True, False, False, False, False, False, False, True, True, False]]


def _oracle_workload(n=68, B=48, seed=5):
    import os, sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from oracle import oracle as orc
    from pnp_solver_test_b200 import patterns as pt
    P, K = pt.pattern_array(pt.synthetic_pattern(n)), pt.default_camera_matrix()
    return orc, P, K, orc.synth(0, B, P, K, cfg=orc.default_synth(seed=seed))


METHODS = ("qeif", "lm", "linear_f2", "linear_f1", "lm_plus", "eif2")


@pytest.mark.parametrize("method", METHODS)
def test_weighted_oracle_with_unit_weights_is_the_oracle_bit_for_bit(method):
    import weighted_oracle as wo
    orc, P, K, w = _oracle_workload()
    a = wo.solve_batch(method, w["uv"], P, K, np.ones((48, 68)))
    b = orc.solve_batch(method, w["uv"], P, K)
    for k in ("R", "t", "euler", "res_norm", "iters"):
        assert np.array_equal(a[k].reshape(b[k].shape), b[k]), k


@pytest.mark.parametrize("method", METHODS)
def test_weighted_oracle_integer_weights_are_repetition_and_zero_is_compaction(method):
    import weighted_oracle as wo
    orc, P, K, w = _oracle_workload()
    rng = np.random.default_rng(1)
    wi = rng.integers(0, 4, size=68).astype(np.float64)
    rep = [j for j in range(68) for _ in range(int(wi[j]))]
    a = wo.solve_batch(method, w["uv"], P, K, np.repeat(wi[None], 48, axis=0))
    r = orc.solve_batch(method, w["uv"][:, rep], P[rep], K)
    keep = [j for j in range(68) if wi[j] > 0]
    ones = np.where(wi > 0, 1.0, 0.0)
    c = wo.solve_batch(method, w["uv"], P, K, np.repeat(ones[None], 48, axis=0))
    cc = orc.solve_batch(method, w["uv"][:, keep], P[keep], K)
    for k in ("R", "t", "res_norm", "iters"):
        assert np.array_equal(c[k].reshape(cc[k].shape), cc[k]), k          # w = 0: the compacted problem, bit for bit
    ok = np.ones(48, bool)
    if method in ("lm", "eif2"):                                            # chaotic / ill-conditioned problems (SURVEY.md 7.3): stable ones only
        for sgn in (1.0, -1.0):
            o = orc.solve_batch(method, w["uv"][:, rep] * (1 + sgn * 1e-13), P[rep], K)
            # a 1e-13 input perturbation moves these problems by < 1e-12: well-conditioned enough for two roundings of the same
            # problem (rows repeated against rows times sqrt(w)) to agree to 1e-11
            ok &= np.abs(o["R"] - r["R"]).reshape(48, -1).max(axis=1) < 1e-12
        assert ok.mean() >= 0.4, ok.mean()
    dR = np.abs(a["R"] - r["R"]).reshape(48, -1).max(axis=1)
    dt = np.abs(a["t"] - r["t"]).max(axis=1) / np.abs(r["t"][:, 2])
    assert dR[ok].max() < 1e-11 and dt[ok].max() < 1e-11, (dR[ok].max(), dt[ok].max())
    assert (np.abs(a["res_norm"] - r["res_norm"]) / r["res_norm"])[ok].max() < 1e-10     # (a difference of sums: one decade more)
    if method not in ("lm", "lm_plus"):
        assert np.array_equal(a["iters"], r["iters"])


def test_weights_accuracy_table_in_the_header():
    """the table beside pnpb200_solve_batch_weighted in include/pnpb200.h is what tests/weights_accuracy.py measures"""
    import os
    import weights_accuracy as wa
    hdr = open(os.path.join(wa.ROOT, "include", "pnpb200.h")).read()
    for line in wa.lines(wa.table()):
        assert (" *   " + line) in hdr, line
