"""Per-problem landmark visibility without a GPU: argument checks of the masked C entries, the packing of the bool mask into
words (torch on the device side, np.packbits on the host side) and the ValueErrors of the Python layer."""
import ctypes as C

import numpy as np
import pytest
import torch

EINVAL = -1


@pytest.fixture(scope="module")
def lib():
    from pnp_solver_test_b200 import _lib
    return _lib.lib


def _K():
    return (C.c_double * 9)(800.0, 0.0, 320.0, 0.0, 800.0, 240.0, 0.0, 0.0, 1.0)


FAKE = C.c_void_p(1 << 20)                                 # 16-byte aligned, never dereferenced: every call below fails its checks first
PI = C.POINTER(C.c_int32)
U32 = C.POINTER(C.c_uint32)


@pytest.mark.parametrize("vis", [None, 2, 1 << 20 | 1])
def test_masked_entries_reject_null_or_misaligned_masks(lib, vis):
    v = None if vis is None else C.cast(C.c_void_p(vis), U32)
    K, bd = _K(), (C.c_double * 4)(10, 10, 10, 10)
    pd = C.cast(FAKE, C.POINTER(C.c_double))
    assert lib.pnpb200_solve_batch_masked(1, 0, 64, 68, 68, FAKE, FAKE, 1, None, K, None, FAKE, FAKE, FAKE, FAKE,
                                          C.cast(FAKE, PI), C.cast(FAKE, PI), v, None) == EINVAL
    assert lib.pnpb200_solve_report_batch_masked(1, 0, 64, 68, 68, FAKE, FAKE, None, K, None, FAKE, FAKE, FAKE, FAKE,
                                                 C.cast(FAKE, PI), pd, bd, pd, 16, 1, None, None, v, None) == EINVAL
    assert lib.pnpb200_report_batch_strided_masked(0, 64, 68, FAKE, FAKE, K, FAKE, FAKE, FAKE, pd, bd, pd, 16, 1, None, None,
                                                   v, None) == EINVAL
    assert lib.pnpb200_check_batch_masked(0, 64, 68, FAKE, 1, FAKE, K, FAKE, FAKE, None, None, 1.0, C.cast(FAKE, PI), None,
                                          v, None) == EINVAL
    if vis is None:                                        # (a misaligned host mask is refused once the pipeline exists)
        assert lib.pnpb200_solve_batch_host_masked(FAKE, 1, 64, 68, 0, FAKE, FAKE, None, K, None, FAKE, FAKE, FAKE, FAKE,
                                                   None, None, v, 0.0, None, None) == EINVAL


def test_masked_workspace_query(lib):
    # the masked moment mapping keeps 10 pattern moments per problem beside the unmasked workspace; the direct mappings take none
    for dtype, esz in ((0, 8), (1, 4)):
        for method in range(6):
            for mapping in (0, 1, 2, 32):
                plain = lib.pnpb200_workspace_bytes(method, dtype, 1 << 20, 1, mapping)
                assert lib.pnpb200_workspace_bytes_masked(method, dtype, 1 << 20, 1, mapping) == (plain + 10 * esz * (1 << 20) if plain else 0)


@pytest.mark.parametrize("n_total", [1, 15, 31, 32, 33, 68, 98, 300])
def test_word_packing_matches_packbits(n_total):
    from pnp_solver_test_b200.solver import visible_words, visible_words_host
    rng = np.random.default_rng(n_total)
    vis = rng.random((37, n_total)) < 0.6
    vis[0] = True
    vis[1] = False
    W = (n_total + 31) // 32
    host = visible_words_host(vis)
    assert host.shape == (37, W) and host.dtype == np.uint32
    pad = np.zeros((37, W * 32), bool)
    pad[:, :n_total] = vis
    np.testing.assert_array_equal(host, np.packbits(pad, axis=1, bitorder="little").view("<u4"))
    dev = visible_words(torch.from_numpy(vis), "cpu")
    assert dev.dtype == torch.int32 and tuple(dev.shape) == (37, W)
    np.testing.assert_array_equal(dev.numpy().view(np.uint32), host)
    np.testing.assert_array_equal(visible_words(vis, "cpu").numpy().view(np.uint32), host)     # NumPy input
    for b in (0, 5, 36):                                   # bit i % 32 of word i / 32, least significant first
        for i in range(n_total):
            assert bool((int(host[b, i // 32]) >> (i % 32)) & 1) == vis[b, i]
    np.testing.assert_array_equal(visible_words_host(torch.from_numpy(vis)), host)


@pytest.mark.parametrize("bad", ["shape", "dtype", "type"])
def test_python_value_errors(bad):
    from pnp_solver_test_b200 import solver, workload as wl
    B, n = 8, 68
    vis = {"shape": np.ones((B, n + 1), bool), "dtype": np.ones((B, n), np.uint8), "type": [[True] * n] * B}[bad]
    with pytest.raises(ValueError):
        solver._check_visible(vis, B, n)
    with pytest.raises(ValueError):
        solver._check_visible(torch.from_numpy(np.ones((B, n), np.int32)) if bad == "dtype" else torch.ones((B + 1, n), dtype=torch.bool), B, n)
    uv, pat = torch.zeros((B, n, 2), dtype=torch.float64), torch.zeros((n, 3), dtype=torch.float64)
    R, t, e, gt = torch.zeros((B, 3, 3), dtype=torch.float64), torch.zeros((B, 3), dtype=torch.float64), \
        torch.zeros((B, 3), dtype=torch.float64), torch.zeros((B, 4), dtype=torch.float64)
    K = np.eye(3)
    # the checks come before any launch: these calls never reach the device
    with pytest.raises(ValueError):
        wl.report_batch(pat, uv, K, R, t, e, gt, visible=vis)
    with pytest.raises(ValueError):
        wl.solve_report_batch("lm", uv, pat, K, gt, visible=vis)
    solver._check_visible(np.ones((B, n), bool), B, n)
    solver._check_visible(torch.ones((B, n), dtype=torch.bool), B, n)


def test_visibility_accuracy_table_in_the_header():
    """the pass rates beside the masked entries of include/pnpb200.h are what tests/visibility_accuracy.py measures"""
    import os
    import re
    import visibility_accuracy as va
    hdr = open(os.path.join(va.ROOT, "include", "pnpb200.h")).read()
    names = {"lm": "LM", "lm_plus": "LM+", "eif2": "EIF2", "qeif": "QEIF"}
    for m, row in va.table().items():
        line = re.search(r"^ \*   %s\s+([0-9.]+) %%\s+([0-9.]+) %%\s+([0-9.]+) %%" % re.escape(names[m]), hdr, re.M)
        assert line, m
        assert [float(x) for x in line.groups()] == [round(v, 1) for v in row], (m, row)
