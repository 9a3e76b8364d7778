"""Argument checks of the solution check entries (pnpb200_check_batch, pnpb200_solve_check_batch_host): every
malformed call is refused before anything touches a device, so these run without a GPU."""
import ctypes as C

import pytest


@pytest.fixture()
def lib():
    from pnp_solver_test_b200 import _lib
    return _lib.lib


K = (C.c_double * 9)(225.7, 0, 160, 0, 225.7, 120, 0, 0, 1)
PI = C.POINTER(C.c_int32)
UV, PAT, R, T, STATUS = (C.c_void_p(a) for a in (0x10000, 0x20000, 0x30000, 0x40000, 0x50000))


def _check(lib, dtype=0, B=4, n=68, pattern=PAT, n_patterns=1, uv=UV, k=K, status=STATUS):
    return lib.pnpb200_check_batch(dtype, B, n, pattern, n_patterns, uv, k, R, T, None, None, 1.0,
                                   C.cast(status, PI) if status else None, None, None)


@pytest.mark.parametrize("bad", [dict(uv=None), dict(uv=C.c_void_p(0x10008)), dict(n_patterns=0), dict(n_patterns=9),
                                 dict(dtype=2), dict(dtype=-1), dict(pattern=None), dict(k=None), dict(status=None),
                                 dict(n=0), dict(B=-1)])
def test_check_batch_rejects_bad_arguments(lib, bad):
    assert _check(lib, **bad) == -1                      # PNPB200_EINVAL


def test_check_batch_accepts_an_empty_batch(lib):
    assert _check(lib, B=0) == 0


def _host(lib, pipe=None, uv=UV, status=STATUS, B=4, n=68):
    return lib.pnpb200_solve_check_batch_host(pipe, 1, B, n, 0, uv, PAT, None, K, None, None, None, None, None, None, None, 1.0,
                                              C.cast(status, PI) if status else None, None)


def test_solve_check_batch_host_rejects_bad_arguments(lib):
    assert _host(lib) == -1                              # null pipeline
    assert _host(lib, pipe=C.c_void_p(0x60000), uv=None) == -1
    assert _host(lib, pipe=C.c_void_p(0x60000), status=None) == -1
    out = C.c_void_p()
    for n_patterns in (0, 9):                           # the pipeline's pattern count
        assert lib.pnpb200_pipeline_create(C.byref(out), 0, 1024, 68, n_patterns, 1) == -1
    assert lib.pnpb200_pipeline_create(C.byref(out), 2, 1024, 68, 1, 1) == -1      # dtype


def test_check_bits_are_exported():
    import pnp_solver_test_b200 as pnp
    assert (pnp.CHECK_NONFINITE, pnp.CHECK_DEPTH, pnp.CHECK_BEHIND, pnp.CHECK_REPROJ) == (1, 2, 4, 8)
