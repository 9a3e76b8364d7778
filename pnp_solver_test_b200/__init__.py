"""pnp_solver_test_b200 -- B200-native batched PnP solver with the entry points of
Benson516/pnp_solver_test's scripts/PNP_SOLVER_LIB.py.

Everything that computes goes through libpnpb200.so (hand-written CUDA for sm_100a behind the C
ABI in include/pnpb200.h).  The library is loaded on first use of any solver symbol and the
import fails loudly if it has not been built (`python -m pnp_solver_test_b200.build`); there is
no CPU fallback.  `patterns` (fixture data) and `build` are importable without the library.
"""
import importlib

from . import patterns  # noqa: F401
from .patterns import get_golden_pattern, synthetic_pattern, LM_KEY_LIST_6  # noqa: F401

__version__ = "0.1.0"

_LAZY = {
    "_lib": ("._lib", None), "solver": (".solver", None), "workload": (".workload", None),
    "METHODS": ("._lib", "METHODS"), "default_params": ("._lib", "default_params"),
    "default_synth": ("._lib", "default_synth"), "PnpB200Error": ("._lib", "PnpB200Error"),
    "PNP_SOLVER": (".solver", "PNP_SOLVER"), "HostPipeline": (".solver", "HostPipeline"), "host_buffer": (".solver", "host_buffer"),
    "solve_batch": (".solver", "solve_batch"), "R_from_euler_batch": (".solver", "R_from_euler_batch"),
    "euler_from_R_batch": (".solver", "euler_from_R_batch"), "project_batch": (".solver", "project_batch"),
    "check_batch": (".solver", "check_batch"), "CHECK_NONFINITE": ("._lib", "CHECK_NONFINITE"),
    "CHECK_DEPTH": ("._lib", "CHECK_DEPTH"), "CHECK_BEHIND": ("._lib", "CHECK_BEHIND"), "CHECK_REPROJ": ("._lib", "CHECK_REPROJ"),
    "solve_robust_batch": (".solver", "solve_robust_batch"), "ROBUST_TOO_FEW": ("._lib", "ROBUST_TOO_FEW"),
    "ROBUST_NOT_CONVERGED": ("._lib", "ROBUST_NOT_CONVERGED"), "hypothesize_batch": (".solver", "hypothesize_batch"),
}


def __getattr__(name):
    if name in _LAZY:
        mod, attr = _LAZY[name]
        m = importlib.import_module(mod, __name__)   # raises ImportError if libpnpb200.so is missing
        return m if attr is None else getattr(m, attr)
    raise AttributeError("module %r has no attribute %r" % (__name__, name))
