"""ctypes binding of libpnpb200.so (the C ABI declared in include/pnpb200.h).

There is no CPU fallback: if the shared library is missing this module raises at import, and
every compute call raises if the library reports an error (e.g. no CUDA device).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# PNPB200_LIB selects another build of the same library (tools/build_variant.py: A/B measurements of kernel variants)
LIB_PATH = os.environ.get("PNPB200_LIB") or os.path.join(_HERE, "libpnpb200.so")

METHOD_QEIF, METHOD_LM, METHOD_LINEAR_F2, METHOD_LINEAR_F1 = 0, 1, 2, 3
METHOD_LM_PLUS = 4
METHOD_EIF2 = 5
METHODS = {"qeif": 0, "lm": 1, "linear_f2": 2, "linear_f1": 3, "lm_plus": 4, "eif2": 5}
DTYPE_F64, DTYPE_F32 = 0, 1
MAP_AUTO, MAP_THREAD, MAP_MOMENT, MAP_WARP = 0, 1, 2, 32
REPORT_WIDTH = 16
FLAG_PROFILE = 1
FLAG_QEIF_DIRECT = 2
FLAG_LM_TRUE_JACOBIAN = 4
MAX_PATTERNS = 8
PIXEL_NATIVE, PIXEL_I16, PIXEL_U16, PIXEL_F32 = 0, 1, 2, 3
# bits of the status word of the solution check (pnpb200_check_batch)
CHECK_NONFINITE, CHECK_DEPTH, CHECK_BEHIND, CHECK_REPROJ = 1, 2, 4, 8
# bits of robust_status of the outlier-robust solve (pnpb200_solve_robust_batch)
ROBUST_TOO_FEW, ROBUST_NOT_CONVERGED = 1, 2

EXPORTS = [
    "pnpb200_version", "pnpb200_launch_count", "pnpb200_last_error", "pnpb200_default_params", "pnpb200_default_synth",
    "pnpb200_device_info", "pnpb200_workspace_bytes", "pnpb200_solve_batch", "pnpb200_pipeline_create", "pnpb200_pipeline_destroy",
    "pnpb200_solve_batch_host", "pnpb200_R_from_euler", "pnpb200_euler_from_R", "pnpb200_project",
    "pnpb200_synth_batch", "pnpb200_report_batch", "pnpb200_report_batch_strided", "pnpb200_stats_pass1", "pnpb200_stats_pass2",
    "pnpb200_fma_peak", "pnpb200_selftest_math", "pnpb200_selftest_sincos", "pnpb200_pipeline_set_packing", "pnpb200_pipeline_last_packed", "pnpb200_pack_i16", "pnpb200_synth_face_variation", "pnpb200_topk_histogram",
    "pnpb200_fragility_accumulate", "pnpb200_write_result_csv", "pnpb200_format_repr", "pnpb200_classify", "pnpb200_classify_drpy", "pnpb200_profile_reset", "pnpb200_profile_read",
    "pnpb200_solve_batch_host_px", "pnpb200_host_alloc", "pnpb200_host_free", "pnpb200_solve_report_batch", "pnpb200_normalise_uvw",
    "pnpb200_check_batch", "pnpb200_solve_check_batch_host",
    "pnpb200_solve_batch_masked", "pnpb200_solve_report_batch_masked", "pnpb200_report_batch_strided_masked",
    "pnpb200_check_batch_masked", "pnpb200_workspace_bytes_masked", "pnpb200_solve_batch_host_masked",
    "pnpb200_default_robust_params", "pnpb200_robust_workspace_bytes", "pnpb200_solve_robust_batch",
    "pnpb200_default_hypothesis_params", "pnpb200_hypothesize_batch", "pnpb200_ransac_workspace_bytes", "pnpb200_solve_ransac_batch",
    "pnpb200_selftest_p3p", "pnpb200_selftest_inliers", "pnpb200_selftest_project",
    "pnpb200_solve_batch_weighted", "pnpb200_workspace_bytes_weighted",
]


class Params(C.Structure):
    """struct pnpb200_params"""
    _fields_ = [("max_it", C.c_int32), ("linear_it", C.c_int32), ("lm_lambda", C.c_double),
                ("exit_tol", C.c_double), ("f_weight", C.c_double), ("meas_sigma_px", C.c_double),
                ("proc_q", C.c_double), ("proc_d", C.c_double), ("omega0", C.c_double),
                ("res_old0", C.c_double), ("mapping", C.c_int32), ("flags", C.c_int32),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_int64)]


class RobustParams(C.Structure):
    """struct pnpb200_robust_params"""
    _fields_ = [("max_rounds", C.c_int32), ("k_median", C.c_double), ("floor_px", C.c_double), ("min_inliers", C.c_int32)]


class HypothesisParams(C.Structure):
    """struct pnpb200_hypothesis_params"""
    _fields_ = [("max_samples", C.c_int32), ("consensus_px", C.c_double), ("confidence", C.c_double), ("seed", C.c_uint64),
                ("idx0", C.c_int64)]


class Synth(C.Structure):
    """struct pnpb200_synth"""
    _fields_ = [("seed", C.c_uint64), ("angle_range_deg", C.c_double), ("depth_min_m", C.c_double),
                ("depth_max_m", C.c_double), ("fov_max_deg", C.c_double), ("is_quantized", C.c_int32),
                ("reserved", C.c_int32), ("quantize_q", C.c_double), ("noise_sigma_px", C.c_double),
                ("roll_center_deg", C.c_double), ("pitch_center_deg", C.c_double), ("yaw_center_deg", C.c_double)]


class PnpB200Error(RuntimeError):
    pass


if not os.path.exists(LIB_PATH):
    raise ImportError(
        "pnp_solver_test_b200: %s is missing.  Build it with `python -m pnp_solver_test_b200.build` "
        "(needs nvcc; there is no CPU fallback)." % LIB_PATH)

lib = C.CDLL(LIB_PATH)
lib.pnpb200_version.restype = C.c_int
lib.pnpb200_last_error.restype = C.c_char_p
for _name in EXPORTS:
    if _name not in ("pnpb200_last_error",):
        getattr(lib, _name).restype = C.c_int
lib.pnpb200_workspace_bytes.restype = C.c_int64
_VP, _PD, _PI = C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int32)
lib.pnpb200_check_batch.argtypes = [C.c_int, C.c_int64, C.c_int, _VP, C.c_int, _VP, _PD, _VP, _VP, _VP, _PI, C.c_double, _PI, _VP,
                                    _VP]
lib.pnpb200_solve_check_batch_host.argtypes = [_VP, C.c_int, C.c_int64, C.c_int, C.c_int, _VP, _VP, _PI, _PD, _VP, _VP, _VP, _VP,
                                               _VP, _PI, _PI, C.c_double, _PI, _VP]
lib.pnpb200_launch_count.restype = C.c_int64
# the masked entries: the unmasked ones plus `const uint32_t* visible` (before the stream)
_U32P = C.POINTER(C.c_uint32)
lib.pnpb200_workspace_bytes_masked.restype = C.c_int64
lib.pnpb200_workspace_bytes_masked.argtypes = [C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int]
lib.pnpb200_solve_batch_masked.argtypes = [C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int, _VP, _VP, C.c_int, _PI, _PD, _VP,
                                           _VP, _VP, _VP, _VP, _PI, _PI, _U32P, _VP]
lib.pnpb200_solve_report_batch_masked.argtypes = [C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int, _VP, _VP, _PI, _PD, _VP,
                                                  _VP, _VP, _VP, _VP, _PI, _PD, _PD, _PD, C.c_int64, C.c_int64, _PI, _PI,
                                                  _U32P, _VP]
lib.pnpb200_report_batch_strided_masked.argtypes = [C.c_int, C.c_int64, C.c_int, _VP, _VP, _PD, _VP, _VP, _VP, _PD, _PD,
                                                    _PD, C.c_int64, C.c_int64, _PI, _PI, _U32P, _VP]
lib.pnpb200_check_batch_masked.argtypes = [C.c_int, C.c_int64, C.c_int, _VP, C.c_int, _VP, _PD, _VP, _VP, _VP, _PI, C.c_double,
                                           _PI, _VP, _U32P, _VP]
lib.pnpb200_solve_batch_host_masked.argtypes = [_VP, C.c_int, C.c_int64, C.c_int, C.c_int, _VP, _VP, _PI, _PD, _VP, _VP, _VP,
                                                _VP, _VP, _PI, _PI, _U32P, C.c_double, _PI, _VP]
# the weighted entry: the unmasked one plus `const float* weights` (before the stream)
lib.pnpb200_workspace_bytes_weighted.restype = C.c_int64
lib.pnpb200_workspace_bytes_weighted.argtypes = [C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int]
lib.pnpb200_solve_batch_weighted.argtypes = lib.pnpb200_solve_batch_masked.argtypes[:-2] + [C.POINTER(C.c_float), _VP]
lib.pnpb200_robust_workspace_bytes.restype = C.c_int64
lib.pnpb200_robust_workspace_bytes.argtypes = [C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int]
# pnpb200_solve_batch_masked's arguments, then the robust parameters and the three outputs
lib.pnpb200_solve_robust_batch.argtypes = [C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int, _VP, _VP, C.c_int, _PI, _PD, _VP,
                                           _VP, _VP, _VP, _VP, _PI, _PI, _U32P, _VP, _U32P, _PI, _PI, _VP]
# the hypothesis stage and the RANSAC solve: the robust entry's arguments, then the hypothesis parameters, consensus and drawn
lib.pnpb200_hypothesize_batch.argtypes = [C.c_int, C.c_int64, C.c_int, C.c_int, _VP, _VP, C.c_int, _PI, _PD, _U32P, _VP, _VP, _VP,
                                          _PI, _U32P, _PI, _PI, _VP]
lib.pnpb200_ransac_workspace_bytes.restype = C.c_int64
lib.pnpb200_ransac_workspace_bytes.argtypes = [C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int]
lib.pnpb200_solve_ransac_batch.argtypes = lib.pnpb200_solve_robust_batch.argtypes[:-1] + [_VP, _PI, _PI, _VP]
lib.pnpb200_selftest_p3p.argtypes = [C.c_int64, _VP, _VP, _VP, _VP, _VP, _VP]
lib.pnpb200_selftest_project.argtypes = [C.c_int, C.c_int64, _VP, _VP, _VP, _VP]
lib.pnpb200_selftest_inliers.argtypes = [C.c_int, C.c_int64, C.c_int, C.c_int, _VP, _VP, C.c_int, _PI, _PD, _U32P, _VP, _VP, _VP,
                                         _PI, _PI, C.c_int, _U32P, _PI, _PI, _VP, _PD, C.c_int, _VP]

_ERR = {-1: "EINVAL (bad argument)", -2: "ECUDA (CUDA runtime error)", -3: "ENODEVICE (no usable CUDA device)",
        -4: "ETOOLARGE (n too large for the selected mapping)"}


def check(rc, what):
    if rc != 0:
        detail = lib.pnpb200_last_error() or b""
        raise PnpB200Error("%s failed: %s %s" % (what, _ERR.get(rc, str(rc)), detail.decode(errors="replace")))


def default_params(**kw):
    p = Params()
    check(lib.pnpb200_default_params(C.byref(p)), "pnpb200_default_params")
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def default_synth(**kw):
    s = Synth()
    check(lib.pnpb200_default_synth(C.byref(s)), "pnpb200_default_synth")
    for k, v in kw.items():
        setattr(s, k, v)
    return s


def ptr(t):
    """device/host pointer of a torch tensor (or None)"""
    return None if t is None else C.c_void_p(t.data_ptr())


# number of kernels of THIS library launched by the Python wrappers (bench.py reports it)
LAUNCHES = [0]


def count_launch(n=1):
    LAUNCHES[0] += int(n)
