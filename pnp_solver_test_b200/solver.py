"""Drop-in mirror of the reference's solver class, backed by the CUDA library.

`PNP_SOLVER` keeps the constructor, method names, argument order, return tuples and side
effects of scripts/PNP_SOLVER_LIB.py:7-4704 for everything on the hot path (SURVEY.md 8b), so
random_stress_test.py / LM_noise_test.py / face_variation_test.py can swap it in for their
per-problem loop; `solve_pnp_batch` is the batched entry point those loops collapse into.
Host code here only packs arguments: every number is computed by libpnpb200.so on the GPU
(PyTorch tensors are used for device memory and streams, nothing else).  No CPU fallback.
"""
import copy
import os
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import lib, check, ptr
_check_rc = check        # HostPipeline.solve's keyword `check` shadows the name there
from .patterns import LM_KEY_LIST_6

_TORCH_DTYPE = {_lib.DTYPE_F64: torch.float64, _lib.DTYPE_F32: torch.float32}


def _dtype_code(dtype):
    if dtype in (torch.float64, "f64", "float64", np.float64, _lib.DTYPE_F64):
        return _lib.DTYPE_F64
    if dtype in (torch.float32, "f32", "float32", np.float32):
        return _lib.DTYPE_F32
    if dtype == _lib.DTYPE_F32:
        return _lib.DTYPE_F32
    raise ValueError("dtype must be float64 or float32")


def _stream_ptr(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _k_host(K):
    K = np.ascontiguousarray(np.asarray(K, dtype=np.float64).reshape(3, 3))
    return K, K.ctypes.data_as(C.POINTER(C.c_double))


def _copy_params(p):
    q = _lib.Params()
    C.memmove(C.byref(q), C.byref(p), C.sizeof(_lib.Params))
    return q


def _check_visible(visible, B, n_total):
    """visible must be a bool [B, n_total] torch tensor or NumPy array"""
    if torch.is_tensor(visible):
        ok = visible.dtype == torch.bool
    elif isinstance(visible, np.ndarray):
        ok = visible.dtype == np.bool_
    else:
        raise ValueError("visible must be a bool torch tensor or NumPy array, not %s" % type(visible).__name__)
    if not ok:
        raise ValueError("visible must have dtype bool, not %s" % (visible.dtype,))
    if tuple(visible.shape) != (B, n_total):
        raise ValueError("visible must be [B, n_total] = [%d, %d], not %s" % (B, n_total, tuple(visible.shape)))


def visible_words(visible, device):
    """bool [B, n_total] visibility -> the [B, ceil(n_total / 32)] words of the masked entries (bit i % 32 of word i / 32 =
    landmark i, least significant bit first), packed with torch ops on `device`: eight landmarks per byte, four bytes per word
    (little-endian), one byte per landmark of temporary memory.  The int32 tensor holds the uint32 bits."""
    if isinstance(visible, np.ndarray):
        visible = torch.from_numpy(np.ascontiguousarray(visible))
    B, n_total = int(visible.shape[0]), int(visible.shape[1])
    W = (n_total + 31) // 32
    u8 = visible.to(device).contiguous().view(torch.uint8)
    if W * 32 != n_total:
        u8 = torch.nn.functional.pad(u8, (0, W * 32 - n_total))
    shifts = torch.arange(8, dtype=torch.uint8, device=device)
    byte = (u8.reshape(B, W * 4, 8) << shifts).sum(-1, dtype=torch.uint8)
    return byte.contiguous().view(torch.int32)


def visible_words_host(visible):
    """the same words on the host, np.packbits(..., bitorder="little"): a [B, ceil(n_total / 32)] uint32 NumPy array"""
    if torch.is_tensor(visible):
        visible = visible.cpu().numpy()
    B, n_total = int(visible.shape[0]), int(visible.shape[1])
    W = (n_total + 31) // 32
    v = np.zeros((B, W * 32), dtype=np.bool_)
    v[:, :n_total] = visible
    return np.ascontiguousarray(np.packbits(v, axis=1, bitorder="little").view("<u4"))


def _u32(t):
    return C.cast(ptr(t), C.POINTER(C.c_uint32))


def _batch_args(method, uv, patterns, point_index, visible):
    """the argument checks and conversions of solve_batch and solve_robust_batch (ValueError before any launch)"""
    m = _lib.METHODS[method] if isinstance(method, str) else int(method)
    if not (uv.is_cuda and patterns.is_cuda):
        raise ValueError("uv and patterns must be CUDA tensors (no CPU fallback)")
    if uv.dtype != patterns.dtype:
        raise ValueError("uv and patterns must share one dtype")
    dt = _dtype_code(uv.dtype)
    uv = uv.contiguous()
    patterns = patterns.contiguous()
    if patterns.dim() == 2:
        patterns = patterns.unsqueeze(0)
    B, n_total = int(uv.shape[0]), int(uv.shape[1])
    if uv.dim() != 3 or uv.shape[2] != 2 or patterns.shape[1] != n_total or patterns.shape[2] != 3:
        raise ValueError("shape mismatch: uv [B,n,2], patterns [P,n,3]")
    if visible is not None:
        _check_visible(visible, B, n_total)
    idx = None if point_index is None else np.ascontiguousarray(np.asarray(point_index, dtype=np.int32))
    return m, dt, uv, patterns, B, n_total, idx


def solve_batch(method, uv, patterns, K, point_index=None, params=None, want=("R", "t", "euler", "res_norm", "iters", "best_pattern"),
                visible=None):
    """pnpb200_solve_batch on device tensors.

    uv [B, n_total, 2] and patterns [P, n_total, 3] are CUDA tensors of the same float dtype;
    K is a host 3x3.  Returns a dict of CUDA tensors: R [B,3,3], t [B,3], euler [B,3] =
    (roll, yaw, pitch) in degrees, res_norm [B], iters [B] int32, best_pattern [B] int32.
    visible: bool [B, n_total] (torch tensor or NumPy array) -> pnpb200_solve_batch_masked: each problem is solved on its
    visible landmarks alone (those of point_index, in its order); hidden pixels are never read, and a problem with fewer
    than 4 of them comes back NaN with iters 0 (include/pnpb200.h)."""
    m, dt, uv, patterns, B, n_total, idx = _batch_args(method, uv, patterns, point_index, visible)
    n, idx_p = (n_total, None) if idx is None else (int(idx.shape[0]), idx.ctypes.data_as(C.POINTER(C.c_int32)))
    dev = uv.device
    o = {}
    if "R" in want: o["R"] = torch.empty((B, 3, 3), dtype=uv.dtype, device=dev)
    if "t" in want: o["t"] = torch.empty((B, 3), dtype=uv.dtype, device=dev)
    if "euler" in want: o["euler"] = torch.empty((B, 3), dtype=uv.dtype, device=dev)
    if "res_norm" in want: o["res_norm"] = torch.empty((B,), dtype=uv.dtype, device=dev)
    if "iters" in want: o["iters"] = torch.empty((B,), dtype=torch.int32, device=dev)
    if "best_pattern" in want: o["best_pattern"] = torch.empty((B,), dtype=torch.int32, device=dev)
    Kh, Kp = _k_host(K)
    if B == 0:
        return o
    # scratch for the moment mapping from torch's caching allocator (stream-ordered, no driver call)
    prm = _lib.default_params() if params is None else params
    ws_query = lib.pnpb200_workspace_bytes if visible is None else lib.pnpb200_workspace_bytes_masked
    ws_bytes = int(ws_query(C.c_int(m), C.c_int(dt), C.c_int64(B), C.c_int(int(patterns.shape[0])), C.c_int(int(prm.mapping))))
    ws = None
    if ws_bytes > 0 and not prm.workspace:
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
        prm = _copy_params(prm)
        prm.workspace, prm.workspace_bytes = ws.data_ptr(), ws_bytes
    params = prm
    if visible is not None:
        words = visible_words(visible, dev)
        with torch.cuda.device(dev):
            rc = lib.pnpb200_solve_batch_masked(
                m, dt, B, n_total, n, ptr(uv), ptr(patterns), int(patterns.shape[0]), idx_p, Kp, C.byref(params),
                ptr(o.get("R")), ptr(o.get("t")), ptr(o.get("euler")), ptr(o.get("res_norm")),
                None if o.get("iters") is None else C.cast(ptr(o["iters"]), C.POINTER(C.c_int32)),
                None if o.get("best_pattern") is None else C.cast(ptr(o["best_pattern"]), C.POINTER(C.c_int32)),
                _u32(words), _stream_ptr(dev))
        check(rc, "pnpb200_solve_batch_masked")
        _lib.count_launch(1)
        return o
    with torch.cuda.device(dev):
        rc = lib.pnpb200_solve_batch(
            C.c_int(m), C.c_int(dt), C.c_int64(B), C.c_int(n_total), C.c_int(n), ptr(uv), ptr(patterns),
            C.c_int(int(patterns.shape[0])), idx_p, Kp, C.byref(params) if params is not None else None,
            ptr(o.get("R")), ptr(o.get("t")), ptr(o.get("euler")), ptr(o.get("res_norm")),
            ptr(o.get("iters")), ptr(o.get("best_pattern")), _stream_ptr(dev))
    check(rc, "pnpb200_solve_batch")
    _lib.count_launch(1 if B > 0 else 0)
    return o


def robust_params(max_rounds=4, k=3.0, floor_px=2.0, min_inliers=6):
    """struct pnpb200_robust_params; ValueError for what pnpb200_solve_robust_batch refuses with EINVAL"""
    max_rounds, min_inliers, k, floor_px = int(max_rounds), int(min_inliers), float(k), float(floor_px)
    if max_rounds < 1:
        raise ValueError("max_rounds must be >= 1, not %d" % max_rounds)
    if min_inliers < 4:
        raise ValueError("min_inliers must be >= 4, not %d" % min_inliers)
    if not (np.isfinite(k) and k >= 0.0):
        raise ValueError("k must be finite and >= 0, not %r" % k)
    if not floor_px >= 0.0:
        raise ValueError("floor_px must be >= 0 (inf allowed), not %r" % floor_px)
    return _lib.RobustParams(max_rounds=max_rounds, k_median=k, floor_px=floor_px, min_inliers=min_inliers)


def hypothesis_params(samples=128, consensus_px=4.0, confidence=0.999, seed=0, idx0=0):
    """struct pnpb200_hypothesis_params; ValueError for what pnpb200_hypothesize_batch refuses with EINVAL"""
    samples, consensus_px, confidence, seed, idx0 = int(samples), float(consensus_px), float(confidence), int(seed), int(idx0)
    if samples < 0:
        raise ValueError("samples must be >= 0, not %d" % samples)
    if not consensus_px >= 0.0:
        raise ValueError("consensus_px must be >= 0 (inf allowed), not %r" % consensus_px)
    if not 0.0 < confidence <= 1.0:
        raise ValueError("confidence must lie in (0, 1], not %r" % confidence)
    if not 0 <= seed < 1 << 64:
        raise ValueError("seed must be a 64-bit unsigned integer, not %d" % seed)
    if idx0 < 0:
        raise ValueError("idx0 must be >= 0, not %d" % idx0)
    return _lib.HypothesisParams(max_samples=samples, consensus_px=consensus_px, confidence=confidence, seed=seed, idx0=idx0)


def hypothesize_batch(uv, patterns, K, point_index=None, visible=None, samples=128, consensus_px=4.0, confidence=0.999, seed=0, idx0=0):
    """pnpb200_hypothesize_batch on device tensors: per problem, minimal samples of 4 candidates (the landmarks of point_index
    that are visible), a P3P pose per sample and pattern tested on the 4th landmark, and the largest consensus set under the
    check's reprojection distance (<= consensus_px).  Returns dict(R [B,3,3], t [B,3] (the winner's pose; NaN where no sample
    survived), best_pattern [B] int32, consensus_mask bool [B, n_total], consensus [B] int32 (its size), drawn [B] int32 (the
    samples taken)).  The rule is in include/pnpb200.h; idx0 = the global index of problem 0 (shards draw what the unsharded
    call draws)."""
    hp = hypothesis_params(samples, consensus_px, confidence, seed, idx0)
    _, dt, uv, patterns, B, n_total, idx = _batch_args(0, uv, patterns, point_index, visible)
    n, idx_p = (n_total, None) if idx is None else (int(idx.shape[0]), idx.ctypes.data_as(C.POINTER(C.c_int32)))
    dev = uv.device
    P = int(patterns.shape[0])
    o = dict(R=torch.empty((B, 3, 3), dtype=uv.dtype, device=dev), t=torch.empty((B, 3), dtype=uv.dtype, device=dev),
             best_pattern=torch.empty((B,), dtype=torch.int32, device=dev), consensus=torch.empty((B,), dtype=torch.int32, device=dev),
             drawn=torch.empty((B,), dtype=torch.int32, device=dev))
    words = torch.empty((B, (n_total + 31) // 32), dtype=torch.int32, device=dev)
    if B == 0:
        o["consensus_mask"] = torch.empty((0, n_total), dtype=torch.bool, device=dev)
        return o
    Kh, Kp = _k_host(K)
    vw = None if visible is None else visible_words(visible, dev)
    PI = C.POINTER(C.c_int32)
    with torch.cuda.device(dev):
        rc = lib.pnpb200_hypothesize_batch(
            dt, B, n_total, n, ptr(uv), ptr(patterns), P, idx_p, Kp, None if vw is None else _u32(vw), C.byref(hp), ptr(o["R"]),
            ptr(o["t"]), C.cast(ptr(o["best_pattern"]), PI), _u32(words), C.cast(ptr(o["consensus"]), PI),
            C.cast(ptr(o["drawn"]), PI), _stream_ptr(dev))
    check(rc, "pnpb200_hypothesize_batch")
    _lib.count_launch(1)
    o["consensus_mask"] = unpack_words(words, n_total)
    return o


def unpack_words(words, n_total):
    """the inverse of visible_words: [B, W] int32 words -> bool [B, n_total] on the words' device"""
    B, W = int(words.shape[0]), int(words.shape[1])
    shifts = torch.arange(8, dtype=torch.uint8, device=words.device)
    bits = (words.contiguous().view(torch.uint8).reshape(B, W * 4, 1) >> shifts) & 1
    return bits.reshape(B, W * 32)[:, :n_total].bool()


def solve_robust_batch(method, uv, patterns, K, point_index=None, params=None, visible=None, max_rounds=4, k=3.0, floor_px=2.0,
                       min_inliers=6, samples=None, consensus_px=4.0, confidence=0.999, seed=0, idx0=0):
    """pnpb200_solve_robust_batch on device tensors: each problem is solved on its candidates (the landmarks of point_index
    that are visible), the landmarks whose reprojection distance exceeds max(floor_px, k * median) are dropped, and the
    problem is solved again on the rest, until the inlier set stops changing or after max_rounds solves.  Returns the dict of
    solve_batch plus inliers (bool [B, n_total]: the landmarks the returned pose was solved on), rounds [B] int32 (solves)
    and robust_status [B] int32 (ROBUST_TOO_FEW, ROBUST_NOT_CONVERGED bits; 0 = converged).  Every output of a problem is
    bit for bit that of solve_batch(..., visible=inliers).  The rule, its defaults and what it rescues are in
    include/pnpb200.h.  The call synchronises the stream once per round.
    samples: None -> the loop starts from all candidates (pnpb200_solve_robust_batch).  An int >= 0 -> pnpb200_solve_ransac_batch:
    the hypothesis stage of hypothesize_batch (samples, consensus_px, confidence, seed, idx0) runs first and the loop starts
    from its consensus set where that holds at least min_inliers landmarks; the dict then also holds consensus and drawn."""
    rp = robust_params(max_rounds, k, floor_px, min_inliers)
    hp = None if samples is None else hypothesis_params(samples, consensus_px, confidence, seed, idx0)
    m, dt, uv, patterns, B, n_total, idx = _batch_args(method, uv, patterns, point_index, visible)
    n, idx_p = (n_total, None) if idx is None else (int(idx.shape[0]), idx.ctypes.data_as(C.POINTER(C.c_int32)))
    dev = uv.device
    P = int(patterns.shape[0])
    o = dict(R=torch.empty((B, 3, 3), dtype=uv.dtype, device=dev), t=torch.empty((B, 3), dtype=uv.dtype, device=dev),
             euler=torch.empty((B, 3), dtype=uv.dtype, device=dev), res_norm=torch.empty((B,), dtype=uv.dtype, device=dev),
             iters=torch.empty((B,), dtype=torch.int32, device=dev), best_pattern=torch.empty((B,), dtype=torch.int32, device=dev))
    words = torch.empty((B, (n_total + 31) // 32), dtype=torch.int32, device=dev)
    o["rounds"] = torch.empty((B,), dtype=torch.int32, device=dev)
    o["robust_status"] = torch.empty((B,), dtype=torch.int32, device=dev)
    if hp is not None:
        o["consensus"] = torch.empty((B,), dtype=torch.int32, device=dev)
        o["drawn"] = torch.empty((B,), dtype=torch.int32, device=dev)
    if B == 0:
        o["inliers"] = torch.empty((0, n_total), dtype=torch.bool, device=dev)
        return o
    Kh, Kp = _k_host(K)
    prm = _lib.default_params() if params is None else params
    ws_query = lib.pnpb200_robust_workspace_bytes if hp is None else lib.pnpb200_ransac_workspace_bytes
    ws_bytes = int(ws_query(m, dt, B, n_total, P, int(prm.mapping)))
    ws = None
    if ws_bytes > 0 and not prm.workspace:
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
        prm = _copy_params(prm)
        prm.workspace, prm.workspace_bytes = ws.data_ptr(), ws_bytes
    vw = None if visible is None else visible_words(visible, dev)
    PI = C.POINTER(C.c_int32)
    args = (m, dt, B, n_total, n, ptr(uv), ptr(patterns), P, idx_p, Kp, C.byref(prm), ptr(o["R"]), ptr(o["t"]), ptr(o["euler"]),
            ptr(o["res_norm"]), C.cast(ptr(o["iters"]), PI), C.cast(ptr(o["best_pattern"]), PI), None if vw is None else _u32(vw),
            C.byref(rp), _u32(words), C.cast(ptr(o["rounds"]), PI), C.cast(ptr(o["robust_status"]), PI))
    with torch.cuda.device(dev):
        if hp is None:
            rc, name = lib.pnpb200_solve_robust_batch(*args, _stream_ptr(dev)), "pnpb200_solve_robust_batch"
        else:
            rc, name = lib.pnpb200_solve_ransac_batch(*args, C.byref(hp), C.cast(ptr(o["consensus"]), PI), C.cast(ptr(o["drawn"]), PI),
                                                      _stream_ptr(dev)), "pnpb200_solve_ransac_batch"
    check(rc, name)
    _lib.count_launch(1)
    o["inliers"] = unpack_words(words, n_total)
    return o


def check_batch(uv, patterns, K, R, t, res_norm=None, best_pattern=None, reproj_limit_px=1.0, visible=None):
    """pnpb200_check_batch on device tensors: the solution check of any pose, without ground truth.

    uv [B, n_total, 2], patterns [P, n_total, 3] (or [n_total, 3]), R [B,3,3], t [B,3] and res_norm [B] are CUDA
    tensors of one float dtype; best_pattern [B] int32 picks each problem's pattern (None: pattern 0); K is a host
    3x3.  Returns dict(status [B] int32 of CHECK_* bits, reproj [B,2] = (mean, max) prediction-vs-landmark distance in
    pixels over all n_total landmarks).  REPROJ is set where the mean exceeds reproj_limit_px (<= 0 turns it off).
    What the bits find, and what they miss (EIF2), is in include/pnpb200.h.
    visible: bool [B, n_total] -> pnpb200_check_batch_masked: reproj and BEHIND over each problem's visible landmarks."""
    if not all(x.is_cuda for x in (uv, patterns, R, t)):
        raise ValueError("uv, patterns, R and t must be CUDA tensors (no CPU fallback)")
    if len({x.dtype for x in (uv, patterns, R, t) + (() if res_norm is None else (res_norm,))}) != 1:
        raise ValueError("uv, patterns, R, t and res_norm must share one dtype")
    if patterns.dim() == 2:
        patterns = patterns.unsqueeze(0)
    B, n_total = int(uv.shape[0]), int(uv.shape[1])
    if uv.dim() != 3 or uv.shape[2] != 2 or patterns.dim() != 3 or tuple(patterns.shape[1:]) != (n_total, 3):
        raise ValueError("shape mismatch: uv [B,n,2], patterns [P,n,3]")
    if R.numel() != 9 * B or t.numel() != 3 * B or (res_norm is not None and res_norm.numel() != B):
        raise ValueError("R [B,3,3], t [B,3] and res_norm [B] must hold B = %d problems" % B)
    if best_pattern is not None and (best_pattern.dtype != torch.int32 or best_pattern.numel() != B or not best_pattern.is_cuda):
        raise ValueError("best_pattern must be a CUDA int32 tensor of B = %d entries" % B)
    if visible is not None:
        _check_visible(visible, B, n_total)
    dev = uv.device
    uv, patterns, R, t = uv.contiguous(), patterns.contiguous(), R.contiguous(), t.contiguous()
    res_norm = None if res_norm is None else res_norm.contiguous()
    best_pattern = None if best_pattern is None else best_pattern.contiguous()
    status = torch.empty((B,), dtype=torch.int32, device=dev)
    reproj = torch.empty((B, 2), dtype=uv.dtype, device=dev)
    if B == 0:
        return dict(status=status, reproj=reproj)
    Kh, Kp = _k_host(K)
    PI = C.POINTER(C.c_int32)
    bp = None if best_pattern is None else C.cast(ptr(best_pattern), PI)
    with torch.cuda.device(dev):
        if visible is None:
            rc = lib.pnpb200_check_batch(_dtype_code(uv.dtype), B, n_total, ptr(patterns), int(patterns.shape[0]), ptr(uv), Kp, ptr(R),
                                         ptr(t), ptr(res_norm), bp, float(reproj_limit_px), C.cast(ptr(status), PI), ptr(reproj),
                                         _stream_ptr(dev))
        else:
            words = visible_words(visible, dev)
            rc = lib.pnpb200_check_batch_masked(_dtype_code(uv.dtype), B, n_total, ptr(patterns), int(patterns.shape[0]), ptr(uv), Kp,
                                                ptr(R), ptr(t), ptr(res_norm), bp, float(reproj_limit_px), C.cast(ptr(status), PI),
                                                ptr(reproj), _u32(words), _stream_ptr(dev))
    check(rc, "pnpb200_check_batch" if visible is None else "pnpb200_check_batch_masked")
    _lib.count_launch()
    return dict(status=status, reproj=reproj)


class HostPipeline(object):
    """Chunked H2D -> solve -> D2H pipeline over host (ideally pinned) buffers:
    pnpb200_pipeline_* / pnpb200_solve_batch_host.  This is the end-to-end call."""

    def __init__(self, dtype, chunk_problems, n_total, n_patterns=1, n_streams=3, device=None, pack_threads=0):
        """pack_threads > 0: chunks whose pixels are whole numbers (quantised detections) may travel as
        int16 -- a second host thread packs chunks from the far end of the batch with that many workers
        while this one sends chunks unchanged from the near end (pnpb200_pipeline_set_packing)."""
        self.dt = _dtype_code(dtype)
        self.n_total, self.n_patterns = int(n_total), int(n_patterns)
        self.chunk = int(chunk_problems)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self._h = C.c_void_p()
        with torch.cuda.device(self.device):
            check(lib.pnpb200_pipeline_create(C.byref(self._h), C.c_int(self.dt), C.c_int64(int(chunk_problems)),
                                              C.c_int(self.n_total), C.c_int(self.n_patterns), C.c_int(int(n_streams))),
                  "pnpb200_pipeline_create")
            if pack_threads:
                self.set_packing(pack_threads)

    def set_packing(self, n_threads):
        with torch.cuda.device(self.device):
            check(lib.pnpb200_pipeline_set_packing(self._h, C.c_int(int(n_threads))), "pnpb200_pipeline_set_packing")

    def last_packed(self):
        """(chunks of the last solve() that travelled as int16, chunks of that call)"""
        a, b = C.c_int64(0), C.c_int64(0)
        check(lib.pnpb200_pipeline_last_packed(self._h, C.byref(a), C.byref(b)), "pnpb200_pipeline_last_packed")
        return int(a.value), int(b.value)

    def close(self):
        if self._h:
            lib.pnpb200_pipeline_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    _PIXEL_TYPES = {torch.int16: _lib.PIXEL_I16, torch.uint16: _lib.PIXEL_U16, torch.float32: _lib.PIXEL_F32}
    _OUT_SHAPES = {"R": (9, None), "t": (3, None), "euler": (3, None), "res_norm": (1, None), "iters": (1, torch.int32),
                   "best_pattern": (1, torch.int32), "status": (1, torch.int32), "reproj": (2, None)}

    def solve(self, method, uv_host, patterns_host, K, out, point_index=None, params=None, check=None, visible=None):
        """uv_host [B,n_total,2], patterns_host [P,n_total,3]: contiguous CPU torch tensors (pinned for overlap).
        uv_host may also be int16, uint16 or float32 whatever the pipeline's dtype (detections as a detector
        delivers them: pnpb200_solve_batch_host_px ships them as they are and widens them on the device).
        out: dict of contiguous CPU tensors to fill among R [B,3,3] / [B,9], t [B,3], euler [B,3], res_norm [B]
        (pipeline dtype), iters [B], best_pattern [B] (int32).  check = a limit in px: each chunk's solve is followed
        by the solution check (pnpb200_solve_check_batch_host), whose status [B] (int32, required then) and
        reproj [B,2] (pipeline dtype) go to out as well.  Everything is checked here: the C side reads and
        writes B * (row size) elements through the raw pointers.
        visible: bool [B, n_total] (NumPy array or torch tensor) -> pnpb200_solve_batch_host_masked: every chunk's mask words
        travel with its pixels, and the solve (and check) of each problem use its visible landmarks alone."""
        m = _lib.METHODS[method] if isinstance(method, str) else int(method)
        tdt = _TORCH_DTYPE[self.dt]
        if not (torch.is_tensor(uv_host) and torch.is_tensor(patterns_host)):
            raise ValueError("uv_host and patterns_host must be CPU torch tensors")
        if uv_host.is_cuda or patterns_host.is_cuda or not uv_host.is_contiguous() or not patterns_host.is_contiguous():
            raise ValueError("uv_host and patterns_host must be contiguous CPU tensors")
        if uv_host.dim() != 3 or tuple(uv_host.shape[1:]) != (self.n_total, 2):
            raise ValueError("uv_host must be [B, %d, 2], not %s" % (self.n_total, tuple(uv_host.shape)))
        if uv_host.dtype == tdt:
            px = _lib.PIXEL_NATIVE
        elif uv_host.dtype in self._PIXEL_TYPES and not (uv_host.dtype == torch.float32 and tdt == torch.float32):
            px = self._PIXEL_TYPES[uv_host.dtype]
        else:
            raise ValueError("uv_host must be %s, int16, uint16 or float32, not %s" % (tdt, uv_host.dtype))
        if patterns_host.dtype != tdt or tuple(patterns_host.shape) != (self.n_patterns, self.n_total, 3):
            raise ValueError("patterns_host must be %s [%d, %d, 3]" % (tdt, self.n_patterns, self.n_total))
        B = int(uv_host.shape[0])
        for k, v in out.items():
            if k not in self._OUT_SHAPES:
                raise ValueError("unknown output %r" % (k,))
            width, dt_k = self._OUT_SHAPES[k]
            if not torch.is_tensor(v) or v.is_cuda or not v.is_contiguous() or v.dtype != (dt_k or tdt) or v.numel() != B * width \
                    or (B and int(v.shape[0]) != B):
                raise ValueError("out[%r] must be a contiguous CPU %s tensor of %d x %d elements" % (k, dt_k or tdt, B, width))
        if check is None and ("status" in out or "reproj" in out):
            raise ValueError("out['status'] / out['reproj'] are the outputs of check=")
        if check is not None and "status" not in out:
            raise ValueError("check= needs out['status']")
        if params is not None and params.workspace:
            raise ValueError("params.workspace is not used by the host pipeline (it owns one scratch per stream)")
        words = None
        if visible is not None:
            _check_visible(visible, B, self.n_total)
            words = visible_words_host(visible)
        if point_index is None:
            n, idx_p = self.n_total, None
        else:
            idx = np.ascontiguousarray(np.asarray(point_index, dtype=np.int32))
            n, idx_p = int(idx.shape[0]), idx.ctypes.data_as(C.POINTER(C.c_int32))
        Kh, Kp = _k_host(K)
        PI = C.POINTER(C.c_int32)
        pi = (lambda k: None if out.get(k) is None else C.cast(ptr(out[k]), PI))
        with torch.cuda.device(self.device):
            if words is not None:
                rc = lib.pnpb200_solve_batch_host_masked(
                    self._h, m, B, n, px, ptr(uv_host), ptr(patterns_host), idx_p, Kp,
                    C.byref(params) if params is not None else None,
                    ptr(out.get("R")), ptr(out.get("t")), ptr(out.get("euler")), ptr(out.get("res_norm")),
                    pi("iters"), pi("best_pattern"), words.ctypes.data_as(C.POINTER(C.c_uint32)),
                    float(check) if check is not None else 0.0, pi("status"), ptr(out.get("reproj")))
            elif check is None:
                rc = lib.pnpb200_solve_batch_host_px(
                    self._h, C.c_int(m), C.c_int64(B), C.c_int(n), C.c_int(px), ptr(uv_host), ptr(patterns_host), idx_p, Kp,
                    C.byref(params) if params is not None else None,
                    ptr(out.get("R")), ptr(out.get("t")), ptr(out.get("euler")), ptr(out.get("res_norm")),
                    ptr(out.get("iters")), ptr(out.get("best_pattern")))
            else:
                rc = lib.pnpb200_solve_check_batch_host(
                    self._h, m, B, n, px, ptr(uv_host), ptr(patterns_host), idx_p, Kp,
                    C.byref(params) if params is not None else None,
                    ptr(out.get("R")), ptr(out.get("t")), ptr(out.get("euler")), ptr(out.get("res_norm")),
                    pi("iters"), pi("best_pattern"), float(check), pi("status"), ptr(out.get("reproj")))
        _check_rc(rc, "pnpb200_solve_batch_host_masked" if words is not None else
                  ("pnpb200_solve_batch_host_px" if check is None else "pnpb200_solve_check_batch_host"))
        _lib.count_launch((B + self.chunk - 1) // self.chunk)
        return out


def host_buffer(shape, dtype, write_combined=False):
    """A page-locked CPU tensor from pnpb200_host_alloc (cudaHostAlloc); write_combined=True for pixel buffers
    the CPU only writes (faster for the device to read, very slow for the CPU to read back).  The memory is
    released when the tensor is garbage-collected."""
    dtype = torch.empty((), dtype=dtype).dtype
    esz = torch.empty((), dtype=dtype).element_size()
    n = 1
    for d in shape:
        n *= int(d)
    p = C.c_void_p()
    check(lib.pnpb200_host_alloc(C.byref(p), C.c_int64(n * esz), C.c_int(int(bool(write_combined)))), "pnpb200_host_alloc")
    buf = (C.c_char * max(n * esz, 1)).from_address(p.value)
    t = torch.frombuffer(buf, dtype=dtype, count=n).view(*shape) if n else torch.empty(shape, dtype=dtype)
    import weakref
    weakref.finalize(buf, lib.pnpb200_host_free, C.c_void_p(p.value))
    return t


def R_from_euler_batch(euler, is_degree=False):
    """euler [B,3] = (roll, yaw, pitch) CUDA tensor -> R [B,3,3]  (PNP_SOLVER_LIB.py:4442-4472)"""
    euler = euler.contiguous()
    B = int(euler.shape[0])
    R = torch.empty((B, 3, 3), dtype=euler.dtype, device=euler.device)
    with torch.cuda.device(euler.device):
        check(lib.pnpb200_R_from_euler(C.c_int(_dtype_code(euler.dtype)), C.c_int64(B), ptr(euler), C.c_int(int(is_degree)),
                                       ptr(R), _stream_ptr(euler.device)), "pnpb200_R_from_euler")
    _lib.count_launch()
    return R


def euler_from_R_batch(R, is_degree=False):
    """R [B,3,3] CUDA tensor -> euler [B,3] = (roll, yaw, pitch)  (PNP_SOLVER_LIB.py:4474-4517)"""
    R = R.contiguous()
    B = int(R.shape[0])
    e = torch.empty((B, 3), dtype=R.dtype, device=R.device)
    with torch.cuda.device(R.device):
        check(lib.pnpb200_euler_from_R(C.c_int(_dtype_code(R.dtype)), C.c_int64(B), ptr(R), C.c_int(int(is_degree)),
                                       ptr(e), _stream_ptr(R.device)), "pnpb200_euler_from_R")
    _lib.count_launch()
    return e


def project_batch(pattern, K, R, t, is_quantized=False, quantize_q=1.0):
    """pattern [n,3], R [B,3,3], t [B,3] CUDA tensors -> uvw [B,n,3]  (PNP_SOLVER_LIB.py:4532-4557)"""
    pattern, R, t = pattern.contiguous(), R.contiguous(), t.contiguous()
    B, n = int(R.shape[0]), int(pattern.shape[0])
    out = torch.empty((B, n, 3), dtype=R.dtype, device=R.device)
    Kh, Kp = _k_host(K)
    with torch.cuda.device(R.device):
        check(lib.pnpb200_project(C.c_int(_dtype_code(R.dtype)), C.c_int64(B), C.c_int(n), ptr(pattern), Kp, ptr(R), ptr(t),
                                  C.c_int(int(is_quantized)), C.c_double(float(quantize_q)), ptr(out),
                                  _stream_ptr(R.device)), "pnpb200_project")
    _lib.count_launch()
    return out


class PNP_SOLVER(object):
    """Same public surface as the reference's PNP_SOLVER (PNP_SOLVER_LIB.py:7).

    Extra keyword arguments (all optional, defaults reproduce the reference):
      device  CUDA device (default: current);  dtype  'f64' (parity) or 'f32';
      method  which single-pattern solver solve_pnp()/solve_pnp_batch() dispatch to
              ('qeif' as in PNP_SOLVER_LIB.py:179, or 'lm', 'linear_f2', 'linear_f1').
    """

    def __init__(self, np_K_camera_est, point_3d_dict_list, pattern_scale_list=None, verbose=False,
                 device=None, dtype="f64", method="qeif"):
        self.verbose = True
        self.np_K_camera_est = copy.deepcopy(np_K_camera_est)
        self.pattern_scale_list = pattern_scale_list
        self.point_3d_dict_list = copy.deepcopy(point_3d_dict_list)
        if self.pattern_scale_list is None:
            self.pattern_scale_list = [1.0 for _ in range(len(self.point_3d_dict_list))]
        elif len(self.pattern_scale_list) < len(self.point_3d_dict_list):
            self.pattern_scale_list += [1.0 for _ in range(len(self.point_3d_dict_list) - len(self.pattern_scale_list))]
        # the reference's pre-transform path is disabled (PNP_SOLVER_LIB.py:27); kept as attributes
        self.is_using_pre_transform = False
        self.pre_trans_R_a_h = np.eye(3)
        self.pre_trans_t_a_h = np.array([[0.0, 0.0, -0.5]]).T
        self.np_R_c_a_est = np.eye(3)
        self.np_t_c_a_est = np.zeros((3, 1))
        self.np_point_3d_dict_list = list()
        self.np_point_3d_pretransfer_dict_list = list()
        self.verbose = verbose   # (the reference prints the pattern table here; we do not)
        for _i in range(len(self.point_3d_dict_list)):
            a, b = self.get_np_point_3d_dict(self.point_3d_dict_list[_i], self.pattern_scale_list[_i])
            self.np_point_3d_dict_list.append(a)
            self.np_point_3d_pretransfer_dict_list.append(b)
        self.set_golden_pattern_id(0)
        # B200 additions
        self.device = str(torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)) \
            if torch.cuda.is_available() else "cuda:0"
        self.dtype_code = _dtype_code(dtype)
        self.method = method
        self.params = None          # optional _lib.Params override
        self.LM_key_list = list(LM_KEY_LIST_6)   # PNP_SOLVER_LIB.py:156
        self.last_iters = None
        self._last_best = 0
        self._dev_cache = {}

    # ---------------------------------------------------------------- pattern store (:66-135)
    def set_golden_pattern_id(self, id):
        self.current_golden_pattern_id = id

    def get_current_golden_pattern(self):
        return self.np_point_3d_dict_list[self.current_golden_pattern_id]

    def get_current_pretransfered_golden_pattern(self):
        return self.np_point_3d_pretransfer_dict_list[self.current_golden_pattern_id]

    def get_np_point_3d_dict(self, point_3d_dict, pattern_scale, is_using_pre_transform=False, pre_trans_R_a_h=None, pre_trans_t_a_h=None):
        d = dict()
        for _k in point_3d_dict:
            d[_k] = np.array(point_3d_dict[_k], dtype=np.float64).reshape((3, 1))
            d[_k] *= pattern_scale
        return (d, copy.deepcopy(d))

    def update_the_selected_golden_pattern(self, id, point_3d_dict, pattern_scale):
        self.pattern_scale_list[id] = pattern_scale
        self.point_3d_dict_list[id] = copy.deepcopy(point_3d_dict)
        a, b = self.get_np_point_3d_dict(self.point_3d_dict_list[id], self.pattern_scale_list[id])
        self.np_point_3d_dict_list[id] = a
        self.np_point_3d_pretransfer_dict_list[id] = b
        self._dev_cache = {}
        return True

    def lib_print(self, str=''):
        if self.verbose:
            print(str)

    def __deepcopy__(self, memo):
        new = self.__class__.__new__(self.__class__)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            new.__dict__[k] = {} if k == "_dev_cache" else copy.deepcopy(v, memo)
        return new

    # ---------------------------------------------------------------- helpers
    def _tdtype(self):
        return _TORCH_DTYPE[self.dtype_code]

    def _pack_patterns(self, dict_list, keys):
        """[P, n, 3] device tensor of the patterns restricted to `keys`, in `keys` order (f2_get_P :3260)."""
        arr = np.stack([np.stack([np.asarray(d[k], dtype=np.float64).reshape(3) for k in keys]) for d in dict_list])
        return torch.from_numpy(arr).to(device=self.device, dtype=self._tdtype())

    def _pack_image_points(self, np_point_image_dict, keys):
        """(uv [1, n, 2] device tensor, K to solve with) -- f2_get_B_xy's input (:3291).  Points are (3,1) homogeneous
        vectors; when a third entry is not 1 (the reference's own projection emits -1 behind the camera, :4548) the
        product K^-1 [u, v, w]^T that the reference forms (:3307) is taken on the device and the solve runs on the
        normalised coordinates with K = I.  Never raises on the numeric path, like the reference."""
        pts = np.zeros((1, len(keys), 3))
        for i, k in enumerate(keys):
            v = np.asarray(np_point_image_dict[k], dtype=np.float64).reshape(-1)
            pts[0, i, 0], pts[0, i, 1] = v[0], v[1]
            pts[0, i, 2] = v[2] if v.shape[0] >= 3 else 1.0
        if (pts[..., 2] == 1.0).all():                           # the ordinary case, decided on the host: no extra device round trip
            return torch.from_numpy(np.ascontiguousarray(pts[..., :2])).to(device=self.device, dtype=self._tdtype()), self.np_K_camera_est
        return self._uv_and_K(torch.from_numpy(pts).to(device=self.device, dtype=self._tdtype()))

    def _uv_and_K(self, pts):
        """pts [B, n, 2] or [B, n, 3] device tensor -> (uv [B, n, 2], K): see _pack_image_points"""
        if pts.shape[-1] == 2:
            return pts.contiguous(), self.np_K_camera_est
        if bool((pts[..., 2] == 1).all()):
            return pts[..., :2].contiguous(), self.np_K_camera_est
        pts = pts.contiguous()
        out = torch.empty(pts.shape[:-1] + (2,), dtype=pts.dtype, device=pts.device)
        Kh, Kp = _k_host(self.np_K_camera_est)
        with torch.cuda.device(pts.device):
            check(lib.pnpb200_normalise_uvw(C.c_int(_dtype_code(pts.dtype)), C.c_int64(int(pts.numel() // 3)), ptr(pts), Kp, ptr(out),
                                            _stream_ptr(pts.device)), "pnpb200_normalise_uvw")
        _lib.count_launch()
        return out, np.eye(3)

    def _finish_single(self, out):
        """device outputs of a B=1 solve -> the reference's 7-tuple, plus its side effects.  One device-to-host
        copy for everything (the scripts call this once per sample)."""
        flat = torch.cat([out["R"].reshape(-1).double(), out["t"].reshape(-1).double(), out["euler"].reshape(-1).double(),
                          out["res_norm"].reshape(-1).double(), out["iters"].double(), out["best_pattern"].double()]).cpu().numpy()
        R = flat[0:9].reshape(3, 3).copy()
        t = flat[9:12].reshape(3, 1).copy()
        e = flat[12:15]
        res = float(flat[15])
        self.last_iters = int(flat[16])
        self._last_best = int(flat[17])
        self.np_R_c_a_est = copy.deepcopy(R)          # :2986-2987
        self.np_t_c_a_est = copy.deepcopy(t)
        return (R, t, float(t[2, 0]), float(e[0]), float(e[1]), float(e[2]), res)

    def _solve_single(self, method, np_point_image_dict, np_point_3d_pretransfer_dict, keys):
        uv, K = self._pack_image_points(np_point_image_dict, keys)
        pat = self._pack_patterns([np_point_3d_pretransfer_dict], keys)
        out = solve_batch(method, uv, pat, K, params=self.params)
        return self._finish_single(out)

    # ---------------------------------------------------------------- solvers
    def solve_pnp(self, np_point_image_dict):
        """PNP_SOLVER_LIB.py:144-203: the 6-landmark subset, every stored pattern, arg-min res_norm."""
        keys = list(self.LM_key_list) if self.LM_key_list is not None else list(self.np_point_3d_pretransfer_dict_list[0].keys())
        if self.method != "qeif":   # only the QEIF solver honours LM_key_list (:2576 vs :2784)
            keys = list(np_point_image_dict.keys())
        uv, K = self._pack_image_points(np_point_image_dict, keys)
        pat = self._pack_patterns(self.np_point_3d_pretransfer_dict_list, keys)
        out = solve_batch(self.method, uv, pat, K, params=self.params)
        ret = self._finish_single(out)
        self.set_golden_pattern_id(self._last_best)                        # :199
        return ret

    def solve_pnp_QEIF_single_pattern(self, np_point_image_dict, np_point_3d_pretransfer_dict, LM_key_list=None):
        """PNP_SOLVER_LIB.py:2771-3025"""
        keys = list(np_point_3d_pretransfer_dict.keys()) if LM_key_list is None else list(LM_key_list)
        return self._solve_single("qeif", np_point_image_dict, np_point_3d_pretransfer_dict, keys)

    def solve_pnp_LM_single_pattern(self, np_point_image_dict, np_point_3d_pretransfer_dict, LM_key_list=None):
        """PNP_SOLVER_LIB.py:2567-2769 (LM_key_list is ignored there too: all points, :2576, :2597)"""
        return self._solve_single("lm", np_point_image_dict, np_point_3d_pretransfer_dict, list(np_point_3d_pretransfer_dict.keys()))

    def solve_pnp_EIF2_single_pattern(self, np_point_image_dict, np_point_3d_pretransfer_dict, LM_key_list=None):
        """PNP_SOLVER_LIB.py:2001-2276 (all points, like LM: f2_get_P / f2_get_B_xy without a key list, :2012, :2045)"""
        return self._solve_single("eif2", np_point_image_dict, np_point_3d_pretransfer_dict, list(np_point_3d_pretransfer_dict.keys()))

    def solve_pnp_formulation_2_single_pattern(self, np_point_image_dict, np_point_3d_pretransfer_dict, LM_key_list=None):
        """PNP_SOLVER_LIB.py:693-953"""
        return self._solve_single("linear_f2", np_point_image_dict, np_point_3d_pretransfer_dict, list(np_point_3d_pretransfer_dict.keys()))

    def solve_pnp_single_pattern(self, np_point_image_dict, np_point_3d_pretransfer_dict, LM_key_list=None):
        """PNP_SOLVER_LIB.py:205-430 (rows follow the image dict's key order, :3069)"""
        return self._solve_single("linear_f1", np_point_image_dict, np_point_3d_pretransfer_dict, list(np_point_image_dict.keys()))

    def solve_pnp_batch(self, uv, method=None, key_list="default", params=None, check=None, visible=None, robust=None):
        """The per-problem script loop as one launch.

        uv: [B, n_total, 2] pixels (or [B, n_total, 3] homogeneous image points, third entry as the reference's
        dicts carry it) in the key order of the stored patterns -- a CUDA tensor, or a NumPy array / CPU tensor
        (copied to the device).  key_list: landmark subset; "default" =
        the 6 keys of solve_pnp() for 'qeif', all points otherwise.  Returns a dict of CUDA
        tensors (see solve_batch) and, like solve_pnp, works over every stored pattern.
        check: a limit in px -> the dict also holds status [B] int32 and reproj [B,2] of check_batch on the
        returned poses, over all n_total landmarks and each problem's winning pattern (0: no REPROJ bit).
        visible: bool [B, n_total] (a detector's per-frame visibility, e.g. isfinite(uv).all(-1)) -> each problem is solved
        and checked on its visible landmarks alone (of key_list, in its order); hidden pixels may hold anything, NaN too.
        robust: None, or a dict of any of max_rounds, k, floor_px, min_inliers -> solve_robust_batch: misplaced landmarks are
        rejected by their reprojection distance and each problem re-solved on its inliers; the dict then also holds inliers,
        rounds and robust_status, and the check (if asked for) runs on the inliers.  With samples (and any of consensus_px,
        confidence, seed, idx0) the loop starts from the hypothesis stage's consensus set (RANSAC), and the dict also holds
        consensus and drawn."""
        method = method or self.method
        if robust is not None:
            hyp_keys = {"samples", "consensus_px", "confidence", "seed", "idx0"}
            unknown = set(robust) - {"max_rounds", "k", "floor_px", "min_inliers"} - hyp_keys
            if unknown:
                raise ValueError("robust takes max_rounds, k, floor_px, min_inliers, samples, consensus_px, confidence, seed, idx0; "
                                 "not %s" % sorted(unknown))
            robust_params(**{k: v for k, v in robust.items() if k not in hyp_keys})
            if robust.get("samples") is not None:
                hypothesis_params(**{k: v for k, v in robust.items() if k in hyp_keys})
        all_keys = list(self.np_point_3d_pretransfer_dict_list[0].keys())
        if isinstance(key_list, str) and key_list == "default":
            key_list = self.LM_key_list if method == "qeif" else None
        idx = None if key_list is None else [all_keys.index(k) for k in key_list]
        if not torch.is_tensor(uv):
            uv = torch.from_numpy(np.ascontiguousarray(uv))
        if visible is not None:
            _check_visible(visible, int(uv.shape[0]), len(all_keys))
        uv, K = self._uv_and_K(uv.to(device=self.device, dtype=self._tdtype()))
        ck = ("all", self.dtype_code)
        if ck not in self._dev_cache:
            self._dev_cache[ck] = self._pack_patterns(self.np_point_3d_pretransfer_dict_list, all_keys)
        prm = params if params is not None else self.params
        if robust is None:
            out = solve_batch(method, uv, self._dev_cache[ck], K, point_index=idx, params=prm, visible=visible)
        else:
            out = solve_robust_batch(method, uv, self._dev_cache[ck], K, point_index=idx, params=prm, visible=visible, **robust)
            visible = out["inliers"]
        if check is not None:
            out.update(check_batch(uv, self._dev_cache[ck], K, out["R"], out["t"], res_norm=out["res_norm"],
                                   best_pattern=out["best_pattern"], reproj_limit_px=check, visible=visible))
        return out

    def solve_pnp_batch_host(self, uv, method=None, key_list="default", params=None, chunk_problems=1 << 16, pack_threads=None,
                             check=None, visible=None):
        """solve_pnp_batch for data that lives on the HOST (what a script that loops over NumPy samples
        has): uv [B, n_total, 2] NumPy array or CPU tensor in; dict of NumPy arrays R [B,3,3], t [B,3],
        euler [B,3] (roll, yaw, pitch, deg.), res_norm [B], iters [B], best_pattern [B] out.  uv may be int16,
        uint16 or float32 (a detector's own output type): it then crosses PCIe as it is.  Runs the
        chunked host pipeline (pnpb200_solve_batch_host: H2D, solve and D2H overlap on three streams);
        pack_threads host threads (default: half the visible cores, at most 8) let chunks of whole-pixel
        landmarks cross PCIe as int16 (lossless, checked per chunk; other chunks travel as they are).
        check: a limit in px -> each chunk's solve is followed by the solution check on the device, and the dict also
        holds status [B] int32 and reproj [B,2] (see solve_pnp_batch); every other output is unchanged.
        visible: bool [B, n_total] -> the masked pipeline (see solve_pnp_batch); a chunk whose hidden pixels are NaN travels
        unpacked."""
        method = method or self.method
        all_keys = list(self.np_point_3d_pretransfer_dict_list[0].keys())
        if isinstance(key_list, str) and key_list == "default":
            key_list = self.LM_key_list if method == "qeif" else None
        idx = None if key_list is None else [all_keys.index(k) for k in key_list]
        tdt = self._tdtype()
        if not torch.is_tensor(uv):
            uv = np.ascontiguousarray(uv)
            uv = torch.from_numpy(uv.view(np.int16)).view(torch.uint16) if uv.dtype == np.uint16 else torch.from_numpy(uv)
        # int16 / uint16 / float32 detections stay what they are (no FP64 round trip): the pipeline widens them on the device
        narrow = uv.dtype in (torch.int16, torch.uint16) or (uv.dtype == torch.float32 and tdt == torch.float64)
        uv_h = uv.to(device="cpu").contiguous() if narrow else uv.to(device="cpu", dtype=tdt).contiguous()
        B, n_total = int(uv_h.shape[0]), int(uv_h.shape[1])
        if n_total != len(all_keys):
            raise ValueError("uv holds %d landmarks per problem, the stored patterns %d" % (n_total, len(all_keys)))
        if visible is not None:
            _check_visible(visible, B, n_total)
        pats = np.stack([np.stack([np.asarray(d[k], dtype=np.float64).reshape(3) for k in all_keys])
                         for d in self.np_point_3d_pretransfer_dict_list])
        pat_h = torch.from_numpy(pats).to(dtype=tdt).contiguous()
        if pack_threads is None:
            cpus = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
            pack_threads = min(8, cpus // 2)
        chunk = int(max(1, min(chunk_problems, 1 << max(0, (B - 1).bit_length()))))    # small batches: next power of two
        key = ("pipe", self.dtype_code, n_total, int(pat_h.shape[0]), chunk)
        pipe = self._dev_cache.get(key)
        if pipe is None:
            pipe = HostPipeline(tdt, chunk_problems=chunk, n_total=n_total, n_patterns=int(pat_h.shape[0]), n_streams=3,
                                device=self.device)
            self._dev_cache[key] = pipe
        pipe.set_packing(int(pack_threads) if (B >= 2 * chunk and not narrow) else 0)
        # results land in page-locked buffers (kept per batch size), so the D2H copies of a chunk are asynchronous and
        # overlap the next chunks' H2D and solve; the arrays handed back are copies the caller owns
        okey = ("host_out", self.dtype_code, B)
        outs = self._dev_cache.get(okey)
        if outs is None:
            for k_old in [k for k in self._dev_cache if k[0] == "host_out"]:
                del self._dev_cache[k_old]
            pin = (lambda t_: t_.pin_memory()) if B > 0 else (lambda t_: t_)
            outs = {"R": pin(torch.empty((B, 3, 3), dtype=tdt)), "t": pin(torch.empty((B, 3), dtype=tdt)),
                    "euler": pin(torch.empty((B, 3), dtype=tdt)), "res_norm": pin(torch.empty((B,), dtype=tdt)),
                    "iters": pin(torch.empty((B,), dtype=torch.int32)), "best_pattern": pin(torch.empty((B,), dtype=torch.int32))}
            self._dev_cache[okey] = outs
        sel = {k: v for k, v in outs.items() if k not in ("status", "reproj")}
        if check is not None:
            if "status" not in outs:
                pin = (lambda t_: t_.pin_memory()) if B > 0 else (lambda t_: t_)
                outs["status"], outs["reproj"] = pin(torch.empty((B,), dtype=torch.int32)), pin(torch.empty((B, 2), dtype=tdt))
            sel["status"], sel["reproj"] = outs["status"], outs["reproj"]
        if B > 0:
            pipe.solve(method, uv_h, pat_h, self.np_K_camera_est, sel, point_index=idx,
                       params=params if params is not None else self.params, check=check, visible=visible)
        return {k: v.numpy().copy() for k, v in sel.items()}

    # ---------------------------------------------------------------- Euler <-> R (:4442-4517)
    def get_rotation_matrix_from_Euler(self, roll, yaw, pitch, is_degree=False):
        e = torch.tensor([[roll, yaw, pitch]], dtype=torch.float64, device=self.device)
        return R_from_euler_batch(e, is_degree)[0].cpu().numpy()

    def get_Euler_from_rotation_matrix(self, R_in, verbose=True, is_degree=False):
        R = torch.from_numpy(np.ascontiguousarray(np.asarray(R_in, dtype=np.float64).reshape(1, 3, 3))).to(self.device)
        e = euler_from_R_batch(R, is_degree)[0].cpu().numpy()
        return (float(e[0]), float(e[1]), float(e[2]))   # (roll, yaw, pitch)

    # ---------------------------------------------------------------- projection (:4520-4621)
    def transform_3D_point(self, point_3D, R_in, t_in):
        return (R_in @ point_3D + t_in)

    def _project(self, pts_n3, np_K_camera, np_R, np_t, is_quantized, quantize_q):
        pat = torch.from_numpy(np.ascontiguousarray(np.asarray(pts_n3, dtype=np.float64).reshape(-1, 3))).to(self.device)
        R = torch.from_numpy(np.ascontiguousarray(np.asarray(np_R, dtype=np.float64).reshape(1, 3, 3))).to(self.device)
        t = torch.from_numpy(np.ascontiguousarray(np.asarray(np_t, dtype=np.float64).reshape(1, 3))).to(self.device)
        q = project_batch(pat, np_K_camera, R, t, is_quantized, quantize_q)[0].cpu().numpy()
        nq = q if not is_quantized else project_batch(pat, np_K_camera, R, t, False, 1.0)[0].cpu().numpy()
        return q, nq

    def perspective_projection(self, np_point_3d, np_K_camera, np_R, np_t, is_quantized=False, quantize_q=1.0, is_returning_homogeneous_vec=True):
        q, nq = self._project(np.asarray(np_point_3d, dtype=np.float64).reshape(1, 3), np_K_camera, np_R, np_t, is_quantized, quantize_q)
        if is_returning_homogeneous_vec:
            return (q[0].reshape(3, 1), nq[0].reshape(3, 1))
        return (q[0, 0:2].copy(), nq[0, 0:2].copy())

    def perspective_projection_obj_axis(self, np_R, np_t, scale=1.0):
        pts = np.array([[0.0, 0.0, 0.0], [scale, 0.0, 0.0], [0.0, scale, 0.0], [0.0, 0.0, scale]])
        q, _ = self._project(pts, self.np_K_camera_est, np_R, np_t, False, 1.0)
        uv_o = q[0, 0:2].copy()
        return (uv_o, q[1, 0:2] - uv_o, q[2, 0:2] - uv_o, q[3, 0:2] - uv_o)

    def perspective_projection_golden_landmarks(self, np_R, np_t, is_quantized=False, quantize_q=1.0, is_pretrans_points=False, is_returning_homogeneous_vec=True):
        src = self.get_current_pretransfered_golden_pattern() if is_pretrans_points else self.get_current_golden_pattern()
        keys = list(src.keys())
        pts = np.stack([np.asarray(src[k]).reshape(3) for k in keys])
        q, _ = self._project(pts, self.np_K_camera_est, np_R, np_t, is_quantized, quantize_q)
        out = dict()
        for i, k in enumerate(keys):
            out[k] = q[i].reshape(3, 1) if is_returning_homogeneous_vec else q[i, 0:2].copy()
        return out

    # ---------------------------------------------------------------- misc (:4666-4675)
    def unit_vec(self, vec_in):
        _norm = np.linalg.norm(vec_in)
        _eps = 10**-7
        _norm_inv = (1 / _eps) if np.abs(_norm) <= 10**-7 else (1.0 / _norm)
        return (vec_in * _norm_inv)
