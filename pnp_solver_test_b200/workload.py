"""Batched workload, error reporting and error statistics around the solve (SURVEY.md 8a rows
a14-a16, 8e): device-side synthetic inputs, per-problem error report, and the statistics of
TEST_TOOLBOX.get_statistic_of_result as two reducible passes so that problem shards on
different GPUs combine with two tiny all-reduces (NCCL over NVLink; gloo in CPU tests).

The solve path itself has no inter-GPU traffic: problems are sharded by global index.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import lib, check, ptr
from .solver import _check_visible, _copy_params, _dtype_code, _k_host, _stream_ptr, _u32, visible_words

# TEST_TOOLBOX.get_classification_parameters("drpy_expand") (TEST_TOOLBOX.py:133-162)
CLASS_BINS = {
    "depth": [30.0 + 20.0 * i for i in range(11)],     # cm; labels 20, 40, ..., 240
    "roll": [-35.0, -15.0, 15.0, 35.0],
    "pitch": [-23.0, -8.0, 8.0, 23.0],
    "yaw": [-30.0, -10.0, 10.0, 30.0],
}
CLASS_LABELS = {
    "depth": [str(20 * (i + 1)) for i in range(12)],
    "roll": ["-45", "-25", "0", "25", "45"],
    "pitch": ["-30", "-15", "0", "15", "30"],
    "yaw": ["-40", "-20", "0", "20", "40"],
}
STAT_KEYS = ("n_data", "m_ratio", "mean", "stddev", "max_dev", "MAE_2_GT", "MAE_2_mean")


def shard_range(total, rank, world_size):
    """Contiguous range of the global problem index owned by `rank` (SURVEY.md 8e)."""
    base, rem = divmod(int(total), int(world_size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def synth_batch(b0, B, pattern, K, cfg=None, dtype=torch.float64, device=None, want_pose=False):
    """Problems b0..b0+B-1 of the global counter-based stream (pnpb200_synth_batch).

    pattern: [n,3] array-like in metres.  Returns dict(uv [B,n,2] dtype, gt [B,4] f64 =
    (distance m, roll, pitch, yaw deg)[, R_gt [B,3,3], t_gt [B,3]])."""
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    pat = torch.as_tensor(np.ascontiguousarray(np.asarray(pattern, dtype=np.float64)), device=device)
    n = int(pat.shape[0])
    uv = torch.empty((B, n, 2), dtype=dtype, device=device)
    gt = torch.empty((B, 4), dtype=torch.float64, device=device)
    Rg = torch.empty((B, 3, 3), dtype=torch.float64, device=device) if want_pose else None
    tg = torch.empty((B, 3), dtype=torch.float64, device=device) if want_pose else None
    Kh, Kp = _k_host(K)
    with torch.cuda.device(device):
        check(lib.pnpb200_synth_batch(C.c_int(_dtype_code(dtype)), C.c_int64(int(b0)), C.c_int64(int(B)), C.c_int(n),
                                      ptr(pat), Kp, C.byref(cfg) if cfg is not None else None, ptr(uv),
                                      C.cast(ptr(gt), C.POINTER(C.c_double)),
                                      C.cast(ptr(Rg), C.POINTER(C.c_double)) if want_pose else None,
                                      C.cast(ptr(tg), C.POINTER(C.c_double)) if want_pose else None,
                                      _stream_ptr(device)), "pnpb200_synth_batch")
    _lib.count_launch()
    out = dict(uv=uv, gt=gt)
    if want_pose:
        out["R_gt"], out["t_gt"] = Rg, tg
    return out


def report_batch(pattern, uv, K, R, t, euler, gt, bounds=(10.0, 10.0, 10.0, 10.0), layout="columns", visible=None):
    """Per-problem error report (pnpb200_report_batch_strided): dict(report [B,16] f64, flags [B,4]
    int32, max_idx [B,3] int32).  Column meaning: include/pnpb200.h.  pattern [n,3], uv [B,n,2]: every
    landmark of the pattern, as in compare_result_and_generate_result_dict (TEST_TOOLBOX.py:291).
    layout="columns" (default): report is the transposed view of a [16,B] array, so report[:, k] is
    contiguous (what the statistics read); layout="rows": a contiguous [B,16] array.
    visible: bool [B, n] -> pnpb200_report_batch_strided_masked: columns 4-9 and max_idx over the visible landmarks."""
    dev = uv.device
    pattern = torch.as_tensor(pattern, device=dev).to(uv.dtype).contiguous()
    B, n = int(uv.shape[0]), int(uv.shape[1])
    if visible is not None:
        _check_visible(visible, B, n)
    if layout == "columns":
        rep = torch.empty((_lib.REPORT_WIDTH, B), dtype=torch.float64, device=dev).t()
    else:
        assert layout == "rows"
        rep = torch.empty((B, _lib.REPORT_WIDTH), dtype=torch.float64, device=dev)
    rs_b, rs_k = max(int(rep.stride(0)), 1), max(int(rep.stride(1)), 1)
    flags = torch.empty((B, 4), dtype=torch.int32, device=dev)
    midx = torch.empty((B, 3), dtype=torch.int32, device=dev)
    Kh, Kp = _k_host(K)
    bd = (C.c_double * 4)(*[float(b) for b in bounds])
    gt = gt.to(torch.float64).contiguous()
    if visible is not None:
        if B == 0:
            return dict(report=rep, flags=flags, max_idx=midx)
        PD, PI = C.POINTER(C.c_double), C.POINTER(C.c_int32)
        words = visible_words(visible, dev)
        with torch.cuda.device(dev):
            check(lib.pnpb200_report_batch_strided_masked(_dtype_code(uv.dtype), B, n, ptr(pattern), ptr(uv.contiguous()), Kp,
                                                          ptr(R.contiguous()), ptr(t.contiguous()), ptr(euler.contiguous()),
                                                          C.cast(ptr(gt), PD), bd, C.cast(ptr(rep), PD), rs_b, rs_k,
                                                          C.cast(ptr(flags), PI), C.cast(ptr(midx), PI), _u32(words),
                                                          _stream_ptr(dev)), "pnpb200_report_batch_strided_masked")
        _lib.count_launch()
        return dict(report=rep, flags=flags, max_idx=midx)
    with torch.cuda.device(dev):
        check(lib.pnpb200_report_batch_strided(C.c_int(_dtype_code(uv.dtype)), C.c_int64(B), C.c_int(n), ptr(pattern),
                                               ptr(uv.contiguous()), Kp, ptr(R.contiguous()), ptr(t.contiguous()),
                                               ptr(euler.contiguous()), C.cast(ptr(gt), C.POINTER(C.c_double)), bd,
                                               C.cast(ptr(rep), C.POINTER(C.c_double)), C.c_int64(rs_b), C.c_int64(rs_k),
                                               C.cast(ptr(flags), C.POINTER(C.c_int32)), C.cast(ptr(midx), C.POINTER(C.c_int32)),
                                               _stream_ptr(dev)), "pnpb200_report_batch_strided")
    _lib.count_launch()
    return dict(report=rep, flags=flags, max_idx=midx)


def solve_report_batch(method, uv, pattern, K, gt, params=None, bounds=(10.0, 10.0, 10.0, 10.0), point_index=None, visible=None):
    """pnpb200_solve_report_batch: solve_batch (one pattern) and report_batch (column layout) of the same problems in
    one call -- the body of the loop of random_stress_test.py:322-377.  With LM / linear F2 over all landmarks the
    residual pass of the solve rides in the report kernel (the pixel rows are read twice instead of three times);
    the results are those of the two separate calls.  uv [B,n,2], pattern [n,3] (or [1,n,3]) CUDA tensors of one
    dtype, gt [B,4] FP64.  Returns the union of both dicts.
    visible: bool [B, n] -> pnpb200_solve_report_batch_masked: the masked solve, then the masked report."""
    m = _lib.METHODS[method] if isinstance(method, str) else int(method)
    dev = uv.device
    uv = uv.contiguous()
    pattern = torch.as_tensor(pattern, device=dev).to(uv.dtype).reshape(-1, 3).contiguous()
    B, n_total = int(uv.shape[0]), int(uv.shape[1])
    if uv.dim() != 3 or uv.shape[2] != 2 or pattern.shape[0] != n_total:
        raise ValueError("shape mismatch: uv [B,n,2], pattern [n,3]")
    if visible is not None:
        _check_visible(visible, B, n_total)
    dt = _dtype_code(uv.dtype)
    if point_index is None:
        n, idx_p = n_total, None
    else:
        idx = np.ascontiguousarray(np.asarray(point_index, dtype=np.int32))
        n, idx_p = int(idx.shape[0]), idx.ctypes.data_as(C.POINTER(C.c_int32))
    o = dict(R=torch.empty((B, 3, 3), dtype=uv.dtype, device=dev), t=torch.empty((B, 3), dtype=uv.dtype, device=dev),
             euler=torch.empty((B, 3), dtype=uv.dtype, device=dev), res_norm=torch.empty((B,), dtype=uv.dtype, device=dev),
             iters=torch.empty((B,), dtype=torch.int32, device=dev),
             report=torch.empty((_lib.REPORT_WIDTH, B), dtype=torch.float64, device=dev).t(),
             flags=torch.empty((B, 4), dtype=torch.int32, device=dev), max_idx=torch.empty((B, 3), dtype=torch.int32, device=dev))
    if B == 0:
        return o
    prm = _lib.default_params() if params is None else params
    ws_query = lib.pnpb200_workspace_bytes if visible is None else lib.pnpb200_workspace_bytes_masked
    ws_bytes = int(ws_query(C.c_int(m), C.c_int(dt), C.c_int64(B), C.c_int(1), C.c_int(int(prm.mapping))))
    ws = None
    if ws_bytes > 0 and not prm.workspace:                 # scratch from torch's caching allocator (stream-ordered, no driver call)
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
        prm = _copy_params(prm)
        prm.workspace, prm.workspace_bytes = ws.data_ptr(), ws_bytes
    Kh, Kp = _k_host(K)
    bd = (C.c_double * 4)(*[float(b) for b in bounds])
    gt = gt.to(torch.float64).contiguous()
    PD, PI = C.POINTER(C.c_double), C.POINTER(C.c_int32)
    rep = o["report"]
    if visible is not None:
        words = visible_words(visible, dev)
        with torch.cuda.device(dev):
            check(lib.pnpb200_solve_report_batch_masked(m, dt, B, n_total, n, ptr(uv), ptr(pattern), idx_p, Kp, C.byref(prm), ptr(o["R"]),
                                                        ptr(o["t"]), ptr(o["euler"]), ptr(o["res_norm"]), C.cast(ptr(o["iters"]), PI),
                                                        C.cast(ptr(gt), PD), bd, C.cast(ptr(rep), PD), max(int(rep.stride(0)), 1),
                                                        max(int(rep.stride(1)), 1), C.cast(ptr(o["flags"]), PI),
                                                        C.cast(ptr(o["max_idx"]), PI), _u32(words), _stream_ptr(dev)),
                  "pnpb200_solve_report_batch_masked")
        _lib.count_launch(2)
        return o
    with torch.cuda.device(dev):
        check(lib.pnpb200_solve_report_batch(C.c_int(m), C.c_int(dt), C.c_int64(B), C.c_int(n_total), C.c_int(n), ptr(uv), ptr(pattern),
                                             idx_p, Kp, C.byref(prm), ptr(o["R"]), ptr(o["t"]), ptr(o["euler"]), ptr(o["res_norm"]),
                                             C.cast(ptr(o["iters"]), PI), C.cast(ptr(gt), PD), bd, C.cast(ptr(rep), PD),
                                             C.c_int64(max(int(rep.stride(0)), 1)), C.c_int64(max(int(rep.stride(1)), 1)),
                                             C.cast(ptr(o["flags"]), PI), C.cast(ptr(o["max_idx"]), PI), _stream_ptr(dev)),
              "pnpb200_solve_report_batch")
    _lib.count_launch(2)
    return o


def classify(values, bins, scale=1.0):
    """np.digitize(values*scale, bins) on the device (TEST_TOOLBOX.classify_drpy, :239-247).
    values: 1-D (possibly strided) FP64 CUDA tensor view."""
    assert values.dtype == torch.float64 and values.dim() == 1
    B = int(values.shape[0])
    cls = torch.empty((B,), dtype=torch.int32, device=values.device)
    bn = (C.c_double * len(bins))(*[float(b) for b in bins])
    with torch.cuda.device(values.device):
        check(lib.pnpb200_classify(C.c_int64(B), C.cast(ptr(values), C.POINTER(C.c_double)), C.c_int64(values.stride(0) if B else 1),
                                   C.c_double(scale), bn, C.c_int(len(bins)), C.cast(ptr(cls), C.POINTER(C.c_int32)),
                                   _stream_ptr(values.device)), "pnpb200_classify")
    _lib.count_launch()
    return cls


def _all_reduce(t, op, group):
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=op, group=group)


def reduce_phase1(s1, group=None):
    """Phase 1: all_reduce(SUM) of the pass-1 sums [..., 4] = (n, sum est/gt, sum e, 0), in place.
    Works on any backend (NCCL on GPUs, gloo in CPU tests)."""
    import torch.distributed as dist
    _all_reduce(s1, dist.ReduceOp.SUM, group)
    return s1


def reduce_phase2(s2, mx, group=None, flat23=None):
    """Phase 2: SUM over ranks of [..., 4] = (sum (e-m)^2, sum |e|, sum |e-m|, 0) and MAX over ranks of max |e-m|,
    in place.  With `flat23` (the contiguous buffer that holds s2 followed by mx, as `statistics` allocates them) the
    two reductions are ONE exchange: an all_gather of the ranks' partials (a few KB) and a local fold -- one collective
    launch instead of two, and the SUM is then taken in rank order on every rank (bit-identical everywhere)."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1):
        return s2, mx
    if flat23 is None:
        _all_reduce(s2, dist.ReduceOp.SUM, group)
        _all_reduce(mx, dist.ReduceOp.MAX, group)
        return s2, mx
    world = dist.get_world_size(group)
    gathered = torch.empty((world * flat23.numel(),), dtype=flat23.dtype, device=flat23.device)
    dist.all_gather_into_tensor(gathered, flat23.reshape(-1), group=group)
    gathered = gathered.view(world, flat23.numel())
    n2 = s2.numel()
    s2.copy_(gathered[:, :n2].sum(dim=0).view_as(s2))
    mx.copy_(gathered[:, n2:].max(dim=0).values.view_as(mx))
    return s2, mx


def finalize_stats(s1, s2, mx):
    """(n, m_ratio, mean, stddev [population], max_dev, MAE_2_GT, MAE_2_mean) per row
    (TEST_TOOLBOX.py:907-915, :928-935), on the host from the three small reduced arrays."""
    s1, s2, mx = (np.asarray(a.detach().cpu().numpy() if torch.is_tensor(a) else a, dtype=np.float64) for a in (s1, s2, mx))
    with np.errstate(divide="ignore", invalid="ignore"):
        n = s1[..., 0]
        out = np.stack([n, s1[..., 1] / n, s1[..., 2] / n, np.sqrt(s2[..., 0] / n), mx, s2[..., 1] / n, s2[..., 2] / n], axis=-1)
    return torch.from_numpy(out)


class PendingStats(object):
    """Statistics whose reduced sums are still on their way to the host (asynchronous D2H into a
    pinned buffer); `.result()` waits for the copy and finalises.  Lets a caller queue many batches
    without a host synchronisation per batch."""
    _pinned = {}

    def __init__(self, flat, nq, rows):
        self.nq, self.rows = nq, rows
        n = int(flat.numel())
        free = PendingStats._pinned.setdefault(n, [])
        self._host = free.pop() if free else torch.empty((n,), dtype=torch.float64).pin_memory()
        self._host.copy_(flat, non_blocking=True)
        self._event = torch.cuda.Event()
        self._event.record(torch.cuda.current_stream(flat.device))
        self._out = None

    def result(self):
        if self._out is None:
            self._event.synchronize()
            nq, rows, h = self.nq, self.rows, self._host
            self._out = finalize_stats(h[:nq * rows * 4].view(nq, rows, 4).clone(), h[nq * rows * 4:nq * rows * 8].view(nq, rows, 4).clone(),
                                       h[nq * rows * 8:].view(nq, rows).clone())
            PendingStats._pinned[int(h.numel())].append(h)
            self._host = None
        return self._out


class DeviceStats(object):
    """Statistics whose reduced sums stay on the device (lazy="device"): nothing but kernels and collectives is
    queued, so the call can be captured in a CUDA graph; `.result()` copies and finalises (synchronises)."""

    def __init__(self, flat, nq, rows):
        self.flat, self.nq, self.rows = flat, nq, rows

    def result(self):
        nq, rows, h = self.nq, self.rows, self.flat.cpu()
        return finalize_stats(h[:nq * rows * 4].view(nq, rows, 4), h[nq * rows * 4:nq * rows * 8].view(nq, rows, 4),
                              h[nq * rows * 8:].view(nq, rows))


def statistics(est, gt=None, class_id=None, n_class=1, group=None, distributed=True, lazy=False):
    """get_statistic_of_result (TEST_TOOLBOX.py:892-937) for up to 4 quantities at once, per class
    and over all problems, over ALL ranks' shards.

    est, gt: lists of 1-D FP64 CUDA views (strided allowed) of this rank's shard (gt entries or gt
    itself may be None); class_id int32 [B] or None.  Two kernels and two reduction phases
    (SURVEY.md 8e): all_reduce(SUM) of [n, sum est/gt, sum e]; the second kernel derives the global
    means from them; all_reduce(SUM) of [sum (e-m)^2, sum |e|, sum |e-m|] and all_reduce(MAX) of
    max |e-m|.  Returns a float64 CPU tensor [nq, n_class+1, 7] in STAT_KEYS order; the last row of
    each quantity is the class 'all'; empty classes have n = 0."""
    if torch.is_tensor(est):
        est, gt = [est], [gt]
    nq = len(est)
    gt = list(gt) if gt is not None else [None] * nq
    dev = est[0].device
    B = int(est[0].shape[0])
    PD = C.POINTER(C.c_double)
    dp = lambda x: None if x is None else C.cast(ptr(x), PD)
    est_a = (PD * nq)(*[dp(e) for e in est])
    gt_a = (PD * nq)(*[dp(g) for g in gt])
    es_a = (C.c_int64 * nq)(*[int(e.stride(0)) if B else 1 for e in est])
    gs_a = (C.c_int64 * nq)(*[(int(g.stride(0)) if B else 1) if g is not None else 0 for g in gt])
    for e in est:
        assert e.dtype == torch.float64 and e.dim() == 1 and int(e.shape[0]) == B
    cid = None if class_id is None else C.cast(ptr(class_id), C.POINTER(C.c_int32))
    rows = n_class + 1
    flat = torch.empty((nq * rows * 9,), dtype=torch.float64, device=dev)      # s1 | s2 | max in one allocation
    s1 = flat[:nq * rows * 4].view(nq, rows, 4)
    s2 = flat[nq * rows * 4:nq * rows * 8].view(nq, rows, 4)
    mx = flat[nq * rows * 8:].view(nq, rows)
    with torch.cuda.device(dev):
        check(lib.pnpb200_stats_pass1(C.c_int64(B), C.c_int(nq), est_a, es_a, gt_a, gs_a, cid, C.c_int(n_class),
                                      dp(s1), _stream_ptr(dev)), "pnpb200_stats_pass1")
    _lib.count_launch()
    if distributed:
        reduce_phase1(s1, group)
    with torch.cuda.device(dev):
        check(lib.pnpb200_stats_pass2(C.c_int64(B), C.c_int(nq), est_a, es_a, gt_a, gs_a, cid, C.c_int(n_class),
                                      dp(s1), dp(s2), dp(mx), _stream_ptr(dev)), "pnpb200_stats_pass2")
    _lib.count_launch()
    if distributed:
        reduce_phase2(s2, mx, group, flat23=flat[nq * rows * 4:])
    if lazy == "device":                                                        # capturable in a CUDA graph: no host buffer, no event
        return DeviceStats(flat, nq, rows)
    pending = PendingStats(flat, nq, rows)
    return pending if lazy else pending.result()                                # .result() is the only synchronisation


def approval_mask(gt, kind):
    """TEST_TOOLBOX.approval_func_small_angle / approval_func_large_angle (:959-970) for a batch:
    gt [B,4] = (depth, roll, pitch, yaw) tensor (any device) -> bool [B].  'small_angle': no ground-truth
    angle beyond 30 degrees in magnitude; 'large_angle': the complement."""
    small = (gt[:, 1].abs() <= 30) & (gt[:, 2].abs() <= 30) & (gt[:, 3].abs() <= 30)
    if kind == "small_angle":
        return small
    if kind == "large_angle":
        return ~small
    raise ValueError("approval must be None, 'small_angle' or 'large_angle', not %r" % (kind,))


def error_statistics(report, gt, group=None, distributed=True, lazy=False, approval=None):
    """The statistics block of TEST_TOOLBOX.data_analysis_and_saving (:1070-1112) for the four
    reported quantities, for class 'all' and per GT-depth class, in two kernels and two all-reduce
    phases.  report: [B,16] from report_batch; gt [B,4].
    approval: None, 'small_angle' or 'large_angle' = the approval_func of get_classified_result
    (:939-970): problems that fail it leave their distance class but stay in 'all', as there.
    Returns {quantity: {'all': stats[7], 'by_depth': stats[12,7]}} (CPU tensors, STAT_KEYS order);
    lazy=True returns an object whose .result() gives that dict (no host sync in this call)."""
    cls = classify(gt[:, 0], CLASS_BINS["depth"], scale=100.0)
    if approval is not None:
        cls = torch.where(approval_mask(gt, approval), cls, torch.full_like(cls, -1))
    # (estimate, GT): depth compares t3_est with distance_GT (:1073), the angles est vs GT
    est = [report[:, 10], report[:, 12], report[:, 13], report[:, 14]]
    ref = [report[:, 11], gt[:, 1], gt[:, 2], gt[:, 3]]
    st = statistics(est, ref, cls, len(CLASS_LABELS["depth"]), group, distributed, lazy=lazy)
    unpack = lambda x: {name: dict(all=x[q, -1], by_depth=x[q, :-1]) for q, name in enumerate(("depth", "roll", "pitch", "yaw"))}
    if lazy:
        return _LazyDict(st, unpack)
    return unpack(st)


DRPY_ORDER = ("depth", "roll", "pitch", "yaw")
DRPY_QUANTITIES = (("depth", "cm", 100.0), ("roll", "deg.", 1.0), ("pitch", "deg.", 1.0), ("yaw", "deg.", 1.0),
                   ("LM_GT_error_average_normalize", "px_m", 1.0))


def drpy_shape():
    return tuple(len(CLASS_LABELS[q]) for q in DRPY_ORDER)


def classify_drpy(gt):
    """Combined (distance, roll, pitch, yaw) class of every problem, one kernel: the key of the nested
    dict of TEST_TOOLBOX.get_all_class_seperated_result (:975-1030) as the mixed-radix integer
    ((cd*nr + cr)*np + cp)*ny + cy.  gt [B,4] (depth m, roll, pitch, yaw deg.) contiguous CUDA FP64."""
    assert gt.dtype == torch.float64 and gt.dim() == 2 and gt.shape[1] == 4 and gt.is_contiguous()
    B = int(gt.shape[0])
    cls = torch.empty((B,), dtype=torch.int32, device=gt.device)
    PD = C.POINTER(C.c_double)
    bins_np = [np.asarray(CLASS_BINS[q], np.float64) for q in DRPY_ORDER]
    bins_a = (PD * 4)(*[b.ctypes.data_as(PD) for b in bins_np])
    nb_a = (C.c_int32 * 4)(*[len(b) for b in bins_np])
    scale_a = (C.c_double * 4)(100.0, 1.0, 1.0, 1.0)                  # the distance class is on centimetres
    with torch.cuda.device(gt.device):
        check(lib.pnpb200_classify_drpy(C.c_int64(B), C.cast(ptr(gt), PD), bins_a, nb_a, scale_a,
                                        C.cast(ptr(cls), C.POINTER(C.c_int32)), _stream_ptr(gt.device)), "pnpb200_classify_drpy")
    _lib.count_launch()
    return cls


def drpy_statistics(report, gt, group=None, distributed=True):
    """get_drpy_statistic (TEST_TOOLBOX.py:1032-1066) for the five quantities data_analysis_and_saving
    tabulates (:1218-1226), over ALL ranks' shards: statistics per (distance, roll, pitch, yaw) class
    combination.  Returns {name: float64 CPU tensor [nd, nr, np, ny, 7]} (STAT_KEYS order; n = 0 where
    the reference's nested dict has no entry)."""
    cls = classify_drpy(gt)
    shape = drpy_shape()
    n_class = int(np.prod(shape))
    st4 = statistics([report[:, 10], report[:, 12], report[:, 13], report[:, 14]], [report[:, 11], gt[:, 1], gt[:, 2], gt[:, 3]],
                     cls, n_class, group, distributed, lazy=True)
    st1 = statistics([report[:, 4]], [None], cls, n_class, group, distributed, lazy=True)
    st4, st1 = st4.result(), st1.result()
    out = {name: st4[q, :-1].reshape(shape + (7,)) for q, name in enumerate(DRPY_ORDER)}
    out["LM_GT_error_average_normalize"] = st1[0, :-1].reshape(shape + (7,))
    return out


class _LazyDict(object):
    def __init__(self, pending, unpack):
        self._pending, self._unpack = pending, unpack

    def result(self):
        return self._unpack(self._pending.result())


# ------------------------------------------------------------------------------------------------
# face_variation_test.py: perturbed-pattern workload and the "most fragile point" analysis
# ------------------------------------------------------------------------------------------------
def synth_face_variation(b0, B, pattern, K, fixed_index, perturb_radius_m=0.02, cfg=None, dtype=torch.float64, device=None):
    """face_variation_test.py:296-356 for problems b0..b0+B-1 of the global stream: pixels of a
    randomly perturbed pattern (unit direction of the 3(n-1) coordinates of every landmark but
    `fixed_index`, times perturb_radius_m).  Returns dict(uv, gt, perturb [B,n,3] f64)."""
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    pat = torch.as_tensor(np.ascontiguousarray(np.asarray(pattern, dtype=np.float64)), device=device)
    n = int(pat.shape[0])
    uv = torch.empty((B, n, 2), dtype=dtype, device=device)
    gt = torch.empty((B, 4), dtype=torch.float64, device=device)
    pert = torch.empty((B, n, 3), dtype=torch.float64, device=device)
    Kh, Kp = _k_host(K)
    PD = C.POINTER(C.c_double)
    with torch.cuda.device(device):
        check(lib.pnpb200_synth_face_variation(C.c_int(_dtype_code(dtype)), C.c_int64(int(b0)), C.c_int64(int(B)), C.c_int(n),
                                               ptr(pat), Kp, C.byref(cfg) if cfg is not None else None,
                                               C.c_double(float(perturb_radius_m)), C.c_int(int(fixed_index)), ptr(uv),
                                               C.cast(ptr(gt), PD), None, None, C.cast(ptr(pert), PD), _stream_ptr(device)),
              "pnpb200_synth_face_variation")
    _lib.count_launch()
    return dict(uv=uv, gt=gt, perturb=pert)


def key_of(values, idx0=0):
    """The selection key of each problem as two NumPy integer arrays (hi uint64 = bits of |value|, NaN as
    +inf; lo uint32 = ~global index): what pnpb200_topk_histogram / pnpb200_fragility_accumulate compare."""
    a = np.abs(np.asarray(values, np.float64))
    hi = np.where(np.isnan(a), np.float64(np.inf), a).view(np.uint64)
    lo = (~(np.arange(a.shape[0], dtype=np.int64) + int(idx0))).astype(np.uint32)
    return hi, lo


def numpy_histogram(values_list, idx0):
    """Host stand-in for pnpb200_topk_histogram (tests, and shards that live in host memory):
    returns hist_fn(prefix_hi, prefix_lo, n_digits) -> int64 [nq, 256]."""
    keys = [key_of(v, idx0) for v in values_list]

    def digit(hi, lo, d):
        return ((hi >> np.uint64(56 - 8 * d)) & np.uint64(0xff)).astype(np.int64) if d < 8 else \
               ((lo >> np.uint32(24 - 8 * (d - 8))) & np.uint32(0xff)).astype(np.int64)

    def fn(pre_hi, pre_lo, nd):
        out = np.zeros((len(keys), 256), np.int64)
        for q, (hi, lo) in enumerate(keys):
            m = np.ones(hi.shape[0], bool)
            for d in range(nd):
                want = (pre_hi[q] >> (56 - 8 * d)) & 0xff if d < 8 else (pre_lo[q] >> (24 - 8 * (d - 8))) & 0xff
                m &= digit(hi, lo, d) == want
            out[q] = np.bincount(digit(hi, lo, nd)[m], minlength=256)
        return out
    return fn


def topk_thresholds(values, k, idx0=0, group=None, hist_fn=None):
    """Exact k-th largest key (|value| bits, then smaller global index first) of each quantity over
    ALL ranks' shards: 12 histogram kernels; the 256-bin histograms are the only thing all-reduced.
    values: list of 1-D FP64 CUDA views of this rank's shard (or, with hist_fn = numpy_histogram(...),
    anything).  Returns (hi [nq] uint64, lo [nq] uint32) as Python ints -- every key >= (hi, lo) is in
    the top k."""
    import torch.distributed as dist
    nq = len(values)
    hi, lo, rem = [0] * nq, [0] * nq, [int(k)] * nq
    if hist_fn is None:
        dev = values[0].device
        B = int(values[0].shape[0])
        PD = C.POINTER(C.c_double)
        val_a = (PD * nq)(*[C.cast(ptr(v), PD) for v in values])
        str_a = (C.c_int64 * nq)(*[int(v.stride(0)) if B else 1 for v in values])
        hist = torch.zeros((nq, 256), dtype=torch.int64, device=dev)
    for d in range(12):
        if hist_fn is None:
            hi_a = (C.c_uint64 * nq)(*hi)
            lo_a = (C.c_uint32 * nq)(*lo)
            with torch.cuda.device(dev):
                check(lib.pnpb200_topk_histogram(C.c_int64(B), C.c_int64(int(idx0)), C.c_int(nq), val_a, str_a, hi_a, lo_a, C.c_int(d),
                                                 C.cast(ptr(hist), C.POINTER(C.c_uint64)), _stream_ptr(dev)), "pnpb200_topk_histogram")
            _lib.count_launch()
        else:
            hist = torch.from_numpy(hist_fn(hi, lo, d))
        _all_reduce(hist, dist.ReduceOp.SUM if dist.is_available() else None, group)
        h = hist.cpu().numpy()
        for q in range(nq):
            digit = 0
            for dg in range(255, -1, -1):                 # from the largest digit down
                if h[q, dg] >= rem[q]:
                    digit = dg
                    break
                rem[q] -= int(h[q, dg])
            if d < 8:
                hi[q] |= digit << (56 - 8 * d)
            else:
                lo[q] |= digit << (24 - 8 * (d - 8))
    return hi, lo


def fragility_analysis(abs_err, perturb, idx0=0, ratio=0.1, k_top_direction=5, total=None, group=None, keys=None):
    """The analysis block of face_variation_test.py (:631-759) on the device, over ALL ranks' shards.

    abs_err: list of up to four 1-D FP64 CUDA views (|depth err|, |roll err|, ...) of this rank's
    shard; perturb [B,n,3] from synth_face_variation; idx0 = global index of the shard's first
    problem; total = number of problems over all ranks (default: this shard).  The top
    int(total * ratio) problems of each quantity are selected exactly as the script's heaps do.
    Returns one dict per quantity with the script's result_dict fields as arrays:
    fragile_point_count [n], fragile_point_order (landmark indices, most fragile first),
    top_perturbation [k_top_direction, n, 3], top_similarity [k_top_direction], value_max,
    top_value_mean, n_selected; with keys (landmark names in pattern order) also
    fragile_point_count_dict and fragile_point_sorted_list = [(count, key)] sorted like the script
    (reverse tuple order, :694-695)."""
    import torch.distributed as dist
    nq = len(abs_err)
    dev = perturb.device
    B, n = int(perturb.shape[0]), int(perturb.shape[1])
    total = B if total is None else int(total)
    k = int(total * ratio)                                                       # :632
    if k < 1:
        raise ValueError("fragility_analysis: nothing to select (total * ratio < 1)")
    hi, lo = topk_thresholds(abs_err, k, idx0, group)
    PD = C.POINTER(C.c_double)
    val_a = (PD * nq)(*[C.cast(ptr(v), PD) for v in abs_err])
    str_a = (C.c_int64 * nq)(*[int(v.stride(0)) if B else 1 for v in abs_err])
    D = 3 * n
    cap = max(1, min(B, k))
    lst = torch.empty((nq, cap), dtype=torch.int64, device=dev)
    nsel = torch.zeros((nq,), dtype=torch.int64, device=dev)
    cnt = torch.zeros((nq, n), dtype=torch.int64, device=dev)
    vsum = torch.zeros((nq,), dtype=torch.float64, device=dev)
    vmax = torch.zeros((nq,), dtype=torch.float64, device=dev)
    gram = torch.zeros((nq, D, D), dtype=torch.float64, device=dev)
    pert = perturb.contiguous()
    PU = C.POINTER(C.c_uint64)
    with torch.cuda.device(dev):
        check(lib.pnpb200_fragility_accumulate(C.c_int64(B), C.c_int64(int(idx0)), C.c_int(nq), val_a, str_a,
                                               (C.c_uint64 * nq)(*hi), (C.c_uint32 * nq)(*lo), C.cast(ptr(pert), PD), C.c_int(n),
                                               C.c_int64(cap), C.cast(ptr(lst), C.POINTER(C.c_int64)), C.cast(ptr(nsel), PU),
                                               C.cast(ptr(cnt), PU), C.cast(ptr(vsum), PD), C.cast(ptr(vmax), PD),
                                               C.cast(ptr(gram), PD), _stream_ptr(dev)), "pnpb200_fragility_accumulate")
    _lib.count_launch(2)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        for t_ in (nsel, cnt, vsum, gram):
            dist.all_reduce(t_, op=dist.ReduceOp.SUM, group=group)
        dist.all_reduce(vmax, op=dist.ReduceOp.MAX, group=group)
    out = []
    G = gram.cpu().numpy()
    for q in range(nq):
        g = np.triu(G[q]) + np.triu(G[q], 1).T                                  # the kernel fills the upper tiles
        w, v = np.linalg.eigh(g)
        order = np.argsort(w)[::-1][:k_top_direction]
        m = int(nsel[q].item())
        c = cnt[q].cpu().numpy()
        out.append(dict(
            n_selected=m, fragile_point_count=c,
            fragile_point_order=np.array(sorted(range(n), key=lambda i: (-int(c[i]), i))),
            top_similarity=np.sqrt(np.maximum(w[order], 0.0)),                    # singular values of the m x 3n matrix
            top_perturbation=v[:, order].T.reshape(-1, n, 3),                     # right singular vectors (sign is arbitrary)
            value_max=float(vmax[q].item()), top_value_mean=float(vsum[q].item()) / max(m, 1)))
        if keys is not None:
            out[-1]["fragile_point_count_dict"] = {key: int(c[i]) for i, key in enumerate(keys)}
            out[-1]["fragile_point_sorted_list"] = sorted([(int(c[i]), key) for i, key in enumerate(keys)], reverse=True)
    return out


# ------------------------------------------------------------------------------------------------
# result writers (TEST_TOOLBOX.py:693-887, :1070-1346)
# ------------------------------------------------------------------------------------------------
def write_result_csv(path, report, flags, max_idx, res_norm, gt, key_names, idx0=0, append=False, n_threads=0):
    """TEST_TOOLBOX.write_result_to_csv (:693-708) for a whole batch: the native writer formats the
    rows from the report arrays (CUDA tensors are copied to the host first; NumPy arrays and CPU
    tensors are used as they are).  key_names: landmark names in pattern order."""
    def host(x, dt):
        if torch.is_tensor(x):
            x = x.detach().to("cpu")
            return np.ascontiguousarray(x.numpy().astype(dt, copy=False))
        return np.ascontiguousarray(np.asarray(x, dtype=dt))
    rep, fl, mi = host(report, np.float64), host(flags, np.int32), host(max_idx, np.int32)
    rn, g = host(res_norm, np.float64).reshape(-1), host(gt, np.float64)
    B = rep.shape[0]
    assert rep.shape == (B, 16) and fl.shape == (B, 4) and mi.shape == (B, 3) and rn.shape == (B,) and g.shape == (B, 4)
    names = [k.encode() for k in key_names]
    name_a = (C.c_char_p * len(names))(*names)
    order = ("depth", "roll", "pitch", "yaw")
    bins_np = [np.asarray(CLASS_BINS[q], np.float64) for q in order]
    PD = C.POINTER(C.c_double)
    bins_a = (PD * 4)(*[b.ctypes.data_as(PD) for b in bins_np])
    nb_a = (C.c_int32 * 4)(*[len(b) for b in bins_np])
    lab_keep = [(C.c_char_p * len(CLASS_LABELS[q]))(*[s.encode() for s in CLASS_LABELS[q]]) for q in order]
    lab_a = (C.POINTER(C.c_char_p) * 4)(*[C.cast(a, C.POINTER(C.c_char_p)) for a in lab_keep])
    check(lib.pnpb200_write_result_csv(str(path).encode(), C.c_int(1 if append else 0), C.c_int64(B), C.c_int64(int(idx0)),
                                       rep.ctypes.data_as(PD), fl.ctypes.data_as(C.POINTER(C.c_int32)),
                                       mi.ctypes.data_as(C.POINTER(C.c_int32)), rn.ctypes.data_as(PD), g.ctypes.data_as(PD),
                                       name_a, C.c_int(len(names)), bins_a, nb_a, lab_a, C.c_int(int(n_threads))),
          "pnpb200_write_result_csv")
    return path


def statistic_dicts(stats, labels, unit, unit_scale):
    """One quantity's statistics (error_statistics()[name]) as the {class label: statis_dict} the
    reference builds with get_statistic_of_result per class (TEST_TOOLBOX.py:928-936, :1090-1101):
    keys n_data, m_ratio, mean(u), stddev(u), max_dev(u), MAE_2_GT(u), MAE_2_mean(u); classes without
    data are absent, 'all' is included."""
    out = {}
    rows = [(lb, stats["by_depth"][i]) for i, lb in enumerate(labels)] + [("all", stats["all"])]
    for lb, r in rows:
        r = [float(x) for x in r]
        if not r[0] > 0:
            continue
        out[lb] = {"n_data": int(r[0]), "m_ratio": r[1], "mean(%s)" % unit: r[2] * unit_scale, "stddev(%s)" % unit: r[3] * unit_scale,
                   "max_dev(%s)" % unit: r[4] * unit_scale, "MAE_2_GT(%s)" % unit: r[5] * unit_scale,
                   "MAE_2_mean(%s)" % unit: r[6] * unit_scale}
    return out


def _class_order(e):
    return float("-inf") if e == "all" else float(e)                 # TEST_TOOLBOX._class_order_func :710-716


def write_statistic_txt(class_statistic_dict, path, class_name="distance", statistic_data_name="depth"):
    """TEST_TOOLBOX.write_statistic_to_txt (:718-752), same text."""
    s = "\nStatistic of [%s] for each [%s] class:\n" % (statistic_data_name, class_name)
    for lb in sorted(class_statistic_dict, key=_class_order):
        s += "[%s]: " % lb + " | ".join("%s=%f" % (k, v) for k, v in class_statistic_dict[lb].items()) + "\n"
    with open(path, "w") as f:
        f.write(s)
    return s


def write_statistic_csv(class_statistic_dict, path, is_horizontal=True):
    """TEST_TOOLBOX.write_statistic_to_csv (:754-820), same rows through the same csv.DictWriter."""
    import csv
    labels = sorted(class_statistic_dict, key=_class_order)
    metrics = list(class_statistic_dict[labels[0]].keys())
    if is_horizontal:
        fields = ["_"] + labels
        rows = [dict([("_", m)] + [(lb, class_statistic_dict[lb][m]) for lb in labels]) for m in metrics]
    else:
        fields = ["_"] + metrics
        rows = [dict([("_", lb)] + [(m, class_statistic_dict[lb][m]) for m in metrics]) for lb in labels]
    with open(path, mode="w") as f:
        w = csv.DictWriter(f, fieldnames=fields, extrasaction="ignore")
        w.writeheader()
        w.writerows(rows)
    return rows


def drpy_statistic_dict(stats5, unit, unit_scale):
    """One quantity of drpy_statistics() as the nested {d: {r: {p: {y: statis_dict}}}} of
    get_drpy_statistic (:1032-1066) plus the four sorted label lists get_all_class_seperated_result
    returns (:1019-1028: labels that occur in the data, numeric order)."""
    a = np.asarray(stats5, dtype=np.float64)
    labs = [CLASS_LABELS[q] for q in DRPY_ORDER]
    present = a[..., 0] > 0
    lists = []
    for ax in range(4):
        occ = present.any(axis=tuple(i for i in range(4) if i != ax))
        lists.append(sorted([labs[ax][i] for i in np.nonzero(occ)[0]], key=_class_order))
    out = {}
    for d, r, p, y in zip(*np.nonzero(present)):
        v = [float(x) for x in a[d, r, p, y]]
        out.setdefault(labs[0][d], {}).setdefault(labs[1][r], {}).setdefault(labs[2][p], {})[labs[3][y]] = {
            "n_data": int(v[0]), "m_ratio": v[1], "mean(%s)" % unit: v[2] * unit_scale, "stddev(%s)" % unit: v[3] * unit_scale,
            "max_dev(%s)" % unit: v[4] * unit_scale, "MAE_2_GT(%s)" % unit: v[5] * unit_scale, "MAE_2_mean(%s)" % unit: v[6] * unit_scale}
    return (out,) + tuple(lists)


def write_drpy_statistic_csv(drpy_dict, path, d_labels, r_labels, p_labels, y_labels, metric_label="mean(cm)"):
    """TEST_TOOLBOX.write_drpy_2_depth_statistic_CSV (:822-887): one block of rows per roll label
    ("r=.., y=.." per yaw label, then an empty row), one group of columns per distance label
    ("d=..", then "d=.., p=.." per pitch label, then a "|count" separator); "-" where the class
    combination holds no data.  Same csv.DictWriter, same text."""
    import csv
    fields, rows = [], []
    def col(name):
        if name not in fields:
            fields.append(name)
        return name
    for r in r_labels:
        for y in y_labels:
            row, bars = {}, 0
            for d in d_labels:
                row[col("d=%s" % d)] = "r=%s, y=%s" % (r, y)
                for p in p_labels:
                    bars += 1
                    leaf = drpy_dict.get(d, {}).get(r, {}).get(p, {}).get(y)
                    row[col("d=%s, p=%s" % (d, p))] = leaf[metric_label] if leaf is not None and metric_label in leaf else "-"
                row[col("|%d" % bars)] = ""
            rows.append(row)
        rows.append({})
    with open(path, mode="w") as f:
        w = csv.DictWriter(f, fieldnames=fields, extrasaction="ignore")
        w.writeheader()
        w.writerows(rows)
    return rows


def drpy_analysis_and_saving(report, gt, result_csv_dir_str, result_statistic_txt_file_prefix_str, data_file_str,
                             group=None, distributed=True, stats=None):
    """The second half of TEST_TOOLBOX.data_analysis_and_saving (:1215-1346): the eleven
    "<prefix><stem>_drpy_to_<quantity>_<metric>.csv" tables (n_data once, mean and stddev for depth,
    roll, pitch, yaw and LM_GT_error_average_normalize).  `stats` = a precomputed drpy_statistics()."""
    st = stats if stats is not None else drpy_statistics(report, gt, group=group, distributed=distributed)
    stem = result_csv_dir_str + result_statistic_txt_file_prefix_str + data_file_str[:-4] + "_drpy_to_"
    dicts, paths = {}, []
    for name, unit, scale in DRPY_QUANTITIES:
        dicts[name] = drpy_statistic_dict(st[name], unit, scale)
    dd, dl, rl, pl, yl = dicts["depth"]
    paths.append(stem + "all_n_data.csv")
    write_drpy_statistic_csv(dd, paths[-1], dl, rl, pl, yl, metric_label="n_data")
    for metric in ("mean", "stddev"):
        for name, unit, _ in DRPY_QUANTITIES:
            label = "%s(%s)" % (metric, unit)
            paths.append(stem + name + "_" + label + ".csv")
            write_drpy_statistic_csv(dicts[name][0], paths[-1], dl, rl, pl, yl, metric_label=label)
    return paths


def data_analysis_and_saving(rep, res_norm, gt, key_names, result_csv_dir_str, result_csv_file_prefix_str,
                             result_statistic_txt_file_prefix_str, data_file_str, is_statistic_csv_horizontal=True,
                             idx0=0, group=None, distributed=True, with_drpy=True):
    """TEST_TOOLBOX.data_analysis_and_saving (:1070-1346) for a batch: the result CSV, for depth,
    roll, pitch and yaw per distance class the statistic TXT and CSV files, and (with_drpy) the eleven
    class-combination tables, with the reference's file names.  rep = report_batch(...) dict.
    Returns the four {label: statis_dict} dicts."""
    stem = data_file_str[:-4]
    write_result_csv(result_csv_dir_str + result_csv_file_prefix_str + stem + ".csv", rep["report"], rep["flags"], rep["max_idx"],
                     res_norm, gt, key_names, idx0=idx0)
    st = error_statistics(rep["report"], gt, group=group, distributed=distributed)
    out = {}
    for name, unit, scale in (("depth", "cm", 100.0), ("roll", "deg.", 1.0), ("pitch", "deg.", 1.0), ("yaw", "deg.", 1.0)):
        d = statistic_dicts(st[name], CLASS_LABELS["depth"], unit, scale)
        base = result_csv_dir_str + result_statistic_txt_file_prefix_str + stem + "_distance_to_%s" % name
        write_statistic_txt(d, base + ".txt", class_name="distance", statistic_data_name=name)
        write_statistic_csv(d, base + ".csv", is_horizontal=is_statistic_csv_horizontal)
        out[name] = d
    if with_drpy:
        drpy_analysis_and_saving(rep["report"], gt, result_csv_dir_str, result_statistic_txt_file_prefix_str, data_file_str,
                                 group=group, distributed=distributed)
    return out
