#!/usr/bin/env python
"""Developer tool: device time of the masked solve (pnpb200_solve_batch_masked) against the solve without a mask, on 1 Mi
problems in FP64: LM and EIF2 on 68 landmarks and QEIF on 6 of 15; then the masked error report and solution check kernels
(pnpb200_report_batch_strided_masked, pnpb200_check_batch_masked) against the unmasked ones on the LM-68 poses.  For each,
three calls alternate in one process: no mask, an all-visible mask and a mask with 25 % of the landmarks hidden (drawn per problem).  Per-kernel times come from CUDA
events (PNPB200_FLAG_PROFILE, pnpb200_profile_read); the call time is a CUDA-event interval around the call.  Prints the
GPU's name and power limit first: the numbers belong to them."""
import ctypes as C
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import pnp_solver_test_b200 as pnp
from pnp_solver_test_b200 import _lib, workload as wl, patterns as pt

B = 1 << 20
REPS = 7

try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=60).stdout.strip()
except (OSError, subprocess.SubprocessError) as e:
    smi = "nvidia-smi unavailable (%s)" % e
print("GPU: %s | nvidia-smi name, power limit, max SM clock: %s" % (torch.cuda.get_device_name(0), smi), flush=True)

K = pt.default_camera_matrix()


def timed(method, uv, pat, idx, vis):
    """(call ms, [kernel ms x 3]) of one profiled call"""
    _lib.lib.pnpb200_profile_reset()
    prm = pnp.default_params(flags=_lib.FLAG_PROFILE)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    pnp.solve_batch(method, uv, pat, K, point_index=idx, params=prm, visible=vis)
    e1.record()
    torch.cuda.synchronize()
    ms = (C.c_float * 3)()
    calls = C.c_int(0)
    _lib.check(_lib.lib.pnpb200_profile_read(ms, C.byref(calls)), "pnpb200_profile_read")
    return e0.elapsed_time(e1), list(ms)


for method, n, subset in (("lm", 68, False), ("eif2", 68, False), ("qeif", 15, True)):
    pat = pt.get_golden_pattern() if n == 15 else pt.synthetic_pattern(n)
    P = pt.pattern_array(pat)
    w = wl.synth_batch(0, B, P, K, dtype=torch.float64)
    patd = torch.from_numpy(P).to("cuda", torch.float64)[None].contiguous()
    idx = [list(pat).index(k) for k in pt.LM_KEY_LIST_6] if subset else None
    sel = idx if subset else list(range(n))
    gen = torch.Generator(device="cuda").manual_seed(1)
    # 25 % of the selected landmarks hidden, drawn per problem (ranks of uniform keys)
    keys = torch.rand((B, len(sel)), generator=gen, device="cuda")
    hide = keys.argsort(dim=1)[:, : len(sel) // 4]
    part = torch.ones((B, n), dtype=torch.bool, device="cuda")
    part.scatter_(1, torch.tensor(sel, device="cuda")[hide], False)
    masks = {"no mask": None, "all visible": torch.ones((B, n), dtype=torch.bool, device="cuda"), "25% hidden": part}
    for v in masks.values():                              # warm-up of every shape
        timed(method, w["uv"], patd, idx, v)
    res = {k: [] for k in masks}
    for _ in range(REPS):
        for k, v in masks.items():
            res[k].append(timed(method, w["uv"], patd, idx, v))
    base = statistics.median(r[0] for r in res["no mask"])
    label = "%s-%s%d" % (method.upper(), "6-of-" if subset else "", n)
    for k, rs in res.items():
        call = statistics.median(r[0] for r in rs)
        kern = [statistics.median(r[1][j] for r in rs) for j in range(3)]
        print("%-12s %-12s %d problems FP64: call %.3f ms (x%.2f of no mask) | kernels (moments | direct solve, iterate, residual) "
              "%.3f %.3f %.3f ms | median of %d alternated calls" % (label, k, B, call, call / base, kern[0], kern[1], kern[2], REPS),
              flush=True)
    if method == "lm":                                    # the report and the check kernels, with the words packed beforehand
        o = pnp.solve_batch(method, w["uv"], patd, K)
        PD, PI, U = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_uint32)
        Kh, bd = (C.c_double * 9)(*K.reshape(-1).tolist()), (C.c_double * 4)(10, 10, 10, 10)
        rep = torch.empty((16, B), dtype=torch.float64, device="cuda").t()
        flags, midx = torch.empty((B, 4), dtype=torch.int32, device="cuda"), torch.empty((B, 3), dtype=torch.int32, device="cuda")
        status, reproj = torch.empty((B,), dtype=torch.int32, device="cuda"), torch.empty((B, 2), dtype=torch.float64, device="cuda")
        gt = w["gt"].contiguous()
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        p_ = _lib.ptr

        def report(words):
            args = (C.c_int(_lib.DTYPE_F64), C.c_int64(B), C.c_int(n), p_(patd), p_(w["uv"]), Kh, p_(o["R"]), p_(o["t"]), p_(o["euler"]),
                    C.cast(p_(gt), PD), bd, C.cast(p_(rep), PD), C.c_int64(1), C.c_int64(B), C.cast(p_(flags), PI), C.cast(p_(midx), PI))
            rc = (_lib.lib.pnpb200_report_batch_strided(*args, st) if words is None else
                  _lib.lib.pnpb200_report_batch_strided_masked(*args, C.cast(p_(words), U), st))
            _lib.check(rc, "report")

        def check(words):
            args = (_lib.DTYPE_F64, B, n, p_(patd), 1, p_(w["uv"]), Kh, p_(o["R"]), p_(o["t"]), p_(o["res_norm"]), None, 1.0,
                    C.cast(p_(status), PI), p_(reproj))
            rc = (_lib.lib.pnpb200_check_batch(*args, st) if words is None else
                  _lib.lib.pnpb200_check_batch_masked(*args, C.cast(p_(words), U), st))
            _lib.check(rc, "check")

        words = {k: (None if v is None else pnp.solver.visible_words(v, "cuda")) for k, v in masks.items()}
        for name, fn in (("k_report_chunk", report), ("k_check_chunk", check)):
            t = {k: [] for k in words}
            for _ in range(3):
                for k, v in words.items():
                    fn(v)
            for _ in range(REPS):
                for k, v in words.items():
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(); fn(v); e1.record()
                    torch.cuda.synchronize()
                    t[k].append(e0.elapsed_time(e1))
            print("%-12s %s: %s | median of %d alternated launches" % (label, name, " | ".join(
                "%s %.3f ms" % (k, statistics.median(v)) for k, v in t.items()), REPS), flush=True)
        del o, rep, flags, midx, status, reproj, words
    del w, masks, part, keys, hide
    torch.cuda.empty_cache()
