#!/usr/bin/env python
"""Developer tool: device time of the weighted solve (pnpb200_solve_batch_weighted) against the masked solve on the same problems,
1 Mi problems: LM, LM+, QEIF and EIF2 on 68 landmarks in FP64, QEIF on 6 of 15 (the direct mapping) and LM-68 in FP32.  For
each, four calls alternate in one process: every landmark visible / every weight 1, and the same 25 % of the landmarks hidden /
of weight 0 (drawn per problem).  Per-kernel times come from CUDA events (PNPB200_FLAG_PROFILE, pnpb200_profile_read); the call
time is a CUDA-event interval around the call.  Each weighted result is also compared bit for bit with its masked twin.  Prints
the GPU's name and power limit first: the numbers belong to them."""
import ctypes as C
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
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


def timed(method, uv, pat, idx, vis, wts):
    """(call ms, [kernel ms x 3], outputs) of one profiled call"""
    _lib.lib.pnpb200_profile_reset()
    prm = pnp.default_params(flags=_lib.FLAG_PROFILE)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = pnp.solve_batch(method, uv, pat, K, point_index=idx, params=prm, visible=vis, weights=wts)
    e1.record()
    torch.cuda.synchronize()
    ms = (C.c_float * 3)()
    calls = C.c_int(0)
    _lib.check(_lib.lib.pnpb200_profile_read(ms, C.byref(calls)), "pnpb200_profile_read")
    return e0.elapsed_time(e1), list(ms), out


def same_bits(a, b):
    return all(torch.equal(a[k].view(torch.uint8) if a[k].is_floating_point() else a[k],
                           b[k].view(torch.uint8) if b[k].is_floating_point() else b[k]) for k in a)


for method, n, subset, dt in (("lm", 68, False, torch.float64), ("lm_plus", 68, False, torch.float64), ("qeif", 68, False, torch.float64),
                              ("eif2", 68, False, torch.float64), ("qeif", 15, True, torch.float64), ("lm", 68, False, torch.float32)):
    pat = pt.get_golden_pattern() if n == 15 else pt.synthetic_pattern(n)
    P = pt.pattern_array(pat)
    w = wl.synth_batch(0, B, P, K, dtype=dt)
    patd = torch.from_numpy(P).to("cuda", dt)[None].contiguous()
    idx = [list(pat).index(k) for k in pt.LM_KEY_LIST_6] if subset else None
    sel = idx if subset else list(range(n))
    gen = torch.Generator(device="cuda").manual_seed(1)
    keys = torch.rand((B, len(sel)), generator=gen, device="cuda")
    hide = keys.argsort(dim=1)[:, : len(sel) // 4]
    part = torch.ones((B, n), dtype=torch.bool, device="cuda")
    part.scatter_(1, torch.tensor(sel, device="cuda")[hide], False)
    allv = torch.ones((B, n), dtype=torch.bool, device="cuda")
    cases = {"masked all visible": (allv, None), "weighted all 1": (None, allv.float()),
             "masked 25% hidden": (part, None), "weighted 25% w=0": (None, part.float())}
    outs = {}
    for k, (v, wt) in cases.items():                      # warm-up of every shape
        outs[k] = timed(method, w["uv"], patd, idx, v, wt)[2]
    ident = (same_bits(outs["weighted all 1"], outs["masked all visible"]), same_bits(outs["weighted 25% w=0"], outs["masked 25% hidden"]))
    del outs
    res = {k: [] for k in cases}
    for _ in range(REPS):
        for k, (v, wt) in cases.items():
            c, kern, o = timed(method, w["uv"], patd, idx, v, wt)
            res[k].append((c, kern))
            del o
    label = "%s-%s%d %s" % (method.upper(), "6-of-" if subset else "", n, "FP64" if dt == torch.float64 else "FP32")
    for k, rs in res.items():
        call = statistics.median(r[0] for r in rs)
        kern = [statistics.median(r[1][j] for r in rs) for j in range(3)]
        print("%-14s %-19s %d problems: call %.3f ms | kernels (moments | direct solve, iterate, residual) %.4f %.4f %.4f ms "
              "(sum %.4f) | median of %d alternated calls" % (label, k, B, call, kern[0], kern[1], kern[2], sum(kern), REPS), flush=True)
    print("%-14s weighted outputs bit-identical to the masked solve: all visible %s, 25%% hidden %s" % (label, ident[0], ident[1]),
          flush=True)
    del w, cases, part, keys, hide, allv
    torch.cuda.empty_cache()
