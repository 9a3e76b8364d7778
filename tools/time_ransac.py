#!/usr/bin/env python
"""Developer tool: device time of the RANSAC solve (pnpb200_solve_ransac_batch) and of its hypothesis stage
(pnpb200_hypothesize_batch, kernel k_hypothesize) on 1 Mi problems x 68 landmarks, FP64 and FP32, default parameters, with 0 /
10 / 30 % of the landmarks of each problem moved by U(30, 150) px and rounded.  The RANSAC call, the robust call
(pnpb200_solve_robust_batch) and the masked solve (all landmarks visible) are timed with CUDA events around the C entries,
alternating in one process; the table gives the median of REPS calls, the mean number of samples drawn, the mean consensus
and the mean number of solves (rounds) of the two robust entries.  Writes its lines to --out (default
profiles/r03e_ransac.log) after the GPU's name and power limit, read in the same run: the numbers belong to them."""
import argparse
import ctypes as C
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import pnp_solver_test_b200 as pnp
from pnp_solver_test_b200 import _lib, workload as wl, patterns as pt
from pnp_solver_test_b200.solver import visible_words

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "r03e_ransac.log"))
ap.add_argument("--methods", default="lm_plus,eif2")
args = ap.parse_args()
B, N = 1 << 20, 68
REPS = 5
lines = []


def say(s):
    print(s, flush=True)
    lines.append(s)


try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=60).stdout.strip()
except (OSError, subprocess.SubprocessError) as e:
    smi = "nvidia-smi unavailable (%s)" % e
say("GPU: %s | nvidia-smi name, power limit, max SM clock: %s" % (torch.cuda.get_device_name(0), smi))

K = pt.default_camera_matrix()
Kh = (C.c_double * 9)(*K.reshape(-1).tolist())
P = pt.pattern_array(pt.synthetic_pattern(N))
w = wl.synth_batch(0, B, P, K, dtype=torch.float64)
PI, U = C.POINTER(C.c_int32), C.POINTER(C.c_uint32)
hp = pnp.solver.hypothesis_params()
rp = pnp.solver.robust_params()


def outliers(uv, f, seed=1):
    """round(f N) landmarks per problem moved by U(30, 150) px in a random direction, rounded (on the device)"""
    k = int(round(f * N))
    if k == 0:
        return uv.clone()
    g = torch.Generator(device="cuda").manual_seed(seed)
    idx = torch.rand((B, N), generator=g, device="cuda").argsort(dim=1)[:, :k]
    r = 30.0 + 120.0 * torch.rand((B, k), generator=g, device="cuda", dtype=torch.float64)
    th = 2 * torch.pi * torch.rand((B, k), generator=g, device="cuda", dtype=torch.float64)
    out = uv.clone()
    d = torch.stack([r * torch.cos(th), r * torch.sin(th)], dim=-1)
    out.scatter_add_(1, idx[..., None].expand(B, k, 2), d)
    return out.round()


def buffers(dt):
    f = lambda *s: torch.empty(s, dtype=dt, device="cuda")          # noqa: E731
    i = lambda *s: torch.empty(s, dtype=torch.int32, device="cuda")  # noqa: E731
    return dict(R=f(B, 9), t=f(B, 3), e=f(B, 3), res=f(B), it=i(B), best=i(B), inl=i(B, 3), rounds=i(B), status=i(B), cons=i(B),
                drawn=i(B), mask=i(B, 3))


def call(kind, m, dtc, uv, pat, o, words, prm):
    if kind == "hyp":
        rc = _lib.lib.pnpb200_hypothesize_batch(dtc, B, N, N, _lib.ptr(uv), _lib.ptr(pat), 1, None, Kh, None, C.byref(hp), _lib.ptr(o["R"]),
                                                _lib.ptr(o["t"]), C.cast(_lib.ptr(o["best"]), PI), C.cast(_lib.ptr(o["mask"]), U),
                                                C.cast(_lib.ptr(o["cons"]), PI), C.cast(_lib.ptr(o["drawn"]), PI), None)
        _lib.check(rc, kind)
        return
    a = (m, dtc, B, N, N, _lib.ptr(uv), _lib.ptr(pat), 1, None, Kh, C.byref(prm[kind]), _lib.ptr(o["R"]), _lib.ptr(o["t"]),
         _lib.ptr(o["e"]), _lib.ptr(o["res"]), C.cast(_lib.ptr(o["it"]), PI), C.cast(_lib.ptr(o["best"]), PI))
    tail = (C.cast(_lib.ptr(o["inl"]), U), C.cast(_lib.ptr(o["rounds"]), PI), C.cast(_lib.ptr(o["status"]), PI))
    if kind == "masked":
        rc = _lib.lib.pnpb200_solve_batch_masked(*a, C.cast(_lib.ptr(words), U), None)
    elif kind == "robust":
        rc = _lib.lib.pnpb200_solve_robust_batch(*a, None, C.byref(rp), *tail, None)
    else:
        rc = _lib.lib.pnpb200_solve_ransac_batch(*a, None, C.byref(rp), *tail, C.byref(hp), C.cast(_lib.ptr(o["cons"]), PI),
                                                 C.cast(_lib.ptr(o["drawn"]), PI), None)
    _lib.check(rc, kind)


def timed(*a):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    call(*a)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


words = visible_words(torch.ones((B, N), dtype=torch.bool, device="cuda"), "cuda")
for dt, dtc in ((torch.float64, 0), (torch.float32, 1)):
    pat = torch.from_numpy(P).to("cuda", dt)[None].contiguous()
    o = buffers(dt)
    for method in args.methods.split(","):
        m = _lib.METHODS[method]
        sizes = dict(masked=int(_lib.lib.pnpb200_workspace_bytes_masked(m, dtc, B, 1, 0)),
                     robust=int(_lib.lib.pnpb200_robust_workspace_bytes(m, dtc, B, N, 1, 0)),
                     ransac=int(_lib.lib.pnpb200_ransac_workspace_bytes(m, dtc, B, N, 1, 0)))
        ws = {k: torch.empty((max(v, 1),), dtype=torch.uint8, device="cuda") for k, v in sizes.items()}
        prm = {k: pnp.default_params(workspace=ws[k].data_ptr(), workspace_bytes=sizes[k]) for k in sizes}
        for f in (0.0, 0.1, 0.3):
            uv = outliers(w["uv"], f).to(dt)
            kinds = ("hyp", "masked", "robust", "ransac")
            for kind in kinds:                            # warm-up
                timed(kind, m, dtc, uv, pat, o, words, prm)
            res = {k: [] for k in kinds}
            stats = {}
            for _ in range(REPS):
                for kind in kinds:
                    res[kind].append(timed(kind, m, dtc, uv, pat, o, words, prm))
                    if kind == "robust":
                        stats["robust_rounds"] = o["rounds"].double().mean().item()
                    if kind == "ransac":
                        stats["ransac_rounds"] = o["rounds"].double().mean().item()
                        stats["drawn"] = o["drawn"].double().mean().item()
                        stats["cons"] = o["cons"].double().mean().item()
            t = {k: statistics.median(v) for k, v in res.items()}
            say("%-8s %s f=%2d%% %d x %d: k_hypothesize %.3f ms (drawn %.2f, consensus %.1f) | RANSAC %.3f ms (%.2f solves) | "
                "robust %.3f ms (%.2f solves) | masked solve %.3f ms | median of %d alternated calls"
                % (method.upper(), "FP64" if dtc == 0 else "FP32", round(100 * f), B, N, t["hyp"], stats["drawn"], stats["cons"],
                   t["ransac"], stats["ransac_rounds"], t["robust"], stats["robust_rounds"], t["masked"], REPS))
os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
with open(args.out, "w") as fh:
    fh.write("\n".join(lines) + "\n")
