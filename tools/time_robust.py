#!/usr/bin/env python
"""Developer tool: device time of the outlier-robust solve (pnpb200_solve_robust_batch) against the masked solve
(pnpb200_solve_batch_masked, all landmarks visible) on 1 Mi problems x 68 landmarks in FP64, QEIF and LM+, with 0 / 10 / 30 % of
the landmarks of each problem moved by U(30, 150) px and rounded.  Calls are timed with CUDA events around the C entries
(arguments prepared beforehand, the two alternating); a separate torch.profiler run of one robust call gives the time of
every kernel, per round for the inlier classification and the compaction (select, gather, scatter).  Prints the GPU's name
and power limit first: the numbers belong to them."""
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

B, N = 1 << 20, 68
REPS = 7

try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=60).stdout.strip()
except (OSError, subprocess.SubprocessError) as e:
    smi = "nvidia-smi unavailable (%s)" % e
print("GPU: %s | nvidia-smi name, power limit, max SM clock: %s" % (torch.cuda.get_device_name(0), smi), flush=True)

K = pt.default_camera_matrix()
Kh = (C.c_double * 9)(*K.reshape(-1).tolist())
P = pt.pattern_array(pt.synthetic_pattern(N))
patd = torch.from_numpy(P).to("cuda", torch.float64)[None].contiguous()
w = wl.synth_batch(0, B, P, K, dtype=torch.float64)
PI, U = C.POINTER(C.c_int32), C.POINTER(C.c_uint32)


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


def buffers():
    f = lambda *s: torch.empty(s, dtype=torch.float64, device="cuda")   # noqa: E731
    i = lambda *s: torch.empty(s, dtype=torch.int32, device="cuda")     # noqa: E731
    return dict(R=f(B, 9), t=f(B, 3), e=f(B, 3), res=f(B), it=i(B), best=i(B), inl=i(B, 3), rounds=i(B), status=i(B))


def call(kind, m, uv, o, words, prm_m, prm_r):
    args = (m, 0, B, N, N, _lib.ptr(uv), _lib.ptr(patd), 1, None, Kh)
    outs = (_lib.ptr(o["R"]), _lib.ptr(o["t"]), _lib.ptr(o["e"]), _lib.ptr(o["res"]), C.cast(_lib.ptr(o["it"]), PI),
            C.cast(_lib.ptr(o["best"]), PI))
    if kind == "masked":
        rc = _lib.lib.pnpb200_solve_batch_masked(*args, C.byref(prm_m), *outs, C.cast(_lib.ptr(words), U), None)
    else:
        rc = _lib.lib.pnpb200_solve_robust_batch(*args, C.byref(prm_r), *outs, None, None, C.cast(_lib.ptr(o["inl"]), U),
                                                 C.cast(_lib.ptr(o["rounds"]), PI), C.cast(_lib.ptr(o["status"]), PI), None)
    _lib.check(rc, kind)


def timed(*a):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    call(*a)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


words = visible_words(torch.ones((B, N), dtype=torch.bool, device="cuda"), "cuda")
for method in ("qeif", "lm_plus"):
    m = _lib.METHODS[method]
    wm = int(_lib.lib.pnpb200_workspace_bytes_masked(m, 0, B, 1, 0))
    wr = int(_lib.lib.pnpb200_robust_workspace_bytes(m, 0, B, N, 1, 0))
    ws_m, ws_r = torch.empty((max(wm, 1),), dtype=torch.uint8, device="cuda"), torch.empty((wr,), dtype=torch.uint8, device="cuda")
    prm_m = pnp.default_params(workspace=ws_m.data_ptr(), workspace_bytes=wm)
    prm_r = pnp.default_params(workspace=ws_r.data_ptr(), workspace_bytes=wr)
    o = buffers()
    for f in (0.0, 0.1, 0.3):
        uv = outliers(w["uv"], f)
        for kind in ("masked", "robust"):                 # warm-up
            timed(kind, m, uv, o, words, prm_m, prm_r)
        res = {"masked": [], "robust": []}
        for _ in range(REPS):
            for kind in res:
                res[kind].append(timed(kind, m, uv, o, words, prm_m, prm_r))
        tm, tr = statistics.median(res["masked"]), statistics.median(res["robust"])
        rounds = o["rounds"].bincount(minlength=5)[1:].tolist()
        status = o["status"].bincount(minlength=3).tolist()
        print("%-8s f=%2d%% %d x %d FP64: masked solve %.3f ms | robust %.3f ms (x%.2f) | problems by solves 1..4 %s | status 0/1/2 %s "
              "| median of %d alternated calls" % (method.upper(), round(100 * f), B, N, tm, tr, tr / tm, rounds, status, REPS), flush=True)
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            call("robust", m, uv, o, words, prm_m, prm_r)
            torch.cuda.synchronize()
        ev = [(e.name, e.device_time_total / 1000.0) for e in prof.events() if e.device_time_total > 0]
        inl = [t for nme, t in ev if "k_inlier" in nme]
        comp = sum(t for nme, t in ev if any(s in nme for s in ("DeviceSelect", "DeviceCompact", "k_robust_gather", "k_robust_scatter")))
        init = sum(t for nme, t in ev if "k_robust_init" in nme)
        total = sum(t for _, t in ev)
        print("    kernels: k_inlier per round %s ms | compaction (select, gather, scatter) %.3f ms | init %.3f ms | solves %.3f ms | "
              "all kernels %.3f ms" % (" ".join("%.3f" % t for t in inl), comp, init, total - comp - init - sum(inl), total), flush=True)
