#!/usr/bin/env python
"""Developer tool: device time of the solution check (pnpb200_check_batch) on the headline workload (1 Mi problems x 68
landmarks, LM poses, FP64 and FP32) against its HBM floor, and the host entry with the check
(pnpb200_solve_check_batch_host) next to the one without (pnpb200_solve_batch_host_px), alternated in one process, with
FP64 and int16 pixels.  Prints the GPU's name and power limit first: the numbers belong to them."""
import ctypes as C
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import pnp_solver_test_b200 as pnp
from pnp_solver_test_b200 import _lib, workload as wl, patterns as pt

B, n, CHUNK = 1 << 20, 68, 1 << 17
HBM_TBS = 6.55          # streaming read rate measured on this GPU model (DESIGN.md section 6)
REPS = 50

try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=60).stdout.strip()
except (OSError, subprocess.SubprocessError) as e:
    smi = "nvidia-smi unavailable (%s)" % e
print("GPU: %s | nvidia-smi name, power limit, max SM clock: %s" % (torch.cuda.get_device_name(0), smi), flush=True)

K = pt.default_camera_matrix()
Kh = (C.c_double * 9)(*K.reshape(-1).tolist())
P = pt.pattern_array(pt.synthetic_pattern(n))
PI = C.POINTER(C.c_int32)
stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

# ---- the kernel alone
for dtype in (torch.float64, torch.float32):
    w = wl.synth_batch(0, B, P, K, dtype=dtype)
    patd = torch.from_numpy(P).to("cuda", dtype)[None].contiguous()
    o = pnp.solve_batch("lm", w["uv"], patd, K)
    status = torch.empty((B,), dtype=torch.int32, device="cuda")
    reproj = torch.empty((B, 2), dtype=dtype, device="cuda")
    dt = _lib.DTYPE_F64 if dtype == torch.float64 else _lib.DTYPE_F32

    def launch():
        rc = _lib.lib.pnpb200_check_batch(dt, B, n, _lib.ptr(patd), 1, _lib.ptr(w["uv"]), Kh, _lib.ptr(o["R"]), _lib.ptr(o["t"]),
                                          _lib.ptr(o["res_norm"]), None, 1.0, C.cast(_lib.ptr(status), PI), _lib.ptr(reproj), stream)
        _lib.check(rc, "pnpb200_check_batch")

    for _ in range(5):
        launch()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(REPS):
        launch()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / REPS
    esz = w["uv"].element_size()
    nbytes = B * (n * 2 * esz + 13 * esz + 4 + 2 * esz)    # pixel rows, R t res_norm in, status reproj out
    floor_ms = nbytes / (HBM_TBS * 1e12) * 1e3
    print("k_check_chunk<%s> %d x %d: %.4f ms per launch (%d launches after 5 warm-up; %.3f GB moved, > L2) = %.2f TB/s; "
          "HBM floor at %.2f TB/s %.4f ms = %.0f %% of it | flagged %.1f %%"
          % ("double" if esz == 8 else "float", B, n, ms, REPS, nbytes / 1e9, nbytes / (ms * 1e-3) / 1e12, HBM_TBS, floor_ms,
             100 * floor_ms / ms, 100 * float((status != 0).double().mean())), flush=True)
    del w, o, status, reproj

# ---- the host entry with and without the check, alternated
w = wl.synth_batch(0, B, P, K)
host64 = torch.empty((B, n, 2), dtype=torch.float64).pin_memory()
host64.copy_(w["uv"])
host16 = pnp.host_buffer((B, n, 2), torch.int16)
host16.copy_(host64.to(torch.int16))
del w
pat_h = torch.from_numpy(P)[None].contiguous()
outs = {"R": torch.empty((B, 3, 3), dtype=torch.float64).pin_memory(), "t": torch.empty((B, 3), dtype=torch.float64).pin_memory(),
        "euler": torch.empty((B, 3), dtype=torch.float64).pin_memory(), "res_norm": torch.empty((B,), dtype=torch.float64).pin_memory(),
        "iters": torch.empty((B,), dtype=torch.int32).pin_memory(), "best_pattern": torch.empty((B,), dtype=torch.int32).pin_memory()}
chk = dict(outs, status=torch.empty((B,), dtype=torch.int32).pin_memory(), reproj=torch.empty((B, 2), dtype=torch.float64).pin_memory())
pipe = pnp.HostPipeline(torch.float64, chunk_problems=CHUNK, n_total=n, n_patterns=1, n_streams=3)


def run(uv, checked):
    t0 = time.perf_counter()
    if checked:
        pipe.solve("lm", uv, pat_h, K, chk, check=1.0)
    else:
        pipe.solve("lm", uv, pat_h, K, outs)
    return 1e3 * (time.perf_counter() - t0)   # the call blocks until the results are in the host buffers


for name, uv in (("fp64", host64), ("int16", host16)):
    for checked in (False, True):
        run(uv, checked)
    t = {False: [], True: []}
    for _ in range(7):
        for checked in (False, True):
            t[checked].append(run(uv, checked))
    R_plain = outs["R"].clone()
    assert torch.equal(chk["R"].view(torch.int64), R_plain.view(torch.int64))
    print("host entry, %s pixels, %d x %d, %d-problem chunks, 3 streams, packing off: median of 7 alternated calls "
          "pnpb200_solve_batch_host_px %.2f ms | pnpb200_solve_check_batch_host %.2f ms (+%.2f ms) | flagged %.1f %%"
          % (name, B, n, CHUNK, statistics.median(t[False]), statistics.median(t[True]),
             statistics.median(t[True]) - statistics.median(t[False]), 100 * float((chk["status"] != 0).double().mean())), flush=True)
pipe.close()
