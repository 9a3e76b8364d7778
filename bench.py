#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric: PnP solves/sec (device-timed) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config.workload): BASELINE.json configs[1] -- 1,048,576 problems x 68-point face
pattern, LM refinement, FP64, per GPU (weak scaling: rank r owns problems [r*B, (r+1)*B) of one
global counter-based synthetic stream, so a sharded run is the slice of the unsharded one).
A "step" is one pass of the hot path over the rank's batch: pnpb200_solve_report_batch (four kernels: pattern
constants; packing, K^-1 normalisation and moments; 14 LM iterations, SO(3) projection, Euler; error report with the
point-wise residual folded in), classification, and the error statistics with their two exchanges (NCCL over NVLink;
the only inter-GPU traffic).  The K timed steps are replays of a CUDA graph of up to 20 captured steps.
Inputs are resident in HBM for `value`; `e2e` runs the same solve through the host-buffer entry
point (pinned host memory -> H2D -> solve -> D2H of all results) inside the timed region; `e2e_i16` the same
for a caller that holds its detections as int16; `extra_configs` (one GPU) times the other BASELINE configs.
--dump-outputs DIR writes what the last timed step returned (see dump_outputs): the inputs are seeded, so two builds
run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

B_PER_GPU = 1 << 20
N_POINTS = 68
METHOD = "lm"
METRIC = "pnp_solves_per_sec"
UNIT = "solves/s"


# ------------------------------------------------------------------------------------------------
# Algorithmic work per solve of the LM path as implemented (DESIGN.md "Kernels"); FMA = 2 flops.
# Moment mapping = three kernels:
#   k_stream_chunk<.,LM,0>  moments: per point 6 theta*theta^T products, bx^2+by^2, 27 FMAs, 2 adds    65 flop/pt   (HBM-bound)
#   k_iterate<.,LM>         14 x [gamma column S u of the reduced system from the constant 9x9 core (kept in shared
#                           memory), its corner u^T S u, right-hand side c - gamma S u + lambda terms 275, nine constraint
#                           rows collected per block (dots, 3 rsqrt/sqrt, 6 + 9 + 9 block entries) 344, LDL^T 10x10
#                           (165 FMA, 55 MUL, 10 reciprocals) 455, two triangular solves 190, delta back-substitution and
#                           update 46] = 14 x 1310
#                           + constant core and c, once per problem 110 + 3x3 SVD, t, Euler ~1000   (FP64 pipe)
#                           (cross-check: the SASS of one iteration is 575 DFMA + 125 DMUL + 35 DADD = 1310)
#   k_stream_chunk<.,LM,1>  residual at the state before the last update: 34 flop/pt                   (HBM-bound)
# ------------------------------------------------------------------------------------------------
def lm_flops_iterate(max_it=14):
    return max_it * (275 + 344 + 455 + 190 + 46) + 110 + 1000


def lm_flops_per_solve(n, max_it=14):
    return n * (65 + 34) + lm_flops_iterate(max_it)


# dram__bytes_read.sum + dram__bytes_write.sum of ONE k_iterate<double, LM> launch over 1,048,576 problems, from the
# committed `ncu --set full` capture (bench.py cannot run ncu on itself); algorithmic bytes are 456 per problem
# (29 moments in; state before the last update, R, t, Euler, iters, best out) = 478 MB.
NCU_TRAFFIC = {"bytes": 243.32e6 + 191.87e6, "problems": 1 << 20, "source": "profiles/r02a_n1024_fp32_ncu.md"}


def hbm_peak_gbs():
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(peaks["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return 6650.0, "fallback 6650 GB/s (B200_PROFILING.md)"


def lm_flops_survey(n, max_it=14):
    return max_it * (212 * n + 1100) + 1000        # SURVEY.md 8(d): per-iteration Jacobians, naive structure


def bytes_per_solve(n, s=8):
    return s * (2 * n + 16) + 8                    # SURVEY.md 8(d)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md).  Started
    before the warm-up (nvidia-smi takes a while to come up); rows are time-stamped on arrival and
    only those inside [mark_begin, mark_end] count (all rows under load if the region is too short)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu_index, self.rows, self.proc = gpu_index, [], None
        self.t0 = self.t1 = None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.gpu_index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))
        except Exception:
            pass

    def wait_first(self, timeout=10.0):
        t = time.perf_counter()
        while not self.rows and time.perf_counter() - t < timeout:
            time.sleep(0.05)

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        inside = [r for ts, r in self.rows if self.t0 is not None and self.t0 <= ts <= (self.t1 or 1e300)]
        scope = "timed region"
        if len(inside) < 3:
            inside, scope = [r for _, r in self.rows], "warm-up + timed region (timed region shorter than 3 samples)"
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": len(inside), "scope": scope}
        sm, reasons = [], set()
        for r in inside:
            try:
                sm.append(float(r[1]))
                out["sm_max_mhz"] = float(r[2])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        if sm:
            out["sm_mhz"] = float(np.median(sm))
            out["sm_mhz_max_seen"] = float(np.max(sm))
        out["reasons"] = sorted(reasons)
        return out


def bind_to_gpu_numa_node(local):
    """Pin this rank's threads (and with them the first-touch placement of the pinned host buffers it is
    about to allocate) to the NUMA node its GPU hangs off -- what `numactl --cpunodebind --membind` does
    in a launcher script.  Matters for the end-to-end arm at N > 1: eight ranks streaming 1 GB per step
    from host memory otherwise cross the socket interconnect.  Returns a description for the JSON line."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read().strip())
        if node < 0:
            return {"gpu": bdf, "node": node, "bound": False}
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return {"gpu": bdf, "node": node, "bound": False}
        os.sched_setaffinity(0, cpus)
        return {"gpu": bdf, "node": node, "bound": True, "cpus": len(cpus)}
    except Exception as e:                                # no sysfs, no permission: run unbound
        return {"bound": False, "why": str(e)[:80]}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's algorithm on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_rate(sample, n_threads=0, method=METHOD, n=N_POINTS, seed=42):
    from oracle import oracle as orc
    from pnp_solver_test_b200 import patterns as pt
    P = pt.pattern_array(pt.synthetic_pattern(n))
    K = pt.default_camera_matrix()
    w = orc.synth(0, sample, P, K, orc.default_synth(seed=seed))
    from pnp_solver_test_b200 import workload as wl
    edges = np.asarray(wl.CLASS_BINS["depth"], np.float64)
    t0 = time.perf_counter()
    # the same step as the GPU arm: solve, error report, statistics of the four quantities for 'all' and per depth class
    o = orc.solve_batch(method, w["uv"], P, K, n_threads=n_threads)
    rep = orc.report_batch(P, w["uv"], K, o["R"], o["t"], o["euler"], w["gt"], n_threads=n_threads)["report"]
    cls = np.digitize(w["gt"][:, 0] * 100.0, edges)
    pairs = ((rep[:, 10], rep[:, 11]), (rep[:, 12], w["gt"][:, 1]), (rep[:, 13], w["gt"][:, 2]), (rep[:, 14], w["gt"][:, 3]))
    for est, ref in pairs:
        orc.stats_of(est, ref)
        for c in np.unique(cls):
            orc.stats_of(est[cls == c], ref[cls == c])
    dt = time.perf_counter() - t0
    return sample / dt, dt


def cpu_baseline_block(target_seconds=12.0):
    from oracle import oracle as orc
    cores = orc.num_threads()
    r0, _ = cpu_rate(max(256, 64 * cores))                      # calibration
    sample = int(max(256, min(B_PER_GPU, r0 * target_seconds)))
    rate, dt = cpu_rate(sample)
    return {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "%d of the %d problems of the workload (first %d of the seeded stream), solve + report + statistics, %.1f s on %d threads; "
                      "oracle/pnp_oracle.c = C port of the reference's NumPy algorithm incl. SVD-based pinv"
                      % (sample, B_PER_GPU, sample, dt, cores)}


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return 0
    from oracle import oracle as orc
    cores = orc.num_threads()
    r0, _ = cpu_rate(max(256, 64 * cores))
    r0, _ = cpu_rate(int(max(256, r0 * 1.5)))                   # second calibration on ~1.5 s of work: thread start-up amortised
    # a step = a bounded sample of the workload: ~8 s of CPU work, less when many steps are asked for, so that
    # the K timed steps take ~90 s in all and the warm-up ~10 s whatever K and W are
    per_step = min(8.0, 90.0 / max(1, args.steps))
    sample = int(max(64, min(B_PER_GPU, r0 * per_step)))
    warm = int(max(64, min(sample, r0 * min(1.0, 10.0 / max(1, args.warmup)))))
    for _ in range(args.warmup):
        cpu_rate(warm)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_rate(sample)
    dt = time.perf_counter() - t0
    rate = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "BASELINE configs[1]: %d-point face pattern, LM refinement (14 it), FP64, random_stress_test pose "
                               "distribution, integer-quantised pixels; a step = solve + error report + statistics of a bounded sample "
                               "(%d problems) of the 1048576-problem batch" % (N_POINTS, sample),
                   "method": METHOD, "n_points": N_POINTS, "problems_per_step": sample},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d problems per step x %d steps on %d host threads, solve + report + statistics (oracle/pnp_oracle.c; "
                                   "the reference is pure Python and is not on this box)" % (sample, args.steps, cores)},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------
# The other BASELINE configs, FP32 mode and the alternative execution shapes: device-timed one by one after the
# timed region of the headline, each with the SM clock seen while it ran.
# ------------------------------------------------------------------------------------------------
def extra_configs(dev, sampler_index=0, min_ms=200.0):
    import ctypes as C
    import torch
    import pnp_solver_test_b200 as pnp
    from pnp_solver_test_b200 import _lib, workload as wl, patterns as pt

    sampler = ClockSampler(sampler_index)
    sampler.start()
    sampler.wait_first()
    K = pt.default_camera_matrix()
    hbm_peak, hbm_src = hbm_peak_gbs()

    def timed(fn, profile=False):
        """ms per call (CUDA events, >= min_ms of work after two warm-up calls), last output, per-kernel ms, clock sample"""
        for _ in range(2):
            out = fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); out = fn(); e1.record()
        torch.cuda.synchronize()
        reps = int(max(3, min(400, min_ms / max(e0.elapsed_time(e1), 1e-3))))
        if profile:
            _lib.lib.pnpb200_profile_reset()
        t0 = time.perf_counter()
        e0.record()
        for _ in range(reps):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        kms = None
        if profile:
            k3, nc = (C.c_float * 3)(), C.c_int(0)
            _lib.lib.pnpb200_profile_read(k3, C.byref(nc))
            kms = [float(k3[0]), float(k3[1]), float(k3[2])]
        rows = [r for ts, r in sampler.rows if t0 <= ts <= t1]
        sm = [float(r[1]) for r in rows if len(r) > 2 and r[1].replace(".", "").isdigit()]
        clock = {"sm_mhz": float(np.median(sm)) if sm else None, "samples": len(sm), "reps": reps}
        return e0.elapsed_time(e1) / reps, out, kms, clock

    res = {}
    B1 = 1 << 20
    # ---- configs[0]: the reference's live path (solve_pnp -> QEIF on 6 of 15 landmarks, PNP_SOLVER_LIB.py:156, :179)
    pat15 = pt.get_golden_pattern("Alexander")
    P15 = pt.pattern_array(pat15)
    idx6 = [list(pat15).index(k) for k in pt.LM_KEY_LIST_6]
    w15 = wl.synth_batch(0, B1, P15, K, device=dev)
    pat15d = torch.from_numpy(P15).to(dev)[None].contiguous()
    ms, o, _, ck = timed(lambda: pnp.solve_batch("qeif", w15["uv"], pat15d, K, point_index=idx6))

    def stress_step():
        so = wl.solve_report_batch("qeif", w15["uv"], pat15d, K, w15["gt"], point_index=idx6)
        return so, wl.error_statistics(so["report"], w15["gt"], lazy="device")
    ms_full, (so, st), _, ck2 = timed(stress_step)
    st = st.result()
    res["configs0_stress_qeif6"] = {
        "workload": "random_stress_test.py: %d problems, Alexander 15 landmarks, QEIF on the 6-key subset (the reference's live solve_pnp), quantised pixels, FP64" % B1,
        "solve_ms": ms, "solves_per_s": B1 / ms * 1e3, "mean_iters": float(o["iters"].double().mean()), "clocks": ck,
        "solve_report_statistics_ms": ms_full, "samples_per_s_incl_report_statistics": B1 / ms_full * 1e3, "clocks_full": ck2,
        "pass_rate_10cm_10deg": float(so["flags"].all(dim=1).double().mean()), "depth_MAE_cm": 100 * float(st["depth"]["all"][5]),
        "yaw_MAE_deg": float(st["yaw"]["all"][5])}

    # ---- configs[3]: n = 1024, 100 k problems: the moments and the residual passes against the measured HBM peak
    n_big, B_big = 1024, 100000
    Pb = pt.pattern_array(pt.synthetic_pattern(n_big))
    wb = wl.synth_batch(0, B_big, Pb, K, device=dev)
    patb = torch.from_numpy(Pb).to(dev)[None].contiguous()
    prof = pnp.default_params(flags=_lib.FLAG_PROFILE)
    big = {"workload": "%d problems x %d points, FP64" % (B_big, n_big), "bytes_per_solve_survey": 8 * (2 * n_big + 16) + 8,
           "hbm_peak_gbs": hbm_peak, "peak_source": hbm_src}
    for method in ("linear_f2", "lm", "qeif", "eif2"):
        ms, o, kms, ck = timed(lambda: pnp.solve_batch(method, wb["uv"], patb, K, params=prof), profile=True)
        b0 = B_big * (16 * n_big + 29 * 8)
        b2 = B_big * (16 * n_big + 12 * 8 + 8)
        big[method] = {"ms": ms, "solves_per_s": B_big / ms * 1e3, "algorithmic_gbs_whole_solve": B_big * big["bytes_per_solve_survey"] / ms / 1e6,
                       "frac_whole_solve": B_big * big["bytes_per_solve_survey"] / ms / 1e6 / hbm_peak,
                       "moments_pass": {"kernel_ms": kms[0], "achieved_gbs": b0 / kms[0] / 1e6, "frac": b0 / kms[0] / 1e6 / hbm_peak},
                       "iterate_ms": kms[1],
                       "residual_pass": {"kernel_ms": kms[2], "achieved_gbs": b2 / kms[2] / 1e6, "frac": b2 / kms[2] / 1e6 / hbm_peak},
                       "clocks": ck}
    res["configs3_n1024"] = big
    del wb

    # ---- configs[2]: FP32 against FP64 -- throughput, pipe roofline and accuracy; noise sweep 0..5 px
    n68 = N_POINTS
    P68 = pt.pattern_array(pt.synthetic_pattern(n68))
    fp = {}
    peaks = {}
    for code, name in ((0, "f64"), (1, "f32")):
        pk = C.c_double(0.0)
        _lib.lib.pnpb200_fma_peak(code, 200000, C.byref(pk))
        peaks[name] = pk.value / 1e12
    outs = {}
    for dt, name in ((torch.float64, "f64"), (torch.float32, "f32")):
        w68 = wl.synth_batch(0, B1, P68, K, dtype=dt, device=dev)
        p68 = torch.from_numpy(P68).to(dev).to(dt)[None].contiguous()
        ms, o, kms, ck = timed(lambda: pnp.solve_batch("lm", w68["uv"], p68, K, params=prof), profile=True)
        outs["lm_" + name] = o
        fp["lm68_" + name] = {"ms": ms, "solves_per_s": B1 / ms * 1e3, "kernel_ms": kms, "clocks": ck,
                              "k_iterate_tflops": lm_flops_iterate() * B1 / kms[1] / 1e9, "fma_peak_tflops": peaks[name],
                              "k_iterate_frac_of_fma_peak": lm_flops_iterate() * B1 / kms[1] / 1e9 / peaks[name]}
        w6 = wl.synth_batch(0, B1, P15, K, dtype=dt, device=dev)
        p6 = pat15d.to(dt)
        ms, o, _, ck = timed(lambda: pnp.solve_batch("qeif", w6["uv"], p6, K, point_index=idx6))
        outs["qeif_" + name] = o
        fp["qeif6_" + name] = {"ms": ms, "solves_per_s": B1 / ms * 1e3, "mean_iters": float(o["iters"].double().mean()), "clocks": ck}
    for m in ("lm", "qeif"):
        a, b = outs[m + "_f64"], outs[m + "_f32"]
        dR = (a["R"] - b["R"].double()).abs().flatten(1).max(dim=1).values
        dtt = (a["t"] - b["t"].double()).abs().max(dim=1).values / a["t"][:, 2].abs()
        ok = torch.isfinite(dR) & torch.isfinite(dtt)
        q = torch.tensor([0.5, 0.9, 0.999], dtype=torch.float64, device=dev)
        fp[m + "_f32_vs_f64"] = {"dR_median_p90_p999": [float(x) for x in torch.quantile(dR[ok][:1 << 20], q)],
                                 "dt_over_t3_median_p90_p999": [float(x) for x in torch.quantile(dtt[ok][:1 << 20], q)],
                                 "same_iteration_count_frac": float((a["iters"] == b["iters"]).double().mean())}
    del outs
    sweep = {"workload": "LM_noise_test.py: yaw 0, t = (0, 0, 1), grid 30/112 px, noise sigma x 30/112 px, %d draws per sigma, QEIF-6" % B1,
             "sigma": [], "f64_yaw_MAE_deg": [], "f32_yaw_MAE_deg": [], "f64_solves_per_s": [], "f32_solves_per_s": []}
    qg = 30.0 / 112.0
    for sg in np.linspace(0.0, 5.0, 6):
        sweep["sigma"].append(float(sg))
        for dt, name in ((torch.float64, "f64"), (torch.float32, "f32")):
            cfg = pnp.default_synth(seed=42, angle_range_deg=0.0, yaw_center_deg=0.0, depth_min_m=1.0, depth_max_m=1.0,
                                    fov_max_deg=0.0, is_quantized=1, quantize_q=qg, noise_sigma_px=float(sg) * qg)
            ws = wl.synth_batch(0, B1, P15, K, cfg=cfg, dtype=dt, device=dev)
            p6 = pat15d.to(dt)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            pnp.solve_batch("qeif", ws["uv"], p6, K, point_index=idx6)
            e0.record()
            o = pnp.solve_batch("qeif", ws["uv"], p6, K, point_index=idx6)
            e1.record()
            torch.cuda.synchronize()
            sweep[name + "_yaw_MAE_deg"].append(float(o["euler"][:, 1].double().abs().mean()))
            sweep[name + "_solves_per_s"].append(B1 / e0.elapsed_time(e1) * 1e3)
    fp["noise_sweep"] = sweep
    res["configs2_fp32_vs_fp64"] = fp

    # ---- SURVEY.md 8(f1): the filters on all 68 landmarks (moment mapping, certified exit decisions) beside LM
    w68 = wl.synth_batch(0, B1, P68, K, device=dev)
    p68 = torch.from_numpy(P68).to(dev)[None].contiguous()
    filt = {}
    for method in ("qeif", "eif2", "lm"):
        def filt_step():
            return wl.solve_report_batch(method, w68["uv"], p68, K, w68["gt"], params=prof)
        ms, so, kms, ck = timed(filt_step, profile=True)
        filt[method] = {"solve_report_ms": ms, "solves_per_s_incl_report": B1 / ms * 1e3, "kernel_ms_moments_iterate_report": kms,
                        "mean_iters": float(so["iters"].double().mean()),
                        "pass_rate_10cm_10deg": float(so["flags"].all(dim=1).double().mean()), "clocks": ck}
    res["filters_68_1Mi"] = filt

    # ---- the execution shapes head to head on the headline workload (north_star: one problem per warp; default: moments)
    shapes = {}
    for name, mp in (("MAP_MOMENT (default: moments -> O(1) iterations -> point-wise residual, one problem per thread)", _lib.MAP_MOMENT),
                     ("MAP_THREAD (one problem per thread, every iteration point-wise)", _lib.MAP_THREAD),
                     ("MAP_WARP (one problem per warp, shuffle-reduced normal equations)", _lib.MAP_WARP)):
        prm = pnp.default_params(mapping=mp)
        ms, o, _, ck = timed(lambda: pnp.solve_batch("lm", w68["uv"], p68, K, params=prm))
        shapes[name] = {"ms": ms, "solves_per_s": B1 / ms * 1e3, "clocks": ck}
    res["mappings_lm68_1Mi"] = shapes

    # ---- configs[4]: the per-GPU shard of the 64 M-problem batch on 8 GPUs (8 Mi problems, 9.1 GB of pixels)
    B8 = 1 << 23
    w8 = wl.synth_batch(0, B8, P68, K, device=dev)

    def shard_step():
        so = wl.solve_report_batch("lm", w8["uv"], p68, K, w8["gt"])
        return wl.error_statistics(so["report"], w8["gt"], lazy="device")
    ms, st, _, ck = timed(shard_step)
    res["configs4_shard_8Mi"] = {"workload": "one GPU's shard of the 64 Mi x 68-point batch over 8 GPUs: %d problems, LM FP64 + report + statistics" % B8,
                                 "ms": ms, "solves_per_s": B8 / ms * 1e3, "clocks": ck, "n_stat": float(st.result()["depth"]["all"][0])}
    sampler.stop()
    return res


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
DUMP_SAMPLE = 1 << 16


def dump_outputs(path, out, stats):
    """Write one step's results as float64 DIR/<name>.npy: every per-problem output of solve_report_batch (R, t, euler,
    res_norm, iters, report, flags, max_idx) for a fixed sample of DUMP_SAMPLE problems of the batch (seeded: the same
    problems in every run with the same --problems; all of them if the batch is smaller), their indices in
    problem_index, and the error statistics [depth, roll, pitch, yaw] x classes x STAT_KEYS of the classes that hold
    problems, listed in statistics_class (depth class 0..11, 12 = all problems; an empty class has no statistics, only
    n = 0).  21 MB at the default sizes.  The per-problem outputs are bit-identical from run to run; the statistics
    agree to rounding only (the kernels sum with FP64 atomics, whose order varies)."""
    import torch
    B = int(out["R"].shape[0])
    idx = np.arange(B) if B <= DUMP_SAMPLE else np.sort(np.random.default_rng(0).choice(B, DUMP_SAMPLE, replace=False))
    sel = torch.from_numpy(idx).to(out["R"].device)
    arrays = {"problem_index": idx}
    for k, v in out.items():
        arrays[k] = v.index_select(0, sel).cpu().numpy()
    st = np.stack([np.concatenate([stats[q]["by_depth"].numpy(), stats[q]["all"].numpy()[None]])
                   for q in ("depth", "roll", "pitch", "yaw")])
    held = st[0, :, 0] > 0                                  # the four quantities share the classes
    arrays["statistics"], arrays["statistics_class"] = st[:, held], np.flatnonzero(held)
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def _largest_divisor(k, cap):
    for d in range(min(k, cap), 0, -1):
        if k % d == 0:
            return d
    return 1


def run_ours(args):
    import ctypes as C
    import torch
    import torch.distributed as dist
    import pnp_solver_test_b200 as pnp
    from pnp_solver_test_b200 import _lib, workload as wl, patterns as pt

    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the CUDA path has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local) if not args.no_numa else {"bound": False, "why": "--no-numa"}
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, n = args.problems, N_POINTS
    K = pt.default_camera_matrix()
    P = pt.pattern_array(pt.synthetic_pattern(n))
    pat = torch.from_numpy(P).to(dev)[None].contiguous()
    params = pnp.default_params(flags=_lib.FLAG_PROFILE)      # CUDA events around each kernel of the solve

    # inputs resident in HBM: this rank's slice of the global stream
    w = wl.synth_batch(rank * B, B, P, K, cfg=pnp.default_synth(seed=42), device=dev)
    uv, gt = w["uv"], w["gt"]
    torch.cuda.synchronize()
    last = {}

    # With several ranks the statistics of a step (two small kernels, two tiny exchanges whose cost is launch latency) go
    # to a second stream: they need the step's report, but the next step's solve does not need them, so the collectives'
    # latency hides under the next solve instead of idling every GPU of the job.
    overlap = world > 1 and not args.no_overlap
    side = torch.cuda.Stream(device=dev) if overlap else None
    keep = []

    def stats_of(out):
        last["stats"] = wl.error_statistics(out["report"], gt, lazy="device")   # two kernels, two exchange phases, nothing on the host
        last["out"] = out

    def step():
        # solve (pattern constants, moments, 14 LM iterations + SO(3) projection + Euler) and the error report with the
        # residual pass folded in: one library call, four kernels
        out = wl.solve_report_batch(METHOD, uv, pat, K, gt, params=params)
        if overlap:
            cur = torch.cuda.current_stream(dev)
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                stats_of(out)
            if torch.cuda.is_current_stream_capturing():
                keep.append(out)                           # inside a capture freed blocks are reused at once: keep every step's outputs
            else:
                for v in out.values():
                    if torch.is_tensor(v):
                        v.record_stream(side)              # allocated on the solve stream, last read on the side stream
        else:
            stats_of(out)
        return out

    def join_side():
        if overlap:
            torch.cuda.current_stream(dev).wait_stream(side)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    sampler.start()
    sampler.wait_first()
    for _ in range(max(args.warmup, 0)):
        step()
    join_side()
    barrier()

    # ---- the K timed steps as replays of a CUDA graph of S steps (kernels, the side-stream fork / join and the NCCL
    # exchanges captured once): the timed region then holds no Python, no allocator and no launch latency of the host, which
    # is what separated 8 ranks sharing one host from a single rank.  Falls back to eager launches if the capture fails.
    S = _largest_divisor(args.steps, 20)
    graph, graph_note, per_graph_launches, g = None, "off (--no-graph)", 0, None
    if not args.no_graph:
        try:
            _lib.check(_lib.lib.pnpb200_profile_reset(), "pnpb200_profile_reset")
            cap_stream = torch.cuda.Stream(device=dev)
            l0 = int(_lib.lib.pnpb200_launch_count())
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=cap_stream):
                for _ in range(S):
                    step()
                join_side()
            per_graph_launches = int(_lib.lib.pnpb200_launch_count()) - l0
            g.replay()                                      # one untimed replay: graph upload, first-use costs
            torch.cuda.synchronize()
            graph, graph_note = g, "on: %d steps per graph" % S
        except Exception as e:                              # noqa: BLE001
            graph, graph_note = None, "off (capture failed: %s)" % (str(e).splitlines()[0][:120] if str(e) else type(e).__name__)
            torch.cuda.synchronize()
    g = None
    barrier()
    if world > 1:                                           # device-side rendezvous: every GPU leaves this all-reduce together, so the
        dist.all_reduce(torch.zeros(1, device=dev))         # timed region starts aligned across ranks whatever the hosts' skew
    sampler.mark_begin()
    l0 = int(_lib.lib.pnpb200_launch_count())               # kernels the library launches, counted by the library itself
    if graph is None:
        _lib.check(_lib.lib.pnpb200_profile_reset(), "pnpb200_profile_reset")
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_start.record()
    if graph is not None:
        for _ in range(args.steps // S):
            graph.replay()
    else:
        for _ in range(args.steps):
            step()
        join_side()                                         # the last steps' statistics are inside the timed region
    t_end.record()
    barrier()
    sampler.mark_end()
    if args.dump_outputs and rank == 0:                     # before anything below can run the step again
        dump_outputs(args.dump_outputs, last["out"], last["stats"].result())
    kms = (C.c_float * 3)()
    ncall = C.c_int(0)
    kernel_times = "CUDA events around each kernel inside the timed region" + \
                   (" (event-record nodes of the graph: the %d steps of its last replay)" % S if graph is not None else "")
    rc = _lib.lib.pnpb200_profile_read(kms, C.byref(ncall))
    if rc != 0 or ncall.value == 0 or not (kms[1] > 0):     # events recorded by graph nodes could not be read: time the kernels eagerly
        _lib.check(_lib.lib.pnpb200_profile_reset(), "pnpb200_profile_reset")
        for _ in range(S):
            step()
        join_side()
        torch.cuda.synchronize()
        _lib.check(_lib.lib.pnpb200_profile_read(kms, C.byref(ncall)), "pnpb200_profile_read")
        kernel_times = "CUDA events around each kernel, %d eager steps right after the timed region" % S
    launches = per_graph_launches * (args.steps // S) if graph is not None else int(_lib.lib.pnpb200_launch_count()) - l0
    clocks = sampler.stop()
    ms_total = t_start.elapsed_time(t_end)
    ms_kernel = float(kms[0]) + float(kms[1]) + float(kms[2])
    tt = torch.tensor([ms_total, ms_kernel], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_total, ms_kernel_max = float(tt[0]), float(tt[1])
    value = world * B * args.steps / (ms_total * 1e-3)
    params.flags = 0
    st = last["stats"].result()
    pass_rate = float(last["out"]["flags"].all(dim=1).double().mean())

    def timed_host(fn, k):
        """wall-clock seconds per call of fn over k calls, barrier on both sides, max over ranks"""
        barrier()
        t_ = time.perf_counter()
        for _ in range(k):
            fn()
        barrier()
        tt_ = torch.tensor([time.perf_counter() - t_], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt_, op=dist.ReduceOp.MAX)
        return float(tt_[0]) / k

    # ---- end to end through the host-buffer entry point (pinned host memory, copies timed)
    e2e = e2e_i16 = None
    if not args.no_e2e:
        host_uv = torch.empty((B, n, 2), dtype=torch.float64).pin_memory()
        host_uv.copy_(uv)
        host_pat = torch.from_numpy(P)[None].contiguous()
        outs = {"R": torch.empty((B, 3, 3), dtype=torch.float64).pin_memory(), "t": torch.empty((B, 3), dtype=torch.float64).pin_memory(),
                "euler": torch.empty((B, 3), dtype=torch.float64).pin_memory(), "res_norm": torch.empty((B,), dtype=torch.float64).pin_memory(),
                "iters": torch.empty((B,), dtype=torch.int32).pin_memory(), "best_pattern": torch.empty((B,), dtype=torch.int32).pin_memory()}
        # packed pixel transfer: the workload's pixels are whole numbers (random_stress_test.py, is_quantized=True), the
        # pipeline checks that per chunk on the host and ships such chunks as int16 (lossless), the rest as FP64
        cpus = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        pack_threads = args.pack_threads if args.pack_threads >= 0 else max(0, min(15, cpus // world - 1))
        if pack_threads < 2:
            pack_threads = 0
        pipe = pnp.HostPipeline(torch.float64, chunk_problems=args.chunk, n_total=n, n_patterns=1, n_streams=3, device=dev,
                                pack_threads=pack_threads)
        solve_host = lambda: pipe.solve(METHOD, host_uv, host_pat, K, outs)     # blocks until the results are on the host
        pack_choice = "off"
        if pack_threads:
            # warm-up decides: packing trades PCIe bytes for host memory traffic, which loses when all the ranks of a box
            # share a host memory system that is already the limit (8 GPUs); every rank takes the same decision
            timed_host(solve_host, 1)
            t_on = timed_host(solve_host, 2)
            pipe.set_packing(0)
            timed_host(solve_host, 1)
            t_off = timed_host(solve_host, 2)
            pack_choice = "on (warm-up: %.1f ms packed, %.1f ms plain)" % (1e3 * t_on, 1e3 * t_off)
            if t_on < t_off:
                pipe.set_packing(pack_threads)
            else:
                pack_choice = "off (warm-up: %.1f ms packed, %.1f ms plain)" % (1e3 * t_on, 1e3 * t_off)
                pack_threads = 0
        timed_host(solve_host, 2)
        e_steps = max(1, min(args.steps, 5))
        e2e_s = timed_host(solve_host, e_steps)
        packed_chunks, n_chunks = pipe.last_packed()
        chunk_bytes = args.chunk * n * 2 * 8
        host_bytes = host_uv.numel() * 8
        h2d = host_bytes - min(packed_chunks * chunk_bytes, host_bytes) * 3 // 4      # a packed chunk travels as int16: a quarter
        d2h = sum(v.numel() * v.element_size() for v in outs.values())
        assert torch.equal(outs["iters"], torch.full((B,), 14, dtype=torch.int32))
        ref_R = outs["R"].clone()

        # what bounds it: the same pixels copied host -> device alone by ALL ranks at once (pinned, one cudaMemcpyAsync per step)
        def copy_alone(src):
            dst = torch.empty(src.shape, dtype=src.dtype, device=dev)
            dst.copy_(src, non_blocking=True)
            barrier()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            for _ in range(3):
                dst.copy_(src, non_blocking=True)
            c1.record()
            torch.cuda.synchronize()
            t_ = torch.tensor([c0.elapsed_time(c1) / 3], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t_, op=dist.ReduceOp.MAX)
            return float(t_[0])
        copy_ms = copy_alone(host_uv)
        e2e_ms = 1e3 * e2e_s
        e2e = {"value": world * B / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "steps": e_steps, "ms_per_step": e2e_ms, "numa": numa,
               "api": "pnpb200_solve_batch_host via HostPipeline.solve (pinned FP64 host buffers, %d-problem chunks, 3 streams%s)"
                      % (args.chunk, "; packed pixel transfer with %d host threads: %d of the %d chunks of the last step were whole "
                                     "pixels packed to int16 on the host inside the timed region, lossless" % (pack_threads, packed_chunks, n_chunks)
                         if pack_threads else ""),
               "host_pixel_bytes_per_step": host_bytes, "pack_threads": pack_threads, "packed_chunks": [packed_chunks, n_chunks],
               "packing": pack_choice,
               "bound": {"what": "host->device copy of the FP64 pixels as they are, all %d rank(s) copying at the same time (max over ranks)" % world,
                         "h2d_copy_alone_ms": copy_ms, "h2d_copy_alone_gbs": host_bytes / (copy_ms * 1e-3) / 1e9,
                         "e2e_over_copy": e2e_ms / copy_ms,
                         "solves_per_s_if_copy_bound": world * B / (copy_ms * 1e-3)}}

        # ---- the same end to end for a caller that keeps its detections as int16 (what a landmark detector delivers; the
        # reference rounds its pixels itself): pnpb200_solve_batch_host_px, no host pass over the pixels at all
        pipe.set_packing(0)
        variants = {}
        for name, wc in (("pinned", False), ("write_combined", True)):
            hb = pnp.host_buffer((B, n, 2), torch.int16, write_combined=wc)
            hb.copy_(host_uv.to(torch.int16))
            fn = lambda: pipe.solve(METHOD, hb, host_pat, K, outs)
            timed_host(fn, 2)
            variants[name] = timed_host(fn, e_steps)
            assert torch.equal(outs["R"].view(torch.int64), ref_R.view(torch.int64))   # bit-identical to the FP64 hand-over
            if name == "write_combined":
                copy16_ms = copy_alone(hb)
            del hb
        best = min(variants, key=variants.get)
        e2e_i16 = {"value": world * B / variants[best], "unit": UNIT, "ms_per_step": 1e3 * variants[best], "steps": e_steps,
                   "h2d_bytes_per_step": B * n * 2 * 2, "d2h_bytes_per_step": d2h, "host_buffer": best,
                   "ms_per_step_by_host_buffer": {k: 1e3 * v for k, v in variants.items()},
                   "api": "pnpb200_solve_batch_host_px(PNPB200_PIXEL_I16) via HostPipeline.solve: int16 pixels cross PCIe as they are and are "
                          "widened on the device; results bit-identical to the FP64 hand-over (asserted)",
                   "bound": {"h2d_copy_alone_ms": copy16_ms, "h2d_copy_alone_gbs": B * n * 4 / (copy16_ms * 1e-3) / 1e9}}
        pipe.close()
        del host_uv, outs

    def leave():
        """A process group whose collectives were captured in a still-alive CUDA graph does not tear down reliably
        (observed: destroy_process_group never returned after a 2-rank graph run).  Drop the graph, let every rank
        reach this point, and leave without the destructor chain."""
        nonlocal graph
        graph = None
        keep.clear()
        sys.stdout.flush()
        try:
            torch.cuda.synchronize()
        except Exception:                                   # noqa: BLE001
            pass
        if world > 1:
            dist.barrier()
            os._exit(0)

    if rank != 0:
        leave()
        return 0

    # ---- roofline of the dominant kernel (k_iterate<double, LM>): FP64 FMA pipe
    ms_mom, ms_it, ms_res = float(kms[0]), float(kms[1]), float(kms[2])
    peak = C.c_double(0.0)
    _lib.check(_lib.lib.pnpb200_fma_peak(0, 200000, C.byref(peak)), "pnpb200_fma_peak")
    fl = lm_flops_iterate()
    achieved_tf = fl * B / (ms_it * 1e-3) / 1e12
    hbm_peak, hbm_src = hbm_peak_gbs()
    mom_bytes = (2 * n * 8 + 29 * 8) * B          # read every pixel once, write 29 moments
    rr_bytes = (2 * n * 8 + 12 * 8 + 15 * 8 + 4 * 8 + 8 + 16 * 8 + 28) * B   # pixels, state, pose, Euler, GT in; res_norm, report, flags, max_idx out
    rr_flop = (34 + 120) * n                       # residual 34 flop/pt + report ~60 FP64 instructions/pt
    roofline = {"bound": "fp64_pipe", "kernel": "k_iterate<double, LM>", "achieved": achieved_tf, "peak": peak.value / 1e12,
                "unit": "TFLOP/s", "frac": achieved_tf / (peak.value / 1e12),
                "traffic": NCU_TRAFFIC["bytes"] * B / NCU_TRAFFIC["problems"], "traffic_unit": "bytes per launch (ncu dram read + write, %s)" % NCU_TRAFFIC["source"],
                "algorithmic_bytes": 456 * B,
                "peak_source": "measured in this run by pnpb200_fma_peak (FP64 FMA microbenchmark; MEASURED_PEAKS.json has no FP64 figure)",
                "flops_per_solve": fl, "kernel_ms": ms_it, "timed_calls": int(ncall.value), "kernel_times": kernel_times,
                "solve_report_kernels_ms": ms_kernel_max, "flops_per_solve_whole_path": lm_flops_per_solve(n),
                "flops_per_solve_survey_formula": lm_flops_survey(n),
                "other_kernels": [
                    {"kernel": "k_stream_chunk<double, LM, 0> (moments)", "bound": "hbm", "kernel_ms": ms_mom,
                     "achieved": mom_bytes / (ms_mom * 1e-3) / 1e9 if ms_mom > 0 else None, "peak": hbm_peak, "unit": "GB/s",
                     "frac": (mom_bytes / (ms_mom * 1e-3) / 1e9 / hbm_peak) if ms_mom > 0 else None, "peak_source": hbm_src},
                    {"kernel": "k_report_chunk<double, 1> (error report with the LM residual pass folded in: the pixel rows are read once for both)",
                     "bound": "fp64_pipe (HBM second)", "kernel_ms": ms_res,
                     "achieved": rr_bytes / (ms_res * 1e-3) / 1e9 if ms_res > 0 else None, "peak": hbm_peak, "unit": "GB/s",
                     "frac": (rr_bytes / (ms_res * 1e-3) / 1e9 / hbm_peak) if ms_res > 0 else None, "peak_source": hbm_src,
                     "fp64_tflops_algorithmic": rr_flop * B / (ms_res * 1e-3) / 1e12 if ms_res > 0 else None}]}
    cpu = cpu_baseline_block() if (world == 1 and not args.no_cpu) else None
    # ---- the other BASELINE configs and the alternative execution shapes, outside the timed region, each device-timed.
    # Last, and fenced: nothing the headline line needs depends on it any more.
    extra = None
    if not args.no_extra and world == 1:
        try:
            extra = extra_configs(dev, sampler_index=local)
        except Exception as e:                              # noqa: BLE001
            extra = {"error": (str(e).splitlines() or [type(e).__name__])[0][:200]}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": "BASELINE configs[1]: %d problems x %d-point face pattern per GPU, LM refinement (14 it), FP64, "
                               "random_stress_test pose distribution, integer-quantised pixels" % (B, n),
                   "method": METHOD, "n_points": n, "problems_per_gpu": B, "global_problems": world * B,
                   "step": "pnpb200_solve_report_batch (pattern constants, moments, iterate, error report + residual: four kernels) + "
                           "classification + error statistics (two kernels, two exchange phases: all_reduce SUM, all_gather of the phase-2 partials)"
                           + ("; the statistics of step i run on a second stream under the solve of step i + 1, all K inside the timed region"
                              if overlap else ""),
                   "cuda_graph": graph_note,
                   "l2": "inputs are %.2f GB per step, larger than the 126 MB L2" % (uv.numel() * 8 / 1e9),
                   "parallelism": "problems sharded by global index, no solve-path traffic"},
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "e2e_i16": e2e_i16, "gpu_launches": launches, "clocks": clocks,
        "quality": {"pass_rate_10cm_10deg": pass_rate,
                    "depth_MAE_m": float(st["depth"]["all"][5]), "yaw_MAE_deg": float(st["yaw"]["all"][5]),
                    "n_stat": float(st["depth"]["all"][0])},
        "extra_configs": extra,
    }
    print(json.dumps(line), flush=True)
    leave()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--problems", type=int, default=B_PER_GPU, help="problems per GPU (default: the BASELINE config)")
    ap.add_argument("--chunk", type=int, default=1 << 17, help="e2e pipeline chunk (problems)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-overlap", action="store_true", help="N > 1: keep report + statistics on the solve stream")
    ap.add_argument("--pack-threads", type=int, default=-1,
                    help="host threads packing whole-pixel chunks to int16 for the e2e transfer (-1: cpus/ranks - 1, at most 15; 0: off)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of CUDA-graph replays")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra_configs block (other BASELINE configs, FP32, mappings)")
    ap.add_argument("--no-numa", action="store_true", help="do not bind the rank to its GPU's NUMA node")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (float64; a fixed sample of %d problems of "
                         "rank 0's batch, and the error statistics)" % DUMP_SAMPLE)
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm keeps no outputs")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
