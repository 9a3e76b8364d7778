#!/usr/bin/env python
"""What the outlier-robust solve rescues (CPU only, C oracle).  8 192 problems of the random_stress_test.py workload (seed 42,
68 landmarks, whole-pixel detections); in each problem a random f % of the landmarks are moved by U(a, b) px in a random
direction and rounded to whole pixels again.  robust_one() restates the rule of pnpb200_solve_robust_batch (include/pnpb200.h)
in NumPy over orc.solve_one on the compacted problems; table() gives the share of problems that pass the 10 cm / 10 deg test of
random_stress_test.py, plain (the round-0 solve) and robust.  The table in include/pnpb200.h is its output
(python tests/outlier_accuracy.py), and tests/test_robust_host.py holds the two to each other."""
import multiprocessing
import os
import sys
from concurrent.futures import ProcessPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import numpy as np

from oracle import oracle as orc
from pnp_solver_test_b200 import patterns as pt

B, N, SEED = 8192, 68, 42
SETTINGS = ((0.0, 0.0, 0.0), (0.1, 5.0, 30.0), (0.3, 5.0, 30.0), (0.1, 30.0, 150.0), (0.3, 30.0, 150.0))   # (f, a, b)
METHODS = ("lm_plus", "qeif", "eif2")
TOO_FEW, NOT_CONVERGED = 1, 2


def add_outliers(uv, f, a, b, seed):
    """a copy of uv [B, n, 2] with round(f n) landmarks per problem moved by U(a, b) px in a random direction, rounded"""
    out = np.array(uv, dtype=np.float64)
    Bn, n = out.shape[0], out.shape[1]
    k = int(round(f * n))
    if k == 0:
        return out
    rng = np.random.default_rng([seed, int(round(1000 * f)), int(a), int(b)])
    idx = np.argsort(rng.random((Bn, n)), axis=1)[:, :k]
    r = rng.uniform(a, b, (Bn, k))
    th = rng.uniform(0.0, 2.0 * np.pi, (Bn, k))
    rows = np.arange(Bn)[:, None]
    out[rows, idx, 0] += r * np.cos(th)
    out[rows, idx, 1] += r * np.sin(th)
    return np.around(out)


def distances(P, uv, K, R, t):
    """the check's prediction-vs-landmark distance of every landmark (pnpb200_check_batch; FP64, without its FMAs)"""
    M, m = K @ R, K @ t
    r = P @ M.T + m
    with np.errstate(all="ignore"):
        inv = np.abs(1.0 / r[:, 2])
        dx, dy = r[:, 0] * inv - uv[:, 0], r[:, 1] * inv - uv[:, 1]
        return np.sqrt(dx * dx + dy * dy + np.where(np.signbit(r[:, 2]), 4.0, 0.0))


def solve_on(method, patterns, uv, K, land):
    """the masked solve of one problem on the landmarks `land` (in solver order): strict-< arg-min over the patterns"""
    if len(land) < 4:
        nan = np.full(3, np.nan)
        return dict(R=np.full((3, 3), np.nan), t=nan, euler=nan, res_norm=np.nan, iters=0), 0
    best = None
    for p in range(patterns.shape[0]):
        o = orc.solve_one(method, patterns[p][land], uv[land], K)
        if best is None or o["res_norm"] < best[0]["res_norm"]:
            best = (o, p)
    return best


def robust_one(method, patterns, uv, K, cand, max_rounds=4, k=3.0, floor_px=2.0, min_inliers=6):
    """the rule for one problem: cand = its candidates in solver order.  Returns (solve output, best pattern, inliers,
    rounds, status, near): near = some distance lay within 1e-9 relative of a threshold (FMA rounding may flip it)"""
    mask = list(cand)
    o, p = solve_on(method, patterns, uv, K, mask)
    rounds, status, near = 1, 0, False
    for r in range(max_rounds):
        d = distances(patterns[p][cand], uv[cand], K, o["R"], o["t"]) if len(cand) else np.zeros(0)
        med = np.sort(d)[(len(d) - 1) // 2] if len(d) else np.nan      # (np.sort puts NaN last)
        s = k * med
        tau = s if (np.isfinite(s) and s > floor_px) else floor_px
        near |= bool(np.any(np.abs(d - tau) <= 1e-9 * max(tau, 1e-300))) or (np.isfinite(s) and abs(s - floor_px) <= 1e-9 * floor_px)
        new = [j for j, dj in zip(cand, d) if dj <= tau]
        if set(new) == set(mask):
            break
        if len(new) < min_inliers:
            status = TOO_FEW
            break
        if r + 1 == max_rounds:
            status = NOT_CONVERGED
            break
        mask = new
        o, p = solve_on(method, patterns, uv, K, mask)
        rounds += 1
    return o, p, mask, rounds, status, near


def _chunk(args):
    method, setting, b0, b1 = args
    P, K = pt.pattern_array(pt.synthetic_pattern(N)), pt.default_camera_matrix()
    w = orc.synth(0, B, P, K, cfg=orc.default_synth(seed=SEED))
    uv = add_outliers(w["uv"], *setting, SEED)[b0:b1]
    plain, robust = [], []
    for b in range(b1 - b0):
        o0, _ = solve_on(method, P[None], uv[b], K, list(range(N)))
        o, _, _, _, _, _ = robust_one(method, P[None], uv[b], K, list(range(N)))
        plain.append(o0)
        robust.append(o)
    ok = []
    for outs in (plain, robust):
        R = np.stack([x["R"] for x in outs]); t = np.stack([x["t"] for x in outs]); e = np.stack([x["euler"] for x in outs])
        r = orc.report_batch(P, w["uv"][b0:b1], K, R, t, e, w["gt"][b0:b1])
        ok.append(int(r["flags"].all(axis=1).sum()))
    return ok


def table(n_workers=None):
    """{method: [(plain %, robust %) per setting]}"""
    orc.build()
    step = 512
    jobs = [(m, s, b0, min(B, b0 + step)) for m in METHODS for s in SETTINGS for b0 in range(0, B, step)]
    # spawned workers: the caller (a test run) may hold threads, which a fork would copy half-way
    with ProcessPoolExecutor(max_workers=n_workers or min(16, os.cpu_count() or 1), mp_context=multiprocessing.get_context("spawn")) as ex:
        res = list(ex.map(_chunk, jobs))
    out = {}
    for m in METHODS:
        row = []
        for s in SETTINGS:
            hits = [r for j, r in zip(jobs, res) if j[0] == m and j[1] == s]
            row.append((100.0 * sum(h[0] for h in hits) / B, 100.0 * sum(h[1] for h in hits) / B))
        out[m] = row
    return out


def header_lines(tab):
    """the table as include/pnpb200.h prints it"""
    lines = []
    for (f, a, b), i in zip(SETTINGS, range(len(SETTINGS))):
        band = "-" if f == 0 else "%d-%d px" % (a, b)
        cells = "  ".join("%5.1f -> %5.1f" % tab[m][i] for m in METHODS)
        lines.append(" *   %-9s %3d %%   %s" % (band, int(round(100 * f)), cells))
    return lines


if __name__ == "__main__":
    print("%d problems, %d landmarks, seed %d, whole pixels; 10 cm / 10 deg pass rate, plain -> robust (defaults)" % (B, N, SEED))
    print(" *   moved by    f      " + "  ".join("%-14s" % m for m in ("LM+", "QEIF", "EIF2")))
    for line in header_lines(table()):
        print(line, flush=True)
