#!/usr/bin/env python
"""What the RANSAC solve rescues (CPU only, C oracle): the counterpart of tests/outlier_accuracy.py on its 8 192 problems (seed
42, 68 landmarks, whole pixels), with a 50 % far-outlier row added.  ransac_one() restates pnpb200_solve_ransac_batch: the
hypothesis stage restated in C (ransac_oracle.hypothesize_one, the rule of pnpb200_hypothesize_batch) gives M0, then the loop of
outlier_accuracy.robust_one runs from M0.  run() gives the 10 cm / 10 deg pass rate plain -> robust -> RANSAC, and the RANSAC
pass rate for each consensus_px in SWEEP, from which best_px() picks the default.  The tables in include/pnpb200.h are its output
(python tests/ransac_accuracy.py), and tests/test_ransac_host.py holds the two to each other."""
import multiprocessing
import os
import sys
from concurrent.futures import ProcessPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.dirname(os.path.abspath(__file__))):
    if p not in sys.path:
        sys.path.insert(0, p)
import numpy as np

import outlier_accuracy as oa
import ransac_oracle as ro
from oracle import oracle as orc
from pnp_solver_test_b200 import patterns as pt

B, N, SEED = oa.B, oa.N, oa.SEED
SETTINGS = oa.SETTINGS + ((0.5, 30.0, 150.0),)
METHODS = oa.METHODS
SWEEP = (2.0, 4.0, 8.0)
SWEEP_SETTINGS = ((0.0, 0.0, 0.0), (0.3, 30.0, 150.0), (0.5, 30.0, 150.0))
DEFAULT_PX = 4.0


def robust_from(method, patterns, uv, K, cand, mask0, max_rounds=4, k=3.0, floor_px=2.0, min_inliers=6):
    """outlier_accuracy.robust_one started from the mask mask0 (a subset of cand) instead of cand"""
    mask = list(mask0)
    o, p = oa.solve_on(method, patterns, uv, K, mask)
    rounds, status = 1, 0
    for r in range(max_rounds):
        d = oa.distances(patterns[p][cand], uv[cand], K, o["R"], o["t"]) if len(cand) else np.zeros(0)
        med = np.sort(d)[(len(d) - 1) // 2] if len(d) else np.nan
        s = k * med
        tau = s if (np.isfinite(s) and s > floor_px) else floor_px
        new = [j for j, dj in zip(cand, d) if dj <= tau]
        if set(new) == set(mask):
            break
        if len(new) < min_inliers:
            status = oa.TOO_FEW
            break
        if r + 1 == max_rounds:
            status = oa.NOT_CONVERGED
            break
        mask = new
        o, p = oa.solve_on(method, patterns, uv, K, mask)
        rounds += 1
    return o, p, mask, rounds, status


def ransac_one(method, patterns, uv, K, cand, g, consensus_px=DEFAULT_PX, samples=128, confidence=0.999, seed=0, min_inliers=6):
    """the rule of pnpb200_solve_ransac_batch for one problem (g = its global index): (solve output, pattern, inliers, rounds,
    status, hypothesis stage's dict)"""
    h = ro.hypothesize_one(uv, patterns, K, cand, g, samples=samples, consensus_px=consensus_px, confidence=confidence, seed=seed)
    mask0 = [j for j in cand if h["mask"][j]] if h["consensus"] >= min_inliers else list(cand)
    return robust_from(method, patterns, uv, K, cand, mask0, min_inliers=min_inliers) + (h,)


def _chunk(args):
    method, setting, b0, b1, pxs = args
    P, K = pt.pattern_array(pt.synthetic_pattern(N)), pt.default_camera_matrix()
    w = orc.synth(0, B, P, K, cfg=orc.default_synth(seed=SEED))
    uv = oa.add_outliers(w["uv"], *setting, SEED)[b0:b1]
    outs = [[], []] + [[] for _ in pxs]
    for b in range(b1 - b0):
        outs[0].append(oa.solve_on(method, P[None], uv[b], K, list(range(N)))[0])
        outs[1].append(oa.robust_one(method, P[None], uv[b], K, list(range(N)))[0])
        for q, px in enumerate(pxs):
            outs[2 + q].append(ransac_one(method, P[None], uv[b], K, list(range(N)), b0 + b, consensus_px=px)[0])
    ok = []
    for o in outs:
        R = np.stack([x["R"] for x in o]); t = np.stack([x["t"] for x in o]); e = np.stack([x["euler"] for x in o])
        r = orc.report_batch(P, w["uv"][b0:b1], K, R, t, e, w["gt"][b0:b1])
        ok.append(int(r["flags"].all(axis=1).sum()))
    return ok


def run(n_workers=None):
    """(table, sweep): table {method: [(plain %, robust %, RANSAC %) per setting]} at DEFAULT_PX; sweep {method: {setting:
    [RANSAC % per consensus_px in SWEEP]}}"""
    orc.build()
    ro.build()
    step = 512
    jobs = [(m, s, b0, min(B, b0 + step), SWEEP if s in SWEEP_SETTINGS else (DEFAULT_PX,))
            for m in METHODS for s in SETTINGS for b0 in range(0, B, step)]
    with ProcessPoolExecutor(max_workers=n_workers or min(16, os.cpu_count() or 1), mp_context=multiprocessing.get_context("spawn")) as ex:
        res = list(ex.map(_chunk, jobs))
    tab, sw = {}, {}
    for m in METHODS:
        tab[m], sw[m] = [], {}
        for s in SETTINGS:
            hits = np.array([r for j, r in zip(jobs, res) if j[0] == m and j[1] == s]).sum(axis=0) * 100.0 / B
            pxs = SWEEP if s in SWEEP_SETTINGS else (DEFAULT_PX,)
            tab[m].append((hits[0], hits[1], hits[2 + pxs.index(DEFAULT_PX)]))
            if s in SWEEP_SETTINGS:
                sw[m][s] = list(hits[2:])
    return tab, sw


def best_px(sw):
    """the smallest consensus_px of the sweep whose pass rate is within 0.1 point of the sweep's best in every cell: a tighter
    threshold keeps near outliers (the 5-30 px rows) out of the consensus set"""
    cells = np.array([[sw[m][s][q] for m in METHODS for s in SWEEP_SETTINGS] for q in range(len(SWEEP))])
    ok = (cells >= cells.max(axis=0) - 0.1).all(axis=1)
    return SWEEP[int(np.flatnonzero(ok)[0])]


def _band(f, a, b):
    return "-" if f == 0 else "%d-%d px" % (a, b)


def header_lines(tab, sw):
    """the two tables as include/pnpb200.h prints them"""
    lines = []
    for i, (f, a, b) in enumerate(SETTINGS):
        cells = "  ".join("%5.1f %5.1f %5.1f" % tab[m][i] for m in METHODS)
        lines.append(" *   %-9s %3d %%   %s" % (_band(f, a, b), int(round(100 * f)), cells))
    for q, px in enumerate(SWEEP):
        cells = "   ".join("%5.1f %5.1f %5.1f" % tuple(sw[m][s][q] for s in SWEEP_SETTINGS) for m in METHODS)
        lines.append(" *   %3.0f px          %s" % (px, cells))
    return lines


if __name__ == "__main__":
    tab, sw = run()
    print("%d problems, %d landmarks, seed %d, whole pixels; 10 cm / 10 deg pass rate, plain  robust  RANSAC (defaults)" % (B, N, SEED))
    print(" *   moved by    f      " + "  ".join("%-17s" % m for m in ("LM+", "QEIF", "EIF2")))
    lines = header_lines(tab, sw)
    for line in lines[:len(SETTINGS)]:
        print(line)
    print("RANSAC pass rate by consensus_px; per method: clean, 30 % and 50 % moved by 30-150 px")
    for line in lines[len(SETTINGS):]:
        print(line)
    print("best consensus_px: %.0f" % best_px(sw), flush=True)
