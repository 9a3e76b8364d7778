#!/usr/bin/env python
"""What per-landmark weights buy (CPU only, the weighted C oracle of tests/weighted_oracle.py): 8 192 problems of the
random_stress_test.py pose distribution (seed 42, 68 landmarks).  Heteroscedastic rows: landmark i of problem b gets
sigma log-uniform on [0.5, 8] px, N(0, sigma^2) noise per coordinate, then whole pixels; weights float32((3 px / sigma)^2).
Homoscedastic control: sigma = 2 px everywhere, every weight 2.25 -- what the absolute scale of the weights alone does.
For each method, unweighted against weighted: the 10 cm / 10 deg pass rate of random_stress_test.py, the median and 95th
percentile of max |d roll, d pitch, d yaw| (deg) and of |d depth| (cm).  The table in include/pnpb200.h is its output
(python tests/weights_accuracy.py), and tests/test_weights_host.py holds the two to each other."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.dirname(os.path.abspath(__file__))):
    if p not in sys.path:
        sys.path.insert(0, p)
import numpy as np

import weighted_oracle as wo
from oracle import oracle as orc
from pnp_solver_test_b200 import patterns as pt

B, N, SEED = 8192, 68, 42
METHODS = ("lm", "lm_plus", "qeif", "eif2")
ROWS = ("hetero", "homo")


def workload(row):
    P, K = pt.pattern_array(pt.synthetic_pattern(N)), pt.default_camera_matrix()
    w = orc.synth(0, B, P, K, cfg=orc.default_synth(seed=SEED, is_quantized=False))
    rng = np.random.default_rng(SEED + (0 if row == "hetero" else 1))
    sigma = np.exp(rng.uniform(np.log(0.5), np.log(8.0), size=(B, N))) if row == "hetero" else np.full((B, N), 2.0)
    uv = np.rint(w["uv"] + rng.standard_normal((B, N, 2)) * sigma[..., None])
    wts = ((3.0 / sigma) ** 2).astype(np.float32).astype(np.float64)
    return P, K, uv, w["gt"], wts


def stats(P, K, uv, gt, o):
    r = orc.report_batch(P, uv, K, o["R"], o["t"], o["euler"], gt)
    ang = np.abs(r["report"][:, 1:4]).max(axis=1)
    dep = np.abs(r["report"][:, 0]) * 100.0
    ang, dep = np.where(np.isfinite(ang), ang, np.inf), np.where(np.isfinite(dep), dep, np.inf)
    return [100.0 * r["flags"].all(axis=1).mean(), np.median(ang), np.percentile(ang, 95), np.median(dep), np.percentile(dep, 95)]


def table():
    """{(row, method): (unweighted stats, weighted stats)}, stats = [pass %, angle median, angle p95, depth median, depth p95]"""
    orc.build()
    out = {}
    for row in ROWS:
        P, K, uv, gt, wts = workload(row)
        for m in METHODS:
            out[(row, m)] = (stats(P, K, uv, gt, orc.solve_batch(m, uv, P, K)), stats(P, K, uv, gt, wo.solve_batch(m, uv, P, K, wts)))
    return out


def lines(tab):
    names = {"lm": "LM", "lm_plus": "LM+", "qeif": "QEIF", "eif2": "EIF2"}
    res = []
    for (row, m), (u, w) in tab.items():
        res.append("%-6s %-5s %5.1f %% -> %5.1f %% | %6.2f %7.2f -> %6.2f %7.2f | %6.2f %7.2f -> %6.2f %7.2f" % (
            row, names[m], u[0], w[0], u[1], u[2], w[1], w[2], u[3], u[4], w[3], w[4]))
    return res


if __name__ == "__main__":
    print("row    method pass unweighted -> weighted | max|d angle| deg median p95 -> ... | |d depth| cm median p95 -> ...")
    for line in lines(table()):
        print(line, flush=True)
