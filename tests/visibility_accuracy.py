#!/usr/bin/env python
"""How much landmark visibility the methods tolerate (CPU only, C oracle): 8 192 problems of the random_stress_test.py
workload (seed 42, quantised noise-free pixels, 68 landmarks); per problem a uniformly drawn subset of 100 %, 75 % or 50 % of
the landmarks is visible, and each method solves the problem made of those landmarks alone -- what the masked entries of
include/pnpb200.h compute.  table() gives the share of problems that pass the 10 cm / 10 deg test of random_stress_test.py
(all four flags of the error report); the table in include/pnpb200.h is its output (python tests/visibility_accuracy.py),
and tests/test_visibility_host.py holds the two to each other."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import numpy as np

from oracle import oracle as orc
from pnp_solver_test_b200 import patterns as pt

B, N, SEED = 8192, 68, 42
FRACTIONS = (1.0, 0.75, 0.5)
METHODS = ("lm", "lm_plus", "eif2", "qeif")


def table():
    """{method: [pass rate in % at 100, 75, 50 % visible]}"""
    orc.build()
    P, K = pt.pattern_array(pt.synthetic_pattern(N)), pt.default_camera_matrix()
    w = orc.synth(0, B, P, K, cfg=orc.default_synth(seed=SEED))
    rng = np.random.default_rng(SEED)
    subsets = {f: [np.sort(rng.permutation(N)[: int(round(f * N))]) for _ in range(B)] for f in FRACTIONS}
    out = {}
    for method in METHODS:
        row = []
        for f in FRACTIONS:
            ok = 0
            for b, c in enumerate(subsets[f]):
                o = orc.solve_one(method, P[c], w["uv"][b][c], K)
                r = orc.report_batch(P[c], w["uv"][b:b + 1, c], K, o["R"][None], o["t"][None], o["euler"][None], w["gt"][b:b + 1])
                ok += int(r["flags"][0].all())
            row.append(100.0 * ok / B)
        out[method] = row
    return out


if __name__ == "__main__":
    print("%d problems, %d landmarks, seed %d, quantised pixels: 10 cm / 10 deg pass rate" % (B, N, SEED))
    print("%-8s %8s %8s %8s" % ("method", "100 %", "75 %", "50 %"))
    for m, row in table().items():
        print("%-8s %7.1f%% %7.1f%% %7.1f%%" % (m, *row), flush=True)
