"""so3_project, the projection the LM and EIF2 solves end with (csrc/pnpb200_math.cuh), against an extended-precision SVD.

It returns R = U diag(1, 1, det(U V^T)) V^T, the rotation that maximises tr(R^T G), and sigma_max = ||G||_2, as
EKF2_reconstruct_R_t_m1 forms them with np.linalg.svd.  The reference is a one-sided Jacobi SVD in NumPy long double,
run to convergence.  R is unique when kappa = sigma_1 / (sigma_2 + sign(det G) sigma_3) is finite; it moves by about
eps * kappa under a perturbation of G of eps.  The kernel's quaternion comes from the adjugate of N - lambda I (N: Horn's
4 x 4 matrix), whose top three eigenvalues cluster when det G < 0 and G is nearly a scaled reflection; there its error
grows by kappa2 = sigma_1 / (sigma_1 + sign(det G) sigma_3) as well.  So R is held to eps * kappa * kappa2 where
kappa <= 1e4 (FP64) or 1e2 (FP32, where the kernel's eigenvalue estimate carries eps kappa^2).  Beyond that (nearly
rank-one G, or det G < 0 with sigma_2 ~ sigma_3), R must still be a rotation whose objective tr(R^T G) is the
reference's to rounding and to that eigenvalue gap, except within eps kappa kappa2 > 1e-3 of a scaled reflection.  Where sigma_2 + sign(det G) sigma_3 is zero to rounding the
maximiser is not unique, and such G are not among the inputs.  sigma_max is held to a few ulp everywhere.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from gpu_util import dev

pytestmark = pytest.mark.gpu
LD = np.longdouble


def _ref(G):
    """R, sigma (descending) and kappa of every G [n, 3, 3], in long double."""
    W = G.astype(LD).copy()
    n = len(W)
    V = np.broadcast_to(np.eye(3, dtype=LD), (n, 3, 3)).copy()
    for _ in range(40):
        for i, j in ((0, 1), (0, 2), (1, 2)):
            a = (W[:, :, i] ** 2).sum(1)
            b = (W[:, :, j] ** 2).sum(1)
            c = (W[:, :, i] * W[:, :, j]).sum(1)
            rot = c != 0
            cs = np.where(rot, c, LD(1))
            zeta = (b - a) / (2 * cs)
            t = np.where(zeta >= 0, 1, -1) / (np.abs(zeta) + np.sqrt(1 + zeta * zeta))
            co = np.where(rot, 1 / np.sqrt(1 + t * t), LD(1))
            si = np.where(rot, co * t, LD(0))
            for M in (W, V):
                mi, mj = M[:, :, i].copy(), M[:, :, j].copy()
                M[:, :, i] = co[:, None] * mi - si[:, None] * mj
                M[:, :, j] = si[:, None] * mi + co[:, None] * mj
    s = np.sqrt((W ** 2).sum(1))
    order = np.argsort(-s.astype(np.float64), axis=1)
    s = np.take_along_axis(s, order, 1)
    U = np.take_along_axis(W, order[:, None, :], 2) / s[:, None, :]
    V = np.take_along_axis(V, order[:, None, :], 2)
    d = np.sign(np.linalg.det(G.astype(np.float64)))
    d = np.where(d == 0, 1, d).astype(LD)
    U[:, :, 2] *= d[:, None]                               # U diag(1, 1, d) V^T, d = det(U V^T) for non-singular G
    R = U @ np.swapaxes(V, 1, 2)
    with np.errstate(divide="ignore"):
        kappa = s[:, 0] / (s[:, 1] + d * s[:, 2])
        kappa2 = s[:, 0] / (s[:, 0] + d * s[:, 2])
    return R, s, np.where(kappa > 0, kappa, np.inf), np.where(kappa2 > 0, kappa2, np.inf)


def _rot(rng, n):
    q = rng.standard_normal((n, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    w, x, y, z = q.T
    return np.stack([w * w + x * x - y * y - z * z, 2 * (x * y - w * z), 2 * (x * z + w * y),
                     2 * (x * y + w * z), w * w - x * x + y * y - z * z, 2 * (y * z - w * x),
                     2 * (x * z - w * y), 2 * (y * z + w * x), w * w - x * x - y * y + z * z], 1).reshape(n, 3, 3)


def _hard(rng):
    """Matrices U diag(s) V^T with chosen singular values (s3 < 0: det G < 0), exact rotations and the LM's final states."""
    spectra = [(1, 1, 1), (2.5, 2.5, 2.5), (3, 1, 1), (3, 1, -0.2), (1, 0.5, 0.25), (1, 0.9, -0.1),
               (1, 1 + 1e-9, 0.3), (1, 1 - 1e-12, 1 - 2e-12), (1, 1 - 1e-7, 1 - 1e-7), (1, 0.3, 0.3 - 1e-10), (1, 1, 1e-8),
               (1, 1, -1e-8), (1, 0.2, 1e-8), (1, 1e-4, 1e-4), (1, 1e-4, -1e-5), (1, 0.5, -0.5 + 1e-9), (1, 1e-8, 1e-8),
               (7e3, 3e3, 1e3), (2e-6, 1e-6, 5e-7), (9e16, 3e16, 1e14)]
    Gs = []
    for s in spectra:
        Gs.append(_rot(rng, 64) @ (np.array(s, float)[None, :, None] * _rot(rng, 64)))
    Gs.append(_rot(rng, 64))                              # exact rotations (up to rounding)
    Gs.append(np.broadcast_to(np.eye(3), (1, 3, 3)))
    Gs.append(np.diag([3.0, 2.0, 1.0])[None])
    # rotations plus noise, as the LM leaves them, and reflections plus noise (nearer to a scaled reflection than 1e-6,
    # the maximiser is all but undetermined, and the kernel's R need not be one: see so3_project)
    base = _rot(rng, 512)
    base[256:, :, 2] *= -1
    noise = 10 ** np.concatenate([rng.uniform(-9, -0.3, 256), rng.uniform(-6, -0.3, 256)])
    Gs.append(base * rng.uniform(0.2, 5, (512, 1, 1)) + rng.standard_normal((512, 3, 3)) * noise[:, None, None])
    return np.concatenate(Gs).astype(np.float64)


def _lm_final_states(n):
    from oracle import oracle as orc
    from pnp_solver_test_b200 import patterns as pt
    P = pt.pattern_array(pt.synthetic_pattern(68))
    K = pt.default_camera_matrix()
    w = orc.synth(0, n, P, K, orc.default_synth(seed=42))
    return np.stack([np.asarray(orc.solve_one("lm", P, w["uv"][b], K, want_trace=True)["trace"][-1][:9]) for b in range(n)]).reshape(n, 3, 3)


def _project(G, dtype):
    from pnp_solver_test_b200 import _lib
    tdt = torch.float64 if dtype == np.float64 else torch.float32
    g = dev(G.reshape(-1, 9), tdt)
    R, s = torch.empty_like(g), torch.empty(len(G), dtype=tdt, device="cuda")
    code = _lib.DTYPE_F64 if dtype == np.float64 else _lib.DTYPE_F32
    _lib.check(_lib.lib.pnpb200_selftest_project(code, C.c_int64(len(G)), C.c_void_p(g.data_ptr()), C.c_void_p(R.data_ptr()),
                                                 C.c_void_p(s.data_ptr()), None), "pnpb200_selftest_project")
    torch.cuda.synchronize()
    return R.cpu().numpy().astype(np.float64).reshape(-1, 3, 3), s.cpu().numpy().astype(np.float64)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_projection_matches_extended_precision_svd(dtype):
    rng = np.random.default_rng(11)
    G = np.concatenate([_hard(rng), _lm_final_states(256)]).astype(dtype)   # the reference sees the values the kernel reads
    eps = float(np.finfo(dtype).eps)
    R, smax = _project(G, dtype)
    Rr, s, kappa, kappa2 = _ref(G)
    assert np.isfinite(R).all() and np.isfinite(smax).all()
    # sigma_max to a few ulp
    ds = np.abs(smax.astype(LD) / s[:, 0] - 1).astype(np.float64)
    assert ds.max() <= 8 * eps, (ds.max() / eps, G[ds.argmax()])
    # a proper rotation
    I = np.swapaxes(R, 1, 2) @ R
    assert np.abs(I - np.eye(3)).max() <= 16 * eps
    assert np.abs(np.linalg.det(R) - 1).max() <= 16 * eps
    # the reference's rotation where it is well defined
    dR = np.abs(R.astype(LD) - Rr).reshape(len(G), -1).max(1).astype(np.float64)
    well = kappa <= (1e4 if dtype == np.float64 else 1e2)
    assert well.sum() > 0.5 * len(G)
    ratio = dR[well] / (eps * (kappa * kappa2)[well].astype(np.float64))
    assert ratio.max() <= 64, (ratio.max(), G[well][ratio.argmax()])
    # elsewhere, short of where eps kappa kappa2 leaves the adjugate no digits: the objective tr(R^T G) is the maximum, to
    # rounding and to the width 2 sigma_1 / kappa of the eigenvalue gap that leaves the maximiser undetermined
    obj = (R.astype(LD) * G.astype(LD)).sum((1, 2))
    best = (Rr * G.astype(LD)).sum((1, 2))
    some = (eps * kappa * kappa2).astype(np.float64) <= 1e-3
    assert some.sum() > 0.75 * len(G)
    assert ((best - obj) / s[:, 0] - 2 / kappa)[some].astype(np.float64).max() <= 32 * eps


def test_projection_of_exact_cases():
    """Rotations project to themselves and sigma_max of a rotation times c is |c|."""
    rng = np.random.default_rng(12)
    Q = _rot(rng, 256)
    c = rng.uniform(0.1, 10, 256)
    R, smax = _project(Q * c[:, None, None], np.float64)
    assert np.abs(R - Q).max() <= 8e-16
    assert np.abs(smax / c - 1).max() <= 1e-15
    R, smax = _project(np.diag([2.0, -3.0, 1.0])[None], np.float64)
    assert smax[0] == pytest.approx(3.0, rel=4e-16)
    assert np.abs(R[0] - np.diag([1.0, -1.0, -1.0])).max() <= 4e-16
