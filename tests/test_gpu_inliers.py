"""The inlier classification of the robust and RANSAC solves (k_inlier_chunk, k_inlier_warp in csrc/pnpb200_robust.cu) against
an extended-precision restatement of the rule of include/pnpb200.h, through the test hook pnpb200_selftest_inliers:
  a. exact geometry (every distance exact in FP64): tau, mask, flag, status and rounds bit for bit, on both kernel shapes;
  b. realistic poses on the synthetic workload: the shapes agree bit for bit, tau within a derived error bound, the decision
     equal but for landmarks within that bound of tau;
  c. invariants of the robust and RANSAC entries that hold for every problem whatever the solver does."""
import ctypes as C

import numpy as np
import pytest
import torch

import outlier_accuracy as oa
from oracle import oracle as orc
from pnp_solver_test_b200 import patterns as pt

from gpu_util import dev, to_np

pytestmark = pytest.mark.gpu

TOO_FEW, NOT_CONVERGED = 1, 2
L = np.longdouble
U = 2.0 ** -53                                      # unit roundoff of FP64: the kernels compute in FP64 for both dtypes


# ------------------------------------------------------------------------------------------------------------------------------
# the reference
# ------------------------------------------------------------------------------------------------------------------------------
def distances(P, uv, K, R, t, best, cand):
    """d [B, n] (np.longdouble; NaN outside C) of every candidate from the exact inputs (P [n_patterns, n, 3], uv [B, n, 2], R
    [B, 3, 3], t [B, 3] in the call's dtype, K FP64), widened as the kernels widen them: the projection through K R and K t,
    division by |z|, +4 under the root where z < 0.  The kernels' FP64 distance is never infinite: where its square is not
    finite (z = 0, a non-finite pixel, an overflow) it is NaN, and so it is here.  Also returns the parts the error bound
    needs: the predicted pixel p [B, n, 2], z [B, n] and A [B, n, 3] = |K| |R| |X| + |K| |t|."""
    Kl, Rl, tl = np.asarray(K, L), np.asarray(R, L), np.asarray(t, L)
    X = np.asarray(P, L)[np.asarray(best)]                              # [B, n, 3]
    M, m = np.einsum("ij,bjk->bik", Kl, Rl), np.einsum("ij,bj->bi", Kl, tl)
    r = np.einsum("bij,bnj->bni", M, X) + m[:, None, :]
    A = np.einsum("bij,bnj->bni", np.einsum("ij,bjk->bik", np.abs(Kl), np.abs(Rl)), np.abs(X)) + \
        np.einsum("ij,bj->bi", np.abs(Kl), np.abs(tl))[:, None, :]
    z = r[..., 2]
    uvl = np.asarray(uv, L)
    with np.errstate(all="ignore"):
        p = r[..., :2] / np.abs(z)[..., None]
        dx, dy = p[..., 0] - uvl[..., 0], p[..., 1] - uvl[..., 1]
        d2 = dx * dx + dy * dy + np.where(np.signbit(z), L(4), L(0))
        d = np.sqrt(d2)
        d[~np.isfinite(d2.astype(np.float64)) | (z == 0)] = np.nan
    d[~cand] = np.nan
    return d, p, z, A


def rule(d, cand, k, floor_px):
    """tau [B] and M' [B, n] of the header's rule over the candidates: the lower median of rank floor((c - 1) / 2) with NaN
    last, tau = max(floor_px, k med) (floor_px where k med is not finite in FP64), M' = {i in C : d_i <= tau}"""
    d = np.where(cand, np.asarray(d, L), L(np.nan))
    B = d.shape[0]
    c = cand.sum(1)
    srt = np.sort(d, axis=1)                                            # NaN last
    med = srt[np.arange(B), np.maximum(c - 1, 0) // 2] if d.shape[1] else np.full(B, L(np.nan))
    med = np.where(c > 0, med, L(np.nan))
    with np.errstate(all="ignore"):
        s = L(k) * med
        use = np.isfinite(s.astype(np.float64)) & (s > L(floor_px))
    tau = np.where(use, s, L(floor_px))
    with np.errstate(invalid="ignore"):
        new = cand & (d <= tau[:, None])
    return tau, new


def decide(new, mask, rounds, status, min_inliers, last_round):
    """the decision on M' against the problem's mask M: (flag, mask, rounds, status) after the pass"""
    same = (new == mask).all(1)
    few = ~same & (new.sum(1) < min_inliers)
    nc = ~same & ~few & bool(last_round)
    acc = ~same & ~few & (not last_round)
    status = np.where(few, TOO_FEW, np.where(nc, NOT_CONVERGED, status))
    return acc.astype(np.uint8), np.where(acc[:, None], new, mask), rounds + acc, status


def distance_bound(d, p, z, A):
    """an upper bound of |d_kernel - d| per landmark: K R and K t folded with <= 2 roundings per entry, each coordinate of the
    projection three FMAs (<= 3 roundings of terms bounded by A), 1 / z within 0.5003 ulp, the division and the difference one
    FMA, the sum of squares two FMAs and the root <= 1 ulp; each step's relative error is at most a few u, and 8 u covers
    their sum with margin.  |dp| <= 8 u ((A_x + |p_x| A_z) / |z| + |p_x|), |dd| <= |dp_u| + |dp_v| + 8 u d."""
    with np.errstate(all="ignore"):
        az = np.abs(z)
        e = 8 * U * ((A[..., 0] + A[..., 1] + (np.abs(p[..., 0]) + np.abs(p[..., 1])) * A[..., 2]) / az +
                     np.abs(p[..., 0]) + np.abs(p[..., 1]) + np.nan_to_num(d, nan=0.0))
    return e.astype(np.float64)


# ------------------------------------------------------------------------------------------------------------------------------
# the hook
# ------------------------------------------------------------------------------------------------------------------------------
def _words(mask):
    """bool [B, n] -> uint32 words [B, W] (bit i % 32 of word i / 32)"""
    B, n = mask.shape
    W = (n + 31) // 32
    v = np.zeros((B, W * 32), bool)
    v[:, :n] = mask
    return np.packbits(v.reshape(B, W, 4, 8), axis=-1, bitorder="little").reshape(B, W * 4).view("<u4").copy()


def _unwords(words, n):
    return np.unpackbits(np.ascontiguousarray(words).view(np.uint8).reshape(len(words), -1), axis=1, bitorder="little")[:, :n].astype(bool)


def hook(dtype, uv, P, K, R, t, best, point_index=None, visible=None, k=3.0, floor_px=2.0, min_inliers=6, idx=None,
         last_round=0, inliers=None, rounds=None, status=None, shape=0):
    """pnpb200_selftest_inliers on NumPy inputs: returns (rc, dict(inliers bool, rounds, status over the problem rows, flag,
    tau over the batch))"""
    from pnp_solver_test_b200 import _lib
    td = torch.float64 if dtype == np.float64 else torch.float32
    B, n_total = uv.shape[0], uv.shape[1]
    sel = None if point_index is None else np.ascontiguousarray(point_index, np.int32)
    n = n_total if sel is None else len(sel)
    g = dict(uv=dev(uv, td), P=dev(P, td), R=dev(R, td), t=dev(t, td))
    best_d = None if best is None else torch.from_numpy(np.ascontiguousarray(best, np.int32)).cuda()
    idx_d = None if idx is None else torch.from_numpy(np.ascontiguousarray(idx, np.int32)).cuda()
    vis_d = None if visible is None else torch.from_numpy(_words(visible).view(np.int32)).cuda()
    inl = torch.from_numpy(_words(inliers).view(np.int32)).cuda()
    rnd = torch.from_numpy(np.ascontiguousarray(rounds, np.int32)).cuda()
    sts = torch.from_numpy(np.ascontiguousarray(status, np.int32)).cuda()
    flag = torch.full((B,), 7, dtype=torch.uint8, device="cuda")
    tau = torch.full((B,), -1.0, dtype=torch.float64, device="cuda")
    Kh = np.ascontiguousarray(K, np.float64)
    rp = _lib.RobustParams(max_rounds=4, k_median=k, floor_px=floor_px, min_inliers=min_inliers)
    vp = lambda x: None if x is None else C.c_void_p(x.data_ptr())
    PI, PU = C.POINTER(C.c_int32), C.POINTER(C.c_uint32)
    rc = _lib.lib.pnpb200_selftest_inliers(
        0 if dtype == np.float64 else 1, B, n_total, n, vp(g["uv"]), vp(g["P"]), int(P.shape[0]),
        None if sel is None else sel.ctypes.data_as(PI), Kh.ctypes.data_as(C.POINTER(C.c_double)),
        None if vis_d is None else C.cast(vp(vis_d), PU), C.byref(rp), vp(g["R"]), vp(g["t"]),
        None if best_d is None else C.cast(vp(best_d), PI), None if idx_d is None else C.cast(vp(idx_d), PI), last_round,
        C.cast(vp(inl), PU), C.cast(vp(rnd), PI), C.cast(vp(sts), PI), vp(flag), C.cast(vp(tau), C.POINTER(C.c_double)), shape, None)
    torch.cuda.synchronize()
    return rc, dict(inliers=_unwords(inl.cpu().numpy(), n_total), rounds=rnd.cpu().numpy(), status=sts.cpu().numpy(),
                    flag=flag.cpu().numpy(), tau=tau.cpu().numpy())


def _same(a, b):
    for key in ("inliers", "rounds", "status", "flag", "tau"):
        assert a[key].tobytes() == b[key].tobytes(), key


# the kernel shapes the dispatcher picks (inlier_launch): the streaming kernel where report_can_fuse holds -- the row tile of
# 32 problems (row_geometry: the row padded to an odd number of 16-byte units) fits 48 KiB and rows stream in whole 16-byte
# units (stream_geometry) -- and one warp per problem otherwise
def _streams(dtype, n):
    esz = 8 if dtype == np.float64 else 4
    units = (n * 2 * esz + 15) // 16
    units += 1 - (units & 1)
    return 32 * units * 16 <= 48 * 1024 and n % (16 // (2 * esz)) == 0


def test_shape_boundaries_are_those_of_the_issue_lists():
    """the n values below sit on both sides of the streaming kernel's limit"""
    assert max(n for n in range(1, 400) if _streams(np.float64, n)) == 95
    assert max(n for n in range(1, 400) if _streams(np.float32, n)) == 190
    assert not _streams(np.float32, 15) and _streams(np.float32, 16) and not _streams(np.float32, 192)


# ------------------------------------------------------------------------------------------------------------------------------
# a. exact geometry
# ------------------------------------------------------------------------------------------------------------------------------
F, CX, CY = 256.0, 160.0, 128.0
K_EXACT = np.array([[F, 0.0, CX], [0.0, F, CY], [0.0, 0.0, 1.0]])
Q = 0.625                                            # the distance unit: 5/8, so (3/8, 4/8) is a 3-4-5 offset
DIRS = np.array([[1.0, 0.0], [0.0, -1.0], [0.6, 0.8], [-0.8, 0.6]])
# behind the camera the distance is sqrt(e^2 + 4): pixel offsets e with an exact root, (e, root) = (b, 2 + b) scaled by 2^-s...
BEHIND = np.array([[0.0, 2.0], [1.5, 2.5], [3.75, 4.25], [7.875, 8.125], [15.9375, 16.0625]])


def _exact_patterns(n):
    """pattern 0: (x, y, 0) on a dyadic grid; pattern 1: the same with landmarks 1, 4, 7, ... behind the camera (z = -2 with
    t = (0, 0, 1): depth -1) and landmark 2 at depth 0 exactly"""
    j = np.arange(n)
    P0 = np.stack([(j % 8) / 16.0 - 0.25, (j // 8) / 32.0 - 0.125, np.zeros(n)], 1)
    P1 = P0.copy()
    P1[1::3, 2] = -2.0
    if n > 2:
        P1[2, 2] = -1.0
    return np.stack([P0, P1])


def _exact_rows(n, rng):
    """rows of (candidates, distance targets, pattern, pixel overrides): ladders in four orders for every c, and edge rows"""
    rows = []
    for order in ("asc", "desc", "rand", "organ"):
        for c in range(n + 1):
            cand = np.zeros(n, bool)
            cand[rng.permutation(n)[:c]] = True
            lad = Q * np.arange(1, c + 1)
            if order == "desc":
                lad = lad[::-1]
            elif order == "rand":
                lad = rng.permutation(lad)
            elif order == "organ":
                lad = np.concatenate([lad[0::2], lad[1::2][::-1]])
            d = np.zeros(n)
            d[cand] = lad
            rows.append((cand, d, 0, {}))
    full = np.ones(n, bool)
    rows.append((full, np.full(n, 5 * Q), 0, {}))                                   # all equal
    m = (n - 1) // 2
    d = Q * np.arange(1, n + 1, dtype=float)
    d[m - 2:m + 3] = d[m]                                                           # duplicates straddling the median
    rows.append((full, rng.permutation(d), 0, {}))
    for h in (n // 2 - 1, n // 2, n // 2 + 1, n - (n - 1) // 2, n - (n - 1) // 2 - 1):     # NaN pixels around half of C
        over = {int(i): (np.nan, 0.0) for i in rng.permutation(n)[:max(h, 0)]}
        rows.append((full, rng.permutation(Q * np.arange(1, n + 1, dtype=float)), 0, over))
    rows.append((full, Q * np.arange(1, n + 1, dtype=float), 0, {0: (np.inf, 0.0), 3: (0.0, -np.inf)}))   # infinite pixels
    for pat_rows in range(3):                                                       # behind the camera, depth 0 (pattern 1)
        rows.append((full, rng.permutation(Q * np.arange(1, n + 1, dtype=float)) * (pat_rows + 1), 1, {}))
    rows.append((full, np.zeros(n), 1, {}))
    return rows


def _exact_batch(dtype, n, seed):
    rng = np.random.default_rng(seed)
    P = _exact_patterns(n)
    rows = _exact_rows(n, rng)
    B = len(rows)
    uv, cand, best, want = np.zeros((B, n, 2)), np.zeros((B, n), bool), np.zeros(B, np.int32), np.zeros((B, n))
    for b, (cm, d, pat, over) in enumerate(rows):
        X = P[pat]
        depth = X[:, 2] + 1.0
        with np.errstate(all="ignore"):
            pred = np.stack([F * X[:, 0] + CX * depth, F * X[:, 1] + CY * depth], 1) / np.abs(depth)[:, None]
        off = DIRS[np.arange(n) % 4] * d[:, None]
        if pat == 1:                                                                # behind: (e, 0) with an exact root
            back = np.flatnonzero(X[:, 2] == -2.0)
            e = BEHIND[np.arange(len(back)) % len(BEHIND)]
            off[back] = np.stack([e[:, 0], np.zeros(len(back))], 1)
            d = d.copy()
            d[back] = e[:, 1]
        want[b] = d
        uv[b] = np.where(np.isfinite(pred), pred + off, 0.0)
        for i, (du, dv) in over.items():
            uv[b, i] += (du, dv)
        cand[b], best[b] = cm, pat
        uv[b, ~cm] = np.nan                                                         # never read
    R = np.tile(np.eye(3), (B, 1, 1))
    t = np.tile([0.0, 0.0, 1.0], (B, 1))
    return P.astype(dtype), uv.astype(dtype), R.astype(dtype), t.astype(dtype), best, cand, want


EXACT_PARAMS = [
    dict(k=1.5, floor_px=1.5 * 5 * Q),       # k med = floor_px exactly at med = 5 Q; under = rank and rank + 1 on the ladders
    dict(k=1.5, floor_px=0.0),               # tau = k med: a rank error moves tau by 1.5 Q; d = tau exactly where med is even
    dict(k=0.0, floor_px=7 * Q),             # tau = floor_px, and the ladder value 7 Q equals it
    dict(k=1.0, floor_px=0.1),               # tau = med itself
    dict(k=1.5, floor_px=float("inf")),      # every finite distance kept, NaN ones (z = 0, infinite pixels) not
    dict(k=1e308, floor_px=1.0),             # k med overflows from med = 1.8 px on: tau = floor_px
]


@pytest.mark.parametrize("dtype,n", [(np.float64, 16), (np.float64, 40), (np.float32, 16), (np.float32, 40)])
@pytest.mark.parametrize("pi", range(len(EXACT_PARAMS)))
def test_exact_geometry_bit_for_bit(dtype, n, pi):
    prm = EXACT_PARAMS[pi]
    P, uv, R, t, best, cand, want = _exact_batch(dtype, n, seed=n + pi)
    B = len(uv)
    d, p, z, A = distances(P, uv, K_EXACT, R, t, best, cand)
    # the construction is exact: every finite distance is the one designed, and NaN ones are there
    fin = np.isfinite(d)
    assert (d[fin] == want[fin]).all() and np.isnan(d[cand]).any()
    tau, new = rule(d, cand, prm["k"], prm["floor_px"])
    assert (tau.astype(np.float64) == tau).all()                       # k med is exact too
    rng = np.random.default_rng(pi)
    mask = cand.copy()
    mask[4::5] = new[4::5]                                              # M = M': flag 0, nothing written
    mask[2::7] &= rng.random((len(mask[2::7]), n)) < 0.7
    rounds = rng.integers(1, 4, B).astype(np.int32)
    status = np.zeros(B, np.int32)
    cnt = new.sum(1)
    changed = (new != mask).any(1) & (cnt >= 4)
    x = int(np.sort(cnt[changed])[changed.sum() // 2])                  # min_inliers = |M'| of a changed row, and |M'| + 1
    for last_round in (0, 1):
        for min_inliers in (x, x + 1):
            flag, m_ref, r_ref, s_ref = decide(new, mask, rounds, status, min_inliers, last_round)
            changed_at = changed & (cnt == x)                          # accepted at x, too few at x + 1
            assert ((s_ref == TOO_FEW) if min_inliers > x else ((flag == 1) | (s_ref == NOT_CONVERGED)))[changed_at].all()
            for shape in (0, 1, 2):
                rc, o = hook(dtype, uv, P, K_EXACT, R, t, best, visible=cand, k=prm["k"], floor_px=prm["floor_px"],
                             min_inliers=min_inliers, last_round=last_round, inliers=mask, rounds=rounds, status=status, shape=shape)
                assert rc == 0, (shape, rc)
                np.testing.assert_array_equal(o["tau"], tau.astype(np.float64))
                np.testing.assert_array_equal(o["inliers"], m_ref)
                np.testing.assert_array_equal(o["flag"], flag)
                np.testing.assert_array_equal(o["status"], s_ref)
                np.testing.assert_array_equal(o["rounds"], r_ref)


# ------------------------------------------------------------------------------------------------------------------------------
# b. realistic poses
# ------------------------------------------------------------------------------------------------------------------------------
CASE_B = {"all": (4113, 3, 0.0), "vis": (33, 1, 0.1), "idx": (31, 3, 0.3), "vis_idx": (1, 1, 0.1)}
N_BOTH = [(np.float64, n) for n in (4, 15, 16, 17, 18, 33, 68, 95)] + [(np.float32, n) for n in (4, 16, 18, 34, 36, 68, 98, 190)]
N_WARP = [(np.float64, n) for n in (96, 98, 300, 1024)] + [(np.float32, n) for n in (15, 192, 300)]


def _realistic(dtype, n, case, seed):
    B, n_pat, f = CASE_B[case]
    if n >= 300 and case == "all":
        B = 1031
    if n == 1024 and case == "all":
        B = 4113
    base = pt.pattern_array(pt.synthetic_pattern(max(n, 15)))[:n]
    P = np.stack([base * (1.0 + 0.03 * j) for j in range(n_pat)])
    K = pt.default_camera_matrix()
    w = orc.synth(0, B, base, K, cfg=orc.default_synth(seed=seed))
    uv = oa.add_outliers(w["uv"], f, 5.0, 150.0, seed)
    rng = np.random.default_rng(seed)
    sel = rng.permutation(n)[: max(4, n - n // 5)] if "idx" in case else None
    vis = (rng.random((B, n)) < 0.85) if "vis" in case else np.ones((B, n), bool)
    cand = vis.copy()
    if sel is not None:
        cand[:, np.setdiff1d(np.arange(n), sel)] = False
    best = rng.integers(0, n_pat, B).astype(np.int32)
    # poses: the ground truth on even rows, a solve on its candidates on odd ones
    import pnp_solver_test_b200 as pnp
    td = torch.float64 if dtype == np.float64 else torch.float32
    s = to_np(pnp.solve_batch("qeif", dev(uv, td), dev(P[:1], td), K, visible=torch.from_numpy(cand).cuda()))
    R = np.where((np.arange(B) % 2 == 0)[:, None, None], w["R_gt"], s["R"])
    t = np.where((np.arange(B) % 2 == 0)[:, None], w["t_gt"], s["t"])
    uv = uv.copy()
    uv[~vis] = np.nan
    return (P.astype(dtype), uv.astype(dtype), K, R.astype(dtype), t.astype(dtype), best, sel,
            None if "vis" not in case else vis, cand)


def _check_realistic(dtype, n, case, shapes):
    P, uv, K, R, t, best, sel, vis, cand = _realistic(dtype, n, case, seed=1000 + n)
    B = len(uv)
    rng = np.random.default_rng(n)
    extra = 5                                            # problem rows no batch entry maps to: canaries
    rows = B + extra
    idx = rng.permutation(rows)[:B].astype(np.int32)     # batch entry k -> problem row idx[k], unsorted
    vis_rows = np.zeros((rows, n), bool)
    vis_rows[idx] = cand if vis is None else vis
    if vis is not None:
        vis_rows[np.setdiff1d(np.arange(rows), idx)] = rng.random((extra, n)) < 0.5
    cand_rows = np.zeros((rows, n), bool)
    cand_rows[idx] = cand
    mask_rows = rng.random((rows, n)) < 0.5                                 # canary rows: arbitrary bits
    mask_rows[idx] = cand
    rounds_rows = rng.integers(1, 4, rows).astype(np.int32)
    status_rows = np.zeros(rows, np.int32)
    status_rows[np.setdiff1d(np.arange(rows), idx)] = 3
    k, floor_px, min_inliers = 3.0, 0.5, 6
    last_round = int(n % 2)
    d, p, z, A = distances(P, uv, K, R, t, best, cand)
    tau, new = rule(d, cand, k, floor_px)
    err = distance_bound(d, p, z, A)
    err = np.where(cand & np.isfinite(d), err, 0.0)
    tau_bound = k * err.max(1) + 2 * U * np.abs(tau.astype(np.float64))
    flag_ref, m_ref, r_ref, s_ref = decide(new, cand, rounds_rows[idx], status_rows[idx], min_inliers, last_round)
    kw = dict(point_index=sel, visible=None if vis is None else vis_rows, k=k, floor_px=floor_px, min_inliers=min_inliers,
              idx=idx, last_round=last_round, inliers=mask_rows, rounds=rounds_rows, status=status_rows)
    outs = {}
    for shape in shapes + [0]:
        rc, outs[shape] = hook(dtype, uv, P, K, R, t, best, shape=shape, **kw)
        assert rc == 0, (shape, rc)
    if 1 not in shapes:
        assert hook(dtype, uv, P, K, R, t, best, shape=1, **kw)[0] == -1             # EINVAL: the streaming kernel cannot run
    _same(outs[0], outs[1 if _streams(dtype, n) else 2])                               # auto = the shape it dispatches to
    for s in shapes[1:]:
        _same(outs[shapes[0]], outs[s])                                                # the shapes agree bit for bit
    o = outs[0]
    canary = np.setdiff1d(np.arange(rows), idx)
    np.testing.assert_array_equal(o["inliers"][canary], mask_rows[canary])
    np.testing.assert_array_equal(o["rounds"][canary], rounds_rows[canary])
    np.testing.assert_array_equal(o["status"][canary], status_rows[canary])
    # tau: within the bound, and the bound no looser than 1e-9 relative (measured on a B200: the worst |tau - tau_ref| / tau_ref
    # over every run here is 5.2e-13, FP64 n = 16, against a bound of 1.0e-11 there)
    gap = np.abs(o["tau"] - tau.astype(np.float64))
    assert (gap <= tau_bound).all(), (gap.max(), tau_bound[np.argmax(gap)])
    assert (tau_bound <= 1e-9 * tau.astype(np.float64)).all()
    print("%s n=%d %s: worst |tau - tau_ref| / tau_ref %.3g, bound %.3g" % (np.dtype(dtype).name, n, case,
          (gap / tau.astype(np.float64)).max(), (tau_bound / tau.astype(np.float64)).max()))
    # the decision: equal but for landmarks within the band of tau
    with np.errstate(invalid="ignore"):
        band = cand & (np.abs(d - tau[:, None]).astype(np.float64) <= err + tau_bound[:, None])
    got_new = o["inliers"][idx]
    ex = band.any(1)
    assert ex.mean() < 1e-3, ex.mean()
    ok = ~ex
    np.testing.assert_array_equal((got_new != m_ref)[ok], False)
    assert not (got_new != m_ref)[~band & ex[:, None]].any()
    np.testing.assert_array_equal(o["flag"][ok], flag_ref[ok])
    np.testing.assert_array_equal(o["status"][idx][ok], s_ref[ok])
    np.testing.assert_array_equal(o["rounds"][idx][ok], r_ref[ok])


@pytest.mark.parametrize("case", list(CASE_B))
@pytest.mark.parametrize("dtype,n", N_BOTH, ids=lambda x: str(x))
def test_realistic_both_shapes(dtype, n, case):
    _check_realistic(dtype, n, case, [1, 2])


@pytest.mark.parametrize("case", list(CASE_B))
@pytest.mark.parametrize("dtype,n", N_WARP, ids=lambda x: str(x))
def test_realistic_warp_shape(dtype, n, case):
    _check_realistic(dtype, n, case, [2])


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_warp_shape_size_limit(dtype):
    """shape 2 at the largest n_total whose shared memory fits (8 warps x (n 8-byte keys + 2 W mask words)) and one above"""
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    fits = lambda n: 8 * (n * 8 + 2 * ((n + 31) // 32) * 4) <= optin
    n_max = max(n for n in range(1, 8192) if fits(n))
    assert not fits(n_max + 1)
    for n, rc_want in ((n_max, 0), (n_max + 1, -4)):
        B = 3
        P = pt.pattern_array(pt.synthetic_pattern(n))[None]
        K = pt.default_camera_matrix()
        w = orc.synth(0, B, P[0], K, cfg=orc.default_synth(seed=5))
        cand = np.ones((B, n), bool)
        args = (dtype, w["uv"].astype(dtype), P.astype(dtype), K, w["R_gt"].astype(dtype), w["t_gt"].astype(dtype), None)
        kw = dict(k=3.0, floor_px=0.5, inliers=cand, rounds=np.ones(B, np.int32), status=np.zeros(B, np.int32))
        rc, o = hook(*args, shape=2, **kw)
        assert rc == rc_want, (n, rc)
        rc0, _ = hook(*args, shape=0, **kw)
        assert rc0 == rc_want                                                          # the dispatcher has no other shape there
        if rc == 0:
            d, p, z, A = distances(P.astype(dtype), w["uv"].astype(dtype), K, w["R_gt"].astype(dtype), w["t_gt"].astype(dtype),
                                   np.zeros(B, np.int32), cand)
            tau, new = rule(d, cand, 3.0, 0.5)
            assert np.allclose(o["tau"], tau.astype(np.float64), rtol=1e-12, atol=0)


# ------------------------------------------------------------------------------------------------------------------------------
# c. invariants of the robust and RANSAC entries
# ------------------------------------------------------------------------------------------------------------------------------
def _entry(method, uv, P, K, td, sel, vis, **kw):
    import pnp_solver_test_b200 as pnp
    out = pnp.solve_robust_batch(method, dev(uv, td), dev(P, td), K, point_index=sel,
                                 visible=None if vis is None else torch.from_numpy(vis).cuda(), **kw)
    torch.cuda.synchronize()
    return to_np(out)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("n", [15, 18, 68, 98, 300])
@pytest.mark.parametrize("method", ["lm", "lm_plus", "qeif", "eif2"])
@pytest.mark.parametrize("case", ["all", "vis", "idx", "vis_idx"])
def test_entry_invariants(method, n, dtype, case):
    import pnp_solver_test_b200 as pnp
    td = torch.float64 if dtype == np.float64 else torch.float32
    B = 256
    pat = pt.get_golden_pattern() if n == 15 else pt.synthetic_pattern(n)
    P, K = pt.pattern_array(pat)[None], pt.default_camera_matrix()
    w = orc.synth(0, B, P[0], K, cfg=orc.default_synth(seed=n))
    uv = oa.add_outliers(w["uv"], 0.2, 5.0, 150.0, n)
    rng = np.random.default_rng(n + 1)
    sel = rng.permutation(n)[: n - n // 5] if "idx" in case else None
    vis = (rng.random((B, n)) < 0.85) if "vis" in case else None
    cand = np.ones((B, n), bool) if vis is None else vis.copy()
    if sel is not None:
        cand[:, np.setdiff1d(np.arange(n), sel)] = False
    if vis is not None:
        uv[~vis] = np.nan
    uvd, Pd = uv.astype(dtype), P.astype(dtype)
    zeros = np.zeros(B, np.int32)

    def classify(out, mask, rounds, last_round):
        rc, o = hook(dtype, uvd, Pd, K, out["R"].astype(dtype), out["t"].astype(dtype), out["best_pattern"], point_index=sel,
                     visible=vis, k=3.0, floor_px=2.0, min_inliers=6, last_round=last_round, inliers=mask, rounds=rounds,
                     status=zeros)
        assert rc == 0
        return o

    # robust_status is the rule on the returned pose, pattern and mask (for the RANSAC entry as well)
    for kw in (dict(), dict(samples=128)):
        got = _entry(method, uv, Pd, K, td, sel, vis, **kw)
        o = classify(got, got["inliers"], got["rounds"], 1)
        np.testing.assert_array_equal(o["inliers"], got["inliers"])
        np.testing.assert_array_equal(o["status"], got["robust_status"])
        assert (got["rounds"][got["robust_status"] == NOT_CONVERGED] == 4).all()
    # max_rounds = 2: the rule on the round-0 pose (the masked solve on C) decides the mask, rounds and (where kept) status
    r0 = to_np(pnp.solve_batch(method, dev(uv, td), dev(Pd, td), K, point_index=sel, visible=torch.from_numpy(cand).cuda()))
    o = classify(r0, cand, np.ones(B, np.int32), 0)
    two = _entry(method, uv, Pd, K, td, sel, vis, max_rounds=2)
    np.testing.assert_array_equal(two["inliers"], o["inliers"])
    np.testing.assert_array_equal(two["rounds"], o["rounds"])
    kept = o["flag"] == 0
    np.testing.assert_array_equal(two["robust_status"][kept], o["status"][kept])
    assert (o["flag"] == 1).any()
    # RANSAC, one round: M0 = the consensus set where it holds min_inliers landmarks, else C
    one = _entry(method, uv, Pd, K, td, sel, vis, samples=128, max_rounds=1)
    hyp = to_np(pnp.hypothesize_batch(dev(uv, td), dev(Pd, td), K, point_index=sel,
                                      visible=None if vis is None else torch.from_numpy(vis).cuda(), samples=128))
    seeded = hyp["consensus"] >= 6
    np.testing.assert_array_equal(one["consensus"], hyp["consensus"])
    np.testing.assert_array_equal(one["inliers"], np.where(seeded[:, None], hyp["consensus_mask"], cand))
    assert (one["rounds"] == 1).all() and seeded.any()
