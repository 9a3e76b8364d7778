"""The error report (pnpb200_report_batch_strided[_masked]) on every kernel shape the dispatcher picks, against the
extended-precision reference of tests/report_ref.py:
  a. realistic poses (near-solved, medium, diverged, behind the camera, non-orthogonal R, ground-truth angles to +-1000 deg)
     at n on both sides of every shape boundary, masked and unmasked, ragged batches: exact columns bit for bit, columns 4-9
     within the derived bound, flags exact, max_idx exact but at near-ties;
  b. exact geometry, where every decision is exact: ties of the maximum, depth 0, t3 = 0, non-finite pixels, the visible
     count at 4, angle and depth errors at their bounds, and depth-flag pairs on which a contracted FMA flips the flag;
  c. strided outputs, NULL flags / max_idx, the stream chunk size, and the identity with the solution check."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import report_ref as rr
from pnp_solver_test_b200 import patterns as pt

from gpu_util import dev

HERE = os.path.dirname(os.path.abspath(__file__))

# ------------------------------------------------------------------------------------------------------------------------------
# the shape map (report_launch, csrc/pnpb200_aux.cu): the streaming kernel k_report_chunk where the row tile of 32 problems
# (row_geometry: the row padded to an odd number of 16-byte units) fits 48 KiB and rows stream in whole 16-byte units
# (stream_geometry); k_report_thread where the tile fits but rows do not stream (FP32, odd n; never masked); k_report (one warp
# per problem) otherwise
# ------------------------------------------------------------------------------------------------------------------------------
N_F64 = [1, 4, 16, 17, 18, 34, 35, 68, 94, 95, 96, 97, 98, 300]
N_F32 = [1, 2, 3, 15, 33, 34, 35, 36, 68, 69, 188, 189, 190, 191, 192, 193, 300]


def shape(dtype, n, masked=False):
    esz = 8 if dtype == np.float64 else 4
    units = (n * 2 * esz + 15) // 16
    units += 1 - (units & 1)
    fits = 32 * units * 16 <= 48 * 1024
    if fits and n % (16 // (2 * esz)) == 0:
        return "chunk"
    return "thread" if fits and not masked else "warp"


def test_shape_map_puts_the_n_lists_on_both_sides_of_every_boundary():
    f64 = {n: shape(np.float64, n) for n in N_F64}
    f32 = {n: shape(np.float32, n) for n in N_F32}
    assert max(n for n in range(1, 400) if shape(np.float64, n) == "chunk") == 95
    assert max(n for n in range(1, 400) if shape(np.float32, n) == "chunk") == 190
    assert max(n for n in range(1, 400) if shape(np.float32, n) == "thread") == 189
    assert f64[95] == "chunk" and f64[96] == "warp" and f64[300] == "warp"
    assert f32[189] == "thread" and f32[190] == "chunk" and f32[191] == "warp" and f32[192] == "warp"
    assert f32[15] == "thread" and shape(np.float32, 15, masked=True) == "warp"
    assert set(f32.values()) == {"chunk", "thread", "warp"} and set(f64.values()) == {"chunk", "warp"}
    # the default chunk is 17 16-byte units: 17 landmarks in FP64, 34 in FP32; the lists straddle one and two chunks
    assert {16, 17, 18, 34, 35} <= set(N_F64) and {33, 34, 35, 68, 69} <= set(N_F32)


# ------------------------------------------------------------------------------------------------------------------------------
# calling the library
# ------------------------------------------------------------------------------------------------------------------------------
F64, F32 = np.float64, np.float32
CANARY = 0x7ff4dead0000beef                        # a signalling NaN no kernel writes


def run(dtype, P, uv, K, R, t, euler, gt, bounds=None, visible=None, strides=None, want_flags=True, want_idx=True):
    """pnpb200_report_batch_strided[_masked] through ctypes on NumPy inputs, into a buffer of canaries: returns (report [B, 16],
    flags, max_idx, the whole buffer); flags and max_idx start at -7"""
    from pnp_solver_test_b200 import _lib
    from pnp_solver_test_b200.solver import visible_words
    td = torch.float64 if dtype == F64 else torch.float32
    B, n = uv.shape[0], uv.shape[1]
    rs_b, rs_k = strides or (1, B)
    buf = torch.empty((max((B - 1) * rs_b + 15 * rs_k + 1, 1),), dtype=torch.float64, device="cuda")
    buf.view(torch.int64).fill_(CANARY)
    flags = torch.full((B, 4), -7, dtype=torch.int32, device="cuda")
    midx = torch.full((B, 3), -7, dtype=torch.int32, device="cuda")
    g = [dev(x, td) for x in (P, uv, R, t, euler)]
    gtd = dev(gt)
    Kh = np.ascontiguousarray(K, np.float64)
    bd = None if bounds is None else (C.c_double * 4)(*[float(b) for b in bounds])
    PD, PI = C.POINTER(C.c_double), C.POINTER(C.c_int32)
    vp = lambda x: C.c_void_p(x.data_ptr())
    args = [C.c_int(0 if dtype == F64 else 1), C.c_int64(B), C.c_int(n), vp(g[0]), vp(g[1]), Kh.ctypes.data_as(PD), vp(g[2]),
            vp(g[3]), vp(g[4]), C.cast(vp(gtd), PD), bd, C.cast(vp(buf), PD), C.c_int64(rs_b), C.c_int64(rs_k),
            C.cast(vp(flags), PI) if want_flags else None, C.cast(vp(midx), PI) if want_idx else None]
    if visible is None:
        rc = _lib.lib.pnpb200_report_batch_strided(*args, None)
    else:
        words = visible_words(torch.from_numpy(np.asarray(visible, bool)).cuda(), torch.device("cuda"))
        rc = _lib.lib.pnpb200_report_batch_strided_masked(*args, C.cast(vp(words), C.POINTER(C.c_uint32)), None)
    torch.cuda.synchronize()
    assert rc == 0, rc
    raw = buf.cpu().numpy()
    ix = np.arange(B)[:, None] * rs_b + np.arange(16)[None, :] * rs_k
    return raw[ix], flags.cpu().numpy(), midx.cpu().numpy(), raw


def _assert_matches(got, ref, label):
    rep, flags, midx = got[:3]
    ok = rr.columns_ok(rep, ref)
    bad = np.argwhere(~ok)
    assert ok.all(), "%s: columns differ at (problem, column) %s: got %s ref %s bound %s" % (
        label, bad[:4].tolist(), rep[tuple(bad[0])], ref["report"][tuple(bad[0])], ref["bound"][tuple(bad[0])])
    fb = np.argwhere(flags != ref["flags"])
    assert len(fb) == 0, "%s: flags differ at %s" % (label, fb[:8].tolist())
    mi = rr.max_idx_ok(midx, ref)
    assert mi.all(), "%s: max_idx differs at %s: got %s ref %s" % (label, np.argwhere(~mi)[:4].tolist(), midx[~mi][:4],
                                                                   ref["max_idx"][~mi][:4])


def _ratio(got, ref):
    with np.errstate(all="ignore"):
        r = np.abs(got[:, 4:10] - ref["report"][:, 4:10]) / ref["bound"][:, 4:10]
    return float(np.nanmax(np.where(ref["bound"][:, 4:10] > 0, r, 0.0), initial=0.0))


# ------------------------------------------------------------------------------------------------------------------------------
# a. realistic poses
# ------------------------------------------------------------------------------------------------------------------------------
def _pattern(n):
    P = pt.pattern_array(pt.synthetic_pattern(max(n, 15)))
    return P[:n]


def _rot(a):
    """rotation matrices from angles [B, 3] (rad), any convention"""
    out = []
    for x, y, z in a:
        cx, sx, cy, sy, cz, sz = np.cos(x), np.sin(x), np.cos(y), np.sin(y), np.cos(z), np.sin(z)
        Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
        Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
        Rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]])
        out.append(Rz @ Ry @ Rx)
    return np.array(out)


def workload(n, B, dtype, seed):
    """pixels from ground-truth poses (quantised on half the problems), estimated poses near-solved / medium / diverged /
    behind the camera / non-orthogonal, ground-truth angles mostly within 45 deg and out to +-1000 deg on a tenth"""
    rng = np.random.default_rng(seed)
    P, K = _pattern(n), pt.default_camera_matrix()
    ang = rng.uniform(-45, 45, (B, 3))
    wide = rng.random(B) < 0.1
    ang[wide] = rng.uniform(-1000, 1000, (wide.sum(), 3))
    dist = rng.uniform(0.2, 2.25, B)
    gt = np.stack([dist, ang[:, 0], ang[:, 1], ang[:, 2]], 1)                  # (dist, roll, pitch, yaw)
    Rg = rr.rot_from_euler_deg(rr.L(1) * ang[:, 0], rr.L(1) * ang[:, 2], rr.L(1) * ang[:, 1]).astype(np.float64)
    tg = np.stack([dist * rng.uniform(-0.4, 0.4, B), dist * rng.uniform(-0.4, 0.4, B), dist], 1)
    X = np.einsum("bij,nj->bni", Rg, P) + tg[:, None, :]
    uv = np.einsum("ij,bnj->bni", K, X)
    uv = uv[..., :2] / np.abs(uv[..., 2:3]) + rng.normal(0, 0.7, (B, n, 2))
    q = rng.random(B) < 0.5
    uv[q] = np.round(uv[q])
    kind = rng.integers(0, 5, B)
    scale = np.array([1e-4, 3e-2, 1.0, 0.3, 0.1])[kind]
    R = np.einsum("bij,bjk->bik", _rot(rng.normal(0, 1, (B, 3)) * scale[:, None]), Rg)
    t = tg * (1 + rng.normal(0, 1, (B, 3)) * scale[:, None] * 0.3)
    flip = kind == 3                                                            # behind the camera: t3 < 0
    t[flip, 2] *= -1
    skew = kind == 4                                                            # not orthogonal
    R[skew] += rng.normal(0, 0.2, (skew.sum(), 3, 3))
    euler = ang[:, [0, 2, 1]] + rng.normal(0, 1, (B, 3)) * scale[:, None] * 20   # (roll, yaw, pitch)
    t[::97, 2] = dist[::97] + rng.choice([-0.1, 0.1], len(t[::97])) + rng.integers(-3, 4, len(t[::97])) * 1e-16
    cast = lambda x: np.asarray(x, dtype).astype(np.float64) if dtype == F32 else np.asarray(x, F64)
    vis = rng.random((B, n)) < 0.85
    vis[1::11] = False
    vis[1::11, :min(n, 4)] = True                                               # exactly 4 visible (fewer where n < 4)
    vis[5::11, :] = False
    vis[5::11, :min(n, 3)] = True                                               # 3 visible
    return dict(P=cast(P), uv=cast(uv), K=K, R=cast(R), t=cast(t), euler=cast(euler), gt=gt, vis=vis)


SWEEP = [(F64, n) for n in N_F64] + [(F32, n) for n in N_F32]
RATIOS = {}


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,n", SWEEP, ids=["%s-n%d" % ("f64" if d == F64 else "f32", n) for d, n in SWEEP])
def test_report_sweep_matches_extended_precision_reference(dtype, n):
    w = workload(n, 1037, dtype, seed=n * 7 + (dtype == F32))
    args = [w[k] for k in ("P", "uv", "K", "R", "t", "euler", "gt")]
    for masked in (False, True):
        vis = w["vis"] if masked else None
        ref = rr.report(*args, visible=vis)
        # the bound is tight: at most 1e-12 of the pixel magnitudes where every depth is well-conditioned
        good = (ref["kappa"] <= 1e3) & np.isfinite(ref["px"])
        lbmax = np.nanmax(np.where(np.isfinite(ref["lm_bound"]), ref["lm_bound"], 0.0), axis=(1, 2))
        assert (lbmax[good] <= 1e-12 * np.maximum(ref["px"][good], 1.0)).all()
        worst = 0.0
        for B in (1, 31, 33, 1037):
            sub = {k: v[:B] for k, v in ref.items()}
            got = run(dtype, args[0], args[1][:B], args[2], *[a[:B] for a in args[3:]], visible=None if vis is None else vis[:B])
            _assert_matches(got, sub, "%s n=%d masked=%s B=%d" % (dtype.__name__, n, masked, B))
            worst = max(worst, _ratio(got[0], sub))
        RATIOS["%s n=%d %s" % (dtype.__name__, n, "masked" if masked else "unmasked")] = worst
        if masked:
            # hidden pixels are never read: NaN / +-Inf there changes no output bit
            uv2 = args[1].copy()
            hid = ~vis
            uv2[hid] = np.array([np.nan, np.inf, -np.inf])[np.arange(hid.sum()) % 3][:, None]
            a = run(dtype, args[0], args[1], *args[2:], visible=vis)
            b = run(dtype, args[0], uv2, *args[2:], visible=vis)
            assert a[0].tobytes() == b[0].tobytes() and a[1].tobytes() == b[1].tobytes() and a[2].tobytes() == b[2].tobytes()
    print("largest error / bound, columns 4-9:", {k: "%.3f" % v for k, v in RATIOS.items() if k.startswith(dtype.__name__ + " n=%d " % n)})


# ------------------------------------------------------------------------------------------------------------------------------
# b. exact geometry
# ------------------------------------------------------------------------------------------------------------------------------
FX, CX, CY = 256.0, 160.0, 128.0
K_EXACT = np.array([[FX, 0.0, CX], [0.0, FX, CY], [0.0, 0.0, 1.0]])


def _grid(n):
    j = np.arange(n)
    return np.stack([(j % 8) / 16.0 - 0.25, (j // 8) / 32.0 - 0.125, np.zeros(n)], 1)


def _rz(q):
    c, s = [(1, 0), (0, 1), (-1, 0), (0, -1)][q % 4]
    return np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])


def exact_cases(n, chunk, rng, dtype=np.float64):
    """rows of an exact batch: (P per row [n, 3], uv, R, t, euler, gt, visible, label).  With R_gt = I (angles 0), t3 = dist a
    power of two (t_gt = t) and z = 0 every projection is dyadic; the pixels sit at (3, 4)-scaled offsets from the estimated
    projection, so every prediction-vs-landmark distance is exact."""
    rows = []
    P0 = _grid(n)

    def row(label, off=None, q=0, t=(0.0625, -0.03125, 1.0), P=None, euler=(0.0, 0.0, 0.0), gta=(0.0, 0.0, 0.0), vis=None,
            dist=None, uvfix=None):
        P = P0 if P is None else P
        R = _rz(q)
        tt = np.array(t)
        Xc = P @ R.T + tt
        with np.errstate(all="ignore"):
            p = (Xc @ K_EXACT.T)[:, :2] / np.abs(Xc[:, 2:3])
        o = np.zeros((n, 2)) if off is None else off
        uv = np.nan_to_num(p, nan=0.0, posinf=0.0, neginf=0.0) + o
        if uvfix is not None:
            for i, v in uvfix.items():
                uv[i] = v
        d = tt[2] if dist is None else dist
        rows.append(dict(P=P, uv=uv, R=R, t=tt, euler=np.array(euler), gt=np.array([d, gta[0], gta[1], gta[2]]),
                         vis=np.ones(n, bool) if vis is None else vis, label=label))

    base = (np.arange(n) % 5 + 1)[:, None] * np.array([0.09375, 0.125])        # distances 0.15625 * (1..5), max 0.78125
    def tie(i, j):
        o = base.copy()
        o[i] = [0.75, 1.0]
        o[j] = [1.0, 0.75] if (i + j) % 2 else [-0.75, 1.0]
        return o
    pairs = [(0, 1), (0, n - 1), (n - 2, n - 1)]
    for i, j in pairs + ([(chunk - 1, chunk), (3, 3 + chunk)] if n > chunk + 3 else []) + ([(2, 34)] if n > 34 else []):
        if 0 <= i < j < n:
            for q in range(4):
                row("tie %d-%d q%d" % (i, j, q), tie(i, j), q=q)
    row("all zero", np.zeros((n, 2)))
    row("all zero q2", np.zeros((n, 2)), q=2)
    if n >= 2:
        P = P0.copy(); P[1, 2] = -2.0                                           # depth -1: behind, +4 under the root
        o = base.copy(); o[1] = [1.5, 0.0]                                      # sqrt(1.5^2 + 4) = 2.5
        row("behind", o, P=P)
        P = P0.copy(); P[n - 1, 2] = -1.0                                       # depth exactly 0
        row("depth 0", base.copy(), P=P)
    row("t3 = 0", base.copy(), t=(0.0625, -0.03125, 0.0), dist=1.0)
    row("t3 = -0", base.copy(), t=(-0.0625, -0.03125, -0.0), dist=1.0)
    row("t3 < 0", base.copy(), t=(0.0625, -0.03125, -1.0), dist=1.0)
    for v in (np.nan, np.inf, -np.inf):
        row("pixel %s" % v, base.copy(), uvfix={n // 2: [v, 5.0]})
    if n >= 5:
        for c in (3, 4, 5):
            vis = np.zeros(n, bool); vis[rng.permutation(n)[:c]] = True
            row("visible %d" % c, base.copy(), vis=vis, uvfix={i: [np.nan, np.inf] for i in np.nonzero(~vis)[0]})
    b = 10.0
    for dv in (-1, 0, 1):
        a = float(np.nextafter(dtype(b), dtype(np.inf * dv))) if dv else b    # 1 ulp of the dtype the kernel reads
        row("angle err %+d ulp" % dv, base.copy(), euler=(a, -a, a), gta=(0.0, 0.0, 0.0))
        row("angle err neg %+d ulp" % dv, base.copy(), euler=(-a, a, -a))
    for d in (0.5, 1.0, 2.0):
        for s in (0.1, -0.1):
            for k in range(-2, 3):
                x = d + s
                x = x + k * np.spacing(x)
                row("depth %.17g vs %g" % (x, d), base.copy(), t=(0.0625, -0.03125, x), dist=d)
    return rows


def flag_pairs(count=96, seed=0):
    """(t3, dist) pairs on which the reference's rule (both products rounded) and the two FMA contractions disagree"""
    L = np.longdouble
    rng = np.random.default_rng(seed)
    out = []
    while len(out) < count:
        d = rng.uniform(0.2, 2.25)
        for s in (0.1, -0.1):
            for k in range(-4, 5):
                t3 = d + s + k * np.spacing(d + s)
                r = abs(t3 * 100.0 - d * 100.0) < 10
                c1 = abs(np.float64(L(t3) * 100 - L(d * 100.0))) < 10
                c2 = abs(np.float64(L(t3 * 100.0) - L(d) * 100)) < 10
                if c1 != r and c2 != r:
                    out.append((t3, d))
    return out[:count]


def test_flag_pairs_exist_and_straddle_the_bound():
    """host side: the search finds pairs; on each the reference's rule and both contractions disagree"""
    pr = flag_pairs()
    assert len(pr) == 96
    for t3, d in pr:
        assert rr.depth_flag(t3, d, 10.0) != (abs(float(np.longdouble(t3) * 100 - np.longdouble(d * 100.0))) < 10)


def _exact_batch(n, dtype, rows):
    Pn = rows[0]["P"]
    same_P = all(r["P"] is Pn or np.array_equal(r["P"], Pn) for r in rows)
    assert same_P
    st = lambda k: np.stack([r[k] for r in rows])
    io = lambda x: np.asarray(x, dtype).astype(np.float64)                     # the values the kernel reads
    return [io(Pn), io(st("uv")), K_EXACT, io(st("R")), io(st("t")), io(st("euler")), st("gt")], st("vis")


EXACT_SHAPES = [(F64, 35), (F64, 68), (F64, 96), (F64, 300), (F32, 15), (F32, 36), (F32, 68), (F32, 189), (F32, 192)]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,n", EXACT_SHAPES, ids=["%s-n%d-%s" % ("f64" if d == F64 else "f32", n, shape(d, n))
                                                       for d, n in EXACT_SHAPES])
def test_exact_geometry_decisions_are_exact(dtype, n):
    rng = np.random.default_rng(n)
    chunk = 17 if dtype == F64 else 34
    rows = exact_cases(n, chunk, rng, dtype)
    groups = {}
    for r in rows:
        groups.setdefault(id(r["P"]) if r["P"] is not rows[0]["P"] else 0, []).append(r)
    for rs in groups.values():
        args, vis = _exact_batch(n, dtype, rs)
        labels = [r["label"] for r in rs]
        masked_rows = ~vis.all(1)
        for bounds in (None, (0.0, 0.0, 0.0, 0.0), (np.inf,) * 4, (np.nan,) * 4, (10.0, 10.0, 10.0, 10.0)):
            for visible in ((None, vis) if masked_rows.any() else (None,)):
                a = list(args)
                if visible is None and masked_rows.any():
                    keep = ~masked_rows
                    a = [a[0], a[1][keep]] + [a[2]] + [x[keep] for x in a[3:]]
                ref = rr.report(*a, bounds=bounds, visible=visible)
                got = run(dtype, *a, bounds=bounds, visible=visible)
                _assert_matches(got, ref, "%s n=%d bounds=%s masked=%s" % (dtype.__name__, n, bounds, visible is not None))
                # prediction-vs-landmark distances are exact: max_idx[1] exact, also at the ties, and columns 6-7 within
                # the bound of an exact sum
                # where t3 = 1 (or 0) every prediction-vs-landmark distance is exact (or NaN): max_idx[1] exact, ties included;
                # where also R = I and dist = t3, the ground truth is the estimate and max_idx[0] is exact too
                lab = np.array(labels)[~masked_rows] if visible is None and masked_rows.any() else np.array(labels)
                t3, R, dist = a[4][:, 2], a[3], a[6][:, 0]
                ex1 = (t3 == 1.0) | (t3 == 0.0)
                ex0 = (t3 == 1.0) & (dist == 1.0) & (R == np.eye(3)).all((1, 2))
                for q, ex in ((1, ex1), (0, ex0)):
                    bad = ex & (got[2][:, q] != ref["max_idx"][:, q])
                    assert not bad.any(), "max_idx[%d] at %s: got %s ref %s" % (q, lab[bad][:4], got[2][bad, q][:4],
                                                                                ref["max_idx"][bad, q][:4])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,n", [(F64, 68), (F64, 300), (F32, 15), (F32, 68), (F32, 192)],
                         ids=["f64-n68", "f64-n300", "f32-n15", "f32-n68", "f32-n192"])
def test_depth_flag_rounds_both_products_as_the_reference(dtype, n):
    """the depth flag is the reference's |t3 * 100 - dist * 100| < 10 with both products rounded: pairs on which an FMA
    contraction flips it, and 1 ulp either side of the boundary"""
    P = _grid(n)
    pairs = flag_pairs()
    for d in (0.5, 0.75, 1.25):
        for s in (0.1, -0.1):
            x = d + s
            pairs += [(x + k * np.spacing(x), d) for k in (-1, 0, 1)]
    t3 = np.array([p[0] for p in pairs])
    if dtype == F32:
        pairs = [(float(np.float32(a)), d) for a, d in pairs]                  # t3 is read in FP32: search on FP32 values
        t3 = np.array([p[0] for p in pairs])
    B = len(pairs)
    t = np.stack([np.full(B, 0.0625), np.full(B, -0.03125), t3], 1)
    gt = np.stack([np.array([p[1] for p in pairs]), np.zeros(B), np.zeros(B), np.zeros(B)], 1)
    uv = np.zeros((B, n, 2)) + 100.0
    R = np.broadcast_to(np.eye(3), (B, 3, 3)).copy()
    ref = rr.report(P, uv, K_EXACT, R, t, np.zeros((B, 3)), gt)
    got = run(dtype, P, uv, K_EXACT, R, t, np.zeros((B, 3)), gt)
    bad = np.nonzero(got[1][:, 0] != ref["flags"][:, 0])[0]
    assert len(bad) == 0, "depth flag differs on %d of %d pairs, e.g. t3 = %r dist = %r: got %d, reference %d" % (
        len(bad), B, t3[bad[0]], gt[bad[0], 0], got[1][bad[0], 0], ref["flags"][bad[0], 0])


# ------------------------------------------------------------------------------------------------------------------------------
# c. strides, NULL outputs, chunk size, the check
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype,n", [(F64, 68), (F64, 96), (F32, 15), (F32, 68), (F32, 192)],
                         ids=["f64-n68", "f64-n96", "f32-n15", "f32-n68", "f32-n192"])
def test_strided_outputs_touch_only_their_cells(dtype, n):
    B = 45
    w = workload(n, B, dtype, seed=5)
    args = [w[k] for k in ("P", "uv", "K", "R", "t", "euler", "gt")]
    ref = rr.report(*args)
    base = None
    for strides in ((16, 1), (1, B), (19, 1), (1, B + 7)):
        for vis in (None, w["vis"]):
            got = run(dtype, *args, strides=strides, visible=vis)
            r = rr.report(*args, visible=vis) if vis is not None else ref
            _assert_matches(got, r, "strides %s" % (strides,))
            raw = got[3]
            own = np.zeros(raw.shape, bool)
            own[(np.arange(B)[:, None] * strides[0] + np.arange(16)[None, :] * strides[1]).ravel()] = True
            assert (raw[~own].view(np.int64) == CANARY).all()
            if vis is None:
                if base is None:
                    base = got
                assert got[0].tobytes() == base[0].tobytes()
    for wf, wi in ((False, True), (True, False), (False, False)):
        got = run(dtype, *args, want_flags=wf, want_idx=wi)
        assert got[0].tobytes() == base[0].tobytes()
        assert (got[1] == (base[1] if wf else -7)).all() and (got[2] == (base[2] if wi else -7)).all()


CHUNK_SHAPES = [(F64, 1), (F64, 16), (F64, 17), (F64, 35), (F64, 95), (F32, 2), (F32, 34), (F32, 36), (F32, 190)]


def _chunk_outputs():
    """the report of every streaming shape of CHUNK_SHAPES, masked and unmasked, in this process: {key: bytes (hex)}"""
    out = {}
    for dtype, n in CHUNK_SHAPES:
        w = workload(n, 70, dtype, seed=n)
        args = [w[k] for k in ("P", "uv", "K", "R", "t", "euler", "gt")]
        for vis in (None, w["vis"]):
            got = run(dtype, *args, visible=vis)
            out["%s-%d-%s" % (dtype.__name__, n, vis is None)] = b"".join(x.tobytes() for x in got[:3]).hex()
    return out


@pytest.mark.gpu
def test_stream_chunk_size_changes_no_bit(tmp_path):
    """PNPB200_STREAM_CHUNK (read once per process) changes only the buffering, not the order in which a lane visits the
    landmarks: every output is bit-identical to the default's"""
    for dtype, n in CHUNK_SHAPES:
        assert shape(dtype, n) == "chunk"
    ref = _chunk_outputs()
    code = ("import json, sys; sys.path[:0] = [%r, %r]; import test_gpu_report as t; json.dump(t._chunk_outputs(), open(sys.argv[1], 'w'))"
            % (HERE, os.path.dirname(HERE)))
    for units in ("1", "3", "127"):
        path = str(tmp_path / ("chunk%s.json" % units))
        env = dict(os.environ, PNPB200_STREAM_CHUNK=units)
        subprocess.run([sys.executable, "-c", code, path], env=env, check=True, cwd=HERE)
        got = json.load(open(path))
        for k in ref:
            assert got[k] == ref[k], (units, k)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [F64, F32], ids=["f64", "f32"])
def test_check_reprojection_is_report_columns_6_7_at_every_streaming_shape(dtype):
    import pnp_solver_test_b200 as pnp
    td = torch.float64 if dtype == F64 else torch.float32
    for n in (N_F64 if dtype == F64 else N_F32):
        if shape(dtype, n) != "chunk":
            continue
        w = workload(n, 300, dtype, seed=3 * n)
        gt1 = w["gt"].copy()
        gt1[:, 0] = 1.0
        for vis in (None, w["vis"]):
            rep = run(dtype, w["P"], w["uv"], w["K"], w["R"], w["t"], w["euler"], gt1, visible=vis)[0]
            c = pnp.check_batch(dev(w["uv"], td), dev(w["P"], td), w["K"], dev(w["R"], td), dev(w["t"], td),
                                visible=None if vis is None else torch.from_numpy(vis).cuda())
            rp = c["reproj"].cpu().numpy()
            want = rep[:, 6:8].astype(dtype)
            assert rp.tobytes() == np.ascontiguousarray(want).tobytes(), (n, vis is None)
