"""The error report (pnpb200_report_batch*, include/pnpb200.h) restated in NumPy extended precision (np.longdouble, 80-bit on
x86-64), with a per-landmark bound of what the kernels k_report, k_report_thread and k_report_chunk compute.

report() takes the inputs as the kernels read them: FP32 arrays are widened to FP64 first, K and gt are FP64.  It follows
pnp_oracle_report (oracle/pnp_oracle.c) with the library's rules for what the reference leaves open:
  - flags use the reference's float64 rule exactly: |t3 * 100 - dist * 100| < bound with both products rounded, strict <,
    and a NaN fails;
  - a landmark distance whose square is not finite (depth exactly 0, a non-finite pixel) is NaN; NaN makes the mean NaN and
    never wins the maximum.  The kernels form the prediction-vs-GT difference as (prediction - pixel) + (pixel - GT), so a
    non-finite visible pixel makes all three of its distances NaN (equal to prediction - GT for a finite pixel);
  - max_idx: strict >, the first landmark wins, -1 when no distance is > 0;
  - masked: means and maxima over the visible landmarks; fewer than 4 of them: columns 4-9 NaN and max_idx -1.

The bound (derived from the kernels' operations; u = 2^-53, every kernel computes in FP64 for both dtypes):
  - projection of X by (R, t): K R and K t are folded (or R X + t then K, in the warp kernel), then three FMAs per
    coordinate: each coordinate r_j is off by <= 6 u A_j, A = |K| |R| |X| + |K| |t|;
  - the ground-truth pose adds its own input error: each entry of R_gt is off by <= u (16 + 4 sum |theta|) (the bounded
    sin / cos <= 2 ulp, the degree -> radian product <= 2 u |theta|, three roundings of the products), and t_gt = t / t3 *
    dist by <= 4 u |t_gt| (the reciprocal <= 0.5003 ulp and two products, or a division and a product);
  - the pixel p = r_xy / |z| is off by <= (dr_xy + |p| dz) / |z| + 2 u |p| (the reciprocal and the rounding of p or of
    the FMA that forms the difference); |z| small against A_z is where the depth's condition number kappa = A_z / |z|
    enters, as in test_gpu_check._within_oracle;
  - the difference to the measured pixel, and the prediction-vs-GT difference, add one rounding each; the sum of squares
    (two roundings) and sqrt_nonneg (~1 ulp) add <= 4 u e to the distance e;
  - summation: lane-sequential (k_report_thread, k_report_chunk) or per lane then a 5-level shuffle tree (k_report): either
    way <= (c + 5) u sum e over c terms; the division by c and the product with dist add 2 u |column|.
The bound of a mean is (sum of the landmarks' bounds + summation bound) / c * dist; of a maximum, the largest landmark bound
times dist."""
import numpy as np

L = np.longdouble
U = 2.0 ** -53
PI = np.arctan(L(1)) * 4


def rot_from_euler_deg(roll, yaw, pitch):
    """R_from_euler_deg_bounded (csrc/pnpb200_math.cuh) in extended precision: [B, 3, 3]"""
    k = PI / 180
    s1, c1 = np.sin(roll * k), np.cos(roll * k)
    s2, c2 = np.sin(-yaw * k), np.cos(-yaw * k)
    s3, c3 = np.sin(pitch * k), np.cos(pitch * k)
    R = np.stack([c1 * c2 + s1 * s3 * s2, s1 * c3, -c1 * s2 + s1 * s3 * c2,
                  -s1 * c2 + c1 * s3 * s2, c1 * c3, s1 * s2 + c1 * s3 * c2,
                  c3 * s2, -s3, c3 * c2], axis=-1)
    return R.reshape(-1, 3, 3)


def _project(Kl, R, t, X, eR, et):
    """r [B, n, 3] and its error bound dr [B, n, 3] (float64)"""
    r = np.einsum("ij,bjk,nk->bni", Kl, R, X) + np.einsum("ij,bj->bi", Kl, t)[:, None, :]
    aK, aX = np.abs(Kl), np.abs(X)
    A = np.einsum("ij,bjk,nk->bni", aK, np.abs(R), aX) + np.einsum("ij,bj->bi", aK, np.abs(t))[:, None, :]
    dr = 6 * U * A + (eR[:, None, None] * aK.sum(1)[None, None, :] * aX.sum(1)[None, :, None]
                      + np.einsum("ij,bj->bi", aK, et)[:, None, :])
    return r, dr.astype(np.float64), A


def depth_flag(t3, dist, bound):
    """the reference's depth test in float64: both products rounded, strict <"""
    t3, dist = np.asarray(t3, np.float64), np.asarray(dist, np.float64)
    with np.errstate(invalid="ignore"):
        return np.abs(t3 * 100.0 - dist * 100.0) < bound


def report(P, uv, K, R, t, euler, gt, bounds=None, visible=None):
    """P [n, 3], uv [B, n, 2], K [3, 3], R [B, 3, 3], t [B, 3], euler [B, 3] (roll, yaw, pitch), gt [B, 4] (dist, roll, pitch,
    yaw); bounds None = the C default (10, 10, 10, 10); visible bool [B, n] or None.
    Returns dict(report [B, 16] f64, flags [B, 4] i32, max_idx [B, 3] i32, e [B, 3, n] longdouble (NaN where hidden),
    bound [B, 16] f64 (0 where the column is exact), lm_bound [B, 3, n] f64, kappa [B] (largest depth condition number of
    a visible landmark), px [B] (largest pixel magnitude |x| + |y| of a visible landmark))"""
    f = lambda a: np.asarray(a, np.float64)
    P, uv, K, R, t, euler, gt = f(P), f(uv), f(K), f(R).reshape(-1, 3, 3), f(t).reshape(-1, 3), f(euler).reshape(-1, 3), f(gt)
    B, n = uv.shape[0], uv.shape[1]
    bd = np.full(4, 10.0) if bounds is None else f(bounds)
    vis = np.ones((B, n), bool) if visible is None else np.asarray(visible, bool)
    t3, dist = t[:, 2], gt[:, 0]
    roll_e, yaw_e, pitch_e = euler[:, 0], euler[:, 1], euler[:, 2]
    rep = np.zeros((B, 16))
    with np.errstate(all="ignore"):
        rep[:, 0] = t3 - dist
        rep[:, 1], rep[:, 2], rep[:, 3] = roll_e - gt[:, 1], pitch_e - gt[:, 2], yaw_e - gt[:, 3]
        rep[:, 10], rep[:, 11], rep[:, 12], rep[:, 13], rep[:, 14] = t3, dist, roll_e, pitch_e, yaw_e
        flags = np.stack([depth_flag(t3, dist, bd[0]), np.abs(rep[:, 1]) < bd[1], np.abs(rep[:, 2]) < bd[2],
                          np.abs(rep[:, 3]) < bd[3]], 1).astype(np.int32)

        Kl, X = L(1) * K, L(1) * P
        gl = L(1) * gt
        Rg = rot_from_euler_deg(gl[:, 1], gl[:, 3], gl[:, 2])
        tl = L(1) * t
        tg = tl / tl[:, 2:3] * gl[:, 0:1]
        theta = (np.abs(gt[:, 1]) + np.abs(gt[:, 2]) + np.abs(gt[:, 3])) * (np.pi / 180)
        eRg = U * (16 + 4 * theta)
        re, dre, Ae = _project(Kl, L(1) * R, tl, X, np.zeros(B), np.zeros((B, 3)))
        rg, drg, Ag = _project(Kl, Rg, tg, X, eRg, 4 * U * np.abs(tg.astype(np.float64)))
        m = L(1) * np.where(vis[..., None], uv, 0.0)

        def pix(r, dr):
            z = r[..., 2]
            az = np.abs(z)
            p = r[..., :2] / az[..., None]
            h = z / az                                                   # +-1; NaN at depth 0
            pa = np.abs(p.astype(np.float64))
            ep = (dr[..., :2] + pa * dr[..., 2:3]) / az.astype(np.float64)[..., None] + 2 * U * pa
            return p, h, ep

        pe, he, epe = pix(re, dre)
        pg, hg, epg = pix(rg, drg)
        one = L(1)

        def dist3(dx, dy, dh):
            e2 = dx * dx + dy * dy + dh * dh
            e = np.sqrt(e2)
            e[~np.isfinite(e2.astype(np.float64))] = np.nan
            return e

        d0 = m - pg                                                      # LM vs GT (:321)
        d1 = pe - m                                                      # prediction vs LM (:326)
        d2 = d1 + d0                                                     # prediction vs GT (:331), through the pixel
        e0 = dist3(d0[..., 0], d0[..., 1], one - hg)
        e1 = dist3(d1[..., 0], d1[..., 1], he - one)
        e2 = dist3(d2[..., 0], d2[..., 1], he - hg)
        a = lambda x: np.abs(x.astype(np.float64)).sum(-1)
        b0 = epg.sum(-1) + U * a(d0)
        b1 = epe.sum(-1) + U * a(d1)
        b2 = epe.sum(-1) + epg.sum(-1) + U * (a(d0) + a(d1))
        e = np.stack([e0, e1, e2], 1)                                    # [B, 3, n]
        lb = np.stack([b0, b1, b2], 1) + 4 * U * np.nan_to_num(e.astype(np.float64), nan=0.0)
        e[~np.broadcast_to(vis[:, None, :], e.shape)] = np.nan
        lb = np.where(vis[:, None, :] & ~np.isnan(e), lb, 0.0)          # a NaN distance is in no mean and no maximum

        c = vis.sum(1)
        few = c < 4 if visible is not None else np.zeros(B, bool)
        hidden = ~vis[:, None, :]
        s = np.where(hidden, L(0), e).sum(-1)                            # NaN if any visible distance is NaN
        ef = np.where(np.isnan(e), L(-1), e)
        mx = ef.max(-1)
        idx = np.where(mx > 0, ef.argmax(-1), -1).astype(np.int32)
        mx = np.maximum(mx, 0)
        mean = s / c[:, None]
        dl = L(1) * dist[:, None]
        rep[:, [4, 6, 8]] = (mean * dl).astype(np.float64)
        rep[:, [5, 7, 9]] = (mx * dl).astype(np.float64)
        esum = np.where(hidden, 0.0, np.nan_to_num(e.astype(np.float64), nan=0.0)).sum(-1)
        ad = np.abs(dist)[:, None]
        bnd = np.zeros((B, 16))
        bnd[:, [4, 6, 8]] = (lb.sum(-1) + (c[:, None] + 5) * U * esum) / np.maximum(c, 1)[:, None] * ad + \
            2 * U * np.abs(rep[:, [4, 6, 8]])
        bnd[:, [5, 7, 9]] = lb.max(-1) * ad + 2 * U * np.abs(rep[:, [5, 7, 9]])
        rep[few, 4:10] = np.nan
        idx[few] = -1
        bnd[few, 4:10] = 0.0

        zz = np.abs(np.concatenate([re[..., 2], rg[..., 2]], 1)).astype(np.float64)
        Az = np.concatenate([Ae[..., 2], Ag[..., 2]], 1).astype(np.float64)
        kap = np.where(np.concatenate([vis, vis], 1), Az / zz, 0.0).max(1)
        pxm = np.where(vis, np.maximum(a(pe), a(pg)), 0.0).max(1)
    return dict(report=rep, flags=flags, max_idx=idx, e=e, bound=bnd, lm_bound=lb, kappa=kap, px=pxm)


def allowed_max_idx(ref):
    """bool [B, 3, n + 1]: the landmarks (index n stands for -1) a kernel may return as max_idx: the reference's, and at a
    near-tie every landmark whose distance is within the sum of its bound and the maximum's bound of the maximum"""
    e, lb, idx = ref["e"], ref["lm_bound"], ref["max_idx"]
    B, _, n = e.shape
    ok = np.zeros((B, 3, n + 1), bool)
    bi, qi = np.meshgrid(np.arange(B), np.arange(3), indexing="ij")
    ok[bi, qi, np.where(idx >= 0, idx, n)] = True
    ef = np.nan_to_num(e.astype(np.float64), nan=-np.inf)
    top = np.where(idx >= 0, np.take_along_axis(ef, np.maximum(idx, 0)[..., None], -1)[..., 0], 0.0)
    btop = np.where(idx >= 0, np.take_along_axis(lb, np.maximum(idx, 0)[..., None], -1)[..., 0], 0.0)
    near = (ef + lb >= (top - btop)[..., None]) & (ef + lb > 0)
    ok[..., :n] |= near
    ok[..., n] |= top - btop <= 0
    return ok


def max_idx_ok(got, ref):
    """bool [B, 3]: the kernel's max_idx is the reference's or one of a near-tie"""
    ok = allowed_max_idx(ref)
    n = ref["e"].shape[-1]
    g = np.where(got >= 0, got, n)
    return np.take_along_axis(ok, g[..., None].astype(np.int64), -1)[..., 0] & (got >= -1) & (got < n)


def columns_ok(got, ref):
    """bool [B, 16]: exact columns bit-equal (NaN = NaN), columns 4-9 within the bound (NaN exactly where the reference's)"""
    r, b = ref["report"], ref["bound"]
    with np.errstate(invalid="ignore"):
        same = (got == r) | (np.isnan(got) & np.isnan(r))
        near = np.abs(got - r) <= b
    ok = same.copy()
    ok[:, 4:10] |= near[:, 4:10]
    exact = [0, 1, 2, 3, 10, 11, 12, 13, 14, 15]
    ok[:, exact] = np.ascontiguousarray(got[:, exact]).view(np.int64) == np.ascontiguousarray(r[:, exact]).view(np.int64)
    nan_r, nan_g = np.isnan(r[:, exact]), np.isnan(got[:, exact])
    ok[:, exact] |= nan_r & nan_g
    return ok
