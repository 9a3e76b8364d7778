// pnpb200_solvers.cuh -- the four per-problem solvers as device functions.
//
// Each solver is written once against a "points" accessor (normalised correspondences of ONE
// problem) and a lanes-per-problem constant LPP:
//   LPP = 1   one problem per thread (32 problems per warp); sums stay in the thread.
//   LPP = 32  one problem per warp; every lane accumulates a strided subset of the points and
//             the partial normal equations are combined with an xor-butterfly of warp shuffles,
//             which leaves bitwise-identical sums in all lanes, so the small dense solves and the
//             convergence decision are warp-uniform by construction.
//
// Math follows SURVEY.md Appendix A; reference line numbers are cited at each step
// (scripts/PNP_SOLVER_LIB.py unless noted).  The O(n) work per iteration is restricted to the
// terms that actually depend on the state: every block of J^T J that is the state-independent
// moment of the correspondences times a power of gamma is accumulated once per problem.
#pragma once
#include "pnpb200_common.cuh"
#include "pnpb200_math.cuh"

namespace pnpb200 {

template <typename T>
struct SolverPrm {
    int max_it, linear_it;
    T lm_lambda, exit_tol, meas_w, proc_q, proc_d, sigma0, res_old0;
};

template <typename T>
struct Result {
    T R[9], t[3], res;
    int iters;
};

// per-pattern constants kept in shared memory (computed once per CTA)
//   [0..5] M0 = sum theta theta^T (packed 3x3)   [6..8] m0 = sum theta   [9] n
//   [10..19] G = (D^T D)^-1, D = [P | 1]  (packed 4x4; f2_get_D_pinv :3283 is G D^T)
// PNP_PATC (= 20) is defined in pnpb200_common.cuh

template <int LPP, typename T>
PNP_DEV T group_sum(T v)
{
#pragma unroll
    for (int m = LPP / 2; m >= 1; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
    return v;
}
template <int LPP, typename T, int N>
PNP_DEV void group_sum_arr(T (&v)[N])
{
    if (LPP > 1) {
#pragma unroll
        for (int k = 0; k < N; ++k) v[k] = group_sum<LPP, T>(v[k]);
    }
}

PNP_DEV constexpr int s3(int a, int b) { return sym<3>(a, b); }

// -------------------------------------------------------------------------------------------
// block reconstruction of (R, t) from phi = [phi_1(3), phi_2(3), delta_1, delta_2]
// reconstruct_R_t_block_reconstruction :4158-4364
// -------------------------------------------------------------------------------------------
template <typename T>
PNP_DEV void block_reconstruct(const T (&phi)[8], T (&R)[9], T (&t)[3], T& t3)
{
    const T K00 = phi[0], K01 = phi[1], K10 = phi[3], K11 = phi[4];
    const T k1 = K00 * K00 + K10 * K10;                   // K^T K (:4205-4211)
    const T k2 = K00 * K01 + K10 * K11;
    const T k3 = K01 * K01 + K11 * K11;
    const T Dd = (k1 - k3) * (k1 - k3) + T(4) * k2 * k2;  // :4215
    const T gamma2 = T(0.5) * ((k1 + k3) + t_sqrt(Dd));
    const T gamma = t_sqrt(gamma2);
    const T e_se = t_sqrt(gamma2 - k1);                   // :4230
    const T sgn = (k2 > T(0)) ? T(1) : ((k2 < T(0)) ? T(-1) : T(0));   // np.sign
    const T d_se = -sgn * t_sqrt(gamma2 - k3);            // :4233
    const T detK = K00 * K11 - K01 * K10;
    const T ds0 = (K11 * e_se - K10 * d_se) / detK;       // inv(K^T) beta (:4242)
    const T ds1 = (-K01 * e_se + K00 * d_se) / detK;
    const T c = detK / gamma;                             // :4247
    const T a0 = -(c * ds0), a1 = -(c * ds1);             // :4249
    const T sim = a0 * phi[2] + a1 * phi[5];              // :4261
    const T se = (sim < T(0)) ? T(-1) : T(1);             // :4266
    const T ig = T(1) / gamma;
    R[0] = K00 / gamma; R[1] = K01 / gamma; R[2] = (se * a0) / gamma;
    R[3] = K10 / gamma; R[4] = K11 / gamma; R[5] = (se * a1) / gamma;
    R[6] = (se * e_se) / gamma; R[7] = (se * d_se) / gamma; R[8] = c / gamma;   // :4326-4340
    t3 = ig;                                              // :4357
    t[0] = phi[6] * t3; t[1] = phi[7] * t3; t[2] = t3;    // :4360
}

// State-independent moments of one problem's correspondences against the pattern:
//   Mx = sum bx th th^T, My = sum by th th^T, Mw = sum (bx^2+by^2) th th^T   (packed 3x3 each)
//   mx = sum bx th, my = sum by th, mw = sum (bx^2+by^2) th, sx0 = sum bx, sy0 = sum by
// Every block of J^T J of the LM problem is one of these (or the pattern constants M0, m0, n)
// times a power of gamma, and so are the sums of the linear stage F2 (its D^T B and D^T (B o P)).
// PNP_NMOM (= 29) is defined in pnpb200_common.cuh
template <typename T>
struct Moments {
    T Mx[6], My[6], Mw[6], mx[3], my[3], mw[3], sx0, sy0;
    T sw0;                                                // sum (bx^2 + by^2): only the filters' moment-form residual reads it
    PNP_DEV void zero()
    {
#pragma unroll
        for (int e = 0; e < 6; ++e) { Mx[e] = T(0); My[e] = T(0); Mw[e] = T(0); }
#pragma unroll
        for (int e = 0; e < 3; ++e) { mx[e] = T(0); my[e] = T(0); mw[e] = T(0); }
        sx0 = T(0); sy0 = T(0); sw0 = T(0);
    }
    // WITH_W = false skips the (bx^2 + by^2)-weighted moments, which the linear stage F2 never reads;
    // WITH_S adds sum (bx^2 + by^2) itself (QEIF / EIF2 in the moment mapping)
    template <bool WITH_W = true, bool WITH_S = false>
    PNP_DEV void add(const T (&th)[3], T bx, T by)
    {
        const T ww = WITH_W ? (bx * bx + by * by) : T(0);
        if (WITH_S) sw0 += ww;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
#pragma unroll
            for (int b = a; b < 3; ++b) {
                const T m = th[a] * th[b];
                Mx[s3(a, b)] = t_fma(bx, m, Mx[s3(a, b)]);
                My[s3(a, b)] = t_fma(by, m, My[s3(a, b)]);
                if (WITH_W) Mw[s3(a, b)] = t_fma(ww, m, Mw[s3(a, b)]);
            }
            mx[a] = t_fma(bx, th[a], mx[a]);
            my[a] = t_fma(by, th[a], my[a]);
            if (WITH_W) mw[a] = t_fma(ww, th[a], mw[a]);
        }
        sx0 += bx; sy0 += by;
    }
    template <int LPP, bool WITH_W = true, bool WITH_S = false>
    PNP_DEV void reduce()
    {
        group_sum_arr<LPP>(Mx); group_sum_arr<LPP>(My);
        group_sum_arr<LPP>(mx); group_sum_arr<LPP>(my);
        if (WITH_W) { group_sum_arr<LPP>(Mw); group_sum_arr<LPP>(mw); }
        sx0 = group_sum<LPP>(sx0); sy0 = group_sum<LPP>(sy0);
        if (WITH_S) sw0 = group_sum<LPP>(sw0);
    }
    PNP_DEV T gMx(int k) const { return Mx[k]; }
    PNP_DEV T gMy(int k) const { return My[k]; }
    PNP_DEV T gMw(int k) const { return Mw[k]; }
    PNP_DEV T gmx(int k) const { return mx[k]; }
    PNP_DEV T gmy(int k) const { return my[k]; }
    PNP_DEV T gmw(int k) const { return mw[k]; }
    PNP_DEV T gsx0() const { return sx0; }
    PNP_DEV T gsy0() const { return sy0; }
    PNP_DEV T gsw0() const { return sw0; }
    static constexpr bool kHasCore = false;               // the constant blocks of the LM system are recomputed per iteration
    PNP_DEV T gcore(int) const { return T(0); }
    PNP_DEV void set_core(int, T) const {}
    // flat order used for the [PNP_NMOM][B] workspace of the moment mapping
    PNP_DEV T& at(int k)
    {
        return k < 6 ? Mx[k] : k < 12 ? My[k - 6] : k < 18 ? Mw[k - 12] : k < 21 ? mx[k - 18] : k < 24 ? my[k - 21]
               : k < 27 ? mw[k - 24] : (k == 27 ? sx0 : (k == 28 ? sy0 : sw0));
    }
};

// The same 29 moments parked in shared memory, one column per thread ([PNP_NMOM][stride], flat
// order of Moments::at): k_iterate keeps them there so that the registers go to the 10x10 system.
template <typename T>
struct MomentsRef {
    const volatile T* base;   // volatile: re-read per use instead of being hoisted into (spilled) registers
    int stride;
    PNP_DEV T gMx(int k) const { return base[k * stride]; }
    PNP_DEV T gMy(int k) const { return base[(6 + k) * stride]; }
    PNP_DEV T gMw(int k) const { return base[(12 + k) * stride]; }
    PNP_DEV T gmx(int k) const { return base[(18 + k) * stride]; }
    PNP_DEV T gmy(int k) const { return base[(21 + k) * stride]; }
    PNP_DEV T gmw(int k) const { return base[(24 + k) * stride]; }
    PNP_DEV T gsx0() const { return base[27 * stride]; }
    PNP_DEV T gsy0() const { return base[28 * stride]; }
    PNP_DEV T gsw0() const { return base[29 * stride]; }
    // the constant blocks of the delta-eliminated LM system (lm_step): S33 (6), S13 (9), S23 (9) behind the moments,
    // computed once per problem by lm_core_from_moments, followed by the constant right-hand side c (9); S11 = S22 depends on the pattern only (PNP_NCORE = 33)
    static constexpr bool kHasCore = true;
    volatile T* core;
    PNP_DEV T gcore(int k) const { return core[k * stride]; }
    PNP_DEV void set_core(int k, T v) const { core[k * stride] = v; }
};

template <typename T, int LPP, typename Pts, bool WITH_W = true, bool WITH_S = false>
PNP_DEV void accumulate_moments(const Pts& pts, const T* __restrict__ sP, int n, int sub, Moments<T>& mom)
{
    mom.zero();
#pragma unroll (LPP == 32 ? 8 : 4)
    for (int i = sub; i < n; i += LPP) {
        if (!pts.vis(i)) continue;
        const T th[3] = { sP[3 * i], sP[3 * i + 1], sP[3 * i + 2] };
        T bx, by;
        pts.get(i, bx, by);
        mom.template add<WITH_W, WITH_S>(th, bx, by);
    }
    mom.template reduce<LPP, WITH_W, WITH_S>();
}

template <typename T>
PNP_DEV void sym3_mv(const T (&M)[6], const T (&v)[3], T (&o)[3])
{
#pragma unroll
    for (int a = 0; a < 3; ++a) o[a] = M[s3(a, 0)] * v[0] + M[s3(a, 1)] * v[1] + M[s3(a, 2)] * v[2];
}
template <typename T>
PNP_DEV T dot3(const T (&a)[3], const T (&b)[3]) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }

// ||z - hx||^2 over the 2n measurement rows from the moments (filters in the moment mapping).  With g1 = P u1 - bx o P u3,
// g2 = P u2 - by o P u3 the residual is (bx - d1 - gamma g1, by - d2 - gamma g2), so
//   res^2 = sum (bx - d1)^2 + (by - d2)^2  -  2 gamma sum [(bx - d1) g1 + (by - d2) g2]  +  gamma^2 sum (g1^2 + g2^2)
//         = sw0 - 2 (d1 sx0 + d2 sy0) + n (d1^2 + d2^2) - 2 gamma (qa - d1 s1 - d2 s2) + gamma^2 sgg
// with s_k = sum g_k, sgg = sum g1^2 + g2^2, qa = sum bx g1 + by g2 = mx.u1 + my.u2 - mw.u3 (QEIF: u = phi(q), gamma = 1).
// A difference of terms ~|z|^2 / res^2 larger than the result: good to ~1e-10 relative on detected (quantised / noisy) pixels,
// where res ~ 1e-2 |z| -- far inside what the filters' early-exit test (|d res / res| < 1e-2, :2952, :2202) needs; rounding
// noise where the residual itself is (noise-free pixels, res ~ 1e-14), exactly as the reference's own decision is there.
// The reported res_norm never comes from here: it is evaluated point by point in the residual pass.
// The moment-form res^2 carries an absolute error of about res2_error_bound() -- the moments are sums of n products (worst
// case n eps / 2 relative each) combined with cancellation -- so an exit decision taken from it is CERTIFIED only when
// | |ratio| - tol | exceeds the error that bound implies for the ratio; otherwise the lane stops and marks its problem
// (iters = -1), and the fix-up pass of the moment mapping re-solves the marked problems point by point with the direct
// kernel's arithmetic.  On detected pixels a few problems per million are marked; on noise-free pixels, where the
// residual falls to rounding noise, most are -- the result is the direct mapping's either way.
template <typename T>
PNP_DEV T res2_error_bound(T n, T sw0, T gam, T d1, T d2, T tr_m0, T tr_mw, T u11_plus_u22, T u33)
{
    const T scale = sw0 + (gam * gam) * t_fma(tr_m0, u11_plus_u22, tr_mw * u33) + n * t_fma(d1, d1, d2 * d2);
    const T eps = (sizeof(T) == 8) ? T(1.1102230246251565e-16) : T(5.9604645e-8);
    return (T(2) * n + T(16)) * eps * scale;
}

template <typename T>
PNP_DEV T res2_combine(T sw0, T sx0, T sy0, T n, T d1, T d2, T gam, T qa, T s1, T s2, T sgg)
{
    const T a0 = t_fma(n, t_fma(d1, d1, d2 * d2), t_fma(T(-2), t_fma(d1, sx0, d2 * sy0), sw0));
    const T a1 = qa - t_fma(d1, s1, d2 * s2);
    const T r2 = t_fma(gam * gam, sgg, t_fma(T(-2) * gam, a1, a0));
    return r2 > T(0) ? r2 : T(0);
}

// is the decision |ratio| < tol safe against the error bounds e_new, e_old of the two squared residuals behind the ratio?
template <typename T>
PNP_DEV bool exit_decision_uncertain(T ratio_abs, T tol, T r2_new, T e_new, T r2_old, T e_old)
{
    if (!(r2_new > T(4) * e_new)) return true;                 // the residual itself is noise (or NaN)
    const T dn = e_new * t_rcp<T>(r2_new);
    const T dold = (e_old > T(0)) ? e_old * t_rcp<T>(r2_old) : T(0);
    return !(t_abs(ratio_abs - tol) > (T(1) + ratio_abs) * (dn + dold));
}

// -------------------------------------------------------------------------------------------
// QEIF -- solve_pnp_QEIF_single_pattern :2771-3025, QEKF_get_hx_H :3902-3983,
//         QEKF_reconstruct_R_t_m1 :3542-3609
// -------------------------------------------------------------------------------------------
template <typename T>
PNP_DEV void qekf_phi(const T (&x)[6], T (&p1)[3], T (&p2)[3], T (&p3)[3], T& gamma)
{
    const T qr = x[0], qi = x[1], qj = x[2], qk = x[3];
    const T nq = t_sqrt(qr * qr + qi * qi + qj * qj + qk * qk);
    gamma = nq * nq;                                      // (np.linalg.norm(q))**2 (:3918)
    const T qii = qi * qi, qjj = qj * qj, qkk = qk * qk;
    const T qij = qi * qj, qjk = qj * qk, qik = qi * qk;
    const T qri = qr * qi, qrj = qr * qj, qrk = qr * qk;
    p1[0] = gamma - 2 * (qjj + qkk); p1[1] = 2 * (qij - qrk); p1[2] = 2 * (qik + qrj);   // :3934
    p2[0] = 2 * (qij + qrk); p2[1] = gamma - 2 * (qii + qkk); p2[2] = 2 * (qjk - qri);   // :3935
    p3[0] = 2 * (qik - qrj); p3[1] = 2 * (qjk + qri); p3[2] = gamma - 2 * (qii + qjj);   // :3936
}

// HYBRID = false: H^T Q^-1 H and H^T Q^-1 (z - hx + H x) are accumulated point by point each
// iteration (best for the 6-landmark subset).  HYBRID = true: they are bilinear forms of the 29
// moments (Q_j q = 2 phi_j, so z - hx + H x = b + (P phi_1 - b o P phi_3): no cancellation), and only
// the residual ||z - hx|| that drives the early-exit test is still evaluated point by point.
// RES_MOM (moment mapping, implies HYBRID): the residual of the early-exit test comes from the moments too
// (res2_combine), no point is touched inside the loop; x_tail receives what the residual pass needs to evaluate the
// reported res_norm point by point -- the measurement model at the state BEFORE the lane's last update, in the
// 12-number form of LM's residual (phi_1, phi_2, phi_3, delta_1, delta_2, gamma = 1).
template <typename T, int LPP, typename Pts, bool HYBRID, bool RES_MOM, bool WANT_TAIL = RES_MOM>
PNP_DEV void qeif_loop(const Pts& pts, const T* __restrict__ sP, const T* __restrict__ sC, int n, int sub,
                       const SolverPrm<T>& prm, const Moments<T>& mom, T (&x_tail)[12], Result<T>& out)
{
    T x[6] = { T(1), T(0), T(0), T(0), T(0), T(0) };      // :2831-2833
    if (WANT_TAIL) {
#pragma unroll
        for (int e = 0; e < 12; ++e) x_tail[e] = (e == 0 || e == 4 || e == 8 || e == 11) ? T(1) : T(0);
    }
    bool flagged = false;                                 // RES_MOM: an exit decision could not be certified
    T r2_old = T(0), e_old = T(0);
    // One 6 x 6 array carries Sigma from one iteration to the next and Omega inside it.  Lanes that have
    // left the loop (done) keep their x, res and iters; what their matrix becomes no longer matters.
    T Om[21];
#pragma unroll
    for (int e = 0; e < 21; ++e) Om[e] = T(0);
#pragma unroll
    for (int i = 0; i < 6; ++i) Om[sidx<6>(i, i)] = prm.sigma0;   // pinv(1e-5 I) (:2836-2837)
    T res_old = prm.res_old0, res = T(1e5);
    bool done = false;
    int iters = 0;
    const T w = prm.meas_w;                               // 1 / (9 / f^2) (:2844-2852)
    const T nT = T(pts.count(n));                        // landmarks taking part (the visible ones under a mask)

    for (int it = 0; it < prm.max_it; ++it) {
        if (LPP == 1) { if (__all_sync(0xffffffffu, done)) break; }
        else          { if (done) break; }
        // ---- predict: Omega = pinv(Sigma + R) (:2887), zeta = Omega x (:2889)
#pragma unroll
        for (int i = 0; i < 6; ++i) Om[sidx<6>(i, i)] += (i < 4) ? prm.proc_q : prm.proc_d;
        spd_inverse<T, 6>(Om);
        T zeta[6];
        sym_matvec<T, 6>(Om, x, zeta);
        // ---- measurement model at x (:3902-3983)
        T p1[3], p2[3], p3[3], gamma;
        qekf_phi<T>(x, p1, p2, p3, gamma);
        const T r2 = 2 * x[0], i2 = 2 * x[1], j2 = 2 * x[2], k2 = 2 * x[3];
        const T Q1[12] = { r2, i2, -j2, -k2, -k2, j2, i2, -r2, j2, k2, r2, i2 };     // :3945
        const T Q2[12] = { k2, j2, i2, r2, r2, -i2, j2, -k2, -i2, -r2, k2, j2 };     // :3949
        const T Q3[12] = { -j2, k2, -r2, i2, i2, r2, k2, j2, r2, -i2, -j2, k2 };     // :3953
        T qq[10], qd1[4], qd2[4], hv[6], res2 = T(0), res2_err = T(0);
        if (!HYBRID) {
#pragma unroll
            for (int e = 0; e < 10; ++e) qq[e] = T(0);
#pragma unroll
            for (int e = 0; e < 4; ++e) { qd1[e] = T(0); qd2[e] = T(0); }
#pragma unroll
            for (int e = 0; e < 6; ++e) hv[e] = T(0);
            for (int i = sub; i < n; i += LPP) {
                if (!pts.vis(i)) continue;
                const T th0 = sP[3 * i], th1 = sP[3 * i + 1], th2 = sP[3 * i + 2];
                T bx, by;
                pts.get(i, bx, by);
                const T P1 = th0 * p1[0] + th1 * p1[1] + th2 * p1[2];
                const T P2 = th0 * p2[0] + th1 * p2[1] + th2 * p2[2];
                const T P3 = th0 * p3[0] + th1 * p3[1] + th2 * p3[2];
                const T dzx = bx - (P1 - bx * P3 + x[4]);     // z - hx (:3969, :2905)
                const T dzy = by - (P2 - by * P3 + x[5]);     // :3970
                T Hx[4], Hy[4];
                T hxq = x[4], hyq = x[5];                     // (H x) rows: Hq . q + delta
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const T a1 = th0 * Q1[c] + th1 * Q1[4 + c] + th2 * Q1[8 + c];
                    const T a2 = th0 * Q2[c] + th1 * Q2[4 + c] + th2 * Q2[8 + c];
                    const T a3 = th0 * Q3[c] + th1 * Q3[4 + c] + th2 * Q3[8 + c];
                    Hx[c] = a1 - bx * a3;                     // :3979
                    Hy[c] = a2 - by * a3;                     // :3980
                    hxq = t_fma(Hx[c], x[c], hxq);
                    hyq = t_fma(Hy[c], x[c], hyq);
                }
                const T vx = dzx + hxq, vy = dzy + hyq;       // z - hx + H x (:2898)
#pragma unroll
                for (int a = 0; a < 4; ++a) {
#pragma unroll
                    for (int b = a; b < 4; ++b)
                        qq[sidx<4>(a, b)] = t_fma(Hx[a], Hx[b], t_fma(Hy[a], Hy[b], qq[sidx<4>(a, b)]));
                    qd1[a] += Hx[a];
                    qd2[a] += Hy[a];
                    hv[a] = t_fma(Hx[a], vx, t_fma(Hy[a], vy, hv[a]));
                }
                hv[4] += vx; hv[5] += vy;
                res2 = t_fma(dzx, dzx, t_fma(dzy, dzy, res2));
            }
            group_sum_arr<LPP>(qq); group_sum_arr<LPP>(qd1); group_sum_arr<LPP>(qd2); group_sum_arr<LPP>(hv);
            res2 = group_sum<LPP>(res2);
        } else {
            if (!RES_MOM) {
                // ---- residual, point by point (:2905-2907)
#pragma unroll 4
                for (int i = sub; i < n; i += LPP) {
                    if (!pts.vis(i)) continue;
                    const T th0 = sP[3 * i], th1 = sP[3 * i + 1], th2 = sP[3 * i + 2];
                    T bx, by;
                    pts.get(i, bx, by);
                    const T P1 = th0 * p1[0] + th1 * p1[1] + th2 * p1[2];
                    const T P2 = th0 * p2[0] + th1 * p2[1] + th2 * p2[2];
                    const T P3 = th0 * p3[0] + th1 * p3[1] + th2 * p3[2];
                    const T dzx = bx - (P1 - bx * P3 + x[4]);
                    const T dzy = by - (P2 - by * P3 + x[5]);
                    res2 = t_fma(dzx, dzx, t_fma(dzy, dzy, res2));
                }
                res2 = group_sum<LPP>(res2);
            }
            // ---- H^T H and H^T (z - hx + H x) from the moments
            const T M0[6] = { sC[0], sC[1], sC[2], sC[3], sC[4], sC[5] };
            const T m0[3] = { sC[6], sC[7], sC[8] };
            T q1[4][3], q2[4][3], q3[4][3], a1[4][3], a2[4][3], bxv[4][3], byv[4][3], cw[4][3];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
#pragma unroll
                for (int k = 0; k < 3; ++k) { q1[c][k] = Q1[4 * k + c]; q2[c][k] = Q2[4 * k + c]; q3[c][k] = Q3[4 * k + c]; }
                sym3_mv<T>(M0, q1[c], a1[c]); sym3_mv<T>(M0, q2[c], a2[c]);
                sym3_mv<T>(mom.Mx, q3[c], bxv[c]); sym3_mv<T>(mom.My, q3[c], byv[c]); sym3_mv<T>(mom.Mw, q3[c], cw[c]);
                qd1[c] = dot3<T>(q1[c], m0) - dot3<T>(q3[c], mom.mx);
                qd2[c] = dot3<T>(q2[c], m0) - dot3<T>(q3[c], mom.my);
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) {
#pragma unroll
                for (int d = c; d < 4; ++d)
                    qq[sidx<4>(c, d)] = dot3<T>(q1[c], a1[d]) + dot3<T>(q2[c], a2[d]) - (dot3<T>(q1[c], bxv[d]) + dot3<T>(q1[d], bxv[c]))
                                        - (dot3<T>(q2[c], byv[d]) + dot3<T>(q2[d], byv[c])) + dot3<T>(q3[c], cw[d]);
            }
            T e1[3], e2[3], e3[3], t1[3], t2[3], t3v[3], t4[3], t5[3], t6[3], t7[3];
            sym3_mv<T>(M0, p1, t1); sym3_mv<T>(mom.Mx, p3, t2);            // M0 phi1, Mx phi3
            sym3_mv<T>(M0, p2, t3v); sym3_mv<T>(mom.My, p3, t4);           // M0 phi2, My phi3
            sym3_mv<T>(mom.Mx, p1, t5); sym3_mv<T>(mom.My, p2, t6); sym3_mv<T>(mom.Mw, p3, t7);
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                e1[k] = mom.mx[k] + t1[k] - t2[k];
                e2[k] = mom.my[k] + t3v[k] - t4[k];
                e3[k] = mom.mw[k] + t5[k] + t6[k] - t7[k];
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) hv[c] = dot3<T>(q1[c], e1) + dot3<T>(q2[c], e2) - dot3<T>(q3[c], e3);
            const T s1 = dot3<T>(m0, p1) - dot3<T>(mom.mx, p3), s2 = dot3<T>(m0, p2) - dot3<T>(mom.my, p3);
            hv[4] = mom.sx0 + s1;
            hv[5] = mom.sy0 + s2;
            if (RES_MOM) {                                    // ||z - hx||^2 from the moments (:2905-2907)
                const T qa = dot3<T>(mom.mx, p1) + dot3<T>(mom.my, p2) - dot3<T>(mom.mw, p3);
                const T sgg = dot3<T>(p1, t1) - T(2) * dot3<T>(p1, t2) + dot3<T>(p2, t3v) - T(2) * dot3<T>(p2, t4) + dot3<T>(p3, t7);
                res2 = res2_combine<T>(mom.sw0, mom.sx0, mom.sy0, nT, x[4], x[5], T(1), qa, s1, s2, sgg);
                res2_err = res2_error_bound<T>(nT, mom.sw0, T(1), x[4], x[5], M0[0] + M0[3] + M0[5], mom.Mw[0] + mom.Mw[3] + mom.Mw[5],
                                               dot3<T>(p1, p1) + dot3<T>(p2, p2), dot3<T>(p3, p3));
            }
        }
        // ---- update: Omega += H^T Q^-1 H, zeta += H^T Q^-1 (z - hx + H x) (:2896-2898)
#pragma unroll
        for (int a = 0; a < 4; ++a) {
#pragma unroll
            for (int b = a; b < 4; ++b) Om[sidx<6>(a, b)] = t_fma(w, qq[sidx<4>(a, b)], Om[sidx<6>(a, b)]);
            Om[sidx<6>(a, 4)] = t_fma(w, qd1[a], Om[sidx<6>(a, 4)]);
            Om[sidx<6>(a, 5)] = t_fma(w, qd2[a], Om[sidx<6>(a, 5)]);
        }
        Om[sidx<6>(4, 4)] = t_fma(w, nT, Om[sidx<6>(4, 4)]);
        Om[sidx<6>(5, 5)] = t_fma(w, nT, Om[sidx<6>(5, 5)]);
#pragma unroll
        for (int a = 0; a < 6; ++a) zeta[a] = t_fma(w, hv[a], zeta[a]);
        const T res_new = t_sqrt_nn<T>(res2);                   // :2905-2907
        // ---- x = pinv(Omega) zeta (:2924-2925)
        spd_inverse<T, 6>(Om);
        T xn[6];
        sym_matvec<T, 6>(Om, zeta, xn);
        if (!done) {
            if (WANT_TAIL) {
#pragma unroll
                for (int k = 0; k < 3; ++k) { x_tail[k] = p1[k]; x_tail[3 + k] = p2[k]; x_tail[6 + k] = p3[k]; }
                x_tail[9] = x[4]; x_tail[10] = x[5]; x_tail[11] = T(1);
            }
#pragma unroll
            for (int e = 0; e < 6; ++e) x[e] = xn[e];
            res = res_new;
            ++iters;
            const T ratio = (res - res_old) * t_rcp<T>(res_old);   // 0 / 0 and x / 0 both end up not-below-tolerance, as in the reference    // :2945
            res_old = res;
            if (t_abs(ratio) < prm.exit_tol) done = true; // :2952
            if (RES_MOM) {
                if (exit_decision_uncertain<T>(t_abs(ratio), prm.exit_tol, res2, res2_err, r2_old, e_old)) { flagged = true; done = true; }
                r2_old = res2; e_old = res2_err;
            }
        }
    }
    // ---- QEKF_reconstruct_R_t_m1 :3590-3605
    T p1[3], p2[3], p3[3], gamma;
    qekf_phi<T>(x, p1, p2, p3, gamma);
#pragma unroll
    for (int k = 0; k < 3; ++k) { out.R[k] = p1[k] / gamma; out.R[3 + k] = p2[k] / gamma; out.R[6 + k] = p3[k] / gamma; }
    const T t3 = T(1) / gamma;
    out.t[0] = x[4] * t3; out.t[1] = x[5] * t3; out.t[2] = t3;
    out.res = res;
    out.iters = flagged ? -1 : iters;
}

template <typename T, int LPP, typename Pts, bool HYBRID>
PNP_DEV void solve_qeif(const Pts& pts, const T* __restrict__ sP, const T* __restrict__ sC, int n, int sub,
                        const SolverPrm<T>& prm, Result<T>& out)
{
    Moments<T> mom;
    if (HYBRID) accumulate_moments<T, LPP, Pts>(pts, sP, n, sub, mom);
    T unused[12];
    qeif_loop<T, LPP, Pts, HYBRID, false>(pts, sP, sC, n, sub, prm, mom, unused, out);
}

template <typename T, int LPP, typename Pts>
PNP_DEV void solve_qeif_with_tail(const Pts& pts, const T* __restrict__ sP, const T* __restrict__ sC, int n, int sub,
                                  const SolverPrm<T>& prm, T (&x_tail)[12], Result<T>& out)
{
    Moments<T> mom;
    accumulate_moments<T, LPP, Pts>(pts, sP, n, sub, mom);
    qeif_loop<T, LPP, Pts, true, false, true>(pts, sP, sC, n, sub, prm, mom, x_tail, out);
}

// No points inside the loop (moment mapping)
struct NoPts {
    template <typename T> PNP_DEV void get(int, T& bx, T& by) const { bx = T(0); by = T(0); }
    PNP_DEV bool vis(int) const { return true; }
    PNP_DEV int count(int n) const { return n; }
};

template <typename T>
PNP_DEV void solve_qeif_from_moments(const Moments<T>& mom, const T* __restrict__ sC, const SolverPrm<T>& prm, T (&x_tail)[12],
                                     Result<T>& out)
{
    NoPts none;
    qeif_loop<T, 1, NoPts, true, true>(none, nullptr, sC, (int)sC[9], 0, prm, mom, x_tail, out);
}

// -------------------------------------------------------------------------------------------
// LM -- solve_pnp_LM_single_pattern :2567-2769, EKF2_get_hx_H :3718-3836,
//       EKF2_reconstruct_R_t_m1 :3500-3540
// state x = [u1(3), u2(3), u3(3), delta_1, delta_2, gamma]
// -------------------------------------------------------------------------------------------
// The gamma column of J^T J as bilinear forms of the moments (terms have the size of the result):
//   sg1 = sum th g1 = M0 u1 - Mx u3;  sg2 = M0 u2 - My u3;  sg3 = sum th (bx g1 + by g2) = Mx u1 + My u2 - Mw u3
//   s1 = sum g1 = m0.u1 - mx.u3;  s2 = m0.u2 - my.u3;  sgg = sum g1^2 + g2^2 = u1.sg1 + u2.sg2 - u3.sg3
template <typename T>
struct GammaCol { T sg1[3], sg2[3], sg3[3], s1, s2, sgg; };

template <typename T, typename M>
PNP_DEV void lm_gamma_column(const T (&x)[12], const M& m, const T* __restrict__ sC, GammaCol<T>& gc)
{
    gc.s1 = T(0); gc.s2 = T(0); gc.sgg = T(0);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        T e1 = T(0), e2 = T(0), e3 = T(0);
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const T mxkj = m.gMx(s3(k, j)), mykj = m.gMy(s3(k, j));
            e1 = t_fma(sC[s3(k, j)], x[j], t_fma(-mxkj, x[6 + j], e1));
            e2 = t_fma(sC[s3(k, j)], x[3 + j], t_fma(-mykj, x[6 + j], e2));
            e3 = t_fma(mxkj, x[j], t_fma(mykj, x[3 + j], t_fma(-m.gMw(s3(k, j)), x[6 + j], e3)));
        }
        gc.sg1[k] = e1; gc.sg2[k] = e2; gc.sg3[k] = e3;
        gc.s1 = t_fma(sC[6 + k], x[k], t_fma(-m.gmx(k), x[6 + k], gc.s1));
        gc.s2 = t_fma(sC[6 + k], x[3 + k], t_fma(-m.gmy(k), x[6 + k], gc.s2));
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) gc.sgg = t_fma(x[k], gc.sg1[k], t_fma(x[3 + k], gc.sg2[k], t_fma(-x[6 + k], gc.sg3[k], gc.sgg)));
}

template <typename T, typename M>
PNP_DEV T res2_from_moments(const M& m, const T* __restrict__ sC, const GammaCol<T>& gc, T qa, T gam, T d1, T d2)
{
    return res2_combine<T>(m.gsw0(), m.gsx0(), m.gsy0(), sC[9], d1, d2, gam, qa, gc.s1, gc.s2, gc.sgg);
}

// J^T (z - hx) of the 2n measurement rows
template <typename T>
struct LmRhs { T r1[3], r2[3], r3[3], q1, q2, qg; };

// ... from the moments (moment mapping).  Unlike the gamma column these are differences of terms
// ~|z|/|z - hx| larger than the result; the rounding this adds to the step is ~1e3 times smaller
// than the effect of a 1e-13 relative input perturbation, which is what defines the parity subset.
template <typename T, typename M>
PNP_DEV void lm_rhs_from_moments(const T (&x)[12], const M& m, const T* __restrict__ sC, const GammaCol<T>& gc, LmRhs<T>& r)
{
    const T gam = x[11], d1 = x[9], d2 = x[10];
    T qa = T(0);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const T mxk = m.gmx(k), myk = m.gmy(k), mwk = m.gmw(k);
        r.r1[k] = mxk - gam * gc.sg1[k] - d1 * sC[6 + k];
        r.r2[k] = myk - gam * gc.sg2[k] - d2 * sC[6 + k];
        r.r3[k] = mwk - gam * gc.sg3[k] - d1 * mxk - d2 * myk;
        qa = t_fma(mxk, x[k], t_fma(myk, x[3 + k], t_fma(-mwk, x[6 + k], qa)));
    }
    r.q1 = m.gsx0() - gam * gc.s1 - sC[9] * d1;
    r.q2 = m.gsy0() - gam * gc.s2 - sC[9] * d2;
    r.qg = qa - gam * gc.sgg - d1 * gc.s1 - d2 * gc.s2;
}

// The per-problem constant blocks of lm_step's system, for moment containers that can hold them
template <typename T, typename M>
PNP_DEV void lm_core_from_moments(const M& m, const T* __restrict__ sC, T ip)
{
    if (!M::kHasCore) return;
    const T m0[3] = { sC[6], sC[7], sC[8] };
    const T mx[3] = { m.gmx(0), m.gmx(1), m.gmx(2) }, my[3] = { m.gmy(0), m.gmy(1), m.gmy(2) };
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int b = a; b < 3; ++b)
            m.set_core(s3(a, b), t_fma(-(mx[a] * ip), mx[b], t_fma(-(my[a] * ip), my[b], m.gMw(s3(a, b)))));
#pragma unroll
        for (int b = 0; b < 3; ++b) {
            m.set_core(6 + a * 3 + b, t_fma(m0[a] * ip, mx[b], -m.gMx(s3(a, b))));
            m.set_core(15 + a * 3 + b, t_fma(m0[a] * ip, my[b], -m.gMy(s3(a, b))));
        }
    }
    // constant part of the reduced right-hand side (lm_step_core): c1 = mx - m0 sx0 / p, c2 = my - m0 sy0 / p,
    // c3 = (mx sx0 + my sy0) / p - mw
    const T sxp = m.gsx0() * ip, syp = m.gsy0() * ip;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        m.set_core(24 + a, t_fma(-m0[a], sxp, mx[a]));
        m.set_core(27 + a, t_fma(-m0[a], syp, my[a]));
        m.set_core(30 + a, t_fma(mx[a], sxp, t_fma(my[a], syp, -m.gmw(a))));
    }
}

// Second half of an LM step, common to both ways of building the reduced system: the nine constraint
// rows are added to A (10 x 10 packed, order y_u1, y_u2, y_u3, d gamma) and g, the system is solved, the
// two deltas are back-substituted and the state is updated.  s_k, q_k: the delta_k column / right-hand side
// of the measurement rows (s1 = sum g1, q1 = sum (z - hx)_x).  Returns max |dx|.
template <typename T, bool TRUE_JAC>
PNP_DEV T lm_finish(T (&x)[12], T (&A)[55], T (&g)[10], const T (&m0)[3], const T (&mx)[3], const T (&my)[3],
                    T s1, T s2, T q1, T q2, T ig, T ip)
{
    constexpr int U1 = 0, U2 = 3, U3 = 6, GG = 9;
    // ---- the nine constraint rows (:3753-3772, Jacobians :3787-3823 incl. the halved ones), times 1 / gamma
    {
        const T u1[3] = { x[0], x[1], x[2] }, u2[3] = { x[3], x[4], x[5] }, u3[3] = { x[6], x[7], x[8] };
        const T u11 = u1[0] * u1[0] + u1[1] * u1[1] + u1[2] * u1[2];
        const T u22 = u2[0] * u2[0] + u2[1] * u2[1] + u2[2] * u2[2];
        const T u33 = u3[0] * u3[0] + u3[1] * u3[1] + u3[2] * u3[2];
        const T u13 = u1[0] * u3[0] + u1[1] * u3[1] + u1[2] * u3[2];
        const T u23 = u2[0] * u3[0] + u2[1] * u3[1] + u2[2] * u3[2];
        const T u12 = u1[0] * u2[0] + u1[1] * u2[1] + u1[2] * u2[2];
        // |u| and 1 / (kn |u|) from one reciprocal square root each
        const T y1 = t_rsqrt<T>(u11), y2 = t_rsqrt<T>(u22), y3 = t_rsqrt<T>(u33);
        const T n1 = t_sqrt_fast<T>(u11, y1), n2 = t_sqrt_fast<T>(u22, y2), n3 = t_sqrt_fast<T>(u33, y3);
        constexpr T kq = TRUE_JAC ? T(2) : T(1), kn = TRUE_JAC ? T(1) : T(2);
        const T w1[3] = { u1[0] * ig, u1[1] * ig, u1[2] * ig };          // u / gamma
        const T w2[3] = { u2[0] * ig, u2[1] * ig, u2[2] * ig };
        const T w3[3] = { u3[0] * ig, u3[1] * ig, u3[2] * ig };
        // The nine rows r_k (each with two non-zero blocks at most) enter as sum_k r_k^T r_k and sum_k r_k^T e_k.
        // Collected per block instead of row by row:
        //   diagonal block i:     w1 w1^T + w2 w2^T + w3 w3^T + (2 kq^2 + h_i^2 - 1) w_i w_i^T
        //   block (i, j), i < j:  w_j w_i^T - kq^2 w_i w_j^T
        //   right-hand side i:    sum_{j != i} w_j e_ij + w_i (kq (+-e_4..6) + h_i (1 - |u_i|))
        // with h_i = 1 / (kn |u_i|): 36 FMAs less than nine rank-one updates, same sums.
        const T h1 = y1 * (T(1) / kn), h2 = y2 * (T(1) / kn), h3 = y3 * (T(1) / kn);
        constexpr T kq2 = kq * kq;
        const T e13 = -u13, e23 = -u23, e12 = -u12;
        const T e4 = u33 - u11, e5 = u33 - u22, e6 = u22 - u11;       // rows 4-6: -(u_ii - u_jj)
        const T c1 = t_fma(h1, h1, T(2) * kq2 - T(1)), c2 = t_fma(h2, h2, T(2) * kq2 - T(1)), c3 = t_fma(h3, h3, T(2) * kq2 - T(1));
        const T q1[3] = { c1 * w1[0], c1 * w1[1], c1 * w1[2] };
        const T q2[3] = { c2 * w2[0], c2 * w2[1], c2 * w2[2] };
        const T q3[3] = { c3 * w3[0], c3 * w3[1], c3 * w3[2] };
        const T k1[3] = { kq2 * w1[0], kq2 * w1[1], kq2 * w1[2] }, k2[3] = { kq2 * w2[0], kq2 * w2[1], kq2 * w2[2] };
        const T f1c = t_fma(h1, T(1) - n1, kq * (e4 + e6));           // rows 4, 6 (+u1) and 7
        const T f2c = t_fma(h2, T(1) - n2, kq * (e5 - e6));           // rows 5 (+u2), 6 (-u2) and 8
        const T f3c = t_fma(h3, T(1) - n3, -kq * (e4 + e5));          // rows 4, 5 (-u3) and 9
#pragma unroll
        for (int a = 0; a < 3; ++a) {
#pragma unroll
            for (int b = a; b < 3; ++b) {
                const T W = t_fma(w1[a], w1[b], t_fma(w2[a], w2[b], w3[a] * w3[b]));
                A[sidx<10>(U1 + a, U1 + b)] += t_fma(q1[a], w1[b], W);
                A[sidx<10>(U2 + a, U2 + b)] += t_fma(q2[a], w2[b], W);
                A[sidx<10>(U3 + a, U3 + b)] += t_fma(q3[a], w3[b], W);
            }
#pragma unroll
            for (int b = 0; b < 3; ++b) {
                A[sidx<10>(U1 + a, U3 + b)] = t_fma(w3[a], w1[b], t_fma(-k1[a], w3[b], A[sidx<10>(U1 + a, U3 + b)]));
                A[sidx<10>(U2 + a, U3 + b)] = t_fma(w3[a], w2[b], t_fma(-k2[a], w3[b], A[sidx<10>(U2 + a, U3 + b)]));
                A[sidx<10>(U1 + a, U2 + b)] = t_fma(w2[a], w1[b], -k1[a] * w2[b]);          // the core has no (u1, u2) block
            }
            g[U1 + a] = t_fma(w3[a], e13, t_fma(w2[a], e12, t_fma(w1[a], f1c, g[U1 + a])));
            g[U2 + a] = t_fma(w3[a], e23, t_fma(w1[a], e12, t_fma(w2[a], f2c, g[U2 + a])));
            g[U3 + a] = t_fma(w1[a], e13, t_fma(w2[a], e23, t_fma(w3[a], f3c, g[U3 + a])));
        }
    }
    ldlt_factor<T, 10>(A);
    ldlt_solve<T, 10>(A, g);
    // ---- back-substitute the two deltas: d_k = (rhs_k - column_k . y) / p; the back substitution
    // delivers g[9] first and g[0] last: consume them in that order
    T e1 = t_fma(-s1, g[GG], q1), e2 = t_fma(-s2, g[GG], q2);
#pragma unroll
    for (int a = 2; a >= 0; --a) { e1 = t_fma(mx[a], g[U3 + a], e1); e2 = t_fma(my[a], g[U3 + a], e2); }
#pragma unroll
    for (int a = 2; a >= 0; --a) { e1 = t_fma(-m0[a], g[U1 + a], e1); e2 = t_fma(-m0[a], g[U2 + a], e2); }
    T step = t_abs(g[GG]);
#pragma unroll
    for (int i = 0; i < 9; ++i) step = fmax(step, t_abs(g[i] * ig));
    step = fmax(step, fmax(t_abs(e1 * ip), t_abs(e2 * ip)));
#pragma unroll
    for (int i = 0; i < 9; ++i) x[i] = t_fma(g[i], ig, x[i]);
    x[9] += e1 * ip; x[10] += e2 * ip; x[11] += g[GG];
    return step;
}

// One damped Gauss-Newton step: A = J^T J + lambda I (:2666-2667) from the moments and the gamma
// column, g = J^T (z - hx) (:2684) from `r`, the nine constraint rows, x += pinv(A) g (:2675, :2702).
//
// Solved in the variables y = (gamma du1, gamma du2, gamma du3, d gamma) -- a diagonal scaling of the
// same linear system.  Every measurement row then has constant coefficients in (y_u, d delta), so
// after delta_1 and delta_2 are eliminated (their pivots are the constant n + lambda, they do not
// couple to each other) the 9 x 9 core of the matrix is a per-problem constant of the moments:
//   S11 = S22 = M0 - m0 m0^T / p,  S12 = 0,  S13 = -Mx + m0 mx^T / p,  S23 = -My + m0 my^T / p,
//   S33 = Mw - (mx mx^T + my my^T) / p,                                        p = n + lambda
// and per iteration only lambda / gamma^2 on its diagonal, the gamma column / row, the right-hand
// side and the nine constraint rows (scaled by 1 / gamma) change.  What is factorised is the
// 10 x 10 Schur complement on (y_u1, y_u2, y_u3, d gamma) -- the LDL^T of the 12 x 12 matrix with the
// two delta columns ordered first, written out.
// TRUE_JAC = false reproduces the reference's constraint Jacobians (rows 4-6 use u, rows 7-9 use
// u/(2|u|)); true uses the actual gradients (2u, u/|u|) and is only used by the non-parity LM+.
// Returns max |dx|.
template <typename T, typename M, bool TRUE_JAC = false>
PNP_DEV T lm_step(T (&x)[12], const M& m, const T* __restrict__ sC, const GammaCol<T>& gc, const LmRhs<T>& r,
                  T lambda, T ip /* 1 / (n + lambda), loop-invariant */)
{
    constexpr int U1 = 0, U2 = 3, U3 = 6, GG = 9;       // order inside the reduced system
    const T gam = x[11];
    const T ig = t_rcp<T>(gam);
    const T lg = lambda * (ig * ig);                    // lambda I in the scaled variables
    const T m0[3] = { sC[6], sC[7], sC[8] };
    const T mx[3] = { m.gmx(0), m.gmx(1), m.gmx(2) }, my[3] = { m.gmy(0), m.gmy(1), m.gmy(2) };
    const T f1 = r.q1 * ip, f2 = r.q2 * ip, s1p = gc.s1 * ip, s2p = gc.s2 * ip;
    T A[55], g[10];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int b = a; b < 3; ++b) {
            const T lam = (a == b) ? lg : T(0);
            const T s11 = t_fma(-(m0[a] * ip), m0[b], sC[s3(a, b)]) + lam;
            A[sidx<10>(U1 + a, U1 + b)] = s11;
            A[sidx<10>(U2 + a, U2 + b)] = s11;
            if (M::kHasCore) A[sidx<10>(U3 + a, U3 + b)] = m.gcore(s3(a, b)) + lam;
            else A[sidx<10>(U3 + a, U3 + b)] = t_fma(-(mx[a] * ip), mx[b], t_fma(-(my[a] * ip), my[b], m.gMw(s3(a, b)))) + lam;
        }
#pragma unroll
        for (int b = 0; b < 3; ++b) {
            if (M::kHasCore) {
                A[sidx<10>(U1 + a, U3 + b)] = m.gcore(6 + a * 3 + b);
                A[sidx<10>(U2 + a, U3 + b)] = m.gcore(15 + a * 3 + b);
            } else {
                A[sidx<10>(U1 + a, U3 + b)] = t_fma(m0[a] * ip, mx[b], -m.gMx(s3(a, b)));
                A[sidx<10>(U2 + a, U3 + b)] = t_fma(m0[a] * ip, my[b], -m.gMy(s3(a, b)));
            }
        }
        A[sidx<10>(U1 + a, GG)] = t_fma(-m0[a], s1p, gc.sg1[a]);
        A[sidx<10>(U2 + a, GG)] = t_fma(-m0[a], s2p, gc.sg2[a]);
        A[sidx<10>(U3 + a, GG)] = t_fma(mx[a], s1p, t_fma(my[a], s2p, -gc.sg3[a]));
        g[U1 + a] = t_fma(-m0[a], f1, r.r1[a]);
        g[U2 + a] = t_fma(-m0[a], f2, r.r2[a]);
        g[U3 + a] = t_fma(mx[a], f1, t_fma(my[a], f2, -r.r3[a]));
    }
    A[sidx<10>(GG, GG)] = t_fma(-gc.s1, s1p, t_fma(-gc.s2, s2p, gc.sgg + lambda));
    g[GG] = t_fma(-gc.s1, f1, t_fma(-gc.s2, f2, r.qg));
    return lm_finish<T, TRUE_JAC>(x, A, g, m0, mx, my, gc.s1, gc.s2, r.q1, r.q2, ig, ip);
}

// The same step for moment containers that hold the constant blocks (k_iterate).  With S the constant
// 9 x 9 core and u = (u1, u2, u3), the gamma column of the reduced system is S u, its corner is
// u^T S u + lambda, and the reduced right-hand side is
//   g_u = c - gamma S u + (lambda / p) (-d1 m0, -d2 m0, d1 mx + d2 my),   g_gamma = c.u - gamma u^T S u - (lambda / p) (d1 s1 + d2 s2)
// with c constant per problem (lm_core_from_moments) -- algebraically what lm_gamma_column,
// lm_rhs_from_moments and lm_step compute from the raw moments, in 45 fewer FP64 instructions.
template <typename T, typename M, bool TRUE_JAC = false>
PNP_DEV T lm_step_core(T (&x)[12], const M& m, const T* __restrict__ sC, T lambda, T ip)
{
    constexpr int U1 = 0, U2 = 3, U3 = 6, GG = 9;
    const T gam = x[11], d1 = x[9], d2 = x[10];
    const T ig = t_rcp<T>(gam);
    const T lg = lambda * (ig * ig);
    const T lp = lambda * ip;
    const T m0[3] = { sC[6], sC[7], sC[8] };
    const T mx[3] = { m.gmx(0), m.gmx(1), m.gmx(2) }, my[3] = { m.gmy(0), m.gmy(1), m.gmy(2) };
    const T u1[3] = { x[0], x[1], x[2] }, u2[3] = { x[3], x[4], x[5] }, u3[3] = { x[6], x[7], x[8] };
    T A[55], g[10];
    T col1[3] = { T(0), T(0), T(0) }, col2[3] = { T(0), T(0), T(0) }, col3[3] = { T(0), T(0), T(0) };
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int b = 0; b < 3; ++b) {
            const T s11 = t_fma(-(m0[a] * ip), m0[b], sC[s3(a, b)]);
            const T s33 = m.gcore(s3(a, b)), s13 = m.gcore(6 + a * 3 + b), s23 = m.gcore(15 + a * 3 + b);
            if (b >= a) {
                const T lam = (a == b) ? lg : T(0);
                A[sidx<10>(U1 + a, U1 + b)] = s11 + lam;
                A[sidx<10>(U2 + a, U2 + b)] = s11 + lam;
                A[sidx<10>(U3 + a, U3 + b)] = s33 + lam;
            }
            A[sidx<10>(U1 + a, U3 + b)] = s13;
            A[sidx<10>(U2 + a, U3 + b)] = s23;
            col1[a] = t_fma(s11, u1[b], t_fma(s13, u3[b], col1[a]));
            col2[a] = t_fma(s11, u2[b], t_fma(s23, u3[b], col2[a]));
            col3[b] = t_fma(s13, u1[a], t_fma(s23, u2[a], col3[b]));      // S13^T u1 + S23^T u2
            col3[a] = t_fma(s33, u3[b], col3[a]);
        }
    }
    T usu = T(0), cu = T(0), s1 = T(0), s2 = T(0);
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const T c1 = m.gcore(24 + a), c2 = m.gcore(27 + a), c3 = m.gcore(30 + a);
        usu = t_fma(u1[a], col1[a], t_fma(u2[a], col2[a], t_fma(u3[a], col3[a], usu)));
        cu = t_fma(c1, u1[a], t_fma(c2, u2[a], t_fma(c3, u3[a], cu)));
        s1 = t_fma(m0[a], u1[a], t_fma(-mx[a], u3[a], s1));
        s2 = t_fma(m0[a], u2[a], t_fma(-my[a], u3[a], s2));
        A[sidx<10>(U1 + a, GG)] = col1[a];
        A[sidx<10>(U2 + a, GG)] = col2[a];
        A[sidx<10>(U3 + a, GG)] = col3[a];
        g[U1 + a] = t_fma(-gam, col1[a], t_fma(-(lp * d1), m0[a], c1));
        g[U2 + a] = t_fma(-gam, col2[a], t_fma(-(lp * d2), m0[a], c2));
        g[U3 + a] = t_fma(-gam, col3[a], t_fma(lp * d1, mx[a], t_fma(lp * d2, my[a], c3)));
    }
    A[sidx<10>(GG, GG)] = usu + lambda;
    g[GG] = t_fma(-gam, usu, t_fma(-lp, t_fma(d1, s1, d2 * s2), cu));
    const T q1 = t_fma(-gam, s1, t_fma(-sC[9], d1, m.gsx0()));          // sum (z - hx)_x = sx0 - gamma s1 - n d1
    const T q2 = t_fma(-gam, s2, t_fma(-sC[9], d2, m.gsy0()));
    return lm_finish<T, TRUE_JAC>(x, A, g, m0, mx, my, s1, s2, q1, q2, ig, ip);
}

// ||z - hx|| over the 2n measurement rows at state x, point by point (:2679-2681)
template <typename T, int LPP, typename Pts>
PNP_DEV T lm_residual_direct(const Pts& pts, const T* __restrict__ sP, int n, int sub, const T (&x)[12])
{
    LmResidualState<T> lr;
    lr.load(x);
    T rr = T(0);
#pragma unroll 4
    for (int i = sub; i < n; i += LPP) {
        if (!pts.vis(i)) continue;
        const T th[3] = { sP[3 * i], sP[3 * i + 1], sP[3 * i + 2] };
        T bx, by;
        pts.get(i, bx, by);
        lr.add(th, bx, by, rr);
    }
    return t_sqrt(group_sum<LPP>(rr));
}

// EKF2_reconstruct_R_t_m1 :3500-3540
template <typename T>
PNP_DEV void lm_reconstruct(const T (&x)[12], Result<T>& out)
{
    T G[9], smax;
#pragma unroll
    for (int e = 0; e < 9; ++e) G[e] = x[e];
    svd3_project<T>(G, out.R, smax);
    const T t3 = T(1) / (smax * x[11]);                   // :3530-3533
    out.t[0] = x[9] * t3; out.t[1] = x[10] * t3; out.t[2] = t3;
}

// Fused form (direct mapping): J^T (z - hx) and the residual are accumulated point by point in
// every iteration; J^T J comes from the moments.
template <typename T, int LPP, typename Pts>
PNP_DEV void solve_lm(const Pts& pts, const T* __restrict__ sP, const T* __restrict__ sC, int n, int sub,
                      const SolverPrm<T>& prm, Result<T>& out)
{
    T x[12] = { T(1), T(0), T(0), T(0), T(1), T(0), T(0), T(0), T(1), T(0), T(0), T(1) };   // :2619-2624
    Moments<T> mom;
    accumulate_moments<T, LPP, Pts>(pts, sP, n, sub, mom);
    T res = T(1e5);
    const T ip = t_rcp<T>(sC[9] + prm.lm_lambda);
    for (int it = 0; it < prm.max_it; ++it) {             // :2642, fixed count, no exit test
        const T gam = x[11], d1 = x[9], d2 = x[10];
        LmRhs<T> r;
#pragma unroll
        for (int e = 0; e < 3; ++e) { r.r1[e] = r.r2[e] = r.r3[e] = T(0); }
        r.q1 = r.q2 = r.qg = T(0);
        T rr = T(0);
        for (int i = sub; i < n; i += LPP) {
            if (!pts.vis(i)) continue;
            const T th[3] = { sP[3 * i], sP[3 * i + 1], sP[3 * i + 2] };
            T bx, by;
            pts.get(i, bx, by);
            const T a = th[0] * x[0] + th[1] * x[1] + th[2] * x[2];
            const T b = th[0] * x[3] + th[1] * x[4] + th[2] * x[5];
            const T c = th[0] * x[6] + th[1] * x[7] + th[2] * x[8];
            const T g1 = a - bx * c, g2 = b - by * c;     // hu1_bar, hu2_bar (:3738-3741)
            const T rx = bx - (gam * g1 + d1);            // z - hx (:3750, :2679)
            const T ry = by - (gam * g2 + d2);
            const T v3 = bx * rx + by * ry;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                r.r1[k] = t_fma(th[k], rx, r.r1[k]); r.r2[k] = t_fma(th[k], ry, r.r2[k]); r.r3[k] = t_fma(th[k], v3, r.r3[k]);
            }
            r.q1 += rx; r.q2 += ry; r.qg = t_fma(g1, rx, t_fma(g2, ry, r.qg));
            rr = t_fma(rx, rx, t_fma(ry, ry, rr));
        }
        group_sum_arr<LPP>(r.r1); group_sum_arr<LPP>(r.r2); group_sum_arr<LPP>(r.r3);
        r.q1 = group_sum<LPP>(r.q1); r.q2 = group_sum<LPP>(r.q2); r.qg = group_sum<LPP>(r.qg); rr = group_sum<LPP>(rr);
        res = t_sqrt(rr);                                 // res_norm of the state BEFORE the update (:2681)
        GammaCol<T> gc;
        lm_gamma_column<T, Moments<T> >(x, mom, sC, gc);
        lm_step<T, Moments<T> >(x, mom, sC, gc, r, prm.lm_lambda, ip);
    }
    lm_reconstruct<T>(x, out);
    out.res = res;
    out.iters = prm.max_it;
}

// Moment form (moment mapping): every iteration is O(1) in the moments; x_prev receives the state
// before the last update, at which the caller evaluates res_norm point by point.
template <typename T, typename M, bool TRUE_JAC = false>
PNP_DEV void solve_lm_from_moments(const M& mom, const T* __restrict__ sC, const SolverPrm<T>& prm, T (&x_prev)[12],
                                   Result<T>& out)
{
    T x[12] = { T(1), T(0), T(0), T(0), T(1), T(0), T(0), T(0), T(1), T(0), T(0), T(1) };   // :2619-2624
#pragma unroll
    for (int e = 0; e < 12; ++e) x_prev[e] = x[e];
    const T ip = t_rcp<T>(sC[9] + prm.lm_lambda);
    lm_core_from_moments<T, M>(mom, sC, ip);
    for (int it = 0; it < prm.max_it; ++it) {
#pragma unroll
        for (int e = 0; e < 12; ++e) x_prev[e] = x[e];
        if (M::kHasCore) {
            lm_step_core<T, M, TRUE_JAC>(x, mom, sC, prm.lm_lambda, ip);
        } else {
            GammaCol<T> gc;
            LmRhs<T> r;
            lm_gamma_column<T, M>(x, mom, sC, gc);
            lm_rhs_from_moments<T, M>(x, mom, sC, gc, r);
            lm_step<T, M, TRUE_JAC>(x, mom, sC, gc, r, prm.lm_lambda, ip);
        }
    }
    lm_reconstruct<T>(x, out);
    out.res = T(0);
    out.iters = prm.max_it;
}

// -------------------------------------------------------------------------------------------
// EIF2 -- solve_pnp_EIF2_single_pattern :2001-2276: the iterated information filter on LM's
// 12-state model (EKF2_get_hx_H :3718-3836) with the state-dependent process covariance of
// EKF2_get_process_covariance_R (:3668-3716) and QEIF's early exit on the residual.
// H^T Q^-1 H and H^T Q^-1 (z - hx + H x) of the 2n measurement rows are bilinear forms of the 29
// moments (z - hx + H x = b + gamma (P phi_1 - b o P phi_3): no cancellation); the nine constraint
// rows are added one by one with their own weights; ||z - hx|| that drives the exit test is evaluated
// point by point.  State order as in the reference: [u1, u2, u3, delta_1, delta_2, gamma].
// -------------------------------------------------------------------------------------------
// M: the moment container (registers in the direct mappings, shared-memory columns in k_iterate).  RES_MOM (moment
// mapping): the residual of the early-exit test comes from the moments (res2_from_moments) and x_tail receives the state
// before the lane's last update, at which the residual pass evaluates the reported res_norm point by point.
template <typename T, int LPP, typename Pts, typename M, bool RES_MOM, bool WANT_TAIL = RES_MOM>
PNP_DEV void eif2_loop(const Pts& pts, const T* __restrict__ sP, const T* __restrict__ sC, int n, int sub,
                       const SolverPrm<T>& prm, const M& mom, T (&x_tail)[12], Result<T>& out)
{
    constexpr int U1 = 0, U2 = 3, U3 = 6, D1 = 9, D2 = 10, GG = 11;
    T x[12] = { T(1), T(0), T(0), T(0), T(1), T(0), T(0), T(0), T(1), T(0), T(0), T(1) };   // :2058-2063
    if (WANT_TAIL) {
#pragma unroll
        for (int e = 0; e < 12; ++e) x_tail[e] = x[e];
    }
    bool flagged = false;                                            // RES_MOM: an exit decision could not be certified
    T r2_new = T(0), e_new = T(0), r2_old = T(0), e_old = T(0);
    // One 12 x 12 array carries Sigma from one iteration to the next and Omega inside it (see solve_qeif)
    T Om[78];
#pragma unroll
    for (int e = 0; e < 78; ++e) Om[e] = T(0);
#pragma unroll
    for (int i = 0; i < 12; ++i) Om[sidx<12>(i, i)] = prm.sigma0;     // pinv(1e-5 I) (:2067-2068)
    T res_old = prm.res_old0, res = T(1e5);                          // :2101-2102
    bool done = false;
    int iters = 0;
    const T w = prm.meas_w;                                          // 1 / (9 / f^2) (:2080-2083)
    const T wc1 = T(1.0 / (1e-2 * 16.0)), wc2 = T(1.0 / (4.0 * 1e-2 * 16.0)), wc3 = T(1);   // :2085-2091
    const T sth = T(60.0 * (3.14159265358979323846 / 180.0));
    const T sth2 = sth * sth, st12 = T(0.05 * 0.05), st3 = T(4.0);   // :3686-3689
    T zeta[12], res_new = T(0);
#pragma unroll
    for (int e = 0; e < 12; ++e) zeta[e] = T(0);

    // An iteration inverts two 12 x 12 matrices (Sigma + R_k -> Omega_bar, :2146-2150; Omega -> Sigma, :2184) and
    // multiplies each inverse by a vector (zeta = Omega_bar x, :2152; x = Sigma zeta, :2185).  The loop below runs
    // one HALF iteration per trip -- predict-side work, THE inversion, THE product, then update-side work or the
    // state update -- so that the unrolled inversion (the bulk of the kernel's instructions) exists once: the first
    // version, with both inversions unrolled in one body, missed the 32 KB instruction cache on every iteration
    // (ncu: 1.26 instruction-fetch stalls per issued instruction, FP64 pipe 42 % busy).
    for (int half = 0; half < 2 * prm.max_it; ++half) {
        const bool update_half = (half & 1) != 0;                    // warp-uniform
        const T u1[3] = { x[0], x[1], x[2] }, u2[3] = { x[3], x[4], x[5] }, u3[3] = { x[6], x[7], x[8] };
        const T gam = x[GG], d1 = x[D1], d2 = x[D2];
        const T u11 = dot3<T>(u1, u1), u22 = dot3<T>(u2, u2), u33 = dot3<T>(u3, u3);
        const T u13 = dot3<T>(u1, u3), u23 = dot3<T>(u2, u3), u12 = dot3<T>(u1, u2);
        if (!update_half) {
            if (LPP == 1) { if (__all_sync(0xffffffffu, done)) break; }
            else          { if (done) break; }
            // ---- predict: Omega = pinv(Sigma + R_k) (:2146-2150)
            // R_k's u blocks: so3(u_i) sigma^2 so3(u_j)^T = sigma^2 ((u_i . u_j) I - u_j u_i^T)   (:3690-3696)
            const T* uu[3] = { u1, u2, u3 };
            const T dd[3][3] = { { u11, u12, u13 }, { u12, u22, u23 }, { u13, u23, u33 } };
#pragma unroll
            for (int bi = 0; bi < 3; ++bi)
#pragma unroll
                for (int bj = bi; bj < 3; ++bj)
#pragma unroll
                    for (int a = 0; a < 3; ++a)
#pragma unroll
                        for (int b = 0; b < 3; ++b) {
                            if (bi == bj && b < a) continue;
                            const T v = ((a == b) ? dd[bi][bj] : T(0)) - uu[bj][a] * uu[bi][b];
                            Om[sidx<12>(3 * bi + a, 3 * bj + b)] = t_fma(sth2, v, Om[sidx<12>(3 * bi + a, 3 * bj + b)]);
                        }
            Om[sidx<12>(D1, D1)] += t_abs(gam) * st12;               // :3700
            Om[sidx<12>(D2, D2)] += t_abs(gam) * st12;
            Om[sidx<12>(GG, GG)] += (gam * gam) * st3;               // :3701
        }
        spd_inverse<T, 12>(Om);
        T y[12];
        {
            T v[12];
#pragma unroll
            for (int e = 0; e < 12; ++e) v[e] = update_half ? zeta[e] : x[e];
            sym_matvec<T, 12>(Om, v, y);                             // zeta = Omega x (:2152)  |  x = pinv(Omega) zeta (:2184-2185)
        }
        if (update_half) {
            if (!done) {
                if (WANT_TAIL) {
#pragma unroll
                    for (int e = 0; e < 12; ++e) x_tail[e] = x[e];
                }
#pragma unroll
                for (int e = 0; e < 12; ++e) x[e] = y[e];
                res = res_new;
                ++iters;
                const T ratio = (res - res_old) * t_rcp<T>(res_old);   // 0 / 0 and x / 0 both end up not-below-tolerance, as in the reference               // :2196
                res_old = res;
                if (t_abs(ratio) < prm.exit_tol) done = true;        // :2202
                if (RES_MOM) {
                    if (exit_decision_uncertain<T>(t_abs(ratio), prm.exit_tol, r2_new, e_new, r2_old, e_old)) { flagged = true; done = true; }
                    r2_old = r2_new; e_old = e_new;
                }
            }
            continue;
        }
#pragma unroll
        for (int e = 0; e < 12; ++e) zeta[e] = y[e];
        // ---- residual over the 2n measurement rows, point by point (:2176-2178)
        T res2 = T(0);
        if (!RES_MOM) {
#pragma unroll 4
            for (int i = sub; i < n; i += LPP) {
                if (!pts.vis(i)) continue;
                const T th0 = sP[3 * i], th1 = sP[3 * i + 1], th2 = sP[3 * i + 2];
                T bx, by;
                pts.get(i, bx, by);
                const T a = th0 * u1[0] + th1 * u1[1] + th2 * u1[2];
                const T b = th0 * u2[0] + th1 * u2[1] + th2 * u2[2];
                const T c = th0 * u3[0] + th1 * u3[1] + th2 * u3[2];
                const T rx = bx - (gam * (a - bx * c) + d1);
                const T ry = by - (gam * (b - by * c) + d2);
                res2 = t_fma(rx, rx, t_fma(ry, ry, res2));
            }
            res2 = group_sum<LPP>(res2);
        }
        // ---- update, measurement rows from the moments (:2157-2164)
        {
            GammaCol<T> gc;
            lm_gamma_column<T, M>(x, mom, sC, gc);
            const T wg = w * gam, wgg = wg * gam;
            const T mxv[3] = { mom.gmx(0), mom.gmx(1), mom.gmx(2) }, myv[3] = { mom.gmy(0), mom.gmy(1), mom.gmy(2) };
            const T mwv[3] = { mom.gmw(0), mom.gmw(1), mom.gmw(2) };
#pragma unroll
            for (int a = 0; a < 3; ++a) {
#pragma unroll
                for (int b = a; b < 3; ++b) {
                    Om[sidx<12>(U1 + a, U1 + b)] = t_fma(wgg, sC[s3(a, b)], Om[sidx<12>(U1 + a, U1 + b)]);
                    Om[sidx<12>(U2 + a, U2 + b)] = t_fma(wgg, sC[s3(a, b)], Om[sidx<12>(U2 + a, U2 + b)]);
                    Om[sidx<12>(U3 + a, U3 + b)] = t_fma(wgg, mom.gMw(s3(a, b)), Om[sidx<12>(U3 + a, U3 + b)]);
                }
#pragma unroll
                for (int b = 0; b < 3; ++b) {
                    Om[sidx<12>(U1 + a, U3 + b)] = t_fma(-wgg, mom.gMx(s3(a, b)), Om[sidx<12>(U1 + a, U3 + b)]);
                    Om[sidx<12>(U2 + a, U3 + b)] = t_fma(-wgg, mom.gMy(s3(a, b)), Om[sidx<12>(U2 + a, U3 + b)]);
                }
                Om[sidx<12>(U1 + a, D1)] = t_fma(wg, sC[6 + a], Om[sidx<12>(U1 + a, D1)]);
                Om[sidx<12>(U2 + a, D2)] = t_fma(wg, sC[6 + a], Om[sidx<12>(U2 + a, D2)]);
                Om[sidx<12>(U3 + a, D1)] = t_fma(-wg, mxv[a], Om[sidx<12>(U3 + a, D1)]);
                Om[sidx<12>(U3 + a, D2)] = t_fma(-wg, myv[a], Om[sidx<12>(U3 + a, D2)]);
                Om[sidx<12>(U1 + a, GG)] = t_fma(wg, gc.sg1[a], Om[sidx<12>(U1 + a, GG)]);
                Om[sidx<12>(U2 + a, GG)] = t_fma(wg, gc.sg2[a], Om[sidx<12>(U2 + a, GG)]);
                Om[sidx<12>(U3 + a, GG)] = t_fma(-wg, gc.sg3[a], Om[sidx<12>(U3 + a, GG)]);
                // H^T Q^-1 (z - hx + H x), z - hx + H x = (bx + gamma g1, by + gamma g2)
                zeta[U1 + a] = t_fma(wg, mxv[a] + gam * gc.sg1[a], zeta[U1 + a]);
                zeta[U2 + a] = t_fma(wg, myv[a] + gam * gc.sg2[a], zeta[U2 + a]);
                zeta[U3 + a] = t_fma(-wg, mwv[a] + gam * gc.sg3[a], zeta[U3 + a]);
            }
            Om[sidx<12>(D1, D1)] = t_fma(w, sC[9], Om[sidx<12>(D1, D1)]);
            Om[sidx<12>(D2, D2)] = t_fma(w, sC[9], Om[sidx<12>(D2, D2)]);
            Om[sidx<12>(D1, GG)] = t_fma(w, gc.s1, Om[sidx<12>(D1, GG)]);
            Om[sidx<12>(D2, GG)] = t_fma(w, gc.s2, Om[sidx<12>(D2, GG)]);
            Om[sidx<12>(GG, GG)] = t_fma(w, gc.sgg, Om[sidx<12>(GG, GG)]);
            const T qa = dot3<T>(mxv, u1) + dot3<T>(myv, u2) - dot3<T>(mwv, u3);
            zeta[D1] = t_fma(w, mom.gsx0() + gam * gc.s1, zeta[D1]);
            zeta[D2] = t_fma(w, mom.gsy0() + gam * gc.s2, zeta[D2]);
            zeta[GG] = t_fma(w, qa + gam * gc.sgg, zeta[GG]);
            if (RES_MOM) {                                           // :2176-2178 from the moments
                res2 = res2_from_moments<T, M>(mom, sC, gc, qa, gam, d1, d2);
                r2_new = res2;
                e_new = res2_error_bound<T>(sC[9], mom.gsw0(), gam, d1, d2, sC[0] + sC[3] + sC[5],
                                            mom.gMw(0) + mom.gMw(3) + mom.gMw(5), u11 + u22, u33);
            }
        }
        // ---- update, the nine constraint rows (:3753-3772, Jacobians :3787-3823), collected per 3 x 3 block.  Row k adds
        // w_k c_k c_k^T to Omega and w_k c_k (z_k - h_k + c_k . x) to zeta; with the rows
        //   1-3 (weight wc1): (u3 | u1) on blocks (U1, U3), (u3 | u2) on (U2, U3), (u2 | u1) on (U1, U2),   v = u_i . u_j
        //   4-6 (weight wc2): (u1 | -u3) on (U1, U3), (u2 | -u3) on (U2, U3), (u1 | -u2) on (U1, U2),     v = 0
        //   7-9 (weight wc3): j_i = u_i / (2 |u_i|) on block U_i,                                         v = 1 - |u_i| + j_i . u_i
        // the diagonal blocks are combinations of the three outer products P_i = u_i u_i^T and the off-diagonal ones of
        // u_i u_j^T: 60 % fewer instructions than nine rank-one updates, same sums up to the order of the additions.
        {
            const T y1 = t_rsqrt<T>(u11), y2 = t_rsqrt<T>(u22), y3 = t_rsqrt<T>(u33);
            const T n1 = t_sqrt_fast<T>(u11, y1), n2 = t_sqrt_fast<T>(u22, y2), n3 = t_sqrt_fast<T>(u33, y3);
            const T h1 = T(0.5) * y1, h2 = T(0.5) * y2, h3 = T(0.5) * y3;             // j_i = h_i u_i (:3819)
            const T c1 = t_fma(wc3 * h1, h1, T(2) * wc2), c2 = t_fma(wc3 * h2, h2, T(2) * wc2), c3 = t_fma(wc3 * h3, h3, T(2) * wc2);
            // zeta: rows 1-3 carry v = u_i . u_j, rows 7-9 v_i = 1 - |u_i| + h_i |u_i|^2 (times h_i), rows 4-6 nothing
            const T g1 = wc3 * h1 * (T(1) - n1 + h1 * u11), g2 = wc3 * h2 * (T(1) - n2 + h2 * u22), g3 = wc3 * h3 * (T(1) - n3 + h3 * u33);
            const T v13 = wc1 * u13, v23 = wc1 * u23, v12 = wc1 * u12;
#pragma unroll
            for (int a = 0; a < 3; ++a) {
#pragma unroll
                for (int b = a; b < 3; ++b) {
                    const T p1 = u1[a] * u1[b], p2 = u2[a] * u2[b], p3 = u3[a] * u3[b];
                    Om[sidx<12>(U1 + a, U1 + b)] += t_fma(c1, p1, wc1 * (p2 + p3));
                    Om[sidx<12>(U2 + a, U2 + b)] += t_fma(c2, p2, wc1 * (p1 + p3));
                    Om[sidx<12>(U3 + a, U3 + b)] += t_fma(c3, p3, wc1 * (p1 + p2));
                }
#pragma unroll
                for (int b = 0; b < 3; ++b) {
                    Om[sidx<12>(U1 + a, U3 + b)] = t_fma(wc1 * u3[a], u1[b], t_fma(-wc2 * u1[a], u3[b], Om[sidx<12>(U1 + a, U3 + b)]));
                    Om[sidx<12>(U2 + a, U3 + b)] = t_fma(wc1 * u3[a], u2[b], t_fma(-wc2 * u2[a], u3[b], Om[sidx<12>(U2 + a, U3 + b)]));
                    Om[sidx<12>(U1 + a, U2 + b)] = t_fma(wc1 * u2[a], u1[b], t_fma(-wc2 * u1[a], u2[b], Om[sidx<12>(U1 + a, U2 + b)]));
                }
                zeta[U1 + a] = t_fma(v13, u3[a], t_fma(v12, u2[a], t_fma(g1, u1[a], zeta[U1 + a])));
                zeta[U2 + a] = t_fma(v23, u3[a], t_fma(v12, u1[a], t_fma(g2, u2[a], zeta[U2 + a])));
                zeta[U3 + a] = t_fma(v13, u1[a], t_fma(v23, u2[a], t_fma(g3, u3[a], zeta[U3 + a])));
            }
        }
        res_new = t_sqrt_nn<T>(res2);
    }
    lm_reconstruct<T>(x, out);
    out.res = res;
    out.iters = flagged ? -1 : iters;
}

template <typename T, int LPP, typename Pts>
PNP_DEV void solve_eif2(const Pts& pts, const T* __restrict__ sP, const T* __restrict__ sC, int n, int sub,
                        const SolverPrm<T>& prm, Result<T>& out)
{
    Moments<T> mom;
    accumulate_moments<T, LPP, Pts>(pts, sP, n, sub, mom);
    T unused[12];
    eif2_loop<T, LPP, Pts, Moments<T>, false>(pts, sP, sC, n, sub, prm, mom, unused, out);
}

// Direct arithmetic (point-wise residual) with the tail the residual pass needs: the fix-up of the moment mapping
template <typename T, int LPP, typename Pts>
PNP_DEV void solve_eif2_with_tail(const Pts& pts, const T* __restrict__ sP, const T* __restrict__ sC, int n, int sub,
                                  const SolverPrm<T>& prm, T (&x_tail)[12], Result<T>& out)
{
    Moments<T> mom;
    accumulate_moments<T, LPP, Pts>(pts, sP, n, sub, mom);
    eif2_loop<T, LPP, Pts, Moments<T>, false, true>(pts, sP, sC, n, sub, prm, mom, x_tail, out);
}

template <typename T, typename M>
PNP_DEV void solve_eif2_from_moments(const M& mom, const T* __restrict__ sC, const SolverPrm<T>& prm, T (&x_tail)[12], Result<T>& out)
{
    NoPts none;
    eif2_loop<T, 1, NoPts, M, true>(none, nullptr, sC, (int)sC[9], 0, prm, mom, x_tail, out);
}

// -------------------------------------------------------------------------------------------
// Linear stage, formulation 2 -- solve_pnp_formulation_2_single_pattern :693-953,
// helpers :3274-3375.  D^+ B = G (D^T B) with the pattern-constant G = (D^T D)^-1, so the
// per-problem work is the moments of (bx, by) against [theta theta^T, theta, 1].
// -------------------------------------------------------------------------------------------
template <typename T>
PNP_DEV void g4_apply(const T* __restrict__ G, const T (&v)[4], T (&o)[4])
{
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        T acc = T(0);
#pragma unroll
        for (int j = 0; j < 4; ++j) acc = t_fma(G[sym<4>(i, j)], v[j], acc);
        o[i] = acc;
    }
}

// residual of f2_cal_res_all (:3368) at (phi_3 old, phi rebuilt from R, t): res_norm_all (:3374)
template <typename T>
struct F2Tail { T phi3[3], pxn[4], pyn[4]; };

template <typename T, int LPP, typename Pts>
PNP_DEV T f2_residual_direct(const Pts& pts, const T* __restrict__ sP, int n, int sub, const F2Tail<T>& f)
{
    T rx2 = T(0), ry2 = T(0);
#pragma unroll 4
    for (int i = sub; i < n; i += LPP) {
        if (!pts.vis(i)) continue;
        const T th0 = sP[3 * i], th1 = sP[3 * i + 1], th2 = sP[3 * i + 2];
        T bx, by;
        pts.get(i, bx, by);
        const T db = T(1) + (th0 * f.phi3[0] + th1 * f.phi3[1] + th2 * f.phi3[2]);
        const T dx = th0 * f.pxn[0] + th1 * f.pxn[1] + th2 * f.pxn[2] + f.pxn[3];
        const T dy = th0 * f.pyn[0] + th1 * f.pyn[1] + th2 * f.pyn[2] + f.pyn[3];
        const T ex = bx * db - dx, ey = by * db - dy;
        rx2 = t_fma(ex, ex, rx2); ry2 = t_fma(ey, ey, ry2);
    }
    rx2 = group_sum<LPP>(rx2); ry2 = group_sum<LPP>(ry2);
    const T nx = t_sqrt(rx2), ny = t_sqrt(ry2);
    return t_sqrt(nx * nx + ny * ny);
}

// The three fixed-point iterations on phi_3 from the moments; `tail` = what the residual of the
// last iteration needs.
template <typename T>
PNP_DEV void solve_f2_from_moments(const Moments<T>& mom, const T* __restrict__ sC, const SolverPrm<T>& prm, F2Tail<T>& tail,
                                   Result<T>& out)
{
    const T* G = sC + 10;
    T v0x[4], v0y[4], Mxm[12], Mym[12];                   // :3314-3328
    {
        const T bxv[4] = { mom.mx[0], mom.mx[1], mom.mx[2], mom.sx0 }, byv[4] = { mom.my[0], mom.my[1], mom.my[2], mom.sy0 };
        g4_apply<T>(G, bxv, v0x);
        g4_apply<T>(G, byv, v0y);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const T cx[4] = { mom.Mx[s3(0, c)], mom.Mx[s3(1, c)], mom.Mx[s3(2, c)], mom.mx[c] };
            const T cy[4] = { mom.My[s3(0, c)], mom.My[s3(1, c)], mom.My[s3(2, c)], mom.my[c] };
            T ox[4], oy[4];
            g4_apply<T>(G, cx, ox);
            g4_apply<T>(G, cy, oy);
#pragma unroll
            for (int k = 0; k < 4; ++k) { Mxm[k * 3 + c] = ox[k]; Mym[k * 3 + c] = oy[k]; }
        }
    }
    T phi3[3] = { T(0), T(0), T(1) };                     // :758
    const int nit = prm.linear_it < 1 ? 1 : prm.linear_it;
    for (int it = 0; it < nit; ++it) {
        T phi[8], t3;
#pragma unroll
        for (int k = 0; k < 4; ++k) {                     // :3337
            const T px = v0x[k] + (Mxm[k * 3] * phi3[0] + Mxm[k * 3 + 1] * phi3[1] + Mxm[k * 3 + 2] * phi3[2]);
            const T py = v0y[k] + (Mym[k * 3] * phi3[0] + Mym[k * 3 + 1] * phi3[1] + Mym[k * 3 + 2] * phi3[2]);
            if (k < 3) { phi[k] = px; phi[3 + k] = py; } else { phi[6] = px; phi[7] = py; }
        }
        block_reconstruct<T>(phi, out.R, out.t, t3);      // :862
        if (it == nit - 1) {                              // (:868-877): phi from (R, t), the OLD phi_3
#pragma unroll
            for (int k = 0; k < 3; ++k) { tail.pxn[k] = out.R[k] / t3; tail.pyn[k] = out.R[3 + k] / t3; tail.phi3[k] = phi3[k]; }
            tail.pxn[3] = out.t[0] / t3; tail.pyn[3] = out.t[1] / t3;
        }
        const T it3 = T(1) / t3;                          // update_phi_3_est_m2 :4002-4010
#pragma unroll
        for (int k = 0; k < 3; ++k) phi3[k] = it3 * out.R[6 + k];
    }
    out.res = T(30);
    out.iters = nit;
}

// LM+ (NOT a reference method; SURVEY.md 8f item 3, the pipeline of BASELINE.json's north star):
// linear stage F2 for the initial pose, then the 12-state damped Gauss-Newton of LM with the true
// constraint gradients and a convergence test (max |dx| <= 1e-10, at most max_it iterations).
// One problem per thread: a warp leaves the loop when all of its lanes have converged.
// x_out = the returned state, at which the caller evaluates res_norm point by point.
template <typename T, typename M>
PNP_DEV void solve_lm_plus_from_moments(const M& mom, const Moments<T>& mom_regs, const T* __restrict__ sC,
                                        const SolverPrm<T>& prm, T (&x_out)[12], Result<T>& out)
{
    F2Tail<T> tail;
    solve_f2_from_moments<T>(mom_regs, sC, prm, tail, out);
    T x[12];
#pragma unroll
    for (int e = 0; e < 9; ++e) x[e] = out.R[e];
    x[9] = out.t[0] / out.t[2]; x[10] = out.t[1] / out.t[2]; x[11] = T(1) / out.t[2];
    bool done = false;
    int iters = 0;
    const T ip = t_rcp<T>(sC[9] + prm.lm_lambda);
    lm_core_from_moments<T, M>(mom, sC, ip);
    for (int it = 0; it < prm.max_it; ++it) {
        if (__all_sync(0xffffffffu, done)) break;
        T xn[12];
#pragma unroll
        for (int e = 0; e < 12; ++e) xn[e] = x[e];
        GammaCol<T> gc;
        LmRhs<T> r;
        lm_gamma_column<T, M>(xn, mom, sC, gc);
        lm_rhs_from_moments<T, M>(xn, mom, sC, gc, r);
        const T step = lm_step<T, M, true>(xn, mom, sC, gc, r, prm.lm_lambda, ip);
        if (!done) {
#pragma unroll
            for (int e = 0; e < 12; ++e) x[e] = xn[e];
            ++iters;
            if (step <= T(sizeof(T) == 8 ? 1e-10 : 1e-5)) done = true;
        }
    }
#pragma unroll
    for (int e = 0; e < 12; ++e) x_out[e] = x[e];
    lm_reconstruct<T>(x, out);
    out.res = T(0);
    out.iters = iters;
}

template <typename T, int LPP, typename Pts>
PNP_DEV void solve_linear_f2(const Pts& pts, const T* __restrict__ sP, const T* __restrict__ sC, int n, int sub,
                             const SolverPrm<T>& prm, Result<T>& out)
{
    Moments<T> mom;
    accumulate_moments<T, LPP, Pts, false>(pts, sP, n, sub, mom);
    F2Tail<T> tail;
    solve_f2_from_moments<T>(mom, sC, prm, tail, out);
    out.res = f2_residual_direct<T, LPP, Pts>(pts, sP, n, sub, tail);
}

// -------------------------------------------------------------------------------------------
// Linear stage, formulation 1 -- solve_pnp_single_pattern :205-430, helpers :3031-3111.
// A(phi_3) has the x rows acting on (phi_1, delta_1) and the y rows on (phi_2, delta_2) with the
// SAME 2n/2 x 4 block, so pinv(A) B is two 4x4 normal-equation solves sharing one matrix.
// -------------------------------------------------------------------------------------------
template <typename T, int LPP, typename Pts>
PNP_DEV void solve_linear_f1(const Pts& pts, const T* __restrict__ sP, int n, int sub,
                             const SolverPrm<T>& prm, Result<T>& out)
{
    T phi3[3] = { T(0), T(0), T(1) };
    T res = T(30);
    const int nit = prm.linear_it < 1 ? 1 : prm.linear_it;
    const T eps = T(1e-7);
    for (int it = 0; it < nit; ++it) {
        T N[10], bxv[4], byv[4];
#pragma unroll
        for (int e = 0; e < 10; ++e) N[e] = T(0);
#pragma unroll
        for (int e = 0; e < 4; ++e) { bxv[e] = T(0); byv[e] = T(0); }
        for (int i = sub; i < n; i += LPP) {
            if (!pts.vis(i)) continue;
            const T th0 = sP[3 * i], th1 = sP[3 * i + 1], th2 = sP[3 * i + 2];
            T bx, by;
            pts.get(i, bx, by);
            T Delta = th0 * phi3[0] + th1 * phi3[1] + th2 * phi3[2] + T(1);   // get_Delta_i :3031-3046
            if (t_abs(Delta) <= eps) Delta = (Delta < T(0)) ? -eps : eps;
            const T iD = t_rcp<T>(Delta);                 // |Delta| >= 1e-7 after the clamp: normal range
            const T a[4] = { th0 * iD, th1 * iD, th2 * iD, iD };                          // get_A_i :3048-3062
#pragma unroll
            for (int p = 0; p < 4; ++p) {
#pragma unroll
                for (int q = p; q < 4; ++q) N[sidx<4>(p, q)] = t_fma(a[p], a[q], N[sidx<4>(p, q)]);
                bxv[p] = t_fma(a[p], bx, bxv[p]);
                byv[p] = t_fma(a[p], by, byv[p]);
            }
        }
        group_sum_arr<LPP>(N); group_sum_arr<LPP>(bxv); group_sum_arr<LPP>(byv);
        ldlt_factor<T, 4>(N);                             // phi = pinv(A) B (:262)
        ldlt_solve<T, 4>(N, bxv);
        ldlt_solve<T, 4>(N, byv);
        const T phi[8] = { bxv[0], bxv[1], bxv[2], byv[0], byv[1], byv[2], bxv[3], byv[3] };
        T t3;
        block_reconstruct<T>(phi, out.R, out.t, t3);      // :365
        if (it == nit - 1) {                              // res = B - A phi_new (:381-387), A from the old phi_3
            T pn[8];
#pragma unroll
            for (int k = 0; k < 3; ++k) { pn[k] = out.R[k] / t3; pn[3 + k] = out.R[3 + k] / t3; }
            pn[6] = out.t[0] / t3; pn[7] = out.t[1] / t3;
            T r2 = T(0);
            for (int i = sub; i < n; i += LPP) {
                if (!pts.vis(i)) continue;
                const T th0 = sP[3 * i], th1 = sP[3 * i + 1], th2 = sP[3 * i + 2];
                T bx, by;
                pts.get(i, bx, by);
                T Delta = th0 * phi3[0] + th1 * phi3[1] + th2 * phi3[2] + T(1);
                if (t_abs(Delta) <= eps) Delta = (Delta < T(0)) ? -eps : eps;
                const T a3 = t_rcp<T>(Delta), a0 = th0 * a3, a1 = th1 * a3, a2 = th2 * a3;
                const T ex = bx - (a0 * pn[0] + a1 * pn[1] + a2 * pn[2] + a3 * pn[6]);
                const T ey = by - (a0 * pn[3] + a1 * pn[4] + a2 * pn[5] + a3 * pn[7]);
                r2 = t_fma(ex, ex, t_fma(ey, ey, r2));
            }
            r2 = group_sum<LPP>(r2);
            res = t_sqrt(r2);
        }
        const T it3 = T(1) / t3;
#pragma unroll
        for (int k = 0; k < 3; ++k) phi3[k] = it3 * out.R[6 + k];
    }
    out.res = res;
    out.iters = nit;
}

}  // namespace pnpb200
