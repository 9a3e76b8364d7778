/*
 * ransac_oracle.c -- TEST INFRASTRUCTURE ONLY: the CPU restatement of the hypothesis stage of the RANSAC solve
 * (pnpb200_hypothesize_batch, include/pnpb200.h) that tests/test_gpu_ransac.py and tests/ransac_accuracy.py compare the
 * device against.  Its P3P has other numerics than the device's Lambda Twist: Grunert's formulation (Haralick et al.,
 * IJCV 1994) as a quartic in v = s3 / s1, solved by Ferrari in complex arithmetic with Newton polish of the real roots and a
 * Newton refinement of the three depths; the pose from the three camera-frame points by orthonormal triads.  The sample
 * draws, distances and stop test restate the device's rule; Philox4x32-10 is the generator of oracle/pnp_oracle.c.
 * Built on first use by tests/ransac_oracle.py.
 */
#include <complex.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

#define RANSAC_API __attribute__((visibility("default")))

/* Philox4x32-10, as oracle/pnp_oracle.c and csrc/pnpb200_math.cuh */
static void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t *out)
{
    int r;
    for (r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}


static double complex csqrt_p(double complex z) { return csqrt(z); }
static double complex ccbrt_p(double complex z) { return cabs(z) == 0.0 ? 0.0 : cpow(z, 1.0 / 3.0); }

/* the four complex roots of v^4 + a v^3 + b v^2 + c v + d (Ferrari) */
static void quartic_roots(double a, double b, double c, double d, double complex *r)
{
    double p = b - 3.0 * a * a / 8.0, q = c - a * b / 2.0 + a * a * a / 8.0;
    double rr = d - a * c / 4.0 + a * a * b / 16.0 - 3.0 * a * a * a * a / 256.0;
    /* resolvent 8 m^3 + 8 p m^2 + (2 p^2 - 8 r) m - q^2 = 0, monic: m^3 + p m^2 + (p^2 / 4 - r) m - q^2 / 8 (Cardano) */
    double B2 = p, B1 = p * p / 4.0 - rr, B0 = -q * q / 8.0;
    double pp = B1 - B2 * B2 / 3.0, qq = 2.0 * B2 * B2 * B2 / 27.0 - B2 * B1 / 3.0 + B0;
    double complex disc = csqrt_p(qq * qq / 4.0 + pp * pp * pp / 27.0);
    double complex u = ccbrt_p(-qq / 2.0 + disc), m = 0.0;
    double complex w = -0.5 + 0.5 * I * sqrt(3.0);
    int k;
    double best = -1.0;
    for (k = 0; k < 3; ++k) {                      /* the resolvent root of largest modulus (m != 0 unless q = 0 and p = r = 0) */
        double complex uk = u * (k == 0 ? 1.0 : (k == 1 ? w : w * w));
        double complex mk = (cabs(uk) == 0.0 ? 0.0 : uk - pp / (3.0 * uk)) - B2 / 3.0;
        if (cabs(mk) > best) { best = cabs(mk); m = mk; }
    }
    {
        double complex s = csqrt_p(2.0 * m);
        double complex h = (cabs(s) == 0.0) ? csqrt_p(p * p / 4.0 - rr) : q / (2.0 * s);
        int sg;
        for (sg = 0; sg < 2; ++sg) {
            /* y^2 - sgn s y + (p / 2 + m + sgn q / (2 s)) = 0 */
            double complex ss = sg ? -s : s;
            double complex c0 = p / 2.0 + m + (sg ? -h : h);
            double complex dd = csqrt_p(ss * ss - 4.0 * c0);
            r[2 * sg] = (ss + dd) / 2.0 - a / 4.0;
            r[2 * sg + 1] = (ss - dd) / 2.0 - a / 4.0;
        }
    }
}

static void unit3(double *v)
{
    double s = sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
    v[0] /= s; v[1] /= s; v[2] /= s;
}

static void cross3(const double *a, const double *b, double *o)
{
    o[0] = a[1] * b[2] - a[2] * b[1]; o[1] = a[2] * b[0] - a[0] * b[2]; o[2] = a[0] * b[1] - a[1] * b[0];
}

/* R, t with R X_k + t = s_k f_k from the three points: R = Ec Ew^T for the orthonormal triads of (p1, p2, p3) */
static void pose_from_points(const double *X, const double *Y, double *R, double *t)
{
    double ew[9], ec[9], e[3];
    int side, i, j;
    for (side = 0; side < 2; ++side) {
        const double *P = side ? Y : X;
        double *E = side ? ec : ew, a[3], b[3], c3[3];
        for (i = 0; i < 3; ++i) { a[i] = P[3 + i] - P[i]; b[i] = P[6 + i] - P[i]; }
        unit3(a);
        cross3(a, b, c3); unit3(c3);
        cross3(c3, a, e);
        for (i = 0; i < 3; ++i) { E[3 * i] = a[i]; E[3 * i + 1] = e[i]; E[3 * i + 2] = c3[i]; }   /* columns a, e, c3 */
    }
    for (i = 0; i < 3; ++i)
        for (j = 0; j < 3; ++j) R[3 * i + j] = ec[3 * i] * ew[3 * j] + ec[3 * i + 1] * ew[3 * j + 1] + ec[3 * i + 2] * ew[3 * j + 2];
    for (i = 0; i < 3; ++i) t[i] = Y[i] - (R[3 * i] * X[0] + R[3 * i + 1] * X[1] + R[3 * i + 2] * X[2]);
}

/* Grunert P3P: X [3,3] pattern points, f [3,3] unit bearings; R [4,9], t [4,3]; returns the number of poses (roots with a
 * non-finite value or a depth <= 0 dropped) */
RANSAC_API int ransac_oracle_p3p(const double *X, const double *f, double *R, double *t)
{
    double a2 = 0, b2 = 0, c2 = 0, ca, cb, cg, amc, apc, A[5];
    double complex r[4];
    int i, k, ns = 0;
    for (k = 0; k < 3; ++k) {
        a2 += (X[3 + k] - X[6 + k]) * (X[3 + k] - X[6 + k]);
        b2 += (X[k] - X[6 + k]) * (X[k] - X[6 + k]);
        c2 += (X[k] - X[3 + k]) * (X[k] - X[3 + k]);
    }
    ca = f[3] * f[6] + f[4] * f[7] + f[5] * f[8];
    cb = f[0] * f[6] + f[1] * f[7] + f[2] * f[8];
    cg = f[0] * f[3] + f[1] * f[4] + f[2] * f[5];
    amc = (a2 - c2) / b2; apc = (a2 + c2) / b2;
    A[0] = (amc - 1) * (amc - 1) - 4 * c2 / b2 * ca * ca;
    A[1] = 4 * (amc * (1 - amc) * cb - (1 - apc) * ca * cg + 2 * c2 / b2 * ca * ca * cb);
    A[2] = 2 * (amc * amc - 1 + 2 * amc * amc * cb * cb + 2 * (b2 - c2) / b2 * ca * ca - 4 * apc * ca * cb * cg + 2 * (b2 - a2) / b2 * cg * cg);
    A[3] = 4 * (-amc * (1 + amc) * cb + 2 * a2 / b2 * cg * cg * cb - (1 - apc) * ca * cg);
    A[4] = (1 + amc) * (1 + amc) - 4 * a2 / b2 * cg * cg;
    quartic_roots(A[1] / A[0], A[2] / A[0], A[3] / A[0], A[4] / A[0], r);
    for (i = 0; i < 4; ++i) {
        double v = creal(r[i]), u, s1, Y[9];
        int it, dup = 0, j;
        if (!(fabs(cimag(r[i])) <= 1e-7 * (1.0 + fabs(v)))) continue;
        for (it = 0; it < 4; ++it) {                 /* Newton polish on the quartic */
            double fv = (((A[0] * v + A[1]) * v + A[2]) * v + A[3]) * v + A[4];
            double fp = ((4 * A[0] * v + 3 * A[1]) * v + 2 * A[2]) * v + A[3];
            double vn = v - fv / fp;
            if (isfinite(vn)) v = vn;
        }
        for (j = 0; j < i; ++j)                      /* a real double root listed twice */
            if (fabs(cimag(r[j])) <= 1e-7 * (1.0 + fabs(creal(r[j]))) && fabs(creal(r[j]) - creal(r[i])) <= 1e-12 * (1.0 + fabs(v))) dup = 1;
        if (dup) continue;
        u = ((-1 + amc) * v * v - 2 * amc * cb * v + 1 + amc) / (2 * (cg - v * ca));
        s1 = sqrt(b2 / (1 + v * v - 2 * v * cb));
        if (!(s1 > 0.0 && u > 0.0 && v > 0.0 && isfinite(s1 * u) && isfinite(s1 * v))) continue;
        {
            /* Newton on the three law-of-cosines constraints in the depths (s1, s2, s3), Cramer's rule */
            double s[3] = { s1, s1 * u, s1 * v };
            for (it = 0; it < 6; ++it) {
                double F[3], J[9], dt, dl[3], Jc[9];
                int col, e;
                F[0] = s[0] * s[0] + s[1] * s[1] - 2 * s[0] * s[1] * cg - c2;
                F[1] = s[0] * s[0] + s[2] * s[2] - 2 * s[0] * s[2] * cb - b2;
                F[2] = s[1] * s[1] + s[2] * s[2] - 2 * s[1] * s[2] * ca - a2;
                J[0] = 2 * s[0] - 2 * s[1] * cg; J[1] = 2 * s[1] - 2 * s[0] * cg; J[2] = 0;
                J[3] = 2 * s[0] - 2 * s[2] * cb; J[4] = 0; J[5] = 2 * s[2] - 2 * s[0] * cb;
                J[6] = 0; J[7] = 2 * s[1] - 2 * s[2] * ca; J[8] = 2 * s[2] - 2 * s[1] * ca;
                dt = J[0] * (J[4] * J[8] - J[5] * J[7]) - J[1] * (J[3] * J[8] - J[5] * J[6]) + J[2] * (J[3] * J[7] - J[4] * J[6]);
                for (col = 0; col < 3; ++col) {
                    memcpy(Jc, J, sizeof(Jc));
                    for (e = 0; e < 3; ++e) Jc[3 * e + col] = F[e];
                    dl[col] = (Jc[0] * (Jc[4] * Jc[8] - Jc[5] * Jc[7]) - Jc[1] * (Jc[3] * Jc[8] - Jc[5] * Jc[6]) +
                               Jc[2] * (Jc[3] * Jc[7] - Jc[4] * Jc[6])) / dt;
                }
                if (!(isfinite(dl[0]) && isfinite(dl[1]) && isfinite(dl[2]))) break;
                for (e = 0; e < 3; ++e) s[e] -= dl[e];
            }
            s1 = s[0]; u = s[1] / s[0]; v = s[2] / s[0];
            if (!(s[0] > 0.0 && s[1] > 0.0 && s[2] > 0.0)) continue;
        }
        for (k = 0; k < 3; ++k) { Y[k] = s1 * f[k]; Y[3 + k] = s1 * u * f[3 + k]; Y[6 + k] = s1 * v * f[6 + k]; }
        pose_from_points(X, Y, R + 9 * ns, t + 3 * ns);
        {
            int fin = 1;
            for (k = 0; k < 9; ++k) fin &= isfinite(R[9 * ns + k]);
            for (k = 0; k < 3; ++k) fin &= isfinite(t[3 * ns + k]);
            if (fin) ++ns;
        }
    }
    return ns;
}

/* the candidate positions of sample s of problem g (c >= 4): u = Philox4x32-10 (g lo, g hi, s, 4) keyed by seed,
 * j_k = u_k mod (c - k), the k-th sample is the j_k-th candidate not yet chosen */
RANSAC_API void ransac_oracle_draw4(int c, uint64_t g, int s, uint64_t seed, int32_t *pos)
{
    uint32_t u[4];
    int srt[4], k, j;
    philox4x32_10((uint32_t)g, (uint32_t)(g >> 32), (uint32_t)s, 4u, (uint32_t)seed, (uint32_t)(seed >> 32), u);
    for (k = 0; k < 4; ++k) {
        int q = (int)(u[k] % (uint32_t)(c - k));
        for (j = 0; j < k; ++j) q += q >= srt[j] ? 1 : 0;   /* srt ascending: step over the chosen positions */
        pos[k] = q;
        for (j = k; j > 0 && srt[j - 1] > q; --j) srt[j] = srt[j - 1];
        srt[j] = q;
    }
}

/* the check's prediction-vs-landmark distance of pattern point Xp at pixel px under (K R, K t) (FP64, no FMA) */
static double check_distance(const double *M, const double *m, const double *Xp, const double *px)
{
    double r0 = M[0] * Xp[0] + M[1] * Xp[1] + M[2] * Xp[2] + m[0];
    double r1 = M[3] * Xp[0] + M[4] * Xp[1] + M[5] * Xp[2] + m[1];
    double r2 = M[6] * Xp[0] + M[7] * Xp[1] + M[8] * Xp[2] + m[2];
    double inv = fabs(1.0 / r2), dx = r0 * inv - px[0], dy = r1 * inv - px[1];
    return sqrt(dx * dx + dy * dy + (signbit(r2) ? 4.0 : 0.0));
}

static void fold_km(const double *K, const double *R, const double *t, double *M, double *m)
{
    int r, c;
    for (r = 0; r < 3; ++r) {
        for (c = 0; c < 3; ++c) M[3 * r + c] = K[3 * r] * R[c] + K[3 * r + 1] * R[3 + c] + K[3 * r + 2] * R[6 + c];
        m[r] = K[3 * r] * t[0] + K[3 * r + 1] * t[1] + K[3 * r + 2] * t[2];
    }
}

static int near_thr(double d, double thr) { return fabs(d - thr) <= 1e-9 * (thr > 1e-300 ? thr : 1e-300); }

static double powi_ex(double q, int e)
{
    double r = 1.0;
    while (e) { if (e & 1) r *= q; q *= q; e >>= 1; }
    return r;
}

/* The rule of pnpb200_hypothesize_batch for one problem: cand [c] its candidates (landmark indices, candidate order), uv
 * [n_total,2], patterns [P,n_total,3], g = idx0 + b.  Outputs the winner's R [9], t [3], pattern, mask [n_total] (0/1),
 * consensus and sample index (-1: none), and near = some decision distance lay within 1e-9 relative of consensus_px or of
 * another root's at the 4th landmark.  Returns the number of samples drawn. */
RANSAC_API int ransac_oracle_hypothesize_one(int c, const int32_t *cand, int n_total, const double *uv, int P, const double *patterns,
                                          const double *K, int max_samples, double consensus_px, double confidence, uint64_t seed,
                                          uint64_t g, double *R, double *t, int32_t *best_pattern, uint8_t *mask, int32_t *consensus,
                                          int32_t *win_s, int32_t *near)
{
    double Ki[9], det, wR[9], wt[3];
    int s, k, i, p, best = 0, win_p = 0, drawn = 0;
    *near = 0; *win_s = -1;
    Ki[0] = K[4] * K[8] - K[5] * K[7]; Ki[1] = K[2] * K[7] - K[1] * K[8]; Ki[2] = K[1] * K[5] - K[2] * K[4];
    Ki[3] = K[5] * K[6] - K[3] * K[8]; Ki[4] = K[0] * K[8] - K[2] * K[6]; Ki[5] = K[2] * K[3] - K[0] * K[5];
    Ki[6] = K[3] * K[7] - K[4] * K[6]; Ki[7] = K[1] * K[6] - K[0] * K[7]; Ki[8] = K[0] * K[4] - K[1] * K[3];
    det = K[0] * Ki[0] + K[1] * Ki[3] + K[2] * Ki[6];
    for (k = 0; k < 9; ++k) Ki[k] /= det;
    for (s = 0; c >= 4 && s < max_samples; ++s) {
        int32_t pos[4];
        int sc = 0, sp = 0;
        double f[9], sR[9], st[3];
        ransac_oracle_draw4(c, g, s, seed, pos);
        for (k = 0; k < 3; ++k) {
            const double *px = uv + 2 * cand[pos[k]];
            for (i = 0; i < 3; ++i) f[3 * k + i] = Ki[3 * i] * px[0] + Ki[3 * i + 1] * px[1] + Ki[3 * i + 2];
            unit3(f + 3 * k);
        }
        for (p = 0; p < P; ++p) {
            const double *Pp = patterns + (size_t)p * n_total * 3;
            double X[9], Rs[36], ts[12], M[9], m[3], bd = INFINITY, d4[4];
            int ns, r, br = -1, cnt = 0;
            for (k = 0; k < 3; ++k) for (i = 0; i < 3; ++i) X[3 * k + i] = Pp[3 * cand[pos[k]] + i];
            ns = ransac_oracle_p3p(X, f, Rs, ts);
            for (r = 0; r < ns; ++r) {
                fold_km(K, Rs + 9 * r, ts + 3 * r, M, m);
                d4[r] = check_distance(M, m, Pp + 3 * cand[pos[3]], uv + 2 * cand[pos[3]]);
                if (d4[r] < bd) { bd = d4[r]; br = r; }
            }
            for (r = 0; r < ns; ++r)
                if (r != br && br >= 0 && near_thr(d4[r], bd)) *near = 1;
            if (br >= 0 && near_thr(bd, consensus_px)) *near = 1;
            if (!(br >= 0 && bd <= consensus_px)) continue;
            fold_km(K, Rs + 9 * br, ts + 3 * br, M, m);
            for (i = 0; i < c; ++i) {
                double d = check_distance(M, m, Pp + 3 * cand[i], uv + 2 * cand[i]);
                if (near_thr(d, consensus_px)) *near = 1;
                cnt += d <= consensus_px;
            }
            if (cnt > sc) {                          /* ties to the lower pattern */
                sc = cnt; sp = p;
                memcpy(sR, Rs + 9 * br, sizeof(sR)); memcpy(st, ts + 3 * br, sizeof(st));
            }
        }
        if (sc > best) {                             /* ties to the lower sample */
            best = sc; win_p = sp; *win_s = s;
            memcpy(wR, sR, sizeof(wR)); memcpy(wt, st, sizeof(wt));
        }
        drawn = s + 1;
        {
            int64_t c2 = (int64_t)c * c, b2 = (int64_t)best * best;
            double q = (double)(c2 * c2 - b2 * b2) / (double)(c2 * c2);
            if (powi_ex(q, s + 1) <= 1.0 - confidence) break;
        }
    }
    memset(mask, 0, (size_t)n_total);
    if (best > 0) {
        const double *Pp = patterns + (size_t)win_p * n_total * 3;
        double M[9], m[3];
        fold_km(K, wR, wt, M, m);
        for (i = 0; i < c; ++i)
            if (check_distance(M, m, Pp + 3 * cand[i], uv + 2 * cand[i]) <= consensus_px) mask[cand[i]] = 1;
        memcpy(R, wR, sizeof(wR)); memcpy(t, wt, sizeof(wt));
    } else {
        for (k = 0; k < 9; ++k) R[k] = NAN;
        for (k = 0; k < 3; ++k) t[k] = NAN;
    }
    *best_pattern = win_p; *consensus = best;
    return drawn;
}
