// pnpb200_p3p.cuh -- the minimal (three-point) pose solver of the hypothesis stage: Lambda Twist (Persson & Nordberg, "Lambda
// Twist: An Accurate Fast Robust Perspective Three Point (P3P) Solver", ECCV 2018), in FP64, with its Gauss-Newton
// refinement of the three depths.  One cubic root, a closed-form eigen step of a 3x3 matrix with one known zero eigenvalue,
// two quadratics: at most 4 poses.  Divisions and square roots are the branch-free ones of pnpb200_math.cuh (DESIGN.md 6):
// a degenerate triple yields non-finite values, and such roots are dropped like roots with a depth <= 0.
#pragma once
#include "pnpb200_math.cuh"

namespace pnpb200 {

// the roots of x^2 + b x + c without cancellation (b^2 >= 4 c): r1 is the one of larger magnitude
PNP_DEV void p3p_root2(double b, double c, double& r1, double& r2)
{
    const double y = sqrt_nonneg(fmax(fma(b, b, -4.0 * c), 0.0));
    const double q = b < 0.0 ? 0.5 * (y - b) : -0.5 * (b + y);   // -(b + sign(b) y) / 2
    r1 = q;
    r2 = c * t_rcp<double>(q);
}

// a real root of x^3 + b x^2 + c x + d: the start of the reference implementation (a second-order model around the
// stationary point that brackets a root), then Newton steps that keep the last finite iterate
PNP_DEV double p3p_cubic(double b, double c, double d)
{
    const double disc = fma(b, b, -3.0 * c);
    const double v = sqrt_nonneg(fmax(disc, 0.0));
    const double t1 = (-b - v) * (1.0 / 3.0), t2 = (v - b) * (1.0 / 3.0);
    const double k1 = fma(fma(t1 + b, t1, c), t1, d);
    const double k2 = fma(fma(t2 + b, t2, c), t2, d);
    const bool left = k1 > 0.0;
    const double tk = left ? t1 : t2, kk = left ? k1 : k2;
    const double step = sqrt_nonneg(fmax(-kk * t_rcp<double>(fma(3.0, tk, b)), 0.0));
    double r = disc >= 0.0 ? (left ? tk - step : tk + step) : -b * (1.0 / 3.0);
    if (!(disc >= 0.0) && fabs(fma(fma(3.0, r, 2.0 * b), r, c)) < 1e-4) r += 1.0;
#pragma unroll 1
    for (int it = 0; it < 12; ++it) {
        const double fx = fma(fma(r + b, r, c), r, d);
        const double fp = fma(fma(3.0, r, 2.0 * b), r, c);
        const double rn = fma(-fx, t_rcp<double>(fp), r);
        r = (rn - rn == 0.0) ? rn : r;
    }
    return r;
}

// Gauss-Newton on the three distance constraints l_i^2 + l_j^2 + b_ij l_i l_j = a_ij; a step is kept only where it lowers
// the residual (the reference's rule, without its early exit: a fixed count of steps)
PNP_DEV void p3p_refine(double (&L)[3], double a12, double a13, double a23, double b12, double b13, double b23)
{
#pragma unroll 1
    for (int it = 0; it < 5; ++it) {
        const double l1 = L[0], l2 = L[1], l3 = L[2];
        const double r1 = fma(l1, l1, fma(l2, l2, fma(b12 * l1, l2, -a12)));
        const double r2 = fma(l1, l1, fma(l3, l3, fma(b13 * l1, l3, -a13)));
        const double r3 = fma(l2, l2, fma(l3, l3, fma(b23 * l2, l3, -a23)));
        const double v0 = fma(2.0, l1, b12 * l2), v1 = fma(2.0, l2, b12 * l1);
        const double v3 = fma(2.0, l1, b13 * l3), v5 = fma(2.0, l3, b13 * l1);
        const double v7 = fma(2.0, l2, b23 * l3), v8 = fma(2.0, l3, b23 * l2);
        const double det = t_rcp<double>(-v0 * v5 * v7 - v1 * v3 * v8);
        const double n1 = l1 - det * (-v5 * v7 * r1 - v1 * v8 * r2 + v1 * v5 * r3);
        const double n2 = l2 - det * (-v3 * v8 * r1 + v0 * v8 * r2 - v0 * v5 * r3);
        const double n3 = l3 - det * (v3 * v7 * r1 - v0 * v7 * r2 - v1 * v3 * r3);
        const double s1 = fma(n1, n1, fma(n2, n2, fma(b12 * n1, n2, -a12)));
        const double s2 = fma(n1, n1, fma(n3, n3, fma(b13 * n1, n3, -a13)));
        const double s3 = fma(n2, n2, fma(n3, n3, fma(b23 * n2, n3, -a23)));
        const bool better = fabs(s1) + fabs(s2) + fabs(s3) < fabs(r1) + fabs(r2) + fabs(r3);
        L[0] = better ? n1 : l1; L[1] = better ? n2 : l2; L[2] = better ? n3 : l3;
    }
}

// Up to 4 poses (R row-major, t) with R X_k + t = l_k f_k, l_k > 0, for the pattern points X[k] (metres) and the unit
// bearings f[k] (K^-1 [u, v, 1] normalised), k = 0..2.  The roots sit in fixed slots (two per sign of the eigen step's
// square root), so that every index is a compile-time one and the poses stay in registers; returns the mask of the valid
// slots.  A root with a non-finite value or a depth <= 0 is not valid.
PNP_DEV unsigned p3p_lambda_twist(const double (&X)[9], const double (&f)[9], double (&R)[4][9], double (&t)[4][3])
{
    const double* y1 = f;
    const double* y2 = f + 3;
    const double* y3 = f + 6;
    const double b12 = -2.0 * (y1[0] * y2[0] + y1[1] * y2[1] + y1[2] * y2[2]);
    const double b13 = -2.0 * (y1[0] * y3[0] + y1[1] * y3[1] + y1[2] * y3[2]);
    const double b23 = -2.0 * (y2[0] * y3[0] + y2[1] * y3[1] + y2[2] * y3[2]);
    double d12[3], d13[3], d23[3], dx[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) { d12[k] = X[k] - X[3 + k]; d13[k] = X[k] - X[6 + k]; d23[k] = X[3 + k] - X[6 + k]; }
    dx[0] = d12[1] * d13[2] - d12[2] * d13[1];
    dx[1] = d12[2] * d13[0] - d12[0] * d13[2];
    dx[2] = d12[0] * d13[1] - d12[1] * d13[0];
    const double a12 = d12[0] * d12[0] + d12[1] * d12[1] + d12[2] * d12[2];
    const double a13 = d13[0] * d13[0] + d13[1] * d13[1] + d13[2] * d13[2];
    const double a23 = d23[0] * d23[0] + d23[1] * d23[1] + d23[2] * d23[2];
    const double c31 = -0.5 * b13, c23 = -0.5 * b23, c12 = -0.5 * b12;
    const double blob = c12 * c23 * c31 - 1.0;
    const double s31 = fma(-c31, c31, 1.0), s23 = fma(-c23, c23, 1.0), s12 = fma(-c12, c12, 1.0);
    // the cubic det(D1 + g D2) = 0 of the two conics, monic
    const double p3 = a13 * (a23 * s31 - a13 * s23);
    const double p2 = 2.0 * blob * a23 * a13 + a13 * (2.0 * a12 + a13) * s23 + a23 * (a23 - a12) * s31;
    const double p1 = a23 * (a13 - a23) * s12 - a12 * a12 * s23 - 2.0 * a12 * (blob * a23 + a13 * s23);
    const double p0 = a12 * (a12 * s23 - a23 * s12);
    const double ip3 = t_rcp<double>(p3);
    const double g = p3p_cubic(p2 * ip3, p1 * ip3, p0 * ip3);
    // D0 = D1 + g D2 (symmetric, one eigenvalue 0): its other two eigenpairs in closed form
    const double A00 = a23 * (1.0 - g), A01 = a23 * b12 * 0.5, A02 = a23 * b13 * g * -0.5;
    const double A11 = a23 - a12 + a13 * g, A12 = b23 * (a13 * g - a12) * 0.5, A22 = g * (a13 - a23) - a12;
    const double tb = -A00 - A11 - A22;
    const double tc = -A01 * A01 - A02 * A02 - A12 * A12 + A00 * (A11 + A22) + A11 * A22;
    double e1, e2;
    p3p_root2(tb, tc, e1, e2);                            // |e1| >= |e2|
    const double mx0011 = -A00 * A11;
    const double prec0 = A01 * A12 - A02 * A11, prec1 = A01 * A02 - A00 * A12;
    double V[3][2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const double e = j == 0 ? e1 : e2;
        const double tmp = t_rcp<double>(e * (A00 + A11) + mx0011 - e * e + A01 * A01);
        const double q1 = -(e * A02 + prec0) * tmp, q2 = -(e * A12 + prec1) * tmp;
        const double rn = t_rsqrt<double>(fma(q1, q1, fma(q2, q2, 1.0)));
        V[0][j] = q1 * rn; V[1][j] = q2 * rn; V[2][j] = rn;
    }
    const double v = sqrt_nonneg(fmax(-e2 * t_rcp<double>(e1), 0.0));
    // the inverse of [d12, d13, d12 x d13] (columns), for R = Y X^-1
    double Xi[9];
    {
        const double m[9] = { d12[0], d13[0], dx[0], d12[1], d13[1], dx[1], d12[2], d13[2], dx[2] };
        Xi[0] = m[4] * m[8] - m[5] * m[7]; Xi[1] = m[2] * m[7] - m[1] * m[8]; Xi[2] = m[1] * m[5] - m[2] * m[4];
        Xi[3] = m[5] * m[6] - m[3] * m[8]; Xi[4] = m[0] * m[8] - m[2] * m[6]; Xi[5] = m[2] * m[3] - m[0] * m[5];
        Xi[6] = m[3] * m[7] - m[4] * m[6]; Xi[7] = m[1] * m[6] - m[0] * m[7]; Xi[8] = m[0] * m[4] - m[1] * m[3];
        const double id = t_rcp<double>(m[0] * Xi[0] + m[1] * Xi[3] + m[2] * Xi[6]);
#pragma unroll
        for (int e = 0; e < 9; ++e) Xi[e] *= id;
    }
    unsigned valid = 0;
#pragma unroll
    for (int sg = 0; sg < 2; ++sg) {
        const double s = sg == 0 ? v : -v;
        const double w2 = t_rcp<double>(s * V[0][1] - V[0][0]);
        const double w0 = (V[1][0] - s * V[1][1]) * w2, w1 = (V[2][0] - s * V[2][1]) * w2;
        const double a = t_rcp<double>((a13 - a12) * w1 * w1 - a12 * b13 * w1 - a12);
        const double qb = (a13 * b12 * w1 - a12 * b13 * w0 - 2.0 * w0 * w1 * (a12 - a13)) * a;
        const double qc = ((a13 - a12) * w0 * w0 + a13 * b12 * w0 + a13) * a;
        const bool real = fma(qb, qb, -4.0 * qc) >= 0.0;
        double tau[2];
        p3p_root2(qb, qc, tau[0], tau[1]);
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const double ta = tau[r];
            const double dd = a23 * t_rcp<double>(fma(ta, b23 + ta, 1.0));
            const double l2 = sqrt_nonneg(fmax(dd, 0.0)), l3 = ta * l2;
            double L[3] = { fma(w0, l2, w1 * l3), l2, l3 };
            const bool root = real && ta > 0.0 && L[0] >= 0.0;
            p3p_refine(L, a12, a13, a23, b12, b13, b23);
            double ry1[3], yd1[3], yd2[3], yx[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                ry1[k] = y1[k] * L[0];
                yd1[k] = ry1[k] - y2[k] * L[1];
                yd2[k] = ry1[k] - y3[k] * L[2];
            }
            yx[0] = yd1[1] * yd2[2] - yd1[2] * yd2[1];
            yx[1] = yd1[2] * yd2[0] - yd1[0] * yd2[2];
            yx[2] = yd1[0] * yd2[1] - yd1[1] * yd2[0];
            double Rr[9], tr[3];
            bool fin = root && L[0] > 0.0 && L[1] > 0.0 && L[2] > 0.0;
#pragma unroll
            for (int i = 0; i < 3; ++i) {
#pragma unroll
                for (int j = 0; j < 3; ++j) {
                    Rr[i * 3 + j] = yd1[i] * Xi[j] + yd2[i] * Xi[3 + j] + yx[i] * Xi[6 + j];
                    fin = fin && Rr[i * 3 + j] - Rr[i * 3 + j] == 0.0;
                }
            }
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                tr[i] = ry1[i] - (Rr[i * 3] * X[0] + Rr[i * 3 + 1] * X[1] + Rr[i * 3 + 2] * X[2]);
                fin = fin && tr[i] - tr[i] == 0.0;
            }
#pragma unroll
            for (int e = 0; e < 9; ++e) R[2 * sg + r][e] = Rr[e];
#pragma unroll
            for (int e = 0; e < 3; ++e) t[2 * sg + r][e] = tr[e];
            valid |= fin ? 1u << (2 * sg + r) : 0u;
        }
    }
    return valid;
}

}  // namespace pnpb200
