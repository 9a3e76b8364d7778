// pnpb200_reproject.cuh -- the projection of a pattern point by a pose and its distance to the measured pixel, as the
// error report (TEST_TOOLBOX.py:252-286), the solution check and the inlier classification of the robust solve compute them.
#pragma once
#include "pnpb200_math.cuh"

namespace pnpb200 {

PNP_DEV void fold_camera(const double* K, const double (&R)[9], const double (&t)[3], double (&M)[9], double (&m)[3])
{
#pragma unroll
    for (int r = 0; r < 3; ++r) {
#pragma unroll
        for (int c = 0; c < 3; ++c) M[r * 3 + c] = K[r * 3] * R[c] + K[r * 3 + 1] * R[3 + c] + K[r * 3 + 2] * R[6 + c];
        m[r] = K[r * 3] * t[0] + K[r * 3 + 1] * t[1] + K[r * 3 + 2] * t[2];
    }
}

// The projection of one point before its division by |z|: o = (r0, r1), inv = 1 / r2 (:4548 divides by |z|; branch-free,
// <= 0.5003 ulp); behind = the homogeneous coordinate z / |z| is -1 (the point is behind the camera)
PNP_DEV void project_folded(const double (&M)[9], const double (&m)[3], double x, double y, double z, double (&o)[2], double& inv, bool& behind)
{
    o[0] = fma(M[0], x, fma(M[1], y, fma(M[2], z, m[0])));
    o[1] = fma(M[3], x, fma(M[4], y, fma(M[5], z, m[1])));
    const double r2 = fma(M[6], x, fma(M[7], y, fma(M[8], z, m[2])));
    inv = t_rcp<double>(r2);
    behind = __double2hiint(r2) < 0;
}

// The three error distances of one landmark (cal_LM_error_distances, TEST_TOOLBOX.py:252-286).  The
// third component of every difference is a difference of homogeneous coordinates that are exactly +-1
// (the measured one is +1), so its square is 0 or 4.  The division of each projection by |z| and its
// difference to the measured pixel are one FMA per coordinate (the absolute value rides on it as an
// operand modifier); the prediction-vs-GT difference is the difference of the other two.
PNP_DEV void px_difference(const double (&r)[2], double inv, double mu, double mv, double& dx, double& dy)
{
    dx = fma(r[0], fabs(inv), -mu); dy = fma(r[1], fabs(inv), -mv);
}
PNP_DEV double homogeneous_distance(double dx, double dy, bool flipped)
{
    return sqrt_nonneg(fma(dx, dx, fma(dy, dy, flipped ? 4.0 : 0.0)));
}
}  // namespace pnpb200
