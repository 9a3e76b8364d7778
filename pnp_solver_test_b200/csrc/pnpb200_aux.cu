// pnpb200_aux.cu -- the kernels either side of the solve: Euler <-> R, pinhole projection,
// the counter-based synthetic workload generator, per-problem error reporting, the two-pass
// error statistics, and the FMA-pipe microbenchmark used for the roofline denominator.
//
// All of these are streaming, HBM-bound kernels: one thread (or one warp) per problem,
// coalesced loads, grids sized from the problem count.
#include "pnpb200_common.cuh"
#include "pnpb200_math.cuh"
#include "pnpb200_tile.cuh"
#include "pnpb200_reproject.cuh"

namespace pnpb200 {

template <typename T> PNP_DEV double ld(const void* p, size_t i) { return (double)((const T*)p)[i]; }
template <typename T> PNP_DEV void st(void* p, size_t i, double v) { ((T*)p)[i] = (T)v; }

static inline unsigned grid_for(long long n, int block)
{
    long long g = (n + block - 1) / block;
    if (g < 1) g = 1;
    if (g > 0x7fffffffLL) g = 0x7fffffffLL;
    return (unsigned)g;
}

// ------------------------------------------------------------------------------------------
// Euler <-> R  (PNP_SOLVER_LIB.py:4442-4517)
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void k_R_from_euler(long long B, const void* euler, int is_degree, void* R)
{
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    double Rm[9];
    R_from_euler(ld<T>(euler, b * 3), ld<T>(euler, b * 3 + 1), ld<T>(euler, b * 3 + 2), is_degree != 0, Rm);
#pragma unroll
    for (int e = 0; e < 9; ++e) st<T>(R, b * 9 + e, Rm[e]);
}

template <typename T>
__global__ void k_euler_from_R(long long B, const void* R, int is_degree, void* euler)
{
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    double Rm[9], e3[3];
#pragma unroll
    for (int e = 0; e < 9; ++e) Rm[e] = ld<T>(R, b * 9 + e);
    euler_from_R(Rm, is_degree != 0, e3);
#pragma unroll
    for (int e = 0; e < 3; ++e) st<T>(euler, b * 3 + e, e3[e]);
}

// ------------------------------------------------------------------------------------------
// projection  (perspective_projection :4532-4557): K (R theta + t) / |z|, optional np.around
// ------------------------------------------------------------------------------------------
PNP_DEV void project_point(const double* K, const double (&R)[9], const double (&t)[3], double x, double y, double z,
                           bool quant, double q, double (&o)[3])
{
    double X[3], ray[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) X[r] = R[r * 3] * x + R[r * 3 + 1] * y + R[r * 3 + 2] * z + t[r];
#pragma unroll
    for (int r = 0; r < 3; ++r) ray[r] = K[r * 3] * X[0] + K[r * 3 + 1] * X[1] + K[r * 3 + 2] * X[2];
    const double az = fabs(ray[2]);                       // :4548
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        double v = ray[r] / az;
        if (quant) v = rint(v / q) * q;                   // half-to-even, like np.around (:4551)
        o[r] = v;
    }
}

// Same projection for the error report (never quantised): one reciprocal instead of three
// divisions; the homogeneous coordinate z/|z| is exactly +-1.
PNP_DEV void project_point_fast(const double* K, const double (&R)[9], const double (&t)[3], double x, double y, double z,
                                double (&o)[3])
{
    double X[3], ray[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) X[r] = R[r * 3] * x + R[r * 3 + 1] * y + R[r * 3 + 2] * z + t[r];
#pragma unroll
    for (int r = 0; r < 3; ++r) ray[r] = K[r * 3] * X[0] + K[r * 3 + 1] * X[1] + K[r * 3 + 2] * X[2];
    const double inv = 1.0 / fabs(ray[2]);
    o[0] = ray[0] * inv; o[1] = ray[1] * inv; o[2] = copysign(1.0, ray[2]);
}

struct KMat { double k[9]; };

template <typename T>
__global__ void k_project(long long B, int n, const void* pattern, KMat K, const void* R, const void* t,
                          int quant, double q, void* uvw)
{
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // (problem, point)
    if (e >= B * n) return;
    const long long b = e / n;
    const int i = (int)(e - b * n);
    double Rm[9], tv[3], o[3];
#pragma unroll
    for (int k = 0; k < 9; ++k) Rm[k] = ld<T>(R, b * 9 + k);
#pragma unroll
    for (int k = 0; k < 3; ++k) tv[k] = ld<T>(t, b * 3 + k);
    project_point(K.k, Rm, tv, ld<T>(pattern, 3 * i), ld<T>(pattern, 3 * i + 1), ld<T>(pattern, 3 * i + 2), quant != 0, q, o);
#pragma unroll
    for (int k = 0; k < 3; ++k) st<T>(uvw, e * 3 + k, o[k]);
}

// ------------------------------------------------------------------------------------------
// synthetic workload  (random_stress_test.py:246-290, LM_noise_test.py noise model)
// Philox4x32-10 keyed by seed, counter = (global problem index, stream id).  Bit-identical to
// the integer part of oracle/pnp_oracle.c; the trigonometry may differ in the last ulp.  (philox4x32_10: pnpb200_math.cuh)
// ------------------------------------------------------------------------------------------
PNP_DEV double u01(uint32_t hi, uint32_t lo)
{
    const unsigned long long v = (((unsigned long long)hi << 32) | lo) >> 11;
    return (double)v * (1.0 / 9007199254740992.0);
}

// three N(0,1) draws for point i of problem gidx (pattern perturbation, face_variation_test.py:324)
PNP_DEV void perturb_normals(uint32_t g0, uint32_t g1, int i, uint32_t k0, uint32_t k1, double (&z)[3])
{
    uint32_t a[4], b[4];
    philox4x32_10(g0, g1, 16u + (uint32_t)i, 2u, k0, k1, a);
    philox4x32_10(g0, g1, 16u + (uint32_t)i, 3u, k0, k1, b);
    const double r1 = sqrt(-2.0 * log(1.0 - u01(a[0], a[1]))), r2 = sqrt(-2.0 * log(1.0 - u01(b[0], b[1])));
    double sn, cs;
    sincos(2.0 * 3.14159265358979323846 * u01(a[2], a[3]), &sn, &cs);
    z[0] = r1 * cs; z[1] = r1 * sn;
    z[2] = r2 * cos(2.0 * 3.14159265358979323846 * u01(b[2], b[3]));
}

template <typename T>
__global__ void k_synth(long long b0, long long B, int n, const double* __restrict__ pattern, KMat K, pnpb200_synth cfg,
                        void* uv, double* gt, double* R_gt, double* t_gt, double perturb_radius, int fixed_idx, double* perturb)
{
    // one warp per problem: lane 0's pose is broadcast, lanes stride over the points
    const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= B) return;
    const unsigned long long gidx = (unsigned long long)(b0 + w);
    const uint32_t k0 = (uint32_t)cfg.seed, k1 = (uint32_t)(cfg.seed >> 32);
    const uint32_t g0 = (uint32_t)gidx, g1 = (uint32_t)(gidx >> 32);
    uint32_t r0[4], r1[4], r2[4];
    philox4x32_10(g0, g1, 0u, 0u, k0, k1, r0);
    philox4x32_10(g0, g1, 1u, 0u, k0, k1, r1);
    philox4x32_10(g0, g1, 2u, 0u, k0, k1, r2);
    const double kD2R = 3.14159265358979323846 / 180.0;
    const double a = cfg.angle_range_deg, f = cfg.fov_max_deg;
    const double roll = cfg.roll_center_deg + (-a + 2.0 * a * u01(r0[0], r0[1]));
    const double pitch = cfg.pitch_center_deg + (-a + 2.0 * a * u01(r0[2], r0[3]));
    const double yaw = cfg.yaw_center_deg + (-a + 2.0 * a * u01(r1[0], r1[1]));
    const double depth = cfg.depth_min_m + (cfg.depth_max_m - cfg.depth_min_m) * u01(r1[2], r1[3]);
    const double fx = -f + 2.0 * f * u01(r2[0], r2[1]);
    const double fy = -f + 2.0 * f * u01(r2[2], r2[3]);
    double Rm[9], tv[3];
    tv[0] = depth * tan(fx * kD2R); tv[1] = depth * tan(fy * kD2R); tv[2] = depth;
    R_from_euler(roll, yaw, pitch, true, Rm);
    // face_variation_test.py:317-345: a random direction of the 3 (n - 1) pattern coordinates (one
    // landmark stays fixed), scaled to perturb_radius, moves the pattern the pixels are generated from
    double pscale = 0.0;
    if (perturb_radius > 0.0) {
        double ss = 0.0;
        for (int i = lane; i < n; i += 32) {
            if (i == fixed_idx) continue;
            double z[3];
            perturb_normals(g0, g1, i, k0, k1, z);
            ss += z[0] * z[0] + z[1] * z[1] + z[2] * z[2];
        }
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, off);
        pscale = perturb_radius / sqrt(ss);
    }
    for (int i = lane; i < n; i += 32) {
        double o[3];
        double px = pattern[3 * i], py = pattern[3 * i + 1], pz = pattern[3 * i + 2];
        if (perturb_radius > 0.0) {
            double z[3] = { 0.0, 0.0, 0.0 };
            if (i != fixed_idx) perturb_normals(g0, g1, i, k0, k1, z);
            const double d0 = pscale * z[0], d1 = pscale * z[1], d2 = pscale * z[2];
            px += d0; py += d1; pz += d2;
            if (perturb) { perturb[((size_t)w * n + i) * 3] = d0; perturb[((size_t)w * n + i) * 3 + 1] = d1; perturb[((size_t)w * n + i) * 3 + 2] = d2; }
        }
        project_point(K.k, Rm, tv, px, py, pz, false, 1.0, o);
        double u = o[0], v = o[1];
        if (cfg.is_quantized) { u = rint(u / cfg.quantize_q) * cfg.quantize_q; v = rint(v / cfg.quantize_q) * cfg.quantize_q; }
        if (cfg.noise_sigma_px > 0.0) {
            uint32_t g[4];
            philox4x32_10(g0, g1, 16u + (uint32_t)i, 1u, k0, k1, g);
            const double ua = u01(g[0], g[1]), ub = u01(g[2], g[3]);
            const double rad = sqrt(-2.0 * log(1.0 - ua));
            double sn, cs;
            sincos(2.0 * 3.14159265358979323846 * ub, &sn, &cs);
            u += cfg.noise_sigma_px * rad * cs;
            v += cfg.noise_sigma_px * rad * sn;
        }
        st<T>(uv, ((size_t)w * n + i) * 2, u);
        st<T>(uv, ((size_t)w * n + i) * 2 + 1, v);
    }
    if (lane == 0) {
        if (gt) { gt[w * 4] = depth; gt[w * 4 + 1] = roll; gt[w * 4 + 2] = pitch; gt[w * 4 + 3] = yaw; }
        if (R_gt) {
#pragma unroll
            for (int e = 0; e < 9; ++e) R_gt[w * 9 + e] = Rm[e];
        }
        if (t_gt) { t_gt[w * 3] = tv[0]; t_gt[w * 3 + 1] = tv[1]; t_gt[w * 3 + 2] = tv[2]; }
    }
}

// ------------------------------------------------------------------------------------------
// error reporting (TEST_TOOLBOX.py:55-62, :252-286, :291-465; random_stress_test.py:353-377)
// one warp per problem: lanes stride over the landmarks, shuffle-reduce sum / max / arg-max
// ------------------------------------------------------------------------------------------
struct Bounds { double b[4]; };

// a masked problem with fewer than kMinVisible visible landmarks: NaN statistics, no worst landmark
PNP_DEV void too_few_for_report(double& s0, double& s1, double& s2, double& m0, double& m1, double& m2, int& i0, int& i1, int& i2)
{
    s0 = s1 = s2 = m0 = m1 = m2 = __longlong_as_double(0x7ff8000000000000LL);
    i0 = i1 = i2 = -1;
}

// check_if_the_sample_passed on depth (TEST_TOOLBOX.py:55-62 with random_stress_test.py:374-377's t3 * 100 and dist_cm):
// both products in centimetres are rounded before their difference, as the reference rounds them (contracting one of
// them into an FMA flips the flag on some pairs within a few ulp of the bound)
PNP_DEV int32_t depth_passed(double t3, double dist, double bound)
{
    return fabs(__dmul_rn(t3, 100.0) - __dmul_rn(dist, 100.0)) < bound;
}

PNP_DEV void warp_sum_max(double& s, double& m, int& im)
{
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, off);
        const double om = __shfl_xor_sync(0xffffffffu, m, off);
        const int oi = __shfl_xor_sync(0xffffffffu, im, off);
        // strict '>' with first-index-wins (cal_LM_error_distances :274)
        if (om > m || (om == m && oi >= 0 && (im < 0 || oi < im))) { m = om; im = oi; }
    }
}

// MASKED: the statistics of columns 4-9 run over the landmarks whose bit is set in vis[b * vis_words ...]
template <typename T, bool MASKED = false>
__global__ void k_report(long long B, int n, const void* pattern, const void* uv, KMat K, const void* R, const void* t,
                         const void* euler, const double* __restrict__ gt, Bounds bounds, double* report,
                         long long rs_b, long long rs_k, int32_t* flags, int32_t* max_idx,
                         const uint32_t* vis = nullptr, int vis_words = 0)
{
    const long long b = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (b >= B) return;
    double Re[9], te[3], Rg[9], tg[3];
#pragma unroll
    for (int k = 0; k < 9; ++k) Re[k] = ld<T>(R, b * 9 + k);
#pragma unroll
    for (int k = 0; k < 3; ++k) te[k] = ld<T>(t, b * 3 + k);
    const double roll_e = ld<T>(euler, b * 3), yaw_e = ld<T>(euler, b * 3 + 1), pitch_e = ld<T>(euler, b * 3 + 2);
    const double dist = gt[b * 4], roll_g = gt[b * 4 + 1], pitch_g = gt[b * 4 + 2], yaw_g = gt[b * 4 + 3];
    const double t3 = te[2];
    R_from_euler_deg_bounded(roll_g, yaw_g, pitch_g, Rg); // random_stress_test.py:365
#pragma unroll
    for (int k = 0; k < 3; ++k) tg[k] = (te[k] / t3) * dist;   // :367-368
    double s0 = 0, s1 = 0, s2 = 0, m0 = 0, m1 = 0, m2 = 0;
    int i0 = -1, i1 = -1, i2 = -1;
    const uint32_t* vw = MASKED ? vis + (size_t)b * vis_words : nullptr;
    const int nv = MASKED ? count_visible(vw, nullptr, n) : 0;
    // sqrt_nonneg, as homogeneous_distance: a distance whose square is not finite (depth 0, where the projection is +-inf;
    // a non-finite pixel) is NaN, as in the streaming kernels, and so never the maximum.  The prediction-vs-GT difference is
    // the sum of the two pixel differences, as in landmark_errors, so a non-finite pixel makes all three distances NaN.
    for (int i = lane; i < n; i += 32) {
        if constexpr (MASKED) { if (!mask_bit(vw, i)) continue; }
        const double x = ld<T>(pattern, 3 * i), y = ld<T>(pattern, 3 * i + 1), z = ld<T>(pattern, 3 * i + 2);
        double pe[3], pg[3];
        project_point_fast(K.k, Re, te, x, y, z, pe);          // TEST_TOOLBOX.py:312
        project_point_fast(K.k, Rg, tg, x, y, z, pg);          // :314
        const double mu = ld<T>(uv, ((size_t)b * n + i) * 2), mv = ld<T>(uv, ((size_t)b * n + i) * 2 + 1), mw = 1.0;
        double d0, d1, d2, e;
        const double g0 = mu - pg[0], g1 = mv - pg[1], g2 = mw - pg[2];   // LM vs GT (:321)
        e = sqrt_nonneg(g0 * g0 + g1 * g1 + g2 * g2); s0 += e; if (e > m0) { m0 = e; i0 = i; }
        d0 = pe[0] - mu; d1 = pe[1] - mv; d2 = pe[2] - mw;     // prediction vs LM (:326)
        e = sqrt_nonneg(d0 * d0 + d1 * d1 + d2 * d2); s1 += e; if (e > m1) { m1 = e; i1 = i; }
        d0 += g0; d1 += g1; d2 = pe[2] - pg[2];                 // prediction vs GT (:331) through the pixel, as landmark_errors
        e = sqrt_nonneg(d0 * d0 + d1 * d1 + d2 * d2); s2 += e; if (e > m2) { m2 = e; i2 = i; }
    }
    warp_sum_max(s0, m0, i0); warp_sum_max(s1, m1, i1); warp_sum_max(s2, m2, i2);
    if constexpr (MASKED) { if (nv < kMinVisible) too_few_for_report(s0, s1, s2, m0, m1, m2, i0, i1, i2); }
    if (lane == 0) {
        double* rp = report + b * rs_b;
        const long long sk = rs_k;
        rp[0] = t3 - dist; rp[sk] = roll_e - roll_g; rp[2 * sk] = pitch_e - pitch_g; rp[3 * sk] = yaw_e - yaw_g;
        rp[4 * sk] = (s0 / (MASKED ? nv : n)) * dist; rp[5 * sk] = m0 * dist;  // :452-453
        rp[6 * sk] = (s1 / (MASKED ? nv : n)) * dist; rp[7 * sk] = m1 * dist;
        rp[8 * sk] = (s2 / (MASKED ? nv : n)) * dist; rp[9 * sk] = m2 * dist;
        rp[10 * sk] = t3; rp[11 * sk] = dist; rp[12 * sk] = roll_e; rp[13 * sk] = pitch_e; rp[14 * sk] = yaw_e; rp[15 * sk] = 0.0;
        if (flags) {                                           // check_if_the_sample_passed (:55-62), depth in cm
            flags[b * 4] = depth_passed(t3, dist, bounds.b[0]);
            flags[b * 4 + 1] = fabs(roll_e - roll_g) < bounds.b[1];
            flags[b * 4 + 2] = fabs(pitch_e - pitch_g) < bounds.b[2];
            flags[b * 4 + 3] = fabs(yaw_e - yaw_g) < bounds.b[3];
        }
        if (max_idx) { max_idx[b * 3] = i0; max_idx[b * 3 + 1] = i1; max_idx[b * 3 + 2] = i2; }
    }
}

// Same report, one problem per thread: the 32 pixel rows of a warp's problems are staged by TMA
// bulk copies (pnpb200_tile.cuh), K is folded into the two poses once per problem (M = K R,
// m = K t), and the Euler -> R trigonometry is done once per problem instead of once per lane.
template <typename T>
struct ReportArgs {
    const T* pattern; const T* uv; const T* R; const T* t; const T* euler;
    const double* gt;
    long long B;
    int n, row_pitch, use_tma;
    double K[9], bounds[4];
    double* report; int32_t* flags; int32_t* max_idx;
    long long rs_b, rs_k;           // element strides of report between problems / between columns
    // fused residual pass of the moment mapping (k_report_chunk<T, RES != 0>): the 12 numbers per problem that
    // k_iterate left in the workspace ([12][ld], LM: the state before the last update; F2: its tail) -> res_norm
    const T* tail; long long ld; T* res; double kinv[6];
    int use_tmap;
    alignas(64) CUtensorMap tmap;   // uv as a 2-D tensor (RowStream), valid when use_tmap
    const uint32_t* vis; int vis_words;   // [B, vis_words] visibility bits (masked kernels only)
};

PNP_DEV void landmark_errors(const double (&re)[2], double inv_e, bool be, const double (&rg)[2], double inv_g, bool bg,
                             double mu, double mv, double& e0, double& e1, double& e2)
{
    double gx, gy, ex, ey;
    px_difference(rg, inv_g, mu, mv, gx, gy);             // GT - LM (:321, squared)
    px_difference(re, inv_e, mu, mv, ex, ey);             // prediction - LM (:326)
    e0 = homogeneous_distance(gx, gy, bg);
    e1 = homogeneous_distance(ex, ey, be);
    e2 = homogeneous_distance(ex - gx, ey - gy, be != bg);   // prediction - GT (:331)
}

template <typename T>
PNP_DEV void load_report_pose(const ReportArgs<T>& a, long long b, double (&Re)[9], double (&te)[3], double (&eu)[3], double (&g4)[4])
{
#pragma unroll
    for (int k = 0; k < 4; ++k) g4[k] = __ldg(a.gt + b * 4 + k);
#pragma unroll
    for (int k = 0; k < 3; ++k) te[k] = (double)__ldg(a.t + b * 3 + k);
#pragma unroll
    for (int k = 0; k < 9; ++k) Re[k] = (double)__ldg(a.R + b * 9 + k);
#pragma unroll
    for (int k = 0; k < 3; ++k) eu[k] = (double)__ldg(a.euler + b * 3 + k);
}

template <typename T>
__global__ void __launch_bounds__(32) k_report_thread(const __grid_constant__ ReportArgs<T> a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    T* sRows = reinterpret_cast<T*>(smem_raw);
    T* sP = sRows + (size_t)kTileProblems * a.row_pitch;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw + ((((size_t)((unsigned char*)(sP + (size_t)a.n * 3) - smem_raw)) + 7) & ~(size_t)7));
    const int lane = threadIdx.x;
    typedef typename Vec2<T>::type V2;
    RowTile<T> tile_buf;
    const double kdummy[6] = { 1, 0, 0, 0, 1, 0 };
    tile_buf.init(sRows, bar, a.uv, a.B, a.n, a.row_pitch, a.use_tma, kdummy, lane, /*normalise=*/false);
    const long long n_tiles = (a.B + kTileProblems - 1) / kTileProblems;
    long long tile = blockIdx.x;
    int valid = (tile < n_tiles) ? tile_buf.issue(tile, lane) : 0;
    for (int e = lane; e < a.n * 3; e += 32) sP[e] = a.pattern[e];
    __syncwarp();
    while (tile < n_tiles) {
        long long b = tile * kTileProblems + lane;
        const bool ok = b < a.B;
        if (!ok) b = a.B - 1;
        double Re[9], te[3], Rg[9], tg[3];
#pragma unroll
        for (int k = 0; k < 9; ++k) Re[k] = (double)a.R[b * 9 + k];
#pragma unroll
        for (int k = 0; k < 3; ++k) te[k] = (double)a.t[b * 3 + k];
        const double roll_e = (double)a.euler[b * 3], yaw_e = (double)a.euler[b * 3 + 1], pitch_e = (double)a.euler[b * 3 + 2];
        const double dist = a.gt[b * 4], roll_g = a.gt[b * 4 + 1], pitch_g = a.gt[b * 4 + 2], yaw_g = a.gt[b * 4 + 3];
        const double t3 = te[2];
        R_from_euler_deg_bounded(roll_g, yaw_g, pitch_g, Rg);   // random_stress_test.py:365
#pragma unroll
        for (int k = 0; k < 3; ++k) tg[k] = (te[k] / t3) * dist;   // :367-368
        double Me[9], me[3], Mg[9], mg[3];
        fold_camera(a.K, Re, te, Me, me);
        fold_camera(a.K, Rg, tg, Mg, mg);
        const V2* row = reinterpret_cast<const V2*>(tile_buf.acquire(lane, valid));
        double s0 = 0, s1 = 0, s2 = 0, m0 = 0, m1 = 0, m2 = 0;
        int i0 = -1, i1 = -1, i2 = -1;
        for (int i = 0; i < a.n; ++i) {
            const double x = (double)sP[3 * i], y = (double)sP[3 * i + 1], z = (double)sP[3 * i + 2];
            double pe[2], pg[2], ie, ig, e0, e1, e2;
            bool be, bg;
            project_folded(Me, me, x, y, z, pe, ie, be);  // TEST_TOOLBOX.py:312
            project_folded(Mg, mg, x, y, z, pg, ig, bg);  // :314
            const V2 px = row[i];
            landmark_errors(pe, ie, be, pg, ig, bg, (double)px.x, (double)px.y, e0, e1, e2);
            s0 += e0; if (e0 > m0) { m0 = e0; i0 = i; }
            s1 += e1; if (e1 > m1) { m1 = e1; i1 = i; }
            s2 += e2; if (e2 > m2) { m2 = e2; i2 = i; }
        }
        if (ok) {
            double* rp = a.report + b * a.rs_b;
            const long long sk = a.rs_k;
            rp[0] = t3 - dist; rp[sk] = roll_e - roll_g; rp[2 * sk] = pitch_e - pitch_g; rp[3 * sk] = yaw_e - yaw_g;
            rp[4 * sk] = (s0 / a.n) * dist; rp[5 * sk] = m0 * dist;
            rp[6 * sk] = (s1 / a.n) * dist; rp[7 * sk] = m1 * dist;
            rp[8 * sk] = (s2 / a.n) * dist; rp[9 * sk] = m2 * dist;
            rp[10 * sk] = t3; rp[11 * sk] = dist; rp[12 * sk] = roll_e; rp[13 * sk] = pitch_e; rp[14 * sk] = yaw_e; rp[15 * sk] = 0.0;
            if (a.flags) {
                a.flags[b * 4] = depth_passed(t3, dist, a.bounds[0]);
                a.flags[b * 4 + 1] = fabs(roll_e - roll_g) < a.bounds[1];
                a.flags[b * 4 + 2] = fabs(pitch_e - pitch_g) < a.bounds[2];
                a.flags[b * 4 + 3] = fabs(yaw_e - yaw_g) < a.bounds[3];
            }
            if (a.max_idx) { a.max_idx[b * 3] = i0; a.max_idx[b * 3 + 1] = i1; a.max_idx[b * 3 + 2] = i2; }
        }
        tile += gridDim.x;
        if (tile < n_tiles) {
            tile_buf.release();
            valid = tile_buf.issue(tile, lane);
        }
    }
}

// Streaming variant of k_report_thread: the rows go through two small chunk buffers (RowStream).
// RES != 0 fuses the last pass of the moment mapping into it (pnpb200_solve_report_batch): the rows are streamed ONCE
// for the error report and for res_norm = ||z - hx|| at the state k_iterate stored (RES = 1: LM, PNP_SOLVER_LIB.py:2679-2681;
// RES = 2: linear F2, :3368-3374) -- the same arithmetic, in the same order, as k_stream_chunk<T, METHOD, 1>.
// SKEW = false: K^-1 has k01 = k10 = 0, the pixels are normalised with one FMA per coordinate (normalise_px).
#ifndef PNP_REPORT_UNROLL
#define PNP_REPORT_UNROLL 4       // landmarks in flight per thread
#endif
#ifndef PNP_REPORT_MINBLOCKS
#define PNP_REPORT_MINBLOCKS 11   // one-warp CTAs per SM the register allocation must allow (11 -> <= 184 registers): the two
                                  // chunk buffers (~19 KB per CTA) admit 11 CTAs per SM, so a tighter cap buys no occupancy
#endif
constexpr int kReportUnroll = PNP_REPORT_UNROLL;
// MASKED (RES = 0 only): columns 4-9 run over the landmarks whose bit is set in a.vis
template <typename T, int RES, bool SKEW, bool MASKED = false>
__global__ void __launch_bounds__(32, PNP_REPORT_MINBLOCKS) k_report_chunk(const __grid_constant__ ReportArgs<T> a)
{
    static_assert(!(MASKED && RES), "the fused residual has no masked form");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    typedef typename Vec2<T>::type V2;
    T* sBuf = reinterpret_cast<T*>(smem_raw);
    T* sP = sBuf + (size_t)2 * kTileProblems * a.row_pitch;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + ((((size_t)((unsigned char*)(sP + (size_t)a.n * 3) - smem_raw)) + 7) & ~(size_t)7));
    const int lane = threadIdx.x;
    const long long n_tiles = (a.B + kTileProblems - 1) / kTileProblems;
    long long tile = blockIdx.x;
    // the per-problem pose loads go out FIRST: their latency then overlaps the barrier set-up, the first
    // bulk copies and the pattern staging instead of following them
    long long b = tile * kTileProblems + lane;
    bool ok = b < a.B;
    if (!ok) b = a.B - 1;
    double Re[9], te[3], eu[3], g4[4];
    T st[RES ? PNP_NTAIL : 1];
    LmResidualState<T> lr;          // RES = 1: the state with gamma folded in, as soon as it is loaded
    load_report_pose(a, b, Re, te, eu, g4);
    if (RES) {
#pragma unroll
        for (int k = 0; k < PNP_NTAIL; ++k) st[k] = __ldg(a.tail + (size_t)k * a.ld + b);
        if constexpr (RES == 1) lr.load(st);
    }
    RowStream<T> rs;
    rs.init(sBuf, bars, a.uv, a.B, a.n, a.use_tma /* chunk */, a.row_pitch, lane, a.use_tmap ? &a.tmap : nullptr);
    if (tile < n_tiles) rs.begin_tile(tile, lane);
    for (int e = lane; e < a.n * 3; e += 32) sP[e] = a.pattern[e];
    __syncwarp();
    const T k00 = (T)a.kinv[0], k01 = (T)a.kinv[1], k02 = (T)a.kinv[2];
    const T k10 = (T)a.kinv[3], k11 = (T)a.kinv[4], k12 = (T)a.kinv[5];
    while (tile < n_tiles) {
        double Rg[9], tg[3];
        const double roll_e = eu[0], yaw_e = eu[1], pitch_e = eu[2];
        const double dist = g4[0], roll_g = g4[1], pitch_g = g4[2], yaw_g = g4[3];
        const double t3 = te[2];
        R_from_euler_deg_bounded(roll_g, yaw_g, pitch_g, Rg);   // random_stress_test.py:365
        const double s3 = t_rcp<double>(t3) * dist;
#pragma unroll
        for (int k = 0; k < 3; ++k) tg[k] = te[k] * s3;   // (t / t3) * distance_GT, :367-368
        double Me[9], me[3], Mg[9], mg[3];
        fold_camera(a.K, Re, te, Me, me);
        fold_camera(a.K, Rg, tg, Mg, mg);
        double s0 = 0, s1 = 0, s2 = 0, m0 = 0, m1 = 0, m2 = 0;
        int i0 = -1, i1 = -1, i2 = -1;
        T acc0 = T(0), acc1 = T(0);
        const uint32_t* vw = MASKED ? a.vis + (size_t)b * a.vis_words : nullptr;
        const int nv = MASKED ? count_visible(vw, nullptr, a.n) : 0;
        for (int c = 0; c < rs.n_chunks; ++c) {
            const V2* row = rs.wait(c, lane);
            const int cnt = rs.count(c), base = c * rs.chunk;
#pragma unroll kReportUnroll
            for (int k = 0; k < cnt; ++k) {
                const int i = base + k;
                if constexpr (MASKED) { if (!mask_bit(vw, i)) continue; }
                const T th[3] = { sP[3 * i], sP[3 * i + 1], sP[3 * i + 2] };
                const double x = (double)th[0], y = (double)th[1], z = (double)th[2];
                double pe[2], pg[2], ie, ig, e0, e1, e2;
                bool be, bg;
                project_folded(Me, me, x, y, z, pe, ie, be);  // TEST_TOOLBOX.py:312
                project_folded(Mg, mg, x, y, z, pg, ig, bg);  // :314
                const V2 px = row[k];
                landmark_errors(pe, ie, be, pg, ig, bg, (double)px.x, (double)px.y, e0, e1, e2);
                s0 += e0; if (e0 > m0) { m0 = e0; i0 = i; }
                s1 += e1; if (e1 > m1) { m1 = e1; i1 = i; }
                s2 += e2; if (e2 > m2) { m2 = e2; i2 = i; }
                if (RES) {
                    T bx, by;                                     // nu = K^-1 [u, v, 1]^T (:3305)
                    normalise_px<T, SKEW>(px.x, px.y, k00, k01, k02, k10, k11, k12, bx, by);
                    if (RES == 1) {
                        lr.add(th, bx, by, acc0);                 // z - hx (:3750, :2679)
                    } else {
                        const T db = T(1) + (th[0] * st[0] + th[1] * st[1] + th[2] * st[2]);
                        const T dx = th[0] * st[3] + th[1] * st[4] + th[2] * st[5] + st[6];
                        const T dy = th[0] * st[7] + th[1] * st[8] + th[2] * st[9] + st[10];
                        const T ex = bx * db - dx, ey = by * db - dy;
                        acc0 = t_fma(ex, ex, acc0); acc1 = t_fma(ey, ey, acc1);
                    }
                }
            }
            rs.done(c, lane);
        }
        if constexpr (MASKED) { if (nv < kMinVisible) too_few_for_report(s0, s1, s2, m0, m1, m2, i0, i1, i2); }
        if (ok) {
            double* rp = a.report + b * a.rs_b;
            const long long sk = a.rs_k;
            rp[0] = t3 - dist; rp[sk] = roll_e - roll_g; rp[2 * sk] = pitch_e - pitch_g; rp[3 * sk] = yaw_e - yaw_g;
            rp[4 * sk] = (s0 / (MASKED ? nv : a.n)) * dist; rp[5 * sk] = m0 * dist;
            rp[6 * sk] = (s1 / (MASKED ? nv : a.n)) * dist; rp[7 * sk] = m1 * dist;
            rp[8 * sk] = (s2 / (MASKED ? nv : a.n)) * dist; rp[9 * sk] = m2 * dist;
            rp[10 * sk] = t3; rp[11 * sk] = dist; rp[12 * sk] = roll_e; rp[13 * sk] = pitch_e; rp[14 * sk] = yaw_e; rp[15 * sk] = 0.0;
            if (a.flags) {
                a.flags[b * 4] = depth_passed(t3, dist, a.bounds[0]);
                a.flags[b * 4 + 1] = fabs(roll_e - roll_g) < a.bounds[1];
                a.flags[b * 4 + 2] = fabs(pitch_e - pitch_g) < a.bounds[2];
                a.flags[b * 4 + 3] = fabs(yaw_e - yaw_g) < a.bounds[3];
            }
            if (a.max_idx) { a.max_idx[b * 3] = i0; a.max_idx[b * 3 + 1] = i1; a.max_idx[b * 3 + 2] = i2; }
            if (RES && a.res) {
                if (RES == 1) a.res[b] = t_sqrt(acc0);                                                       // :2681
                else { const T nx = t_sqrt(acc0), ny = t_sqrt(acc1); a.res[b] = t_sqrt(nx * nx + ny * ny); }   // :3374
            }
        }
        tile += gridDim.x;
        if (tile < n_tiles) {
            fence_proxy_async();
            rs.begin_tile(tile, lane);
            b = tile * kTileProblems + lane;
            ok = b < a.B;
            if (!ok) b = a.B - 1;
            load_report_pose(a, b, Re, te, eu, g4);
            if (RES) {
#pragma unroll
                for (int k = 0; k < PNP_NTAIL; ++k) st[k] = __ldg(a.tail + (size_t)k * a.ld + b);
                if constexpr (RES == 1) lr.load(st);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// solution check without ground truth (SURVEY.md 5, failure detection): per problem, over all n landmarks, the
// prediction-vs-landmark distance of cal_LM_error_distances (TEST_TOOLBOX.py:252-286) -- report columns 6, 7 with
// distance_GT = 1, computed as e1 of landmark_errors -- and a status word (PNPB200_CHECK_*).  Problem b is checked
// against pattern best[b] (pattern 0 without best).
// ------------------------------------------------------------------------------------------
template <typename T>
struct CheckArgs {
    const T* pattern; const T* uv; const T* R; const T* t; const T* res; const int32_t* best;
    long long B;
    int n, n_patterns, row_pitch, chunk;
    double K[9], limit;             // limit > 0: the REPROJ bit is on
    int32_t* status; T* reproj;
    int use_tmap;
    alignas(64) CUtensorMap tmap;   // uv as a 2-D tensor (RowStream), valid when use_tmap
    const uint32_t* vis; int vis_words;   // [B, vis_words] visibility bits (masked kernels only)
};

template <typename T>
PNP_DEV void load_check_pose(const CheckArgs<T>& a, long long b, double (&R)[9], double (&t)[3], double& res, int& pat)
{
#pragma unroll
    for (int k = 0; k < 3; ++k) t[k] = (double)__ldg(a.t + b * 3 + k);
#pragma unroll
    for (int k = 0; k < 9; ++k) R[k] = (double)__ldg(a.R + b * 9 + k);
    res = a.res ? (double)__ldg(a.res + b) : 0.0;
    pat = a.best ? __ldg(a.best + b) : 0;
}

// mean = NaN marks a best_pattern entry outside [0, n_patterns): the problem was checked against nothing
PNP_DEV int32_t check_status(const double (&R)[9], const double (&t)[3], double res, double mean, double mx, bool behind, double limit)
{
    double z = (res - res) + (mean - mean) + (mx - mx);   // x - x is 0 for finite x and NaN for NaN and +-Inf
#pragma unroll
    for (int k = 0; k < 9; ++k) z += R[k] - R[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) z += t[k] - t[k];
    int32_t s = 0;
    if (!(z == 0.0)) s |= PNPB200_CHECK_NONFINITE;
    if (t[2] <= 0.0) s |= PNPB200_CHECK_DEPTH;
    if (behind) s |= PNPB200_CHECK_BEHIND;
    if (limit > 0.0 && mean > limit) s |= PNPB200_CHECK_REPROJ;
    return s;
}

// n_visible: the landmarks the sum ran over (MASKED), else a.n
template <typename T, bool MASKED = false>
PNP_DEV void store_check(const CheckArgs<T>& a, long long b, const double (&R)[9], const double (&t)[3], double res, bool bad,
                         double sum, double mx, bool behind, int n_visible = 0)
{
    double mean = sum / (MASKED ? n_visible : a.n);       // (s1 / n) * distance_GT of the report, distance_GT = 1
    if (bad) mean = mx = __longlong_as_double(0x7ff8000000000000LL);
    if (a.reproj) { a.reproj[b * 2] = (T)mean; a.reproj[b * 2 + 1] = (T)mx; }
    a.status[b] = check_status(R, t, res, mean, mx, behind, a.limit);
}

// The streaming shape of k_report_chunk: one-warp CTAs, lane <-> problem, the rows through RowStream, every pattern in
// shared memory.  The landmark loop is the report's e1 in the same order, so mean and max are the report's bits.
#ifndef PNP_CHECK_MINBLOCKS
#define PNP_CHECK_MINBLOCKS 16
#endif
// MASKED: mean, max and BEHIND over the landmarks whose bit is set in a.vis; fewer than kMinVisible of them: NaN, NONFINITE
template <typename T, bool MASKED = false>
__global__ void __launch_bounds__(32, PNP_CHECK_MINBLOCKS) k_check_chunk(const __grid_constant__ CheckArgs<T> a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    typedef typename Vec2<T>::type V2;
    T* sBuf = reinterpret_cast<T*>(smem_raw);
    T* sP = sBuf + (size_t)2 * kTileProblems * a.row_pitch;
    uint64_t* bars = carve_bar<T>(smem_raw, sP + (size_t)a.n_patterns * a.n * 3);
    const int lane = threadIdx.x;
    const long long n_tiles = (a.B + kTileProblems - 1) / kTileProblems;
    long long tile = blockIdx.x;
    long long b = tile * kTileProblems + lane;
    bool ok = b < a.B;
    if (!ok) b = a.B - 1;
    double R[9], t[3], res;
    int pat;
    load_check_pose(a, b, R, t, res, pat);
    RowStream<T> rs;
    rs.init(sBuf, bars, a.uv, a.B, a.n, a.chunk, a.row_pitch, lane, a.use_tmap ? &a.tmap : nullptr);
    if (tile < n_tiles) rs.begin_tile(tile, lane);
    for (int e = lane; e < a.n_patterns * a.n * 3; e += 32) sP[e] = a.pattern[e];
    __syncwarp();
    while (tile < n_tiles) {
        const bool bad = (unsigned)pat >= (unsigned)a.n_patterns;
        const T* P = sP + (size_t)(bad ? 0 : pat) * a.n * 3;
        double M[9], m[3];
        fold_camera(a.K, R, t, M, m);
        double s = 0, mx = 0;
        bool behind = false;
        const uint32_t* vw = MASKED ? a.vis + (size_t)b * a.vis_words : nullptr;
        const int nv = MASKED ? count_visible(vw, nullptr, a.n) : 0;
        for (int c = 0; c < rs.n_chunks; ++c) {
            const V2* row = rs.wait(c, lane);
            const int cnt = rs.count(c), base = c * rs.chunk;
#pragma unroll kReportUnroll
            for (int k = 0; k < cnt; ++k) {
                const int i = base + k;
                if constexpr (MASKED) { if (!mask_bit(vw, i)) continue; }
                double pe[2], ie, ex, ey;
                bool be;
                project_folded(M, m, (double)P[3 * i], (double)P[3 * i + 1], (double)P[3 * i + 2], pe, ie, be);   // TEST_TOOLBOX.py:312
                const V2 px = row[k];
                px_difference(pe, ie, (double)px.x, (double)px.y, ex, ey);                                           // :326
                const double e = homogeneous_distance(ex, ey, be);
                s += e; if (e > mx) mx = e;
                behind |= be;
            }
            rs.done(c, lane);
        }
        if (ok) store_check<T, MASKED>(a, b, R, t, res, bad || (MASKED && nv < kMinVisible), s, mx, behind, nv);
        tile += gridDim.x;
        if (tile < n_tiles) {
            fence_proxy_async();
            rs.begin_tile(tile, lane);
            b = tile * kTileProblems + lane;
            ok = b < a.B;
            if (!ok) b = a.B - 1;
            load_check_pose(a, b, R, t, res, pat);
        }
    }
}

// Rows the streaming shape cannot take (large n, FP32 rows that are not 16-byte granular): one warp per problem, the
// lanes stride over the landmarks, the patterns are read from global memory.
template <typename T, bool MASKED = false>
__global__ void __launch_bounds__(256) k_check_warp(const __grid_constant__ CheckArgs<T> a)
{
    const long long b = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (b >= a.B) return;                                 // whole warps
    double R[9], t[3], res;
    int pat;
    load_check_pose(a, b, R, t, res, pat);
    const bool bad = (unsigned)pat >= (unsigned)a.n_patterns;
    const T* P = a.pattern + (size_t)(bad ? 0 : pat) * a.n * 3;
    double M[9], m[3];
    fold_camera(a.K, R, t, M, m);
    double s = 0, mx = 0;
    bool behind = false;
    const uint32_t* vw = MASKED ? a.vis + (size_t)b * a.vis_words : nullptr;
    const int nv = MASKED ? count_visible(vw, nullptr, a.n) : 0;
    for (int i = lane; i < a.n; i += 32) {
        if constexpr (MASKED) { if (!mask_bit(vw, i)) continue; }
        double pe[2], ie, ex, ey;
        bool be;
        project_folded(M, m, (double)__ldg(P + 3 * i), (double)__ldg(P + 3 * i + 1), (double)__ldg(P + 3 * i + 2), pe, ie, be);
        const T* px = a.uv + ((size_t)b * a.n + i) * 2;
        px_difference(pe, ie, (double)__ldg(px), (double)__ldg(px + 1), ex, ey);
        const double e = homogeneous_distance(ex, ey, be);
        s += e; if (e > mx) mx = e;
        behind |= be;
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, off);
        const double o = __shfl_xor_sync(0xffffffffu, mx, off);
        if (o > mx) mx = o;
    }
    behind = __any_sync(0xffffffffu, behind);
    if (lane == 0) store_check<T, MASKED>(a, b, R, t, res, bad || (MASKED && nv < kMinVisible), s, mx, behind, nv);
}

// ------------------------------------------------------------------------------------------
// statistics (get_statistic_of_result, TEST_TOOLBOX.py:892-937), two SUM/MAX-reducible passes,
// for up to 4 quantities at once, per class and (last row) over all problems.
//   pass 1 row = (n, sum est/gt, sum e, 0);  pass 2 row = (sum (e-m)^2, sum |e|, sum |e-m|, max |e-m|)
// No floating-point atomics on shared memory: lanes of a warp that share a class take turns
// (rank among equal-class lanes via __match_any_sync), each turn is conflict-free; the "all"
// row is accumulated in registers.  One RED per (block, row, column) to global memory at the end.
// ------------------------------------------------------------------------------------------
constexpr int kStatBlock = 256;
constexpr int kStatWarps = kStatBlock / 32;
constexpr int kStatMaxClass = 64;
constexpr int kStatMaxQ = 4;

struct StatIn {
    const double* est[kStatMaxQ];
    const double* gt[kStatMaxQ];
    long long es[kStatMaxQ], gs[kStatMaxQ];
    int nq;
};

PNP_DEV void atomic_max_double(double* addr, double v)   // v >= 0: the bit pattern is monotone
{
    atomicMax(reinterpret_cast<unsigned long long*>(addr), (unsigned long long)__double_as_longlong(v));
}

template <int PASS>
__global__ void __launch_bounds__(kStatBlock) k_stats(long long B, StatIn in, const int32_t* __restrict__ cls, int n_class,
                                                     const double* __restrict__ sums1, double* out, double* out_max)
{
    extern __shared__ double sh[];                        // [warp][n_class][nq][4]
    const int nq = in.nq, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int rows = n_class + 1;                         // + the "all" row
    const int per_warp = n_class * nq * 4;
    __shared__ double sMean[kStatMaxQ * (kStatMaxClass + 1)];
    for (int e = threadIdx.x; e < kStatWarps * per_warp; e += blockDim.x) sh[e] = 0.0;
    if (PASS == 2) {                                      // mean = sum e / n from the (all-reduced) pass-1 sums
        for (int e = threadIdx.x; e < nq * rows; e += blockDim.x) {
            const double cnt = sums1[e * 4];
            sMean[e] = cnt > 0.0 ? sums1[e * 4 + 2] / cnt : 0.0;
        }
    }
    __syncthreads();
    const double* mean = sMean;
    double* mine = sh + warp * per_warp;
    double all[kStatMaxQ][4];
#pragma unroll
    for (int q = 0; q < kStatMaxQ; ++q) all[q][0] = all[q][1] = all[q][2] = all[q][3] = 0.0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long b_start = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    // all lanes of a warp iterate together (the match below needs the full warp)
    for (long long base = b_start - lane; base < B; base += stride) {
        const long long b = base + lane;
        const bool ok = b < B;
        int c = -1;
        double v[kStatMaxQ][4];
#pragma unroll
        for (int q = 0; q < kStatMaxQ; ++q) v[q][0] = v[q][1] = v[q][2] = v[q][3] = 0.0;
        if (ok) {
            c = cls ? cls[b] : 0;
            if (c < 0 || c >= n_class) c = -1;
#pragma unroll
            for (int q = 0; q < kStatMaxQ; ++q) {
                if (q < nq) {
                    const double ev = in.est[q][b * in.es[q]];
                    double ratio, err;
                    if (in.gt[q]) { const double g = in.gt[q][b * in.gs[q]]; ratio = ev / g; err = ev - g; }
                    else          { ratio = ev; err = ev; }
                    if (PASS == 1) { v[q][0] = 1.0; v[q][1] = ratio; v[q][2] = err; }
                    else {
                        if (c >= 0) { const double d = err - mean[q * rows + c]; v[q][0] = d * d; v[q][1] = fabs(err); v[q][2] = fabs(d); v[q][3] = fabs(d); }
                    }
                    // the "all" row (its own mean in pass 2)
                    if (PASS == 1) { all[q][0] += 1.0; all[q][1] += ratio; all[q][2] += err; }
                    else {
                        const double d = err - mean[q * rows + n_class];
                        all[q][0] += d * d; all[q][1] += fabs(err); all[q][2] += fabs(d); all[q][3] = fmax(all[q][3], fabs(d));
                    }
                }
            }
        }
        const unsigned same = __match_any_sync(0xffffffffu, c);
        const int rank = __popc(same & ((1u << lane) - 1u));
        const unsigned any_valid = __ballot_sync(0xffffffffu, c >= 0);
        int max_rank = 0;
        {
            int r = (c >= 0) ? rank : 0;
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) r = max(r, __shfl_xor_sync(0xffffffffu, r, off));
            max_rank = r;
        }
        if (any_valid) {
            for (int turn = 0; turn <= max_rank; ++turn) {
                if (c >= 0 && rank == turn) {
                    double* row = mine + (size_t)c * nq * 4;
#pragma unroll
                    for (int q = 0; q < kStatMaxQ; ++q) {
                        if (q < nq) {
                            row[q * 4 + 0] += v[q][0]; row[q * 4 + 1] += v[q][1]; row[q * 4 + 2] += v[q][2];
                            if (PASS == 2) row[q * 4 + 3] = fmax(row[q * 4 + 3], v[q][3]);
                        }
                    }
                }
                __syncwarp();
            }
        }
    }
    __syncthreads();
    // classes: sum over the block's warps, one RED per value
    for (int e = threadIdx.x; e < per_warp; e += blockDim.x) {
        double acc = 0.0;
        const bool is_max = (PASS == 2) && ((e & 3) == 3);
        for (int w = 0; w < kStatWarps; ++w) acc = is_max ? fmax(acc, sh[w * per_warp + e]) : acc + sh[w * per_warp + e];
        const int c = e / (nq * 4), r = e - c * nq * 4, q = r >> 2, k = r & 3;
        if (is_max) atomic_max_double(out_max + (size_t)q * rows + c, acc);
        else if (acc != 0.0) atomicAdd(out + ((size_t)q * rows + c) * 4 + k, acc);
    }
    // "all" row: warp shuffle reduction, then one RED per warp
#pragma unroll
    for (int q = 0; q < kStatMaxQ; ++q) {
        if (q < nq) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                double a = all[q][k];
                const bool is_max = (PASS == 2) && (k == 3);
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) {
                    const double o = __shfl_xor_sync(0xffffffffu, a, off);
                    a = is_max ? fmax(a, o) : a + o;
                }
                if (lane == 0) {
                    if (is_max) atomic_max_double(out_max + (size_t)q * rows + n_class, a);
                    else if (a != 0.0) atomicAdd(out + ((size_t)q * rows + n_class) * 4 + k, a);
                }
            }
        }
    }
}

// Fast path of the same two passes when the per-class tables fit in shared memory with one private
// column per LANE ([warp][class][value][32 lanes]: every lane adds to its own 8-byte word, so there
// is no conflict, no matching and no turn-taking whatever the class pattern is).  Each WARP works on
// ONE quantity (warp % nq), so its table is a quarter of the all-quantities one and up to 16 warps
// fit per SM (one block per SM): the first version had 4 warps per SM doing all four quantities and
// sat on exposed load / shared-memory latency (issue slots 18 % busy, 82 us for 36 MB).
constexpr int kStatLaneMaxWarps = 16;
#ifndef PNP_STAT_UNROLL
#define PNP_STAT_UNROLL 8
#endif
constexpr int kStatUnroll = PNP_STAT_UNROLL;

template <int PASS>
__global__ void __launch_bounds__(kStatLaneMaxWarps * 32) k_stats_lane(long long B, StatIn in, const int32_t* __restrict__ cls, int n_class,
                                                                   const double* __restrict__ sums1, double* out, double* out_max)
{
    extern __shared__ double sh[];                        // [warp][n_class][NV][32]
    constexpr int NV = (PASS == 1) ? 3 : 4;
    const int nq = in.nq, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    const int q = warp % nq, group = warp / nq, n_groups = n_warps / nq;     // blockDim.x is a multiple of 32 nq
    const int rows = n_class + 1;
    const int entries = n_class * NV;                     // per warp, times 32 lanes
    __shared__ double sMean[kStatMaxQ * (kStatMaxClass + 1)];
    for (int e = threadIdx.x; e < n_warps * entries * 32; e += blockDim.x) sh[e] = 0.0;
    if (PASS == 2) {
        for (int e = threadIdx.x; e < nq * rows; e += blockDim.x) {
            const double cnt = sums1[e * 4];
            sMean[e] = cnt > 0.0 ? sums1[e * 4 + 2] / cnt : 0.0;
        }
    }
    __syncthreads();
    double* mine = sh + (size_t)warp * entries * 32 + lane;
    const double* __restrict__ est = in.est[0];
    const double* __restrict__ gtp = in.gt[0];
    long long es = in.es[0], gs = in.gs[0];
#pragma unroll
    for (int k = 1; k < kStatMaxQ; ++k)
        if (k == q) { est = in.est[k]; gtp = in.gt[k]; es = in.es[k]; gs = in.gs[k]; }
    const double mean_all = (PASS == 2) ? sMean[q * rows + n_class] : 0.0;
    double all0 = 0.0, all1 = 0.0, all2 = 0.0, all3 = 0.0;
    const long long stride = (long long)gridDim.x * n_groups * 32;
    // one element's contribution (c = -2: no problem there; outside [0, n_class): counted in the "all" row only)
    auto account = [&](int c, double e, double g) {
        if (c == -2) return;
        const bool in_class = (unsigned)c < (unsigned)n_class;
        const double err = gtp ? e - g : e;
        if (PASS == 1) {
            const double ratio = gtp ? e / g : e;
            all0 += 1.0; all1 += ratio; all2 += err;
            if (in_class) {
                double* p = mine + (size_t)(c * NV) * 32;
                p[0] += 1.0; p[32] += ratio; p[64] += err;
            }
        } else {
            const double da = err - mean_all;
            all0 += da * da; all1 += fabs(err); all2 += fabs(da); all3 = fmax(all3, fabs(da));
            if (in_class) {
                const double d = err - sMean[q * rows + c];
                double* p = mine + (size_t)(c * NV) * 32;
                p[0] += d * d; p[32] += fabs(err); p[64] += fabs(d); p[96] = fmax(p[96], fabs(d));
            }
        }
    };
    // Running pointers instead of 64-bit index products per load (the first version spent 42 of its 153 instructions per
    // element on them, ncu r02x), and full batches of kStatUnroll elements without a bounds test per element.
    // (A missing class / ground-truth array reads `est` at stride 0 instead -- a valid address whose value is not used -- so
    // that the loads and the pointer steps carry no null tests.)
    long long b0 = ((long long)blockIdx.x * n_groups + group) * 32 + lane;
    const bool has_gt = gtp != nullptr, has_cls = cls != nullptr;
    const double* pe = est + b0 * es;
    const double* pg = has_gt ? gtp + b0 * gs : est;
    const int32_t* pc = has_cls ? cls + b0 : reinterpret_cast<const int32_t*>(est);
    const long long se = stride * es, sg = has_gt ? stride * gs : 0, sc = has_cls ? stride : 0;
    for (; b0 + (kStatUnroll - 1) * stride < B; b0 += stride * kStatUnroll) {
        int c[kStatUnroll];
        double ev[kStatUnroll], gv[kStatUnroll];
#pragma unroll
        for (int u = 0; u < kStatUnroll; ++u) {           // all loads first
            c[u] = *pc; ev[u] = *pe; gv[u] = *pg;
            pc += sc; pe += se; pg += sg;
        }
#pragma unroll
        for (int u = 0; u < kStatUnroll; ++u) account(has_cls ? c[u] : 0, ev[u], gv[u]);
    }
    if (b0 < B) {                                         // the ragged end as ONE more batch: its loads are in flight together too
        int c[kStatUnroll];
        double ev[kStatUnroll], gv[kStatUnroll];
#pragma unroll
        for (int u = 0; u < kStatUnroll; ++u) {
            c[u] = -2; ev[u] = 0.0; gv[u] = 1.0;          // -2: no problem there
            if (b0 + u * stride < B) { c[u] = has_cls ? *pc : 0; ev[u] = *pe; gv[u] = *pg; }
            pc += sc; pe += se; pg += sg;
        }
#pragma unroll
        for (int u = 0; u < kStatUnroll; ++u) account(c[u], ev[u], gv[u]);
    }
    __syncthreads();
    // classes: entry e = (quantity, class, value): add the warps that worked on that quantity per lane, then across lanes
    for (int e = warp; e < nq * entries; e += n_warps) {
        const int qq = e / entries, r = e - qq * entries, cidx = r / NV, k = r - cidx * NV;
        const bool is_max = (PASS == 2) && (k == 3);
        double a = 0.0;
        for (int g = 0; g < n_groups; ++g) {
            const double v = sh[((size_t)(g * nq + qq) * entries + r) * 32 + lane];
            a = is_max ? fmax(a, v) : a + v;
        }
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) {
            const double o = __shfl_xor_sync(0xffffffffu, a, off);
            a = is_max ? fmax(a, o) : a + o;
        }
        if (lane == 0) {
            if (is_max) atomic_max_double(out_max + (size_t)qq * rows + cidx, a);
            else if (a != 0.0) atomicAdd(out + ((size_t)qq * rows + cidx) * 4 + k, a);
        }
    }
    {                                                     // the "all" row of this warp's quantity
        double av[4] = { all0, all1, all2, all3 };
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            double a = av[k];
            const bool is_max = (PASS == 2) && (k == 3);
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) {
                const double o = __shfl_xor_sync(0xffffffffu, a, off);
                a = is_max ? fmax(a, o) : a + o;
            }
            if (lane == 0) {
                if (is_max) atomic_max_double(out_max + (size_t)q * rows + n_class, a);
                else if (a != 0.0) atomicAdd(out + ((size_t)q * rows + n_class) * 4 + k, a);
            }
        }
    }
}

// The same two passes for MANY classes (the 12 x 5 x 5 x 5 distance / roll / pitch / yaw grid of
// TEST_TOOLBOX.get_all_class_seperated_result, :975-1030): the tables do not fit shared memory, and with
// ~1500 classes two problems rarely meet in one, so every problem adds straight into the global table
// with FP64 reductions (RED.ADD.F64); the means of pass 2 are read from the pass-1 table.
template <int PASS>
__global__ void __launch_bounds__(256) k_stats_global(long long B, StatIn in, const int32_t* __restrict__ cls, int n_class,
                                                      const double* __restrict__ sums1, double* out, double* out_max)
{
    const int nq = in.nq, rows = n_class + 1;
    double all[kStatMaxQ][4];
#pragma unroll
    for (int q = 0; q < kStatMaxQ; ++q) all[q][0] = all[q][1] = all[q][2] = all[q][3] = 0.0;
    for (long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
        int c = cls ? cls[b] : 0;
        if (c < 0 || c >= n_class) c = -1;
#pragma unroll
        for (int q = 0; q < kStatMaxQ; ++q) {
            if (q < nq) {
                const double ev = in.est[q][b * in.es[q]];
                double ratio, err;
                if (in.gt[q]) { const double g = in.gt[q][b * in.gs[q]]; ratio = ev / g; err = ev - g; }
                else          { ratio = ev; err = ev; }
                if (PASS == 1) {
                    all[q][0] += 1.0; all[q][1] += ratio; all[q][2] += err;
                    if (c >= 0) {
                        double* o = out + ((size_t)q * rows + c) * 4;
                        atomicAdd(o, 1.0); atomicAdd(o + 1, ratio); atomicAdd(o + 2, err);
                    }
                } else {
                    const double na = sums1[((size_t)q * rows + n_class) * 4];
                    const double da = err - (na > 0.0 ? sums1[((size_t)q * rows + n_class) * 4 + 2] / na : 0.0);
                    all[q][0] += da * da; all[q][1] += fabs(err); all[q][2] += fabs(da); all[q][3] = fmax(all[q][3], fabs(da));
                    if (c >= 0) {
                        const double* s1 = sums1 + ((size_t)q * rows + c) * 4;
                        const double d = err - (s1[0] > 0.0 ? s1[2] / s1[0] : 0.0);
                        double* o = out + ((size_t)q * rows + c) * 4;
                        atomicAdd(o, d * d); atomicAdd(o + 1, fabs(err)); atomicAdd(o + 2, fabs(d));
                        atomic_max_double(out_max + (size_t)q * rows + c, fabs(d));
                    }
                }
            }
        }
    }
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int q = 0; q < kStatMaxQ; ++q) {                 // the "all" row
        if (q < nq) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                double a = all[q][k];
                const bool is_max = (PASS == 2) && (k == 3);
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) {
                    const double o = __shfl_xor_sync(0xffffffffu, a, off);
                    a = is_max ? fmax(a, o) : a + o;
                }
                if (lane == 0) {
                    if (is_max) atomic_max_double(out_max + (size_t)q * rows + n_class, a);
                    else if (a != 0.0) atomicAdd(out + ((size_t)q * rows + n_class) * 4 + k, a);
                }
            }
        }
    }
}

// Combined class of the four ground-truth quantities, mixed radix in the order (distance, roll, pitch, yaw):
// ((cd * nr + cr) * np + cp) * ny + cy with c = np.digitize(value * scale, bins) (classify_drpy :239-247)
struct Bins4 { double b[4][32]; int n[4]; double scale[4]; };
__global__ void k_classify_drpy(long long B, const double* __restrict__ gt, Bins4 bins, int32_t* cls)
{
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    int id = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const double x = gt[b * 4 + q] * bins.scale[q];
        int c = 0;
        for (int i = 0; i < bins.n[q]; ++i) c += (bins.b[q][i] <= x) ? 1 : 0;
        id = id * (bins.n[q] + 1) + c;
    }
    cls[b] = id;
}

struct Bins { double b[32]; int n; };
__global__ void k_classify(long long B, const double* __restrict__ v, long long stride, double scale, Bins bins, int32_t* cls)
{
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const double x = v[b * stride] * scale;
    int c = 0;
    for (int i = 0; i < bins.n; ++i) c += (bins.b[i] <= x) ? 1 : 0;   // np.digitize, right=False
    cls[b] = c;
}

// ------------------------------------------------------------------------------------------
// FMA pipe microbenchmark: 8 independent accumulators per thread, `iters` rounds of 8 FMAs
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void k_fma_peak(int iters, T seed, T* out)
{
    T a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const T m = T(0.999999), c = T(1e-6);
#pragma unroll 16
    for (int i = 0; i < iters; ++i) {
        a0 = t_fma(a0, m, c); a1 = t_fma(a1, m, c); a2 = t_fma(a2, m, c); a3 = t_fma(a3, m, c);
        a4 = t_fma(a4, m, c); a5 = t_fma(a5, m, c); a6 = t_fma(a6, m, c); a7 = t_fma(a7, m, c);
    }
    const T s = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
    if (s == T(-12345)) out[0] = s;   // never true; keeps the chain alive
}

// the branch-free reciprocal / reciprocal square root of pnpb200_math.cuh, exposed for the tests
__global__ void k_selftest_math(long long n_signed, const double* __restrict__ in, double* rcp, double* rsq, double* sq)
{
    const long long n = n_signed;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double a = in[i];
    const double y = t_rsqrt<double>(a);
    rcp[i] = t_rcp<double>(a); rsq[i] = y;
    sq[i] = (i & 1) ? sqrt_nonneg(a) : t_sqrt_fast<double>(a, y);   // both square roots in use (report / LM constraint rows)
}

// Narrow pixels -> T (int16 of the packed transfer, pnpb200_pack.cpp; int16 / uint16 / float32 detections handed to
// pnpb200_solve_batch_host_px): every thread widens the 16 bytes of one vector load, 8 or 4 values.
template <typename Tin> PNP_DEV void unpack16(const int4& v, double (&o)[8]);
template <> PNP_DEV void unpack16<int16_t>(const int4& v, double (&o)[8])
{
    const int w[4] = { v.x, v.y, v.z, v.w };
#pragma unroll
    for (int k = 0; k < 4; ++k) { o[2 * k] = (double)(int16_t)(w[k] & 0xffff); o[2 * k + 1] = (double)(int16_t)(w[k] >> 16); }
}
template <> PNP_DEV void unpack16<uint16_t>(const int4& v, double (&o)[8])
{
    const unsigned w[4] = { (unsigned)v.x, (unsigned)v.y, (unsigned)v.z, (unsigned)v.w };
#pragma unroll
    for (int k = 0; k < 4; ++k) { o[2 * k] = (double)(w[k] & 0xffffu); o[2 * k + 1] = (double)(w[k] >> 16); }
}
template <> PNP_DEV void unpack16<float>(const int4& v, double (&o)[8])
{
    o[0] = (double)__int_as_float(v.x); o[1] = (double)__int_as_float(v.y);
    o[2] = (double)__int_as_float(v.z); o[3] = (double)__int_as_float(v.w);
    o[4] = o[5] = o[6] = o[7] = 0.0;
}

template <typename Tin, typename T>
__global__ void __launch_bounds__(256) k_widen(long long n, const Tin* __restrict__ in, T* __restrict__ out)
{
    constexpr int kPer = 16 / (int)sizeof(Tin);                // values per 16-byte load
    const long long g = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * kPer;
    if (g >= n) return;
    if (g + kPer <= n) {
        const int4 v = __ldg(reinterpret_cast<const int4*>(in + g));
        double o[8];
        unpack16<Tin>(v, o);                                   // exact: every int16 / uint16 / float32 is a double (and the
        if (sizeof(T) == 8) {                                  // 16-bit integers are floats)
            double2* d = reinterpret_cast<double2*>(out + g);
#pragma unroll
            for (int k = 0; k < kPer / 2; ++k) d[k] = make_double2(o[2 * k], o[2 * k + 1]);
        } else {
            float4* d = reinterpret_cast<float4*>(out + g);
#pragma unroll
            for (int k = 0; k < kPer / 4; ++k) d[k] = make_float4((float)o[4 * k], (float)o[4 * k + 1], (float)o[4 * k + 2], (float)o[4 * k + 3]);
        }
    } else {
        for (long long i = g; i < n; ++i) out[i] = (T)in[i];
    }
}

// f2_get_B_xy (PNP_SOLVER_LIB.py:3291-3312) for image points whose homogeneous coordinate is not 1: nu = K^-1 [u, v, w]^T,
// (B_x, B_y) = (nu_0, nu_1) -- the reference multiplies whatever it is given (:3307), and perspective_projection emits
// w = -1 for points behind the camera (:4548).  The solve kernels then run with K = I on these normalised coordinates.
template <typename T>
__global__ void __launch_bounds__(256) k_normalise_uvw(long long n, const T* __restrict__ uvw, KMat kinv, T* __restrict__ out)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double u = (double)uvw[3 * i], v = (double)uvw[3 * i + 1], w = (double)uvw[3 * i + 2];
    out[2 * i] = (T)(kinv.k[0] * u + kinv.k[1] * v + kinv.k[2] * w);
    out[2 * i + 1] = (T)(kinv.k[3] * u + kinv.k[4] * v + kinv.k[5] * w);
}

__global__ void k_selftest_sincos(long long n, const double* __restrict__ in, double* s, double* c)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    sincos_bounded(in[i], s[i], c[i]);
}

template <typename T>
__global__ void k_selftest_project(long long n, const T* __restrict__ G, T* __restrict__ R, T* __restrict__ smax)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    T g[9], r[9];
#pragma unroll
    for (int e = 0; e < 9; ++e) g[e] = G[9 * i + e];
    so3_project<T>(g, r, smax[i]);
#pragma unroll
    for (int e = 0; e < 9; ++e) R[9 * i + e] = r[e];
}

}  // namespace pnpb200

namespace pnpb200 {
template <typename Tin>
static int widen_typed(int dtype, long long n_values, const void* in, void* out, cudaStream_t stream)
{
    constexpr int kPer = 16 / (int)sizeof(Tin);
    const unsigned grid = grid_for((n_values + kPer - 1) / kPer, 256);
    if (dtype == PNPB200_DTYPE_F64) k_widen<Tin, double><<<grid, 256, 0, stream>>>(n_values, (const Tin*)in, (double*)out);
    else                            k_widen<Tin, float><<<grid, 256, 0, stream>>>(n_values, (const Tin*)in, (float*)out);
    count_kernel_launches(1);
    PNP_CUDA_OK(cudaGetLastError());
    return PNPB200_OK;
}

int widen_launch(int pixel_type, int dtype, long long n_values, const void* in, void* out, cudaStream_t stream)
{
    if (n_values <= 0) return PNPB200_OK;
    switch (pixel_type) {
    case PNPB200_PIXEL_I16: return widen_typed<int16_t>(dtype, n_values, in, out, stream);
    case PNPB200_PIXEL_U16: return widen_typed<uint16_t>(dtype, n_values, in, out, stream);
    case PNPB200_PIXEL_F32: return widen_typed<float>(dtype, n_values, in, out, stream);
    default: return PNPB200_EINVAL;
    }
}
}  // namespace pnpb200

using namespace pnpb200;

#define DISPATCH_DTYPE(dtype, CALL_F64, CALL_F32)            \
    if ((dtype) == PNPB200_DTYPE_F64) { CALL_F64; }          \
    else if ((dtype) == PNPB200_DTYPE_F32) { CALL_F32; }     \
    else return PNPB200_EINVAL;

namespace pnpb200 {

template <typename T, int RES, bool SKEW, bool MASKED = false>
int launch_report_chunk(const ReportArgs<T>& a, unsigned grid, size_t smem, cudaStream_t st)
{
    PNP_CUDA_OK(set_dynamic_smem((const void*)k_report_chunk<T, RES, SKEW, MASKED>, smem));
    k_report_chunk<T, RES, SKEW, MASKED><<<grid, 32, smem, st>>>(a);
    return PNPB200_OK;
}

bool report_can_fuse(int dtype, int n)
{
    const RowGeom g = (dtype == PNPB200_DTYPE_F64) ? row_geometry<double>(n) : row_geometry<float>(n);
    const StreamGeom sg = (dtype == PNPB200_DTYPE_F64) ? stream_geometry<double>(n) : stream_geometry<float>(n);
    return g.tile_bytes <= 48 * 1024 && sg.use_stream;
}

// fuse != nullptr (only where report_can_fuse): the streaming report kernel also evaluates res_norm from the state in the workspace
int report_launch(int dtype, int64_t B, int n, const void* pattern, const void* uv, const double* K,
                  const void* R, const void* t, const void* euler_deg, const double* gt, const double* bounds,
                  double* report, int64_t report_stride_problem, int64_t report_stride_column,
                  int32_t* flags, int32_t* max_idx, const ReportFuse* fuse, cudaStream_t st, const uint32_t* vis)
{
    if (B < 0 || n < 1 || !pattern || !uv || !K || !R || !t || !euler_deg || !gt || !report) return PNPB200_EINVAL;
    if (vis && (fuse || !vis_aligned(vis))) return PNPB200_EINVAL;         // the fused residual has no masked form
    if (report_stride_problem < 1 || report_stride_column < 1) return PNPB200_EINVAL;
    const long long rs_b = report_stride_problem, rs_k = report_stride_column;
    if (((uintptr_t)uv & 15u) != 0) return PNPB200_EINVAL;   // rows are staged with 16-byte bulk copies
    if (fuse && !report_can_fuse(dtype, n)) return PNPB200_EINVAL;
    if (B == 0) return PNPB200_OK;
    KMat km;
    for (int e = 0; e < 9; ++e) km.k[e] = K[e];
    Bounds bd;
    for (int e = 0; e < 4; ++e) bd.b[e] = bounds ? bounds[e] : 10.0;
    const size_t esz = (dtype == PNPB200_DTYPE_F64) ? 8 : 4;
    const RowGeom g = (dtype == PNPB200_DTYPE_F64) ? row_geometry<double>(n) : row_geometry<float>(n);
    const size_t smem = g.tile_bytes + (size_t)n * 3 * esz + 16;
    const StreamGeom sg = (dtype == PNPB200_DTYPE_F64) ? stream_geometry<double>(n) : stream_geometry<float>(n);
    if (g.tile_bytes <= 48 * 1024 && sg.use_stream) {
        const long long n_tiles = (B + kTileProblems - 1) / kTileProblems;
        const unsigned grid = (unsigned)(n_tiles < 0x7fffffffLL ? n_tiles : 0x7fffffffLL);
        const size_t csmem = 2 * sg.buf_bytes + (size_t)n * 3 * esz + 32;
        const int res_mode = fuse ? fuse->res_mode : 0;
        const bool skew = fuse && (fuse->kinv[1] != 0.0 || fuse->kinv[3] != 0.0);
#define LAUNCH_REPORT_CHUNK(TT)                                                                                         \
        {                                                                                                               \
            ReportArgs<TT> a;                                                                                           \
            a.pattern = (const TT*)pattern; a.uv = (const TT*)uv; a.R = (const TT*)R; a.t = (const TT*)t;              \
            a.euler = (const TT*)euler_deg; a.gt = gt; a.B = B; a.n = n; a.row_pitch = sg.pitch; a.use_tma = sg.chunk;  \
            for (int e = 0; e < 9; ++e) a.K[e] = K[e];                                                                  \
            for (int e = 0; e < 4; ++e) a.bounds[e] = bd.b[e];                                                          \
            a.report = report; a.flags = flags; a.max_idx = max_idx; a.rs_b = rs_b; a.rs_k = rs_k;                      \
            a.tail = fuse ? (const TT*)fuse->tail : nullptr; a.ld = fuse ? fuse->ld : 0; a.res = fuse ? (TT*)fuse->res : nullptr; \
            for (int e = 0; e < 6; ++e) a.kinv[e] = fuse ? fuse->kinv[e] : 0.0;                                         \
            a.use_tmap = (sg.pitch == sg.chunk * 2) ? make_row_tensor_map(&a.tmap, uv, (int)sizeof(TT), B, n, sg.chunk) : 0; \
            a.vis = vis; a.vis_words = (n + 31) / 32;                                                                   \
            const int rc = vis ? launch_report_chunk<TT, 0, true, true>(a, grid, csmem, st) : (res_mode == 1) ? (skew ? launch_report_chunk<TT, 1, true>(a, grid, csmem, st)               \
                                                   : launch_report_chunk<TT, 1, false>(a, grid, csmem, st))             \
                         : (res_mode == 2) ? (skew ? launch_report_chunk<TT, 2, true>(a, grid, csmem, st)               \
                                                   : launch_report_chunk<TT, 2, false>(a, grid, csmem, st))             \
                                           : launch_report_chunk<TT, 0, true>(a, grid, csmem, st);                      \
            if (rc != PNPB200_OK) return rc;                                                                            \
            count_kernel_launches(1);                                                                                   \
        }
        DISPATCH_DTYPE(dtype, LAUNCH_REPORT_CHUNK(double), LAUNCH_REPORT_CHUNK(float));
#undef LAUNCH_REPORT_CHUNK
    } else if (g.tile_bytes <= 48 * 1024 && !vis) {
        const long long n_tiles = (B + kTileProblems - 1) / kTileProblems;
        const unsigned grid = (unsigned)(n_tiles < 0x7fffffffLL ? n_tiles : 0x7fffffffLL);
#define LAUNCH_REPORT_THREAD(TT)                                                                                        \
        {                                                                                                               \
            ReportArgs<TT> a;                                                                                           \
            a.pattern = (const TT*)pattern; a.uv = (const TT*)uv; a.R = (const TT*)R; a.t = (const TT*)t;              \
            a.euler = (const TT*)euler_deg; a.gt = gt; a.B = B; a.n = n; a.row_pitch = g.row_pitch; a.use_tma = g.use_tma; \
            for (int e = 0; e < 9; ++e) a.K[e] = K[e];                                                                  \
            for (int e = 0; e < 4; ++e) a.bounds[e] = bd.b[e];                                                          \
            a.report = report; a.flags = flags; a.max_idx = max_idx; a.use_tmap = 0; a.rs_b = rs_b; a.rs_k = rs_k;      \
            a.tail = nullptr; a.ld = 0; a.res = nullptr;                                                                \
            PNP_CUDA_OK(set_dynamic_smem((const void*)k_report_thread<TT>, smem));                                      \
            k_report_thread<TT><<<grid, 32, smem, st>>>(a); count_kernel_launches(1);                                   \
        }
        DISPATCH_DTYPE(dtype, LAUNCH_REPORT_THREAD(double), LAUNCH_REPORT_THREAD(float));
#undef LAUNCH_REPORT_THREAD
    } else if (vis) {                                         // masked rows the streaming kernel cannot take: one warp per problem
        const unsigned grid = grid_for(B * 32, 256);
        const int W = (n + 31) / 32;
        DISPATCH_DTYPE(dtype,
                       (k_report<double, true><<<grid, 256, 0, st>>>(B, n, pattern, uv, km, R, t, euler_deg, gt, bd, report, rs_b, rs_k, flags, max_idx, vis, W)),
                       (k_report<float, true><<<grid, 256, 0, st>>>(B, n, pattern, uv, km, R, t, euler_deg, gt, bd, report, rs_b, rs_k, flags, max_idx, vis, W))); count_kernel_launches(1);
    } else {
        const unsigned grid = grid_for(B * 32, 256);
        DISPATCH_DTYPE(dtype,
                       (k_report<double><<<grid, 256, 0, st>>>(B, n, pattern, uv, km, R, t, euler_deg, gt, bd, report, rs_b, rs_k, flags, max_idx)),
                       (k_report<float><<<grid, 256, 0, st>>>(B, n, pattern, uv, km, R, t, euler_deg, gt, bd, report, rs_b, rs_k, flags, max_idx))); count_kernel_launches(1);
    }
    PNP_CUDA_OK(cudaGetLastError());
    return PNPB200_OK;
}

// the execution shape of report_launch: the streaming kernel where report_can_fuse, one warp per problem otherwise
int check_launch(int dtype, int64_t B, int n, const void* pattern, int n_patterns, const void* uv, const double* K,
                 const void* R, const void* t, const void* res_norm, const int32_t* best_pattern, double limit,
                 int32_t* status, void* reproj, cudaStream_t st, const uint32_t* vis)
{
    if (B < 0 || n < 1 || !pattern || !uv || !K || !R || !t || !status) return PNPB200_EINVAL;
    if (vis && !vis_aligned(vis)) return PNPB200_EINVAL;
    if (n_patterns < 1 || n_patterns > PNPB200_MAX_PATTERNS) return PNPB200_EINVAL;
    if (dtype != PNPB200_DTYPE_F64 && dtype != PNPB200_DTYPE_F32) return PNPB200_EINVAL;
    if (((uintptr_t)uv & 15u) != 0) return PNPB200_EINVAL;   // rows are staged with 16-byte bulk copies
    if (B == 0) return PNPB200_OK;
#define LAUNCH_CHECK(TT)                                                                                                \
    {                                                                                                                   \
        CheckArgs<TT> a;                                                                                                \
        a.pattern = (const TT*)pattern; a.uv = (const TT*)uv; a.R = (const TT*)R; a.t = (const TT*)t;                  \
        a.res = (const TT*)res_norm; a.best = best_pattern; a.B = B; a.n = n; a.n_patterns = n_patterns;              \
        for (int e = 0; e < 9; ++e) a.K[e] = K[e];                                                                      \
        a.limit = (limit > 0.0) ? limit : 0.0;                                                                          \
        a.status = status; a.reproj = (TT*)reproj; a.use_tmap = 0;                                                      \
        a.vis = vis; a.vis_words = (n + 31) / 32;                                                                       \
        const StreamGeom sg = stream_geometry<TT>(n);                                                                   \
        if (report_can_fuse(dtype, n)) {                                                                                \
            DeviceProps dp;                                                                                             \
            const int rc = get_device_props(&dp);                                                                       \
            if (rc != PNPB200_OK) return rc;                                                                            \
            const size_t smem = 2 * sg.buf_bytes + sizeof(TT) * (size_t)n_patterns * n * 3 + 32;                        \
            if (smem > (size_t)dp.max_smem_optin) return PNPB200_ETOOLARGE;   /* every pattern stays in shared memory */ \
            a.row_pitch = sg.pitch; a.chunk = sg.chunk;                                                                 \
            a.use_tmap = (sg.pitch == sg.chunk * 2) ? make_row_tensor_map(&a.tmap, uv, (int)sizeof(TT), B, n, sg.chunk) : 0; \
            const long long n_tiles = (B + kTileProblems - 1) / kTileProblems;                                          \
            const unsigned grid = (unsigned)(n_tiles < 0x7fffffffLL ? n_tiles : 0x7fffffffLL);                          \
            if (vis) {                                                                                                  \
                PNP_CUDA_OK(set_dynamic_smem((const void*)k_check_chunk<TT, true>, smem));                              \
                k_check_chunk<TT, true><<<grid, 32, smem, st>>>(a);                                                     \
            } else {                                                                                                    \
                PNP_CUDA_OK(set_dynamic_smem((const void*)k_check_chunk<TT>, smem));                                    \
                k_check_chunk<TT><<<grid, 32, smem, st>>>(a);                                                           \
            }                                                                                                           \
        } else {                                                                                                        \
            a.row_pitch = 0; a.chunk = 0;                                                                               \
            if (vis) k_check_warp<TT, true><<<grid_for(B * 32, 256), 256, 0, st>>>(a);                                  \
            else     k_check_warp<TT><<<grid_for(B * 32, 256), 256, 0, st>>>(a);                                        \
        }                                                                                                               \
        count_kernel_launches(1);                                                                                       \
    }
    DISPATCH_DTYPE(dtype, LAUNCH_CHECK(double), LAUNCH_CHECK(float));
#undef LAUNCH_CHECK
    PNP_CUDA_OK(cudaGetLastError());
    return PNPB200_OK;
}

}  // namespace pnpb200

extern "C" {

int pnpb200_check_batch(int dtype, int64_t B, int n_total, const void* pattern, int n_patterns, const void* uv, const double* K,
                        const void* R, const void* t, const void* res_norm, const int32_t* best_pattern, double reproj_limit_px,
                        int32_t* status, void* reproj, void* stream)
{
    return check_launch(dtype, B, n_total, pattern, n_patterns, uv, K, R, t, res_norm, best_pattern, reproj_limit_px, status,
                        reproj, (cudaStream_t)stream);
}

int pnpb200_check_batch_masked(int dtype, int64_t B, int n_total, const void* pattern, int n_patterns, const void* uv,
                               const double* K, const void* R, const void* t, const void* res_norm, const int32_t* best_pattern,
                               double reproj_limit_px, int32_t* status, void* reproj, const uint32_t* visible, void* stream)
{
    if (!visible) return PNPB200_EINVAL;
    return check_launch(dtype, B, n_total, pattern, n_patterns, uv, K, R, t, res_norm, best_pattern, reproj_limit_px, status,
                        reproj, (cudaStream_t)stream, visible);
}

int pnpb200_default_synth(pnpb200_synth* s)
{
    if (!s) return PNPB200_EINVAL;
    s->seed = 42; s->angle_range_deg = 45.0; s->depth_min_m = 0.20; s->depth_max_m = 2.25; s->fov_max_deg = 45.0;
    s->is_quantized = 1; s->reserved = 0; s->quantize_q = 1.0; s->noise_sigma_px = 0.0;
    s->roll_center_deg = 0.0; s->pitch_center_deg = 0.0; s->yaw_center_deg = 0.0;
    return PNPB200_OK;
}

int pnpb200_R_from_euler(int dtype, int64_t B, const void* euler, int is_degree, void* R, void* stream)
{
    if (B < 0 || !euler || !R) return PNPB200_EINVAL;
    if (B == 0) return PNPB200_OK;
    cudaStream_t st = (cudaStream_t)stream;
    DISPATCH_DTYPE(dtype, (k_R_from_euler<double><<<grid_for(B, 128), 128, 0, st>>>(B, euler, is_degree, R)),
                   (k_R_from_euler<float><<<grid_for(B, 128), 128, 0, st>>>(B, euler, is_degree, R))); count_kernel_launches(1);
    PNP_CUDA_OK(cudaGetLastError());
    return PNPB200_OK;
}

int pnpb200_euler_from_R(int dtype, int64_t B, const void* R, int is_degree, void* euler, void* stream)
{
    if (B < 0 || !euler || !R) return PNPB200_EINVAL;
    if (B == 0) return PNPB200_OK;
    cudaStream_t st = (cudaStream_t)stream;
    DISPATCH_DTYPE(dtype, (k_euler_from_R<double><<<grid_for(B, 128), 128, 0, st>>>(B, R, is_degree, euler)),
                   (k_euler_from_R<float><<<grid_for(B, 128), 128, 0, st>>>(B, R, is_degree, euler))); count_kernel_launches(1);
    PNP_CUDA_OK(cudaGetLastError());
    return PNPB200_OK;
}

int pnpb200_project(int dtype, int64_t B, int n, const void* pattern, const double* K, const void* R, const void* t,
                    int is_quantized, double quantize_q, void* uvw, void* stream)
{
    if (B < 0 || n < 1 || !pattern || !K || !R || !t || !uvw) return PNPB200_EINVAL;
    if (B == 0) return PNPB200_OK;
    KMat km;
    for (int e = 0; e < 9; ++e) km.k[e] = K[e];
    cudaStream_t st = (cudaStream_t)stream;
    DISPATCH_DTYPE(dtype,
                   (k_project<double><<<grid_for(B * n, 256), 256, 0, st>>>(B, n, pattern, km, R, t, is_quantized, quantize_q, uvw)),
                   (k_project<float><<<grid_for(B * n, 256), 256, 0, st>>>(B, n, pattern, km, R, t, is_quantized, quantize_q, uvw))); count_kernel_launches(1);
    PNP_CUDA_OK(cudaGetLastError());
    return PNPB200_OK;
}

static int synth_launch(int dtype, int64_t b0, int64_t B, int n, const void* pattern_f64, const double* K,
                        const pnpb200_synth* cfg, void* uv, double* gt, double* R_gt, double* t_gt, double radius, int fixed_idx,
                        double* perturb, void* stream)
{
    if (B < 0 || n < 1 || !pattern_f64 || !K || !uv || radius < 0.0) return PNPB200_EINVAL;
    if (B == 0) return PNPB200_OK;
    pnpb200_synth c;
    if (cfg) c = *cfg; else pnpb200_default_synth(&c);
    KMat km;
    for (int e = 0; e < 9; ++e) km.k[e] = K[e];
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned grid = grid_for(B * 32, 256);
    DISPATCH_DTYPE(dtype,
                   (k_synth<double><<<grid, 256, 0, st>>>(b0, B, n, (const double*)pattern_f64, km, c, uv, gt, R_gt, t_gt, radius, fixed_idx, perturb)),
                   (k_synth<float><<<grid, 256, 0, st>>>(b0, B, n, (const double*)pattern_f64, km, c, uv, gt, R_gt, t_gt, radius, fixed_idx, perturb))); count_kernel_launches(1);
    PNP_CUDA_OK(cudaGetLastError());
    return PNPB200_OK;
}

int pnpb200_synth_batch(int dtype, int64_t b0, int64_t B, int n, const void* pattern_f64, const double* K,
                        const pnpb200_synth* cfg, void* uv, double* gt, double* R_gt, double* t_gt, void* stream)
{
    return synth_launch(dtype, b0, B, n, pattern_f64, K, cfg, uv, gt, R_gt, t_gt, 0.0, -1, nullptr, stream);
}

int pnpb200_synth_face_variation(int dtype, int64_t b0, int64_t B, int n, const void* pattern_f64, const double* K,
                                 const pnpb200_synth* cfg, double perturb_radius_m, int fixed_index, void* uv, double* gt,
                                 double* R_gt, double* t_gt, double* perturb, void* stream)
{
    if (!(perturb_radius_m > 0.0) || fixed_index >= n || (fixed_index < 0 ? n < 1 : n < 2)) return PNPB200_EINVAL;
    return synth_launch(dtype, b0, B, n, pattern_f64, K, cfg, uv, gt, R_gt, t_gt, perturb_radius_m, fixed_index, perturb, stream);
}

int pnpb200_report_batch(int dtype, int64_t B, int n, const void* pattern, const void* uv, const double* K,
                         const void* R, const void* t, const void* euler_deg, const double* gt, const double* bounds,
                         double* report, int32_t* flags, int32_t* max_idx, void* stream)
{
    return pnpb200_report_batch_strided(dtype, B, n, pattern, uv, K, R, t, euler_deg, gt, bounds, report, PNPB200_REPORT_WIDTH, 1,
                                        flags, max_idx, stream);
}

int pnpb200_report_batch_strided(int dtype, int64_t B, int n, const void* pattern, const void* uv, const double* K,
                                 const void* R, const void* t, const void* euler_deg, const double* gt, const double* bounds,
                                 double* report, int64_t report_stride_problem, int64_t report_stride_column,
                                 int32_t* flags, int32_t* max_idx, void* stream)
{
    return report_launch(dtype, B, n, pattern, uv, K, R, t, euler_deg, gt, bounds, report, report_stride_problem,
                         report_stride_column, flags, max_idx, nullptr, (cudaStream_t)stream);
}

int pnpb200_report_batch_strided_masked(int dtype, int64_t B, int n, const void* pattern, const void* uv, const double* K,
                                        const void* R, const void* t, const void* euler_deg, const double* gt, const double* bounds,
                                        double* report, int64_t report_stride_problem, int64_t report_stride_column,
                                        int32_t* flags, int32_t* max_idx, const uint32_t* visible, void* stream)
{
    if (!visible) return PNPB200_EINVAL;
    return report_launch(dtype, B, n, pattern, uv, K, R, t, euler_deg, gt, bounds, report, report_stride_problem,
                         report_stride_column, flags, max_idx, nullptr, (cudaStream_t)stream, visible);
}

}  // extern "C"

static int stats_grid(int64_t B)
{
    DeviceProps dp;
    if (get_device_props(&dp) != PNPB200_OK) return 148;
    long long g = (B + kStatBlock - 1) / kStatBlock;
    const long long cap = (long long)dp.sm_count * 8;
    return (int)(g < cap ? (g < 1 ? 1 : g) : cap);
}

template <int PASS>
static int stats_launch(int64_t B, int nq, const double* const* est, const int64_t* es, const double* const* gt,
                        const int64_t* gs, const int32_t* class_id, int n_class, const double* sums1, double* sums,
                        double* sums_max, cudaStream_t st)
{
    if (B < 0 || nq < 1 || nq > kStatMaxQ || !est || !es || !sums || n_class < 1 || n_class > (1 << 20)) return PNPB200_EINVAL;
    if (PASS == 2 && (!sums1 || !sums_max)) return PNPB200_EINVAL;
    StatIn in;
    in.nq = nq;
    for (int q = 0; q < kStatMaxQ; ++q) {
        in.est[q] = (q < nq) ? est[q] : nullptr;
        in.gt[q] = (q < nq && gt) ? gt[q] : nullptr;
        in.es[q] = (q < nq) ? es[q] : 0;
        in.gs[q] = (q < nq && gs) ? gs[q] : 0;
        if (q < nq && !in.est[q]) return PNPB200_EINVAL;
    }
    PNP_CUDA_OK(cudaMemsetAsync(sums, 0, sizeof(double) * 4 * (size_t)nq * (n_class + 1), st));
    if (PASS == 2) PNP_CUDA_OK(cudaMemsetAsync(sums_max, 0, sizeof(double) * (size_t)nq * (n_class + 1), st));
    if (B == 0) return PNPB200_OK;
    DeviceProps dp;
    int rc = get_device_props(&dp);
    if (rc != PNPB200_OK) return rc;
    if (n_class > kStatMaxClass) {                        // many classes: reductions straight into the global table
        k_stats_global<PASS><<<stats_grid(B), 256, 0, st>>>(B, in, class_id, n_class, sums1, sums, sums_max); count_kernel_launches(1);
        PNP_CUDA_OK(cudaGetLastError());
        return PNPB200_OK;
    }
    const size_t per_warp = sizeof(double) * (size_t)n_class * (PASS == 1 ? 3 : 4) * 32;
    int warps = (int)(((size_t)dp.max_smem_optin - 4096) / per_warp);
    if (warps > kStatLaneMaxWarps) warps = kStatLaneMaxWarps;
    warps -= warps % nq;                                  // every quantity gets the same number of warps
    if (warps >= nq) {                                    // lane-private tables fit: one block per SM
        const size_t lane_smem = per_warp * warps;
        PNP_CUDA_OK(set_dynamic_smem((const void*)k_stats_lane<PASS>, lane_smem));
        const int per_block = (warps / nq) * 32;          // problems a block covers per sweep
        long long g = (B + per_block - 1) / per_block;
        if (g > dp.sm_count) g = dp.sm_count;
        k_stats_lane<PASS><<<(unsigned)g, warps * 32, lane_smem, st>>>(B, in, class_id, n_class, sums1, sums, sums_max); count_kernel_launches(1);
    } else {
        const size_t smem = sizeof(double) * (size_t)kStatWarps * n_class * nq * 4;
        if (smem > 48 * 1024) PNP_CUDA_OK(set_dynamic_smem((const void*)k_stats<PASS>, smem));
        k_stats<PASS><<<stats_grid(B), kStatBlock, smem, st>>>(B, in, class_id, n_class, sums1, sums, sums_max); count_kernel_launches(1);
    }
    PNP_CUDA_OK(cudaGetLastError());
    return PNPB200_OK;
}

extern "C" {

int pnpb200_stats_pass1(int64_t B, int nq, const double* const* est, const int64_t* est_stride, const double* const* gt,
                        const int64_t* gt_stride, const int32_t* class_id, int n_class, double* sums1, void* stream)
{
    return stats_launch<1>(B, nq, est, est_stride, gt, gt_stride, class_id, n_class, nullptr, sums1, nullptr, (cudaStream_t)stream);
}

int pnpb200_stats_pass2(int64_t B, int nq, const double* const* est, const int64_t* est_stride, const double* const* gt,
                        const int64_t* gt_stride, const int32_t* class_id, int n_class, const double* sums1, double* sums2,
                        double* max2, void* stream)
{
    return stats_launch<2>(B, nq, est, est_stride, gt, gt_stride, class_id, n_class, sums1, sums2, max2, (cudaStream_t)stream);
}

int pnpb200_classify(int64_t B, const double* values, int64_t stride, double scale, const double* bins, int n_bins,
                     int32_t* class_id, void* stream)
{
    if (B < 0 || !values || !bins || !class_id || n_bins < 0 || n_bins > 32) return PNPB200_EINVAL;
    if (B == 0) return PNPB200_OK;
    Bins bn;
    bn.n = n_bins;
    for (int i = 0; i < 32; ++i) bn.b[i] = (i < n_bins) ? bins[i] : 0.0;
    k_classify<<<grid_for(B, 256), 256, 0, (cudaStream_t)stream>>>(B, values, stride, scale, bn, class_id); count_kernel_launches(1);
    PNP_CUDA_OK(cudaGetLastError());
    return PNPB200_OK;
}

int pnpb200_classify_drpy(int64_t B, const double* gt, const double* const* bins, const int32_t* n_bins, const double* scale,
                          int32_t* class_id, void* stream)
{
    if (B < 0 || !gt || !bins || !n_bins || !class_id) return PNPB200_EINVAL;
    Bins4 b4;
    long long total = 1;
    for (int q = 0; q < 4; ++q) {
        if (!bins[q] || n_bins[q] < 0 || n_bins[q] > 32) return PNPB200_EINVAL;
        b4.n[q] = n_bins[q];
        b4.scale[q] = scale ? scale[q] : 1.0;
        for (int i = 0; i < 32; ++i) b4.b[q][i] = (i < n_bins[q]) ? bins[q][i] : 0.0;
        total *= n_bins[q] + 1;
    }
    if (total > (1 << 20)) return PNPB200_EINVAL;
    if (B == 0) return PNPB200_OK;
    k_classify_drpy<<<grid_for(B, 256), 256, 0, (cudaStream_t)stream>>>(B, gt, b4, class_id); count_kernel_launches(1);
    PNP_CUDA_OK(cudaGetLastError());
    return PNPB200_OK;
}

int pnpb200_normalise_uvw(int dtype, int64_t n_points, const void* uvw, const double* K, void* uv_normalised, void* stream)
{
    if (n_points < 0 || !uvw || !K || !uv_normalised) return PNPB200_EINVAL;
    if (n_points == 0) return PNPB200_OK;
    KMat ki;
    host_inv3(K, ki.k);
    for (int e = 0; e < 9; ++e)
        if (!(ki.k[e] - ki.k[e] == 0.0)) return PNPB200_EINVAL;
    const unsigned grid = grid_for(n_points, 256);
    DISPATCH_DTYPE(dtype, (k_normalise_uvw<double><<<grid, 256, 0, (cudaStream_t)stream>>>(n_points, (const double*)uvw, ki, (double*)uv_normalised)),
                   (k_normalise_uvw<float><<<grid, 256, 0, (cudaStream_t)stream>>>(n_points, (const float*)uvw, ki, (float*)uv_normalised)));
    count_kernel_launches(1);
    PNP_CUDA_OK(cudaGetLastError());
    return PNPB200_OK;
}

int pnpb200_selftest_math(int64_t n, const double* in, double* rcp, double* rsqrt, double* sqrt_out, void* stream)
{
    if (n < 0 || !in || !rcp || !rsqrt || !sqrt_out) return PNPB200_EINVAL;
    if (n == 0) return PNPB200_OK;
    k_selftest_math<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(n, in, rcp, rsqrt, sqrt_out); count_kernel_launches(1);
    PNP_CUDA_OK(cudaGetLastError());
    return PNPB200_OK;
}

int pnpb200_selftest_sincos(int64_t n, const double* in, double* sin_out, double* cos_out, void* stream)
{
    if (n < 0 || !in || !sin_out || !cos_out) return PNPB200_EINVAL;
    if (n == 0) return PNPB200_OK;
    k_selftest_sincos<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(n, in, sin_out, cos_out); count_kernel_launches(1);
    PNP_CUDA_OK(cudaGetLastError());
    return PNPB200_OK;
}

int pnpb200_selftest_project(int dtype, int64_t n, const void* G, void* R, void* sigma_max, void* stream)
{
    if (n < 0 || !G || !R || !sigma_max || (dtype != PNPB200_DTYPE_F64 && dtype != PNPB200_DTYPE_F32)) return PNPB200_EINVAL;
    if (n == 0) return PNPB200_OK;
    if (dtype == PNPB200_DTYPE_F64)
        k_selftest_project<double><<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(n, (const double*)G, (double*)R, (double*)sigma_max);
    else
        k_selftest_project<float><<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(n, (const float*)G, (float*)R, (float*)sigma_max);
    count_kernel_launches(1);
    PNP_CUDA_OK(cudaGetLastError());
    return PNPB200_OK;
}

int pnpb200_fma_peak(int dtype, int iters, double* flops_per_s)
{
    if (!flops_per_s || iters < 1) return PNPB200_EINVAL;
    DeviceProps dp;
    int rc = get_device_props(&dp);
    if (rc != PNPB200_OK) return rc;
    void* out = nullptr;
    PNP_CUDA_OK(cudaMalloc(&out, 64));
    cudaEvent_t e0, e1;
    PNP_CUDA_OK(cudaEventCreate(&e0));
    PNP_CUDA_OK(cudaEventCreate(&e1));
    const int block = 256, grid = dp.sm_count * 8;
    float best_ms = 1e30f;
    for (int rep = 0; rep < 4; ++rep) {
        PNP_CUDA_OK(cudaEventRecord(e0, 0));
        if (dtype == PNPB200_DTYPE_F64) k_fma_peak<double><<<grid, block>>>(iters, 1.0, (double*)out);
        else                            k_fma_peak<float><<<grid, block>>>(iters, 1.0f, (float*)out);
        count_kernel_launches(1);
        PNP_CUDA_OK(cudaEventRecord(e1, 0));
        PNP_CUDA_OK(cudaEventSynchronize(e1));
        float ms = 0.f;
        PNP_CUDA_OK(cudaEventElapsedTime(&ms, e0, e1));
        if (rep > 0 && ms < best_ms) best_ms = ms;
    }
    PNP_CUDA_OK(cudaGetLastError());
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(out);
    const double fmas = (double)grid * block * (double)iters * 8.0;
    *flops_per_s = 2.0 * fmas / (best_ms * 1e-3);
    return PNPB200_OK;
}

}  // extern "C"
