// pnpb200_ransac.cu -- the hypothesis stage of the RANSAC solve (pnpb200_hypothesize_batch, include/pnpb200.h): per problem,
// minimal samples of 4 candidates drawn with Philox, a Lambda Twist P3P pose per sample and pattern (pnpb200_p3p.cuh) tested
// on the 4th landmark, and the consensus of the surviving hypotheses under the check's reprojection distance.
#include "pnpb200_common.cuh"
#include "pnpb200_math.cuh"
#include "pnpb200_p3p.cuh"
#include "pnpb200_reproject.cuh"

namespace pnpb200 {
namespace {

constexpr int kHypMaxN = 1024;   // candidates (landmarks of point_index) a problem may have: their list travels in the arguments
constexpr int kHypWarps = 4;     // problems per CTA, one warp each

struct HypArgs {                 // uv, pattern, R, t: the dtype of the call (the kernel's T)
    const void* uv; const void* pattern; const uint32_t* vis;
    void* R; void* t; int32_t* best; uint32_t* mask; int32_t* consensus; int32_t* drawn;
    long long B, idx0;
    unsigned long long seed;
    int n_total, n, n_patterns, W, max_samples, warp_bytes;
    double consensus_px, one_minus_conf;
    double K[9], Ki[9];
    uint16_t idx[kHypMaxN];      // the landmarks of point_index, in solver order
};

// the check's prediction-vs-landmark distance (k_check_chunk's arithmetic) of pattern point (x, y, z) at pixel (u, v)
PNP_DEV double hyp_distance(const double (&M)[9], const double (&m)[3], double x, double y, double z, double u, double v)
{
    double pe[2], ie, ex, ey;
    bool be;
    project_folded(M, m, x, y, z, pe, ie, be);
    px_difference(pe, ie, u, v, ex, ey);
    return homogeneous_distance(ex, ey, be);
}

// q^e by binary powering: the same products in the same order as tests/ransac_oracle.c
PNP_DEV double hyp_powi(double q, int e)
{
    double r = 1.0;
    while (e) {
        if (e & 1) r *= q;
        q *= q;
        e >>= 1;
    }
    return r;
}

// the stop test after sample s: (1 - w^4)^(s + 1) <= 1 - confidence, w = best / c; 1 - w^4 = (c^4 - best^4) / c^4 with both
// integers exact in FP64 (c <= 1024) and one correctly rounded division
PNP_DEV bool hyp_enough(int best, int c, int s, double one_minus_conf)
{
    const long long c2 = (long long)c * c, b2 = (long long)best * best;
    const double q = (double)(c2 * c2 - b2 * b2) / (double)(c2 * c2);
    return hyp_powi(q, s + 1) <= one_minus_conf;
}

// the candidate positions of sample s: u = philox(g, s, 4), j_k = u_k mod (c - k), the j_k-th candidate not yet chosen
PNP_DEV void hyp_draw(uint32_t g0, uint32_t g1, uint32_t s, uint32_t k0, uint32_t k1, int c, int (&pos)[4])
{
    uint32_t u[4];
    philox4x32_10(g0, g1, s, 4u, k0, k1, u);
    int srt[4];                                           // the chosen positions, ascending
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        int p = (int)(u[k] % (uint32_t)(c - k));
#pragma unroll
        for (int i = 0; i < k; ++i) p += p >= srt[i] ? 1 : 0;
        pos[k] = p;
        srt[k] = p;
#pragma unroll
        for (int i = k; i > 0; --i) {                      // insertion into the ascending list
            const int lo = min(srt[i - 1], srt[i]), hi = max(srt[i - 1], srt[i]);
            srt[i - 1] = lo; srt[i] = hi;
        }
    }
}

template <typename T>
PNP_DEV void hyp_point(const HypArgs& a, int p, int j, double& x, double& y, double& z)
{
    const T* q = (const T*)a.pattern + ((size_t)p * a.n_total + j) * 3;
    x = (double)__ldg(q); y = (double)__ldg(q + 1); z = (double)__ldg(q + 2);
}

// One warp per problem.  The candidates (index and pixel) go to shared memory in candidate order.  Per batch of 32 samples,
// lane l draws sample base + l and solves P3P for every pattern (lanes <-> samples); a pattern's hypothesis is the root
// closest to the 4th landmark and survives where that distance is <= consensus_px.  The survivors are then scored in sample
// order by the whole warp (lanes <-> candidates), and the stop test runs after every sample.
template <typename T>
__global__ void __launch_bounds__(kHypWarps * 32) k_hypothesize(const __grid_constant__ HypArgs a)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long b = (long long)blockIdx.x * kHypWarps + warp;
    if (b >= a.B) return;                                 // whole warps
    double* sHyp = reinterpret_cast<double*>(smem_raw + (size_t)warp * a.warp_bytes);   // [P][12][32] surviving poses
    double2* sPx = reinterpret_cast<double2*>(sHyp + (size_t)a.n_patterns * 12 * 32);  // [n] candidate pixels
    uint32_t* sMask = reinterpret_cast<uint32_t*>(sPx + a.n);                          // [W]
    uint16_t* sIdx = reinterpret_cast<uint16_t*>(sMask + a.W);                         // [n] candidate landmarks
    const uint32_t* vis = a.vis ? a.vis + (size_t)b * a.W : nullptr;
    int c = 0;
    for (int k0 = 0; k0 < a.n; k0 += 32) {
        const int k = k0 + lane;
        int j = 0;
        bool v = false;
        if (k < a.n) {
            j = a.idx[k];
            v = !vis || ((__ldg(vis + (j >> 5)) >> (j & 31)) & 1u);
        }
        const unsigned bal = __ballot_sync(0xffffffffu, v);
        if (v) {                                          // hidden pixels are never read
            const int pos = c + __popc(bal & ((1u << lane) - 1u));
            const T* px = (const T*)a.uv + ((size_t)b * a.n_total + j) * 2;
            sIdx[pos] = (uint16_t)j;
            sPx[pos] = make_double2((double)__ldg(px), (double)__ldg(px + 1));
        }
        c += __popc(bal);
    }
    for (int w = lane; w < a.W; w += 32) sMask[w] = 0u;
    __syncwarp();

    const unsigned long long g = (unsigned long long)(a.idx0 + b);
    const uint32_t g0 = (uint32_t)g, g1 = (uint32_t)(g >> 32), k0 = (uint32_t)a.seed, k1 = (uint32_t)(a.seed >> 32);
    int best = 0, win_p = 0, drawn = 0;
    double wR[9], wt[3];
    bool done = c < 4;
    for (int base = 0; !done && base < a.max_samples; base += 32) {
        const int s = base + lane;
        unsigned surv = 0;
        if (s < a.max_samples) {
            int pos[4];
            hyp_draw(g0, g1, (uint32_t)s, k0, k1, c, pos);
            double f[9];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const double2 px = sPx[pos[k]];
                double bx, by;
                normalise_px<double>(px.x, px.y, a.Ki[0], a.Ki[1], a.Ki[2], a.Ki[3], a.Ki[4], a.Ki[5], bx, by);
                const double bz = fma(a.Ki[6], px.x, fma(a.Ki[7], px.y, a.Ki[8]));
                const double r = t_rsqrt<double>(fma(bx, bx, fma(by, by, bz * bz)));
                f[3 * k] = bx * r; f[3 * k + 1] = by * r; f[3 * k + 2] = bz * r;
            }
            const double2 px4 = sPx[pos[3]];
            const int j4 = sIdx[pos[3]];
            for (int p = 0; p < a.n_patterns; ++p) {
                double X[9], x4, y4, z4;
#pragma unroll
                for (int k = 0; k < 3; ++k) hyp_point<T>(a, p, sIdx[pos[k]], X[3 * k], X[3 * k + 1], X[3 * k + 2]);
                hyp_point<T>(a, p, j4, x4, y4, z4);
                double Rs[4][9], ts[4][3];
                const unsigned valid = p3p_lambda_twist(X, f, Rs, ts);
                double bd = __longlong_as_double(0x7ff0000000000000ll);   // +inf: a NaN distance never wins
                double hR[9], ht[3];
#pragma unroll
                for (int r = 0; r < 4; ++r) {               // strict <: the first root wins ties
                    double M[9], m[3];
                    fold_camera(a.K, Rs[r], ts[r], M, m);
                    const double d = hyp_distance(M, m, x4, y4, z4, px4.x, px4.y);
                    const bool take = ((valid >> r) & 1u) && d < bd;
                    bd = take ? d : bd;
#pragma unroll
                    for (int e = 0; e < 9; ++e) hR[e] = take ? Rs[r][e] : hR[e];
#pragma unroll
                    for (int e = 0; e < 3; ++e) ht[e] = take ? ts[r][e] : ht[e];
                }
                if (bd <= a.consensus_px) {
                    double* h = sHyp + (size_t)p * 12 * 32 + lane;
#pragma unroll
                    for (int e = 0; e < 9; ++e) h[e * 32] = hR[e];
#pragma unroll
                    for (int e = 0; e < 3; ++e) h[(9 + e) * 32] = ht[e];
                    surv |= 1u << p;
                }
            }
        }
        __syncwarp();
        const int nb = min(32, a.max_samples - base);
        for (int l = 0; l < nb; ++l) {
            const unsigned bits = __shfl_sync(0xffffffffu, surv, l);
            int sc = 0, sp = 0;
            for (int p = 0; p < a.n_patterns; ++p) {
                if (!((bits >> p) & 1u)) continue;
                const double* h = sHyp + (size_t)p * 12 * 32 + l;
                double R[9], t[3], M[9], m[3];
#pragma unroll
                for (int e = 0; e < 9; ++e) R[e] = h[e * 32];
#pragma unroll
                for (int e = 0; e < 3; ++e) t[e] = h[(9 + e) * 32];
                fold_camera(a.K, R, t, M, m);
                int cnt = 0;
                for (int i = lane; i < c; i += 32) {
                    double x, y, z;
                    hyp_point<T>(a, p, sIdx[i], x, y, z);
                    const double2 px = sPx[i];
                    cnt += hyp_distance(M, m, x, y, z, px.x, px.y) <= a.consensus_px ? 1 : 0;
                }
                cnt = __reduce_add_sync(0xffffffffu, cnt);
                if (cnt > sc) {                            // ties go to the lower pattern
                    sc = cnt; sp = p;
                }
            }
            if (sc > best) {                               // ties go to the lower sample
                best = sc; win_p = sp;
                const double* h = sHyp + (size_t)sp * 12 * 32 + l;
#pragma unroll
                for (int e = 0; e < 9; ++e) wR[e] = h[e * 32];
#pragma unroll
                for (int e = 0; e < 3; ++e) wt[e] = h[(9 + e) * 32];
            }
            drawn = base + l + 1;
            if (hyp_enough(best, c, base + l, a.one_minus_conf)) { done = true; break; }
        }
        __syncwarp();                                     // the next batch overwrites sHyp
    }
    if (best > 0) {
        double M[9], m[3];
        fold_camera(a.K, wR, wt, M, m);
        for (int i = lane; i < c; i += 32) {
            double x, y, z;
            const int j = sIdx[i];
            hyp_point<T>(a, win_p, j, x, y, z);
            const double2 px = sPx[i];
            if (hyp_distance(M, m, x, y, z, px.x, px.y) <= a.consensus_px) atomicOr(sMask + (j >> 5), 1u << (j & 31));
        }
    } else {
        const double nan = __longlong_as_double(0x7ff8000000000000ll);
#pragma unroll
        for (int e = 0; e < 9; ++e) wR[e] = nan;
#pragma unroll
        for (int e = 0; e < 3; ++e) wt[e] = nan;
    }
    __syncwarp();
    for (int w = lane; w < a.W; w += 32) a.mask[(size_t)b * a.W + w] = sMask[w];
    if (lane < 9) ((T*)a.R)[b * 9 + lane] = (T)wR[lane];
    else if (lane < 12) ((T*)a.t)[b * 3 + lane - 9] = (T)wt[lane - 9];
    else if (lane == 12) {
        a.consensus[b] = best;
        if (a.best) a.best[b] = win_p;
        if (a.drawn) a.drawn[b] = drawn;
    }
}

// the P3P solver of the hypothesis stage, exposed for the tests: one triple per thread
__global__ void k_selftest_p3p(long long m, const double* __restrict__ X, const double* __restrict__ f, double* R, double* t, int32_t* n_sol)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    double x[9], y[9], Rs[4][9], ts[4][3];
#pragma unroll
    for (int e = 0; e < 9; ++e) { x[e] = X[i * 9 + e]; y[e] = f[i * 9 + e]; }
    const unsigned valid = p3p_lambda_twist(x, y, Rs, ts);
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    int ns = 0;                                           // the valid roots first, in slot order, then NaN
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        if (!((valid >> r) & 1u)) continue;
        for (int e = 0; e < 9; ++e) R[(i * 4 + ns) * 9 + e] = Rs[r][e];
        for (int e = 0; e < 3; ++e) t[(i * 4 + ns) * 3 + e] = ts[r][e];
        ++ns;
    }
    for (int r = ns; r < 4; ++r) {
        for (int e = 0; e < 9; ++e) R[(i * 4 + r) * 9 + e] = nan;
        for (int e = 0; e < 3; ++e) t[(i * 4 + r) * 3 + e] = nan;
    }
    n_sol[i] = ns;
}

template <typename T>
int hyp_launch(HypArgs& a, cudaStream_t st)
{
    DeviceProps dp;
    const int rc = get_device_props(&dp);
    if (rc != PNPB200_OK) return rc;
    a.warp_bytes = (int)(((size_t)a.n_patterns * 12 * 32 * 8 + (size_t)a.n * 16 + (size_t)a.W * 4 + (size_t)a.n * 2 + 15) & ~(size_t)15);
    const size_t smem = (size_t)kHypWarps * a.warp_bytes;
    if (smem > (size_t)dp.max_smem_optin) return PNPB200_ETOOLARGE;
    PNP_CUDA_OK(set_dynamic_smem((const void*)k_hypothesize<T>, smem));
    k_hypothesize<T><<<(unsigned)((a.B + kHypWarps - 1) / kHypWarps), kHypWarps * 32, smem, st>>>(a);
    count_kernel_launches(1);
    PNP_CUDA_OK(cudaGetLastError());
    return PNPB200_OK;
}

}  // namespace

bool hypothesis_params_ok(const pnpb200_hypothesis_params& h)
{
    return h.max_samples >= 0 && h.consensus_px >= 0.0 && h.confidence > 0.0 && h.confidence <= 1.0;
}

void fill_default_hypothesis(pnpb200_hypothesis_params* h)
{
    h->max_samples = 128; h->consensus_px = 4.0; h->confidence = 0.999; h->seed = 0; h->idx0 = 0;
}

int hypothesize_impl(int dtype, int64_t B, int n_total, int n, const void* uv, const void* pattern, int n_patterns,
                     const int32_t* point_index, const double* K, const uint32_t* visible, const pnpb200_hypothesis_params& hp,
                     void* R, void* t, int32_t* best_pattern, uint32_t* consensus_mask, int32_t* consensus, int32_t* drawn,
                     cudaStream_t st)
{
    if (!hypothesis_params_ok(hp)) return PNPB200_EINVAL;
    if (B < 0 || n_total < 1 || n < 1 || (!point_index && n != n_total) || !uv || !pattern || !K) return PNPB200_EINVAL;
    if (!R || !t || !consensus_mask || !consensus || (n_patterns > 1 && !best_pattern)) return PNPB200_EINVAL;
    if (n_patterns < 1 || n_patterns > PNPB200_MAX_PATTERNS) return PNPB200_EINVAL;
    if (dtype != PNPB200_DTYPE_F64 && dtype != PNPB200_DTYPE_F32) return PNPB200_EINVAL;
    if ((visible && !vis_aligned(visible)) || !vis_aligned(consensus_mask)) return PNPB200_EINVAL;
    HypArgs ad;
    for (int i = 0; i < n && i < kHypMaxN; ++i) {
        const int j = point_index ? point_index[i] : i;
        if (j < 0 || j >= n_total) return PNPB200_EINVAL;
        ad.idx[i] = (uint16_t)j;
    }
    if (n > kHypMaxN || n_total > 65536) return PNPB200_ETOOLARGE;
    double Ki[9];
    host_inv3(K, Ki);
    for (int e = 0; e < 9; ++e)
        if (!(Ki[e] - Ki[e] == 0.0)) return PNPB200_EINVAL;
    if (B == 0) return PNPB200_OK;
    ad.uv = uv; ad.pattern = pattern; ad.vis = visible;
    ad.R = R; ad.t = t; ad.best = best_pattern; ad.mask = consensus_mask; ad.consensus = consensus; ad.drawn = drawn;
    ad.B = B; ad.idx0 = hp.idx0; ad.seed = hp.seed;
    ad.n_total = n_total; ad.n = n; ad.n_patterns = n_patterns; ad.W = (n_total + 31) / 32; ad.max_samples = hp.max_samples;
    ad.consensus_px = hp.consensus_px; ad.one_minus_conf = 1.0 - hp.confidence;
    for (int e = 0; e < 9; ++e) { ad.K[e] = K[e]; ad.Ki[e] = Ki[e]; }
    return dtype == PNPB200_DTYPE_F64 ? hyp_launch<double>(ad, st) : hyp_launch<float>(ad, st);
}

}  // namespace pnpb200

using namespace pnpb200;

extern "C" {

int pnpb200_default_hypothesis_params(pnpb200_hypothesis_params* p)
{
    if (!p) return PNPB200_EINVAL;
    fill_default_hypothesis(p);
    return PNPB200_OK;
}

int pnpb200_hypothesize_batch(int dtype, int64_t B, int n_total, int n, const void* uv, const void* pattern, int n_patterns,
                              const int32_t* point_index, const double* K, const uint32_t* visible,
                              const pnpb200_hypothesis_params* hyp, void* R, void* t, int32_t* best_pattern,
                              uint32_t* consensus_mask, int32_t* consensus, int32_t* drawn, void* stream)
{
    pnpb200_hypothesis_params hp;
    if (hyp) hp = *hyp; else fill_default_hypothesis(&hp);
    return hypothesize_impl(dtype, B, n_total, n, uv, pattern, n_patterns, point_index, K, visible, hp, R, t, best_pattern,
                            consensus_mask, consensus, drawn, (cudaStream_t)stream);
}

int pnpb200_selftest_p3p(int64_t m, const double* X, const double* f, double* R, double* t, int32_t* n_sol, void* stream)
{
    if (m < 0 || !X || !f || !R || !t || !n_sol) return PNPB200_EINVAL;
    if (m == 0) return PNPB200_OK;
    k_selftest_p3p<<<(unsigned)((m + 127) / 128), 128, 0, (cudaStream_t)stream>>>(m, X, f, R, t, n_sol);
    count_kernel_launches(1);
    PNP_CUDA_OK(cudaGetLastError());
    return PNPB200_OK;
}

}  // extern "C"
