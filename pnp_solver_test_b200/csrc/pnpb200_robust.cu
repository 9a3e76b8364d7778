// pnpb200_robust.cu -- the outlier-robust solve (pnpb200_solve_robust_batch, include/pnpb200.h): masked solve of every
// problem on its candidates, then per round the inlier classification (k_inlier_*, pnpb200_aux.cu), a stable selection of
// the problems whose mask changed, and the masked solve of that compacted batch, scattered back.
#include <cub/device/device_select.cuh>
#include <vector>

#include "pnpb200_common.cuh"
#include "pnpb200_math.cuh"
#include "pnpb200_reproject.cuh"
#include "pnpb200_tile.cuh"

namespace pnpb200 {
namespace {

// ------------------------------------------------------------------------------------------
// inlier classification of the outlier-robust solve (pnpb200_solve_robust_batch): per problem, over its candidates C (the
// landmarks of point_index that are visible), the check's prediction-vs-landmark distance d_i of the pose just solved, the
// lower median med of {d_i} (rank floor((|C| - 1) / 2), NaN last), tau = max(floor_px, k med) (floor_px where k med is not
// finite) and M' = {i in C : d_i <= tau}.  M' = M (the mask the pose was solved on): converged; |M'| < min_inliers:
// TOO_FEW, M kept; last round: NOT_CONVERGED, M kept; otherwise M' replaces M, the round count grows and the problem is
// flagged for the next solve.  Batch entry k is problem idx[k] of the call (inliers, vis, rounds, status are indexed by it);
// flag and tau (where non-null: the threshold of the entry) by k.
// ------------------------------------------------------------------------------------------
constexpr int kInlierUnroll = 4;                          // landmarks in flight per thread, as k_check_chunk
template <typename T>
struct InlierArgs {
    const T* pattern; const T* uv; const T* R; const T* t; const int32_t* best;
    const int32_t* idx; const uint32_t* sel; const uint32_t* vis;
    uint32_t* inliers; int32_t* rounds; int32_t* status; uint8_t* flag; double* tau;
    long long B;
    int n, n_patterns, row_pitch, chunk, vis_words, last_round, min_inliers;
    double K[9], k_median, floor_px;
    int use_tmap;
    alignas(64) CUtensorMap tmap;   // uv as a 2-D tensor (RowStream), valid when use_tmap
};

// the distances as ordered integer keys: d >= 0, so its bits order like its value; NaN is the largest key
PNP_DEV unsigned long long distance_key(double d)
{
    return d != d ? ~0ull : ((unsigned long long)__double_as_longlong(d) & 0x7fffffffffffffffull);
}
PNP_DEV double inlier_threshold(unsigned long long med_key, double k, double floor_px)
{
    const double s = k * __longlong_as_double((long long)med_key);     // (the NaN key is a NaN)
    return (s - s == 0.0 && s > floor_px) ? s : floor_px;
}
// fl(k d) <= floor_px holds on a prefix of the distances in key order, and where it holds at the median tau is floor_px
PNP_DEV bool under_floor(double d, double k, double floor_px) { return k * d <= floor_px; }

// the decision on M' (words nw, W of them) against the mask M of problem o; returns the flag of batch entry k
template <typename T>
PNP_DEV uint8_t decide_inliers(const InlierArgs<T>& a, long long o, const uint32_t* nw, int stride)
{
    const int W = a.vis_words;
    uint32_t* m = a.inliers + (size_t)o * W;
    bool same = true;
    int cnt = 0;
    for (int w = 0; w < W; ++w) {
        same &= nw[(size_t)w * stride] == m[w];
        cnt += __popc(nw[(size_t)w * stride]);
    }
    if (same) return 0;
    if (cnt < a.min_inliers) { a.status[o] = PNPB200_ROBUST_TOO_FEW; return 0; }
    if (a.last_round) { a.status[o] = PNPB200_ROBUST_NOT_CONVERGED; return 0; }
    for (int w = 0; w < W; ++w) m[w] = nw[(size_t)w * stride];
    a.rounds[o] += 1;
    return 1;
}

template <typename T>
PNP_DEV void load_inlier_pose(const InlierArgs<T>& a, long long b, double (&R)[9], double (&t)[3], int& pat)
{
#pragma unroll
    for (int k = 0; k < 3; ++k) t[k] = (double)__ldg(a.t + b * 3 + k);
#pragma unroll
    for (int k = 0; k < 9; ++k) R[k] = (double)__ldg(a.R + b * 9 + k);
    pat = a.best ? __ldg(a.best + b) : 0;
}

// The streaming shape of k_check_chunk (lane <-> problem, rows through RowStream, every pattern in shared memory), plus per
// lane a column of shared memory for the keys of its candidates and their landmark indices, and its candidate / new mask
// words.  Where at least rank + 1 distances lie under floor_px / k, tau = floor_px without a selection; otherwise the lane
// selects the median from its column (Wirth's FIND: exact, in place).
template <typename T>
__global__ void __launch_bounds__(32) k_inlier_chunk(const __grid_constant__ InlierArgs<T> a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    typedef typename Vec2<T>::type V2;
    const int W = a.vis_words;
    unsigned long long* sKey = reinterpret_cast<unsigned long long*>(smem_raw);               // [n][32]
    uint32_t* sCw = reinterpret_cast<uint32_t*>(sKey + (size_t)a.n * kTileProblems);           // [W][32] candidates
    uint32_t* sNw = sCw + (size_t)W * kTileProblems;                                          // [W][32] M'
    uint16_t* sIdx = reinterpret_cast<uint16_t*>(sNw + (size_t)W * kTileProblems);            // [n][32]
    T* sBuf = reinterpret_cast<T*>(smem_raw + ((((size_t)((unsigned char*)(sIdx + (size_t)a.n * kTileProblems) - smem_raw)) + 127) & ~(size_t)127));
    T* sP = sBuf + (size_t)2 * kTileProblems * a.row_pitch;
    uint64_t* bars = carve_bar<T>(smem_raw, sP + (size_t)a.n_patterns * a.n * 3);
    const int lane = threadIdx.x;
    const long long n_tiles = (a.B + kTileProblems - 1) / kTileProblems;
    long long tile = blockIdx.x;
    long long b = tile * kTileProblems + lane;
    bool ok = b < a.B;
    if (!ok) b = a.B - 1;
    double R[9], t[3];
    int pat;
    load_inlier_pose(a, b, R, t, pat);
    RowStream<T> rs;
    rs.init(sBuf, bars, a.uv, a.B, a.n, a.chunk, a.row_pitch, lane, a.use_tmap ? &a.tmap : nullptr);
    if (tile < n_tiles) rs.begin_tile(tile, lane);
    for (int e = lane; e < a.n_patterns * a.n * 3; e += 32) sP[e] = a.pattern[e];
    __syncwarp();
    while (tile < n_tiles) {
        const long long o = __ldg(a.idx + b);
        for (int w = 0; w < W; ++w) {
            sCw[w * kTileProblems + lane] = __ldg(a.sel + w) & (a.vis ? __ldg(a.vis + (size_t)o * W + w) : ~0u);
            sNw[w * kTileProblems + lane] = 0u;
        }
        const T* P = sP + (size_t)pat * a.n * 3;          // (best_pattern comes from the solve: always in range)
        double M[9], m[3];
        fold_camera(a.K, R, t, M, m);
        int c = 0, under = 0;
        for (int ch = 0; ch < rs.n_chunks; ++ch) {
            const V2* row = rs.wait(ch, lane);
            const int cnt = rs.count(ch), base = ch * rs.chunk;
#pragma unroll kInlierUnroll
            for (int k = 0; k < cnt; ++k) {
                const int i = base + k;
                if (!((sCw[(i >> 5) * kTileProblems + lane] >> (i & 31)) & 1u)) continue;
                double pe[2], ie, ex, ey;
                bool be;
                project_folded(M, m, (double)P[3 * i], (double)P[3 * i + 1], (double)P[3 * i + 2], pe, ie, be);   // as k_check_chunk
                const V2 px = row[k];
                px_difference(pe, ie, (double)px.x, (double)px.y, ex, ey);
                const double d = homogeneous_distance(ex, ey, be);
                under += under_floor(d, a.k_median, a.floor_px) ? 1 : 0;
                sKey[(size_t)c * kTileProblems + lane] = distance_key(d);
                sIdx[(size_t)c * kTileProblems + lane] = (uint16_t)i;
                ++c;
            }
            rs.done(ch, lane);
        }
        double tau = a.floor_px;
        const int rank = (c - 1) / 2;
        if (c > 0 && under <= rank) {                     // the median lies above floor_px / k: select it
            int l = 0, r = c - 1;
            while (l < r) {
                const unsigned long long x = sKey[(size_t)rank * kTileProblems + lane];
                int i = l, j = r;
                do {
                    while (sKey[(size_t)i * kTileProblems + lane] < x) ++i;
                    while (x < sKey[(size_t)j * kTileProblems + lane]) --j;
                    if (i <= j) {
                        const unsigned long long ki = sKey[(size_t)i * kTileProblems + lane];
                        sKey[(size_t)i * kTileProblems + lane] = sKey[(size_t)j * kTileProblems + lane];
                        sKey[(size_t)j * kTileProblems + lane] = ki;
                        const uint16_t ii = sIdx[(size_t)i * kTileProblems + lane];
                        sIdx[(size_t)i * kTileProblems + lane] = sIdx[(size_t)j * kTileProblems + lane];
                        sIdx[(size_t)j * kTileProblems + lane] = ii;
                        ++i; --j;
                    }
                } while (i <= j);
                if (j < rank) l = i;
                if (rank < i) r = j;
            }
            tau = inlier_threshold(sKey[(size_t)rank * kTileProblems + lane], a.k_median, a.floor_px);
        }
        for (int p = 0; p < c; ++p) {
            if (__longlong_as_double((long long)sKey[(size_t)p * kTileProblems + lane]) <= tau) {
                const int i = sIdx[(size_t)p * kTileProblems + lane];
                sNw[(i >> 5) * kTileProblems + lane] |= 1u << (i & 31);
            }
        }
        if (ok) {
            if (a.tau) a.tau[b] = tau;
            a.flag[b] = decide_inliers(a, o, sNw + lane, kTileProblems);
        }
        tile += gridDim.x;
        if (tile < n_tiles) {
            fence_proxy_async();
            rs.begin_tile(tile, lane);
            b = tile * kTileProblems + lane;
            ok = b < a.B;
            if (!ok) b = a.B - 1;
            load_inlier_pose(a, b, R, t, pat);
        }
    }
}

// Rows the streaming shape cannot take: one warp per problem, landmark i on lane i % 32 (so word w of a mask is one
// ballot), the keys in a per-warp row of shared memory, the median by rank counting across the lanes.
constexpr int kInlierWarps = 8;
template <typename T>
__global__ void __launch_bounds__(kInlierWarps * 32) k_inlier_warp(const __grid_constant__ InlierArgs<T> a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int W = a.vis_words;
    unsigned long long* sKey = reinterpret_cast<unsigned long long*>(smem_raw) + (size_t)warp * a.n;
    uint32_t* sCw = reinterpret_cast<uint32_t*>(reinterpret_cast<unsigned long long*>(smem_raw) + (size_t)kInlierWarps * a.n) + (size_t)warp * 2 * W;
    uint32_t* sNw = sCw + W;
    const long long b = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= a.B) return;                                 // whole warps
    const long long o = __ldg(a.idx + b);
    double R[9], t[3];
    int pat;
    load_inlier_pose(a, b, R, t, pat);
    const T* P = a.pattern + (size_t)pat * a.n * 3;
    double M[9], m[3];
    fold_camera(a.K, R, t, M, m);
    for (int w = lane; w < W; w += 32) sCw[w] = __ldg(a.sel + w) & (a.vis ? __ldg(a.vis + (size_t)o * W + w) : ~0u);
    __syncwarp();
    int c = 0, under = 0;
    for (int i = lane; i < (W << 5); i += 32) {
        const bool cand = i < a.n && ((sCw[i >> 5] >> lane) & 1u);
        c += __popc(__ballot_sync(0xffffffffu, cand));
        if (!cand) continue;
        double pe[2], ie, ex, ey;
        bool be;
        project_folded(M, m, (double)__ldg(P + 3 * i), (double)__ldg(P + 3 * i + 1), (double)__ldg(P + 3 * i + 2), pe, ie, be);
        const T* px = a.uv + ((size_t)b * a.n + i) * 2;
        px_difference(pe, ie, (double)__ldg(px), (double)__ldg(px + 1), ex, ey);
        const double d = homogeneous_distance(ex, ey, be);
        under += under_floor(d, a.k_median, a.floor_px) ? 1 : 0;
        sKey[i] = distance_key(d);
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) under += __shfl_xor_sync(0xffffffffu, under, off);
    __syncwarp();
    double tau = a.floor_px;
    const int rank = (c - 1) / 2;
    if (c > 0 && under <= rank) {                         // the median lies above floor_px / k: rank counting
        unsigned long long med = 0;
        bool found = false;
        for (int i = lane; i < a.n; i += 32) {
            if (!((sCw[i >> 5] >> (i & 31)) & 1u)) continue;
            const unsigned long long ki = sKey[i];
            int less = 0, eq = 0;
            for (int j = 0; j < a.n; ++j) {
                if (!((sCw[j >> 5] >> (j & 31)) & 1u)) continue;
                const unsigned long long kj = sKey[j];
                less += kj < ki ? 1 : 0;
                eq += kj == ki ? 1 : 0;
            }
            if (less <= rank && rank < less + eq) { med = ki; found = true; }
        }
        const unsigned has = __ballot_sync(0xffffffffu, found);
        med = __shfl_sync(0xffffffffu, med, __ffs(has) - 1);
        tau = inlier_threshold(med, a.k_median, a.floor_px);
    }
    for (int w = 0; w < W; ++w) {
        const int i = (w << 5) + lane;
        const bool in = i < a.n && ((sCw[w] >> lane) & 1u) && __longlong_as_double((long long)sKey[i]) <= tau;
        const unsigned word = __ballot_sync(0xffffffffu, in);
        if (lane == 0) sNw[w] = word;
    }
    __syncwarp();
    if (lane == 0) {
        if (a.tau) a.tau[b] = tau;
        a.flag[b] = decide_inliers(a, o, sNw, 1);
    }
}


__global__ void __launch_bounds__(256) k_robust_init(long long B, int W, const uint32_t* __restrict__ sel, const uint32_t* __restrict__ vis,
                                                     uint32_t* inliers, int32_t* idx, int32_t* rounds, int32_t* status)
{
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    for (int w = 0; w < W; ++w) inliers[b * W + w] = sel[w] & (vis ? vis[b * W + w] : ~0u);
    idx[b] = (int32_t)b;
    rounds[b] = 1;
    status[b] = 0;
}

// the RANSAC solve's M0: the hypothesis stage's consensus set where it holds at least min_inliers landmarks (else C, as set
// by k_robust_init)
__global__ void __launch_bounds__(256) k_ransac_seed(long long B, int W, int min_inliers, const int32_t* __restrict__ consensus,
                                                     const uint32_t* __restrict__ cmask, uint32_t* inliers)
{
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B || consensus[b] < min_inliers) return;
    for (int w = 0; w < W; ++w) inliers[b * W + w] = cmask[b * W + w];
}

// compact entry k <- problem idx[k]: its pixel row and its mask (16-byte rows; the mask as words)
template <typename T>
__global__ void __launch_bounds__(256) k_robust_gather(long long m, int n_total, const int32_t* __restrict__ idx, const T* __restrict__ uv,
                                                       const uint32_t* __restrict__ inliers, T* uv_c, uint32_t* mask_c)
{
    const int W = (n_total + 31) / 32;
    const long long row = (long long)n_total * 2;
    const long long per = row + W;                        // elements of work per problem
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < m * per; e += (long long)gridDim.x * blockDim.x) {
        const long long k = e / per, j = e - k * per;
        const long long o = idx[k];
        if (j < row) uv_c[k * row + j] = uv[o * row + j];
        else mask_c[k * W + (j - row)] = inliers[o * W + (j - row)];
    }
}

// problem idx[k] <- the compact solve's outputs of entry k
template <typename T>
__global__ void __launch_bounds__(256) k_robust_scatter(long long m, const int32_t* __restrict__ idx, const T* __restrict__ cR,
                                                        const T* __restrict__ ct, const T* __restrict__ ce, const T* __restrict__ cres,
                                                        const int32_t* __restrict__ cit, const int32_t* __restrict__ cbest,
                                                        T* R, T* t, T* e, T* res, int32_t* it, int32_t* best)
{
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= m) return;
    const long long o = idx[k];
#pragma unroll
    for (int j = 0; j < 9; ++j) R[o * 9 + j] = cR[k * 9 + j];
#pragma unroll
    for (int j = 0; j < 3; ++j) t[o * 3 + j] = ct[k * 3 + j];
    if (e) {
#pragma unroll
        for (int j = 0; j < 3; ++j) e[o * 3 + j] = ce[k * 3 + j];
    }
    if (res) res[o] = cres[k];
    if (it) it[o] = cit[k];
    if (best) best[o] = cbest[k];
}

// the execution shapes of the check (check_launch): k_inlier_chunk where the check streams, k_inlier_warp otherwise.
// shape (pnpb200_selftest_inliers): 0 that choice, 1 k_inlier_chunk (EINVAL where it cannot run), 2 k_inlier_warp.
template <typename T>
int inlier_launch(InlierArgs<T> a, cudaStream_t st, int shape)
{
    if (a.B == 0) return PNPB200_OK;
    DeviceProps dp;
    const int rc = get_device_props(&dp);
    if (rc != PNPB200_OK) return rc;
    const StreamGeom sg = stream_geometry<T>(a.n);
    const size_t words = (size_t)a.vis_words * kTileProblems * sizeof(uint32_t);
    const size_t smem = (size_t)a.n * kTileProblems * (sizeof(unsigned long long) + sizeof(uint16_t)) + 2 * words + 128 +
                        2 * sg.buf_bytes + sizeof(T) * (size_t)a.n_patterns * a.n * 3 + 32;
    a.use_tmap = 0;
    const bool chunk = report_can_fuse(sizeof(T) == 8 ? PNPB200_DTYPE_F64 : PNPB200_DTYPE_F32, a.n) && smem <= (size_t)dp.max_smem_optin;
    if (shape == 1 && !chunk) return PNPB200_EINVAL;
    if (chunk && shape != 2) {
        a.row_pitch = sg.pitch; a.chunk = sg.chunk;
        a.use_tmap = (sg.pitch == sg.chunk * 2) ? make_row_tensor_map(&a.tmap, a.uv, (int)sizeof(T), a.B, a.n, sg.chunk) : 0;
        PNP_CUDA_OK(set_dynamic_smem((const void*)k_inlier_chunk<T>, smem));
        k_inlier_chunk<T><<<(unsigned)((a.B + kTileProblems - 1) / kTileProblems), 32, smem, st>>>(a);
    } else {
        const size_t wsmem = (size_t)kInlierWarps * ((size_t)a.n * sizeof(unsigned long long) + 2 * (size_t)a.vis_words * sizeof(uint32_t));
        if (wsmem > (size_t)dp.max_smem_optin) return PNPB200_ETOOLARGE;
        a.row_pitch = 0; a.chunk = 0;
        PNP_CUDA_OK(set_dynamic_smem((const void*)k_inlier_warp<T>, wsmem));
        k_inlier_warp<T><<<(unsigned)((a.B + kInlierWarps - 1) / kInlierWarps), kInlierWarps * 32, wsmem, st>>>(a);
    }
    count_kernel_launches(1);
    PNP_CUDA_OK(cudaGetLastError());
    return PNPB200_OK;
}

unsigned blocks_for(long long n) { return (unsigned)((n + 255) / 256 < 1 ? 1 : ((n + 255) / 256 < 0x7fffffffLL ? (n + 255) / 256 : 0x7fffffffLL)); }

size_t up256(size_t x) { return (x + 255) & ~(size_t)255; }

// the robust scratch behind the masked solve's: index lists, flags, count, cub's storage, the compacted batch; for the
// RANSAC solve (ransac) then the hypothesis stage's pose, pattern, consensus mask and sample count
struct RobustLayout {
    size_t solve, idx_a, idx_b, flag, count, sel, cub, cub_bytes, uv, mask, R, t, e, res, it, best, hR, ht, hbest, hmask, hdrawn, total;
};

RobustLayout robust_layout(int method, int dtype, int64_t B, int n_total, int n_patterns, int mapping, bool ransac = false)
{
    RobustLayout L;
    const size_t esz = (dtype == PNPB200_DTYPE_F32) ? 4 : 8, b = (size_t)B, W = ((size_t)n_total + 31) / 32;
    size_t cub_bytes = 0;
    cub::DeviceSelect::Flagged(nullptr, cub_bytes, (const int32_t*)nullptr, (const uint8_t*)nullptr, (int32_t*)nullptr, (int32_t*)nullptr,
                               (int)B);
    size_t o = 0;
    L.solve = o; o += up256((size_t)pnpb200_workspace_bytes_masked(method, dtype, B, n_patterns, mapping));
    L.idx_a = o; o += up256(4 * b);
    L.idx_b = o; o += up256(4 * b);
    L.flag = o; o += up256(b);
    L.count = o; o += 256;
    L.sel = o; o += up256(4 * W);
    L.cub = o; L.cub_bytes = cub_bytes; o += up256(cub_bytes);
    L.uv = o; o += up256(esz * b * n_total * 2);
    L.mask = o; o += up256(4 * W * b);
    L.R = o; o += up256(esz * 9 * b);
    L.t = o; o += up256(esz * 3 * b);
    L.e = o; o += up256(esz * 3 * b);
    L.res = o; o += up256(esz * b);
    L.it = o; o += up256(4 * b);
    L.best = o; o += up256(4 * b);
    if (ransac) {
        L.hR = o; o += up256(esz * 9 * b);
        L.ht = o; o += up256(esz * 3 * b);
        L.hbest = o; o += up256(4 * b);
        L.hmask = o; o += up256(4 * W * b);
        L.hdrawn = o; o += up256(4 * b);
    } else {
        L.hR = L.ht = L.hbest = L.hmask = L.hdrawn = o;
    }
    L.total = o;
    return L;
}

// the candidate words of point_index (all n_total landmarks where NULL); false for an index outside [0, n_total)
bool candidate_words(int n, int n_total, const int32_t* point_index, std::vector<uint32_t>& sel)
{
    sel.assign((size_t)(n_total + 31) / 32, 0u);
    for (int i = 0; i < n; ++i) {
        const int j = point_index ? point_index[i] : i;
        if (j < 0 || j >= n_total) return false;
        sel[(size_t)(j >> 5)] |= 1u << (j & 31);
    }
    return true;
}

bool robust_params_ok(const pnpb200_robust_params& r)
{
    return r.max_rounds >= 1 && r.min_inliers >= 4 && r.k_median >= 0.0 && r.k_median - r.k_median == 0.0 && r.floor_px >= 0.0;
}

void fill_default_robust(pnpb200_robust_params* r)
{
    r->max_rounds = 4; r->k_median = 3.0; r->floor_px = 2.0; r->min_inliers = 6;
}

// one pinned word per calling thread: the number of problems a round re-solves
int32_t* pinned_count()
{
    static thread_local int32_t* p = nullptr;
    if (!p && cudaMallocHost((void**)&p, sizeof(int32_t)) != cudaSuccess) p = nullptr;
    return p;
}

template <typename T>
void launch_gather(long long m, int n_total, const int32_t* idx, const void* uv, const uint32_t* inliers, void* uv_c, uint32_t* mask_c,
                   cudaStream_t st)
{
    const long long g = (m * ((long long)n_total * 2 + (n_total + 31) / 32) + 255) / 256;
    k_robust_gather<T><<<(unsigned)(g < 148 * 64 ? g : 148 * 64), 256, 0, st>>>(m, n_total, idx, (const T*)uv, inliers, (T*)uv_c, mask_c);
    count_kernel_launches(1);
}

template <typename T>
void launch_scatter(long long m, const int32_t* idx, void* const* c, void* const* out, const int32_t* cit, const int32_t* cbest,
                    int32_t* it, int32_t* best, cudaStream_t st)
{
    k_robust_scatter<T><<<blocks_for(m), 256, 0, st>>>(m, idx, (const T*)c[0], (const T*)c[1], (const T*)c[2], (const T*)c[3], cit, cbest,
                                                        (T*)out[0], (T*)out[1], (T*)out[2], (T*)out[3], it, best);
    count_kernel_launches(1);
}

// The loop of the robust entry.  hp = NULL: the robust solve, from M0 = C.  Otherwise the RANSAC solve: the hypothesis stage
// first, and M0 = its consensus set where that holds at least min_inliers landmarks.
int robust_run(int method, int dtype, int64_t B, int n_total, int n, const void* uv, const void* pattern, int n_patterns,
               const int32_t* point_index, const double* K, const pnpb200_params* params, void* R, void* t, void* euler_deg,
               void* res_norm, int32_t* iters, int32_t* best_pattern, const uint32_t* visible, const pnpb200_robust_params* robust,
               uint32_t* inliers, int32_t* rounds, int32_t* robust_status, const pnpb200_hypothesis_params* hp, int32_t* consensus,
               int32_t* drawn, cudaStream_t st)
{
    pnpb200_robust_params rp;
    if (robust) rp = *robust; else fill_default_robust(&rp);
    if (!robust_params_ok(rp)) return PNPB200_EINVAL;
    if (hp && (!hypothesis_params_ok(*hp) || !consensus)) return PNPB200_EINVAL;
    if (B < 0 || n_total < 1 || n < 1 || (!point_index && n != n_total) || !uv || !pattern || !K) return PNPB200_EINVAL;
    if (!R || !t || !inliers || !rounds || !robust_status || (n_patterns > 1 && !best_pattern)) return PNPB200_EINVAL;
    if (n_patterns < 1 || n_patterns > PNPB200_MAX_PATTERNS) return PNPB200_EINVAL;
    if (method < 0 || method > 5 || (dtype != PNPB200_DTYPE_F64 && dtype != PNPB200_DTYPE_F32)) return PNPB200_EINVAL;
    if ((visible && !vis_aligned(visible)) || !vis_aligned(inliers) || ((uintptr_t)uv & 15u)) return PNPB200_EINVAL;
    if (B > 0x7fffffffLL) return PNPB200_ETOOLARGE;       // int32 problem indices in the selection
    const int W = (n_total + 31) / 32;
    std::vector<uint32_t> sel;
    if (!candidate_words(n, n_total, point_index, sel)) return PNPB200_EINVAL;
    if (B == 0) return PNPB200_OK;
    pnpb200_params prm;
    if (params) prm = *params; else fill_default_params(&prm);
    prm.flags &= ~PNP_FLAG_INTERNAL_NO_RESIDUAL;
    const RobustLayout L = robust_layout(method, dtype, B, n_total, n_patterns, prm.mapping, hp != nullptr);
    char* ws = nullptr;
    const bool own_ws = !(prm.workspace && prm.workspace_bytes >= (int64_t)L.total);
    if (own_ws) PNP_CUDA_OK(cudaMallocAsync((void**)&ws, L.total, st));
    else ws = (char*)prm.workspace;
    struct Guard { void* p; cudaStream_t st; ~Guard() { if (p) cudaFreeAsync(p, st); } } guard = { own_ws ? ws : nullptr, st };
    prm.workspace_bytes = (int64_t)(L.idx_a - L.solve);      // (0 where the mapping takes none)
    prm.workspace = prm.workspace_bytes > 0 ? (void*)(ws + L.solve) : nullptr;
    int32_t* idx_cur = (int32_t*)(ws + L.idx_a);
    int32_t* idx_next = (int32_t*)(ws + L.idx_b);
    uint8_t* flag = (uint8_t*)(ws + L.flag);
    int32_t* d_count = (int32_t*)(ws + L.count);
    uint32_t* d_sel = (uint32_t*)(ws + L.sel);
    void* c[4] = { ws + L.R, ws + L.t, euler_deg ? ws + L.e : nullptr, res_norm ? ws + L.res : nullptr };
    void* out[4] = { R, t, euler_deg, res_norm };
    int32_t* cit = iters ? (int32_t*)(ws + L.it) : nullptr;
    int32_t* cbest = best_pattern ? (int32_t*)(ws + L.best) : nullptr;
    int32_t* h_count = pinned_count();
    if (!h_count) return PNPB200_ECUDA;

    PNP_CUDA_OK(cudaMemcpyAsync(d_sel, sel.data(), sizeof(uint32_t) * (size_t)W, cudaMemcpyHostToDevice, st));
    int rc;
    if (hp) {
        rc = hypothesize_impl(dtype, B, n_total, n, uv, pattern, n_patterns, point_index, K, visible, *hp, ws + L.hR, ws + L.ht,
                              (int32_t*)(ws + L.hbest), (uint32_t*)(ws + L.hmask), consensus, drawn ? drawn : (int32_t*)(ws + L.hdrawn), st);
        if (rc != PNPB200_OK) return rc;
    }
    k_robust_init<<<blocks_for(B), 256, 0, st>>>(B, W, d_sel, visible, inliers, idx_cur, rounds, robust_status);
    count_kernel_launches(1);
    PNP_CUDA_OK(cudaGetLastError());
    if (hp) {
        k_ransac_seed<<<blocks_for(B), 256, 0, st>>>(B, W, rp.min_inliers, consensus, (const uint32_t*)(ws + L.hmask), inliers);
        count_kernel_launches(1);
        PNP_CUDA_OK(cudaGetLastError());
    }
    rc = solve_batch_impl(method, dtype, B, n_total, n, uv, pattern, n_patterns, point_index, K, prm, R, t, euler_deg, res_norm,
                              iters, best_pattern, st, inliers);
    if (rc != PNPB200_OK) return rc;
    // the batch the next classification reads: the whole call first, then each round's compacted problems
    const bool f64 = dtype == PNPB200_DTYPE_F64;
    InlierArgs<double> ad;
    InlierArgs<float> af;
    ad.pattern = (const double*)pattern; af.pattern = (const float*)pattern;
    ad.idx = af.idx = idx_cur;
    ad.sel = af.sel = d_sel; ad.vis = af.vis = visible; ad.inliers = af.inliers = inliers; ad.rounds = af.rounds = rounds;
    ad.status = af.status = robust_status; ad.flag = af.flag = flag; ad.tau = af.tau = nullptr; ad.B = af.B = B; ad.n = af.n = n_total;
    ad.n_patterns = af.n_patterns = n_patterns; ad.vis_words = af.vis_words = W; ad.min_inliers = af.min_inliers = rp.min_inliers;
    for (int e = 0; e < 9; ++e) ad.K[e] = af.K[e] = K[e];
    ad.k_median = af.k_median = rp.k_median; ad.floor_px = af.floor_px = rp.floor_px;
    const void *b_uv = uv, *b_R = R, *b_t = t;
    const int32_t* b_best = best_pattern;
    for (int r = 0;; ++r) {
        ad.uv = (const double*)b_uv; ad.R = (const double*)b_R; ad.t = (const double*)b_t;
        af.uv = (const float*)b_uv; af.R = (const float*)b_R; af.t = (const float*)b_t;
        ad.best = af.best = b_best;
        ad.last_round = af.last_round = (r + 1 >= rp.max_rounds) ? 1 : 0;
        rc = f64 ? inlier_launch<double>(ad, st, 0) : inlier_launch<float>(af, st, 0);
        if (rc != PNPB200_OK) return rc;
        if (ad.last_round) break;
        size_t cub_bytes = L.cub_bytes;
        PNP_CUDA_OK(cub::DeviceSelect::Flagged(ws + L.cub, cub_bytes, ad.idx, flag, idx_next, d_count, (int)ad.B, st));
        PNP_CUDA_OK(cudaMemcpyAsync(h_count, d_count, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        PNP_CUDA_OK(cudaStreamSynchronize(st));
        const long long m = *h_count;
        if (m == 0) break;
        void* uv_c = ws + L.uv;
        uint32_t* mask_c = (uint32_t*)(ws + L.mask);
        if (f64) launch_gather<double>(m, n_total, idx_next, uv, inliers, uv_c, mask_c, st);
        else     launch_gather<float>(m, n_total, idx_next, uv, inliers, uv_c, mask_c, st);
        PNP_CUDA_OK(cudaGetLastError());
        rc = solve_batch_impl(method, dtype, m, n_total, n, uv_c, pattern, n_patterns, point_index, K, prm, c[0], c[1], c[2], c[3], cit,
                              cbest, st, mask_c);
        if (rc != PNPB200_OK) return rc;
        if (f64) launch_scatter<double>(m, idx_next, c, out, cit, cbest, iters, best_pattern, st);
        else     launch_scatter<float>(m, idx_next, c, out, cit, cbest, iters, best_pattern, st);
        PNP_CUDA_OK(cudaGetLastError());
        b_uv = uv_c; b_R = c[0]; b_t = c[1]; b_best = cbest;
        ad.idx = af.idx = idx_next; ad.B = af.B = m;
        int32_t* sw = idx_cur; idx_cur = idx_next; idx_next = sw;
    }
    return PNPB200_OK;
}

// one classification pass of the robust loop over the caller's poses (pnpb200_selftest_inliers)
template <typename T>
int inlier_pass(int64_t B, int n_total, const void* uv, const void* pattern, int n_patterns, const double* K, const uint32_t* visible,
                const pnpb200_robust_params& rp, const void* R, const void* t, const int32_t* best, const int32_t* idx,
                const uint32_t* sel, int last_round, uint32_t* inliers, int32_t* rounds, int32_t* status, uint8_t* flag, double* tau,
                int shape, cudaStream_t st)
{
    InlierArgs<T> a;
    a.pattern = (const T*)pattern; a.uv = (const T*)uv; a.R = (const T*)R; a.t = (const T*)t; a.best = best;
    a.idx = idx; a.sel = sel; a.vis = visible; a.inliers = inliers; a.rounds = rounds; a.status = status; a.flag = flag; a.tau = tau;
    a.B = B; a.n = n_total; a.n_patterns = n_patterns; a.vis_words = (n_total + 31) / 32;
    a.last_round = last_round ? 1 : 0; a.min_inliers = rp.min_inliers;
    for (int e = 0; e < 9; ++e) a.K[e] = K[e];
    a.k_median = rp.k_median; a.floor_px = rp.floor_px;
    return inlier_launch<T>(a, st, shape);
}

}  // namespace
}  // namespace pnpb200

using namespace pnpb200;

extern "C" {

int pnpb200_default_robust_params(pnpb200_robust_params* p)
{
    if (!p) return PNPB200_EINVAL;
    fill_default_robust(p);
    return PNPB200_OK;
}

int64_t pnpb200_robust_workspace_bytes(int method, int dtype, int64_t B, int n_total, int n_patterns, int mapping)
{
    if (B <= 0 || B > 0x7fffffffLL || n_total < 1) return 0;
    return (int64_t)robust_layout(method, dtype, B, n_total, n_patterns, mapping).total;
}

int64_t pnpb200_ransac_workspace_bytes(int method, int dtype, int64_t B, int n_total, int n_patterns, int mapping)
{
    if (B <= 0 || B > 0x7fffffffLL || n_total < 1) return 0;
    return (int64_t)robust_layout(method, dtype, B, n_total, n_patterns, mapping, true).total;
}

int pnpb200_solve_robust_batch(int method, int dtype, int64_t B, int n_total, int n, const void* uv, const void* pattern,
                               int n_patterns, const int32_t* point_index, const double* K, const pnpb200_params* params,
                               void* R, void* t, void* euler_deg, void* res_norm, int32_t* iters, int32_t* best_pattern,
                               const uint32_t* visible, const pnpb200_robust_params* robust, uint32_t* inliers, int32_t* rounds,
                               int32_t* robust_status, void* stream)
{
    return robust_run(method, dtype, B, n_total, n, uv, pattern, n_patterns, point_index, K, params, R, t, euler_deg, res_norm, iters,
                      best_pattern, visible, robust, inliers, rounds, robust_status, nullptr, nullptr, nullptr, (cudaStream_t)stream);
}

int pnpb200_solve_ransac_batch(int method, int dtype, int64_t B, int n_total, int n, const void* uv, const void* pattern,
                               int n_patterns, const int32_t* point_index, const double* K, const pnpb200_params* params,
                               void* R, void* t, void* euler_deg, void* res_norm, int32_t* iters, int32_t* best_pattern,
                               const uint32_t* visible, const pnpb200_robust_params* robust, uint32_t* inliers, int32_t* rounds,
                               int32_t* robust_status, const pnpb200_hypothesis_params* hyp, int32_t* consensus, int32_t* drawn,
                               void* stream)
{
    pnpb200_hypothesis_params hp;
    if (hyp) hp = *hyp; else fill_default_hypothesis(&hp);
    return robust_run(method, dtype, B, n_total, n, uv, pattern, n_patterns, point_index, K, params, R, t, euler_deg, res_norm, iters,
                      best_pattern, visible, robust, inliers, rounds, robust_status, &hp, consensus, drawn, (cudaStream_t)stream);
}

int pnpb200_selftest_inliers(int dtype, int64_t B, int n_total, int n, const void* uv, const void* pattern, int n_patterns,
                             const int32_t* point_index, const double* K, const uint32_t* visible,
                             const pnpb200_robust_params* robust, const void* R, const void* t, const int32_t* best_pattern,
                             const int32_t* idx, int last_round, uint32_t* inliers, int32_t* rounds, int32_t* robust_status,
                             uint8_t* flag, double* tau, int shape, void* stream)
{
    pnpb200_robust_params rp;
    if (robust) rp = *robust; else fill_default_robust(&rp);
    if (!robust_params_ok(rp) || shape < 0 || shape > 2) return PNPB200_EINVAL;
    if (dtype != PNPB200_DTYPE_F64 && dtype != PNPB200_DTYPE_F32) return PNPB200_EINVAL;
    if (B < 0 || n_total < 1 || n < 1 || (!point_index && n != n_total) || !uv || !pattern || !K || !R || !t) return PNPB200_EINVAL;
    if (!inliers || !rounds || !robust_status || !flag || n_patterns < 1 || n_patterns > PNPB200_MAX_PATTERNS) return PNPB200_EINVAL;
    if ((visible && !vis_aligned(visible)) || !vis_aligned(inliers) || ((uintptr_t)uv & 15u)) return PNPB200_EINVAL;
    if (B > 0x7fffffffLL) return PNPB200_ETOOLARGE;
    std::vector<uint32_t> sel;
    if (!candidate_words(n, n_total, point_index, sel)) return PNPB200_EINVAL;
    if (B == 0) return PNPB200_OK;
    const cudaStream_t st = (cudaStream_t)stream;
    const size_t W = sel.size(), sel_bytes = up256(4 * W);
    char* buf = nullptr;
    PNP_CUDA_OK(cudaMallocAsync((void**)&buf, sel_bytes + (idx ? 0 : 4 * (size_t)B), st));
    struct Guard { void* p; cudaStream_t st; ~Guard() { cudaFreeAsync(p, st); } } guard = { buf, st };
    uint32_t* d_sel = (uint32_t*)buf;
    PNP_CUDA_OK(cudaMemcpyAsync(d_sel, sel.data(), 4 * W, cudaMemcpyHostToDevice, st));
    if (!idx) {                                           // the identity: batch entry k is problem k
        std::vector<int32_t> id((size_t)B);
        for (int64_t k = 0; k < B; ++k) id[(size_t)k] = (int32_t)k;
        PNP_CUDA_OK(cudaMemcpyAsync(buf + sel_bytes, id.data(), 4 * (size_t)B, cudaMemcpyHostToDevice, st));   // (pageable: staged)
        idx = (const int32_t*)(buf + sel_bytes);
    }
    return dtype == PNPB200_DTYPE_F64
        ? inlier_pass<double>(B, n_total, uv, pattern, n_patterns, K, visible, rp, R, t, best_pattern, idx, d_sel, last_round, inliers,
                              rounds, robust_status, flag, tau, shape, st)
        : inlier_pass<float>(B, n_total, uv, pattern, n_patterns, K, visible, rp, R, t, best_pattern, idx, d_sel, last_round, inliers,
                             rounds, robust_status, flag, tau, shape, st);
}

}  // extern "C"
