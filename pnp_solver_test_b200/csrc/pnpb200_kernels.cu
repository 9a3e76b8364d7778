// pnpb200_kernels.cu -- the hot path: batched PnP solve kernels for sm_100a and their launchers.
// Compiled once per (PNP_F64 = 0|1, PNP_GROUP = 0|1|2|3); the C ABI lives in pnpb200_api.cu.
//
// Two execution shapes share the solver code in pnpb200_solvers.cuh:
//
//  k_solve_thread  one problem per thread.  A CTA is ONE warp that owns 32 consecutive
//                  problems.  Each lane issues one TMA bulk copy (cp.async.bulk, completion on
//                  an mbarrier) of its problem's [n_total, 2] pixel row from HBM into a padded
//                  shared-memory row (row pitch = odd multiple of 16 B, so the per-lane 16-byte
//                  reads of the 14 solver passes are bank-conflict free), then normalises its
//                  row in place with K^-1 (f2_get_B_xy, PNP_SOLVER_LIB.py:3291-3312).  The
//                  pattern sits in shared memory too and is read as a warp-wide broadcast.
//                  All normal equations, factorisations and SO(3) work stay in the thread's
//                  registers; no shuffles are needed at all.  Several such one-warp CTAs are
//                  resident per SM, so the copy of one overlaps the FP64 work of the others.
//  k_solve_warp    one problem per warp for large n (n = 1024): lanes stride over the points
//                  with coalesced vector loads straight from global memory (L1/L2 resident
//                  across iterations), partial sums are combined with shuffle butterflies.
//
// No tensor cores on purpose: the per-problem systems are 6x6 / 12x12.
#include <string.h>

#include "pnpb200_common.cuh"
#include "pnpb200_solvers.cuh"
#include "pnpb200_tile.cuh"

#ifndef PNP_TUNE_VARIANTS
#define PNP_TUNE_VARIANTS 0   // 1: also build the experimental k_iterate occupancy variants (tools/time_solve.py --tune)
#endif
#ifndef PNP_F64
#error "compile with -DPNP_F64=0|1 -DPNP_GROUP=0|1|2|3"
#endif

namespace pnpb200 {

// ------------------------------------------------------------------------------------------
// kernel arguments
// ------------------------------------------------------------------------------------------
// internal kernel variant: QEIF with H^T H / H^T v from the moments (chosen for n >= 12 landmarks)
#define PNP_METHOD_QEIF_HYBRID 100
// internal kernel variant: LM exactly as the reference runs it (identity start, 14 iterations, constant lambda) but with the TRUE
// gradients of the nine constraint rows (PNPB200_FLAG_LM_TRUE_JACOBIAN; not a parity mode)
#define PNP_METHOD_LM_TRUEJAC 101

// what a method's passes of the moment mapping compute
__host__ __device__ constexpr bool method_with_w(int m) { return m != PNPB200_METHOD_LINEAR_F2; }                              // the (bx^2 + by^2)-weighted moments
__host__ __device__ constexpr bool method_with_s(int m) { return m == PNP_METHOD_QEIF_HYBRID || m == PNPB200_METHOD_EIF2; }   // sum (bx^2 + by^2): the filters' residual
__host__ __device__ constexpr int method_nmom(int m) { return method_with_s(m) ? PNP_NMOM : PNP_NMOM_LM; }                    // rows of the moment workspace in use
__host__ __device__ constexpr bool method_lm_residual(int m) { return m != PNPB200_METHOD_LINEAR_F2; }                         // residual of the 12-number measurement model (else: F2's)
__host__ __device__ constexpr bool method_has_core(int m) { return m == PNPB200_METHOD_LM || m == PNPB200_METHOD_LM_PLUS || m == PNP_METHOD_LM_TRUEJAC; }   // k_iterate parks the constant LM blocks in shared memory

template <typename T>
struct SolveArgs {
    const T* uv;            // [B, n_total, 2]
    const T* pattern;       // [P, n_total, 3]
    const int32_t* idx;     // [n] device (large selections), or nullptr
    int idx_mode;           // 0: all landmarks, 1: idx_inline, 2: idx (device)
    int32_t idx_inline[PNP_MAX_INLINE_IDX];
    long long B;
    int n_total, n, n_patterns;
    int row_pitch;          // thread mapping: shared-memory row pitch in elements of T
    int use_tma;            // rows are 16-byte aligned multiples of 16 bytes -> cp.async.bulk
    double kinv[6];         // first two rows of K^-1
    SolverPrm<T> prm;
    T* R; T* t; T* euler; T* res;
    int32_t* iters; int32_t* best;
    void* ws; size_t ws_bytes;   // optional caller scratch (moment mapping)
    int profile, tune;
    int skip_residual;           // moment mapping: leave res_norm to the caller's fused report pass (pnpb200_solve_report_batch)
    const uint32_t* vis;         // [B, vis_words] per-problem visibility bits (masked kernels only)
    int vis_words;
};

// raw pixels of one problem in global memory, normalised on the fly (warp mapping)
template <typename T>
struct PtsGlobal {
    const T* row;          // &uv[b, 0, 0]
    const int32_t* idx;    // shared-memory copy of the selection, or nullptr
    T k00, k01, k02, k10, k11, k12;
    PNP_DEV void get(int i, T& bx, T& by) const
    {
        const int j = idx ? idx[i] : i;
        const typename Vec2<T>::type p = __ldg(reinterpret_cast<const typename Vec2<T>::type*>(row) + j);
        normalise_px<T>(p.x, p.y, k00, k01, k02, k10, k11, k12, bx, by);
    }
    PNP_DEV bool vis(int) const { return true; }
    PNP_DEV int count(int n) const { return n; }
};

// Pattern constants (PNP_PATC per pattern) by one warp: M0, m0, n and G = (D^T D)^-1.
// Accumulated in double whatever T is (they are shared by every problem of the launch).
template <typename T>
PNP_DEV void pattern_constants(const T* __restrict__ sP, int n, T* __restrict__ sC, int lane)
{
    double acc[9];
#pragma unroll
    for (int e = 0; e < 9; ++e) acc[e] = 0.0;
    for (int i = lane; i < n; i += 32) {
        const double th[3] = { (double)sP[3 * i], (double)sP[3 * i + 1], (double)sP[3 * i + 2] };
#pragma unroll
        for (int a = 0; a < 3; ++a) {
#pragma unroll
            for (int b = a; b < 3; ++b) acc[s3(a, b)] = fma(th[a], th[b], acc[s3(a, b)]);
            acc[6 + a] += th[a];
        }
    }
#pragma unroll
    for (int e = 0; e < 9; ++e) acc[e] = group_sum<32, double>(acc[e]);
    if (lane == 0) {
        double G[10];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
#pragma unroll
            for (int b = a; b < 3; ++b) G[sidx<4>(a, b)] = acc[s3(a, b)];
            G[sidx<4>(a, 3)] = acc[6 + a];
        }
        G[sidx<4>(3, 3)] = (double)n;
        spd_inverse<double, 4>(G);
#pragma unroll
        for (int e = 0; e < 9; ++e) sC[e] = (T)acc[e];
        sC[9] = (T)n;
#pragma unroll
        for (int e = 0; e < 10; ++e) sC[10 + e] = (T)G[e];
    }
}

// Sum theta theta^T (6), sum theta (3) and the count (pm[9]) over the visible landmarks of ONE problem (masked kernels; LPP = 1:
// one thread, 32: one warp, every lane ends with the sums).  The moment mapping keeps them per problem in the workspace.
constexpr int kPatternMoments = PNP_NPMOM;
template <typename T, int LPP, typename Pts>
PNP_DEV void pattern_moments_masked(const Pts& pts, const T* __restrict__ sP, int n, int sub, double (&pm)[kPatternMoments])
{
#pragma unroll
    for (int e = 0; e < 9; ++e) pm[e] = 0.0;
    for (int i = sub; i < n; i += LPP) {
        if (!pts.vis(i)) continue;
        const double th[3] = { (double)sP[3 * i], (double)sP[3 * i + 1], (double)sP[3 * i + 2] };
#pragma unroll
        for (int a = 0; a < 3; ++a) {
#pragma unroll
            for (int b = a; b < 3; ++b) pm[s3(a, b)] = fma(th[a], th[b], pm[s3(a, b)]);
            pm[6 + a] += th[a];
        }
    }
#pragma unroll
    for (int e = 0; e < 9; ++e) pm[e] = group_sum<LPP, double>(pm[e]);
    pm[9] = (double)pts.count(n);
}

// the PNP_PATC constants of one problem from its pattern moments: M0, m0, n and G = (D^T D)^-1 (pattern_constants, per problem).
// n in sC[9] is the number of visible landmarks: it enters LM's and the filters' systems as well.
template <typename T>
PNP_DEV void constants_from_pattern_moments(const double (&pm)[kPatternMoments], T* __restrict__ sC)
{
    double G[10];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int b = a; b < 3; ++b) G[sidx<4>(a, b)] = pm[s3(a, b)];
        G[sidx<4>(a, 3)] = pm[6 + a];
    }
    G[sidx<4>(3, 3)] = pm[9];
    spd_inverse<double, 4>(G);
#pragma unroll
    for (int e = 0; e < 10; ++e) sC[e] = (T)pm[e];
#pragma unroll
    for (int e = 0; e < 10; ++e) sC[10 + e] = (T)G[e];
}

template <typename T, int LPP, typename Pts>
PNP_DEV void pattern_constants_masked(const Pts& pts, const T* __restrict__ sP, int n, T* __restrict__ sC, int sub)
{
    double pm[kPatternMoments];
    pattern_moments_masked<T, LPP>(pts, sP, n, sub, pm);
    if (sub == 0) constants_from_pattern_moments<T>(pm, sC);
}

// methods whose direct solvers read the pattern constants
__host__ __device__ constexpr bool method_uses_patc(int m)
{
    return m == PNPB200_METHOD_LM || m == PNPB200_METHOD_LINEAR_F2 || m == PNP_METHOD_QEIF_HYBRID || m == PNPB200_METHOD_EIF2;
}

// fewer than 4 visible landmarks: no solve.  NaN pose and res_norm, 0 iterations, pattern 0.
template <typename T>
PNP_DEV T nan_of() { return (T)__longlong_as_double(0x7ff8000000000000LL); }

template <typename T>
PNP_DEV void too_few_landmarks(Result<T>& r, int& best_p)
{
    const T q = nan_of<T>();
#pragma unroll
    for (int e = 0; e < 9; ++e) r.R[e] = q;
#pragma unroll
    for (int e = 0; e < 3; ++e) r.t[e] = q;
    r.res = q;
    r.iters = 0;
    best_p = 0;
}

template <typename T, int METHOD, int LPP, typename Pts>
PNP_DEV void run_method(const Pts& pts, const T* sP, const T* sC, int n, int sub, const SolverPrm<T>& prm,
                        Result<T>& out)
{
    if (METHOD == PNPB200_METHOD_QEIF)           solve_qeif<T, LPP, Pts, false>(pts, sP, sC, n, sub, prm, out);
    else if (METHOD == PNP_METHOD_QEIF_HYBRID)   solve_qeif<T, LPP, Pts, true>(pts, sP, sC, n, sub, prm, out);
    else if (METHOD == PNPB200_METHOD_LM)        solve_lm<T, LPP, Pts>(pts, sP, sC, n, sub, prm, out);
    else if (METHOD == PNPB200_METHOD_LINEAR_F2) solve_linear_f2<T, LPP, Pts>(pts, sP, sC, n, sub, prm, out);
    else if (METHOD == PNPB200_METHOD_EIF2)      solve_eif2<T, LPP, Pts>(pts, sP, sC, n, sub, prm, out);
    else                                         solve_linear_f1<T, LPP, Pts>(pts, sP, n, sub, prm, out);
}

// solve_pnp's loop over patterns with the strict-'<' arg-min on res_norm (:166-199)
template <typename T, int METHOD, int LPP, typename Pts>
PNP_DEV void solve_all_patterns(const Pts& pts, const T* sP, const T* sC, int n, int n_patterns, int sub,
                                const SolverPrm<T>& prm, Result<T>& best, int& best_p)
{
    // ONE inlined copy of the solver (a separate first call doubled every kernel's code: 12 416 instructions for EIF2)
    best_p = 0;
#pragma unroll 1
    for (int p = 0; p < n_patterns; ++p) {
        Result<T> cand;
        run_method<T, METHOD, LPP, Pts>(pts, sP + (size_t)p * n * 3, sC + p * PNP_PATC, n, sub, prm, cand);
        if (p == 0 || cand.res < best.res) { best = cand; best_p = p; }
    }
}

template <typename T>
PNP_DEV void write_result(const SolveArgs<T>& a, long long b, const Result<T>& r, int best_p)
{
    if (a.R) {
#pragma unroll
        for (int e = 0; e < 9; ++e) a.R[b * 9 + e] = r.R[e];
    }
    if (a.t) {
#pragma unroll
        for (int e = 0; e < 3; ++e) a.t[b * 3 + e] = r.t[e];
    }
    if (a.euler) {
        double Rd[9], e3[3];
#pragma unroll
        for (int e = 0; e < 9; ++e) Rd[e] = (double)r.R[e];
        euler_from_R(Rd, true, e3);                       // degrees, (roll, yaw, pitch) (:2998)
#pragma unroll
        for (int e = 0; e < 3; ++e) a.euler[b * 3 + e] = (T)e3[e];
    }
    if (a.res) a.res[b] = r.res;
    if (a.iters) a.iters[b] = r.iters;
    if (a.best) a.best[b] = best_p;
}

// the landmark selection: small ones travel inside the kernel arguments (no allocation, no copy)
template <typename A>
PNP_DEV const int32_t* selection_of(const A& a)
{
    return a.idx_mode == 1 ? a.idx_inline : (a.idx_mode == 2 ? a.idx : nullptr);
}

// pattern (restricted to the selected landmarks, in selection order) and the selection -> shared memory
template <typename T>
PNP_DEV void load_pattern(const T* __restrict__ pattern, const int32_t* __restrict__ idx, int n_total, int n, int n_patterns,
                          T* sP, int32_t* sIdx, int tid, int nthreads)
{
    if (idx) {
        for (int i = tid; i < n; i += nthreads) sIdx[i] = idx[i];
        __syncthreads();
    }
    for (int e = tid; e < n_patterns * n * 3; e += nthreads) {
        const int p = e / (n * 3), r = e - p * (n * 3), i = r / 3, c = r - 3 * i;
        const int src = idx ? sIdx[i] : i;
        sP[e] = pattern[((size_t)p * n_total + src) * 3 + c];
    }
    __syncthreads();
}

// ------------------------------------------------------------------------------------------
// direct mapping, one problem per thread; CTA = 1 warp = 32 consecutive problems
// ------------------------------------------------------------------------------------------
// MASKED: problem b sees only its visible landmarks (a.vis); every lane keeps its own constants, computed per tile
template <typename T, int METHOD, bool MASKED = false>
__global__ void __launch_bounds__(32) k_solve_thread(const __grid_constant__ SolveArgs<T> a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    // [tile rows | pattern | constants (masked: per lane) | index | mbarrier]
    T* sRows = reinterpret_cast<T*>(smem_raw);
    T* sP = sRows + (size_t)kTileProblems * a.row_pitch;
    T* sC = sP + (size_t)a.n_patterns * a.n * 3;
    int32_t* sIdx = reinterpret_cast<int32_t*>(sC + (MASKED ? kTileProblems : 1) * a.n_patterns * PNP_PATC);
    const int lane = threadIdx.x;
    const int32_t* sel = selection_of(a);
    RowTile<T> tile_buf;
    tile_buf.init(sRows, carve_bar<T>(smem_raw, sIdx + (sel ? a.n : 0)), a.uv, a.B, a.n_total, a.row_pitch, a.use_tma, a.kinv, lane);

    const long long n_tiles = (a.B + kTileProblems - 1) / kTileProblems;
    long long tile = blockIdx.x;
    // kick off the first tile's copies before touching the pattern so the two overlap
    int valid = (tile < n_tiles) ? tile_buf.issue(tile, lane) : 0;
    load_pattern<T>(a.pattern, sel, a.n_total, a.n, a.n_patterns, sP, sIdx, lane, 32);
    if (!MASKED && method_uses_patc(METHOD)) {
        for (int p = 0; p < a.n_patterns; ++p) pattern_constants<T>(sP + (size_t)p * a.n * 3, a.n, sC + p * PNP_PATC, lane);
        __syncwarp();
    }
    while (tile < n_tiles) {
        const long long b0 = tile * kTileProblems;
        Result<T> best;
        int best_p;
        if constexpr (MASKED) {
            // spare lanes of a ragged tile shadow the last problem, as their rows do (RowTile::acquire)
            PtsMasked<PtsRow<T> > pts;
            pts.row = tile_buf.acquire(lane, valid);
            pts.idx = sel ? sIdx : nullptr;
            pts.words = a.vis + (size_t)(b0 + (lane < valid ? lane : valid - 1)) * a.vis_words;
            pts.nvis = count_visible(pts.words, pts.idx, a.n);
            T* myC = sC + (size_t)lane * a.n_patterns * PNP_PATC;
            if (method_uses_patc(METHOD))
                for (int p = 0; p < a.n_patterns; ++p) pattern_constants_masked<T, 1>(pts, sP + (size_t)p * a.n * 3, a.n, myC + p * PNP_PATC, 0);
            solve_all_patterns<T, METHOD, 1, PtsMasked<PtsRow<T> > >(pts, sP, myC, a.n, a.n_patterns, 0, a.prm, best, best_p);
            if (pts.nvis < kMinVisible) too_few_landmarks<T>(best, best_p);
        } else {
            PtsRow<T> pts;
            pts.row = tile_buf.acquire(lane, valid);
            pts.idx = sel ? sIdx : nullptr;
            solve_all_patterns<T, METHOD, 1, PtsRow<T> >(pts, sP, sC, a.n, a.n_patterns, 0, a.prm, best, best_p);
        }
        const long long b = b0 + lane;
        if (b < a.B) write_result<T>(a, b, best, best_p);
        tile += gridDim.x;
        if (tile < n_tiles) {
            tile_buf.release();
            valid = tile_buf.issue(tile, lane);
        }
    }
}

// ------------------------------------------------------------------------------------------
// moment mapping (LM and linear F2, one pattern): three streaming kernels
//   k_moments_*   uv -> 29 moments per problem            (HBM-bound: reads every pixel once)
//   k_iterate     moments -> pose, one problem per thread (FP64 pipe; no shared-memory residency,
//                 so occupancy is bounded by registers only)
//   k_residual_*  uv + state before the last update -> res_norm, point by point (HBM-bound)
// Workspace (stream-ordered allocation): mom [PNP_NMOM][B], tail [PNP_NTAIL][B], patc [PNP_PATC].
// ------------------------------------------------------------------------------------------

template <typename T>
struct MomArgs {
    const T* uv; const T* pattern; const int32_t* idx;
    int idx_mode;
    int32_t idx_inline[PNP_MAX_INLINE_IDX];
    long long B;            // problems of this launch (a slice of the call's batch)
    long long ld;           // leading dimension of the SoA workspace arrays mom / tail (problems of the whole call)
    int n_total, n, row_pitch, use_tma;
    double kinv[6];
    SolverPrm<T> prm;
    T* mom; T* tail; T* patc;
    T* R; T* t; T* euler; T* res;
    int32_t* iters; int32_t* best;
    int fix_warp_max;       // filters: up to this many marked tiles the fix-up runs one problem per WARP (latency), above per thread
    int32_t* fix_list;      // filters: [0] = number of 32-problem tiles with a marked problem, [1..] = those tiles (k_iterate appends)
    int use_tmap;
    alignas(64) CUtensorMap tmap;   // uv of this launch as a 2-D tensor (RowStream), valid when use_tmap
    // masked kernels: [B, vis_words] visibility bits, and the per-problem pattern moments [kPatternMoments][ld] in the workspace
    const uint32_t* vis; int vis_words;
    T* pmom;
};

template <typename T>
__global__ void __launch_bounds__(32) k_pattern_constants(const __grid_constant__ MomArgs<T> a)
{
    // one warp; reads the (selected) pattern straight from global memory
    const int lane = threadIdx.x;
    const T* __restrict__ pattern = a.pattern;
    const int32_t* idx = selection_of(a);
    const int n = a.n;
    T* patc = a.patc;
    double acc[9];
#pragma unroll
    for (int e = 0; e < 9; ++e) acc[e] = 0.0;
    for (int i = lane; i < n; i += 32) {
        const int j = idx ? idx[i] : i;
        const double th[3] = { (double)pattern[3 * j], (double)pattern[3 * j + 1], (double)pattern[3 * j + 2] };
#pragma unroll
        for (int a = 0; a < 3; ++a) {
#pragma unroll
            for (int b = a; b < 3; ++b) acc[s3(a, b)] = fma(th[a], th[b], acc[s3(a, b)]);
            acc[6 + a] += th[a];
        }
    }
#pragma unroll
    for (int e = 0; e < 9; ++e) acc[e] = group_sum<32, double>(acc[e]);
    if (lane == 0) {
        double G[10];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
#pragma unroll
            for (int b = a; b < 3; ++b) G[sidx<4>(a, b)] = acc[s3(a, b)];
            G[sidx<4>(a, 3)] = acc[6 + a];
        }
        G[sidx<4>(3, 3)] = (double)n;
        spd_inverse<double, 4>(G);
#pragma unroll
        for (int e = 0; e < 9; ++e) patc[e] = (T)acc[e];
        patc[9] = (T)n;
#pragma unroll
        for (int e = 0; e < 10; ++e) patc[10 + e] = (T)G[e];
    }
}

// PASS 0: moments.  PASS 1: residual at the stored state (LM: x before the last update; F2: tail).
// MASKED: over each problem's visible landmarks; PASS 0 also stores the problem's pattern moments (a.pmom).
template <typename T, int METHOD, int PASS, bool MASKED = false>
__global__ void __launch_bounds__(32) k_stream_thread(const __grid_constant__ MomArgs<T> a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    T* sRows = reinterpret_cast<T*>(smem_raw);
    T* sP = sRows + (size_t)kTileProblems * a.row_pitch;
    int32_t* sIdx = reinterpret_cast<int32_t*>(sP + (size_t)a.n * 3);
    const int lane = threadIdx.x;
    const int32_t* sel = selection_of(a);
    RowTile<T> tile_buf;
    tile_buf.init(sRows, carve_bar<T>(smem_raw, sIdx + (sel ? a.n : 0)), a.uv, a.B, a.n_total, a.row_pitch, a.use_tma, a.kinv, lane);
    const long long n_tiles = (a.B + kTileProblems - 1) / kTileProblems;
    long long tile = blockIdx.x;
    int valid = (tile < n_tiles) ? tile_buf.issue(tile, lane) : 0;
    load_pattern<T>(a.pattern, sel, a.n_total, a.n, 1, sP, sIdx, lane, 32);
    while (tile < n_tiles) {
        const long long b0 = tile * kTileProblems;
        long long b = b0 + lane;
        const bool ok = b < a.B;
        if (!ok) b = a.B - 1;
        T st[PNP_NTAIL];
        if (PASS == 1) {                                  // issue the state loads before waiting on the tile
#pragma unroll
            for (int k = 0; k < PNP_NTAIL; ++k) st[k] = a.tail[(size_t)k * a.ld + b];
        }
        PtsRow<T> pts;
        pts.row = tile_buf.acquire(lane, valid);
        pts.idx = sel ? sIdx : nullptr;
        if constexpr (MASKED) {
            PtsMasked<PtsRow<T> > pm;
            static_cast<PtsRow<T>&>(pm) = pts;
            pm.words = a.vis + (size_t)b * a.vis_words;
            pm.nvis = count_visible(pm.words, pm.idx, a.n);
            if (PASS == 0) {
                Moments<T> mom;
                accumulate_moments<T, 1, PtsMasked<PtsRow<T> >, method_with_w(METHOD), method_with_s(METHOD)>(pm, sP, a.n, 0, mom);
                double pmo[kPatternMoments];
                pattern_moments_masked<T, 1>(pm, sP, a.n, 0, pmo);
                if (ok) {
#pragma unroll
                    for (int k = 0; k < method_nmom(METHOD); ++k) a.mom[(size_t)k * a.ld + b] = mom.at(k);
#pragma unroll
                    for (int k = 0; k < kPatternMoments; ++k) a.pmom[(size_t)k * a.ld + b] = (T)pmo[k];
                }
            } else {
                T res;
                if (method_lm_residual(METHOD)) {
                    T x[12];
#pragma unroll
                    for (int k = 0; k < 12; ++k) x[k] = st[k];
                    res = lm_residual_direct<T, 1, PtsMasked<PtsRow<T> > >(pm, sP, a.n, 0, x);
                } else {
                    F2Tail<T> f;
#pragma unroll
                    for (int k = 0; k < 3; ++k) f.phi3[k] = st[k];
#pragma unroll
                    for (int k = 0; k < 4; ++k) { f.pxn[k] = st[3 + k]; f.pyn[k] = st[7 + k]; }
                    res = f2_residual_direct<T, 1, PtsMasked<PtsRow<T> > >(pm, sP, a.n, 0, f);
                }
                if (pm.nvis < kMinVisible) res = nan_of<T>();     // not solved (a sum over no landmark would read 0)
                if (ok && a.res) a.res[b] = res;
            }
        } else if (PASS == 0) {
            Moments<T> mom;
            accumulate_moments<T, 1, PtsRow<T>, method_with_w(METHOD), method_with_s(METHOD)>(pts, sP, a.n, 0, mom);
            if (ok) {
#pragma unroll
                for (int k = 0; k < method_nmom(METHOD); ++k) a.mom[(size_t)k * a.ld + b] = mom.at(k);
            }
        } else {
            T res;
            if (method_lm_residual(METHOD)) {
                T x[12];
#pragma unroll
                for (int k = 0; k < 12; ++k) x[k] = st[k];
                res = lm_residual_direct<T, 1, PtsRow<T> >(pts, sP, a.n, 0, x);
            } else {
                F2Tail<T> f;
#pragma unroll
                for (int k = 0; k < 3; ++k) f.phi3[k] = st[k];
#pragma unroll
                for (int k = 0; k < 4; ++k) { f.pxn[k] = st[3 + k]; f.pyn[k] = st[7 + k]; }
                res = f2_residual_direct<T, 1, PtsRow<T> >(pts, sP, a.n, 0, f);
            }
            if (ok && a.res) a.res[b] = res;
        }
        tile += gridDim.x;
        if (tile < n_tiles) {
            tile_buf.release();
            valid = tile_buf.issue(tile, lane);
        }
    }
}

// Streaming variant of k_stream_thread (all landmarks, rows a multiple of 16 bytes): chunks of the
// rows go through two small buffers (RowStream), K^-1 is applied on the fly.
#ifndef PNP_STREAM_UNROLL
#define PNP_STREAM_UNROLL 2       // points in flight per thread in the chunk-streaming passes
#endif
constexpr int kStreamUnroll = PNP_STREAM_UNROLL;
// MASKED: over each problem's visible landmarks (a running mask word per chunk); PASS 0 also stores the pattern moments
template <typename T, int METHOD, int PASS, bool MASKED = false>
__global__ void __launch_bounds__(32) k_stream_chunk(const __grid_constant__ MomArgs<T> a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    typedef typename Vec2<T>::type V2;
    T* sBuf = reinterpret_cast<T*>(smem_raw);
    T* sP = sBuf + (size_t)2 * kTileProblems * a.row_pitch;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + ((((size_t)((unsigned char*)(sP + (size_t)a.n * 3) - smem_raw)) + 7) & ~(size_t)7));
    const int lane = threadIdx.x;
    RowStream<T> rs;
    rs.init(sBuf, bars, a.uv, a.B, a.n_total, a.use_tma /* chunk */, a.row_pitch, lane, a.use_tmap ? &a.tmap : nullptr);
    const long long n_tiles = (a.B + kTileProblems - 1) / kTileProblems;
    long long tile = blockIdx.x;
    if (tile < n_tiles) rs.begin_tile(tile, lane);
    for (int e = lane; e < a.n * 3; e += 32) sP[e] = a.pattern[e];
    __syncwarp();
    const T k00 = (T)a.kinv[0], k01 = (T)a.kinv[1], k02 = (T)a.kinv[2];
    const T k10 = (T)a.kinv[3], k11 = (T)a.kinv[4], k12 = (T)a.kinv[5];
    while (tile < n_tiles) {
        long long b = tile * kTileProblems + lane;
        const bool ok = b < a.B;
        if (!ok) b = a.B - 1;
        Moments<T> mom;
        LmResidualState<T> lr;
        F2Tail<T> f;
        T acc0 = T(0), acc1 = T(0);
        if (PASS == 0) mom.zero();
        else {
            T st[PNP_NTAIL];
#pragma unroll
            for (int k = 0; k < PNP_NTAIL; ++k) st[k] = a.tail[(size_t)k * a.ld + b];
            if (method_lm_residual(METHOD)) {
                lr.load(st);
            } else {
#pragma unroll
                for (int k = 0; k < 3; ++k) f.phi3[k] = st[k];
#pragma unroll
                for (int k = 0; k < 4; ++k) { f.pxn[k] = st[3 + k]; f.pyn[k] = st[7 + k]; }
            }
        }
        const uint32_t* vw = MASKED ? a.vis + (size_t)b * a.vis_words : nullptr;
        double pmo[kPatternMoments];
        if constexpr (MASKED && PASS == 0) {
#pragma unroll
            for (int e = 0; e < kPatternMoments; ++e) pmo[e] = 0.0;
        }
        for (int c = 0; c < rs.n_chunks; ++c) {
            const V2* row = rs.wait(c, lane);
            const int cnt = rs.count(c), i0 = c * rs.chunk;
            uint32_t word = 0;                                // MASKED: bit 0 = landmark i0 + k
            if constexpr (MASKED) word = __ldg(vw + (i0 >> 5)) >> (i0 & 31);
#pragma unroll kStreamUnroll
            for (int k = 0; k < cnt; ++k) {
                if constexpr (MASKED) {
                    const int i = i0 + k;
                    const bool v = word & 1u;
                    word = ((i + 1) & 31) ? (word >> 1) : ((i + 1 < a.n) ? __ldg(vw + ((i + 1) >> 5)) : 0u);
                    if (!v) continue;
                }
                const V2 px = row[k];
                T bx, by;                                     // nu = K^-1 [u, v, 1]^T (:3305)
                normalise_px<T>(px.x, px.y, k00, k01, k02, k10, k11, k12, bx, by);
                const T th[3] = { sP[3 * (i0 + k)], sP[3 * (i0 + k) + 1], sP[3 * (i0 + k) + 2] };
                if constexpr (MASKED && PASS == 0) {
#pragma unroll
                    for (int p = 0; p < 3; ++p) {
#pragma unroll
                        for (int q = p; q < 3; ++q) pmo[s3(p, q)] = fma((double)th[p], (double)th[q], pmo[s3(p, q)]);
                        pmo[6 + p] += (double)th[p];
                    }
                    pmo[9] += 1.0;
                }
                if (PASS == 0) {
                    mom.template add<method_with_w(METHOD), method_with_s(METHOD)>(th, bx, by);
                } else if (method_lm_residual(METHOD)) {
                    lr.add(th, bx, by, acc0);                 // z - hx (:3750, :2679)
                } else {
                    const T db = T(1) + (th[0] * f.phi3[0] + th[1] * f.phi3[1] + th[2] * f.phi3[2]);
                    const T dx = th[0] * f.pxn[0] + th[1] * f.pxn[1] + th[2] * f.pxn[2] + f.pxn[3];
                    const T dy = th[0] * f.pyn[0] + th[1] * f.pyn[1] + th[2] * f.pyn[2] + f.pyn[3];
                    const T ex = bx * db - dx, ey = by * db - dy;
                    acc0 = t_fma(ex, ex, acc0); acc1 = t_fma(ey, ey, acc1);
                }
            }
            rs.done(c, lane);
        }
        if (ok) {
            if (PASS == 0) {
#pragma unroll
                for (int k = 0; k < method_nmom(METHOD); ++k) a.mom[(size_t)k * a.ld + b] = mom.at(k);
                if constexpr (MASKED) {
#pragma unroll
                    for (int k = 0; k < kPatternMoments; ++k) a.pmom[(size_t)k * a.ld + b] = (T)pmo[k];
                }
            } else if (a.res) {
                if (method_lm_residual(METHOD)) a.res[b] = t_sqrt(acc0);   // :2681
                else { const T nx = t_sqrt(acc0), ny = t_sqrt(acc1); a.res[b] = t_sqrt(nx * nx + ny * ny); }   // :3374
                if constexpr (MASKED) {
                    if (count_visible(vw, nullptr, a.n) < kMinVisible) a.res[b] = nan_of<T>();   // not solved
                }
            }
        }
        tile += gridDim.x;
        if (tile < n_tiles) {
            fence_proxy_async();
            rs.begin_tile(tile, lane);
        }
    }
}

// MASKED: over each problem's visible landmarks; PASS 0 also stores the pattern moments
template <typename T, int METHOD, int PASS, bool MASKED = false>
__global__ void __launch_bounds__(256) k_stream_warp(const __grid_constant__ MomArgs<T> a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    T* sP = reinterpret_cast<T*>(smem_raw);
    int32_t* sIdx = reinterpret_cast<int32_t*>(sP + (size_t)a.n * 3);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int32_t* sel = selection_of(a);
    load_pattern<T>(a.pattern, sel, a.n_total, a.n, 1, sP, sIdx, threadIdx.x, blockDim.x);
    PtsGlobal<T> pts;
    pts.idx = sel ? sIdx : nullptr;
    pts.k00 = (T)a.kinv[0]; pts.k01 = (T)a.kinv[1]; pts.k02 = (T)a.kinv[2];
    pts.k10 = (T)a.kinv[3]; pts.k11 = (T)a.kinv[4]; pts.k12 = (T)a.kinv[5];
    for (long long b = (long long)blockIdx.x * nwarps + warp; b < a.B; b += (long long)gridDim.x * nwarps) {
        pts.row = a.uv + (size_t)b * a.n_total * 2;
        if constexpr (MASKED) {
            PtsMasked<PtsGlobal<T> > pm;
            static_cast<PtsGlobal<T>&>(pm) = pts;
            pm.words = a.vis + (size_t)b * a.vis_words;
            pm.nvis = count_visible(pm.words, pm.idx, a.n);
            if (PASS == 0) {
                Moments<T> mom;
                accumulate_moments<T, 32, PtsMasked<PtsGlobal<T> >, method_with_w(METHOD), method_with_s(METHOD)>(pm, sP, a.n, lane, mom);
                double pmo[kPatternMoments];
                pattern_moments_masked<T, 32>(pm, sP, a.n, lane, pmo);
                T mine = T(0);
#pragma unroll
                for (int k = 0; k < method_nmom(METHOD); ++k) if (lane == k) mine = mom.at(k);
                if (lane < method_nmom(METHOD)) a.mom[(size_t)lane * a.ld + b] = mine;
                double pmine = 0.0;
#pragma unroll
                for (int k = 0; k < kPatternMoments; ++k) if (lane == k) pmine = pmo[k];
                if (lane < kPatternMoments) a.pmom[(size_t)lane * a.ld + b] = (T)pmine;
            } else {
                T res;
                if (method_lm_residual(METHOD)) {
                    T x[12];
#pragma unroll
                    for (int k = 0; k < 12; ++k) x[k] = a.tail[(size_t)k * a.ld + b];
                    res = lm_residual_direct<T, 32, PtsMasked<PtsGlobal<T> > >(pm, sP, a.n, lane, x);
                } else {
                    F2Tail<T> f;
#pragma unroll
                    for (int k = 0; k < 3; ++k) f.phi3[k] = a.tail[(size_t)k * a.ld + b];
#pragma unroll
                    for (int k = 0; k < 4; ++k) { f.pxn[k] = a.tail[(size_t)(3 + k) * a.ld + b]; f.pyn[k] = a.tail[(size_t)(7 + k) * a.ld + b]; }
                    res = f2_residual_direct<T, 32, PtsMasked<PtsGlobal<T> > >(pm, sP, a.n, lane, f);
                }
                if (pm.nvis < kMinVisible) res = nan_of<T>();     // not solved (a sum over no landmark would read 0)
                if (lane == 0 && a.res) a.res[b] = res;
            }
            continue;
        }
        if (PASS == 0) {
            Moments<T> mom;
            accumulate_moments<T, 32, PtsGlobal<T>, method_with_w(METHOD), method_with_s(METHOD)>(pts, sP, a.n, lane, mom);
            // after the butterfly every lane holds every sum: lane k writes moment k
            T mine = T(0);
#pragma unroll
            for (int k = 0; k < method_nmom(METHOD); ++k) if (lane == k) mine = mom.at(k);
            if (lane < method_nmom(METHOD)) a.mom[(size_t)lane * a.ld + b] = mine;
        } else {
            T res;
            if (method_lm_residual(METHOD)) {
                T x[12];
#pragma unroll
                for (int k = 0; k < 12; ++k) x[k] = a.tail[(size_t)k * a.ld + b];
                res = lm_residual_direct<T, 32, PtsGlobal<T> >(pts, sP, a.n, lane, x);
            } else {
                F2Tail<T> f;
#pragma unroll
                for (int k = 0; k < 3; ++k) f.phi3[k] = a.tail[(size_t)k * a.ld + b];
#pragma unroll
                for (int k = 0; k < 4; ++k) { f.pxn[k] = a.tail[(size_t)(3 + k) * a.ld + b]; f.pyn[k] = a.tail[(size_t)(7 + k) * a.ld + b]; }
                res = f2_residual_direct<T, 32, PtsGlobal<T> >(pts, sP, a.n, lane, f);
            }
            if (lane == 0 && a.res) a.res[b] = res;
        }
    }
}


// ------------------------------------------------------------------------------------------
// One problem per warp for large n, rows staged by TMA bulk copies: each warp streams its problems'
// rows through a ring of kRingSlots shared-memory slots of kRingPoints points (one cp.async.bulk per
// slot, issued by lane 0, completion on the slot's mbarrier), kRingSlots - 1 copies ahead of the
// arithmetic and straight across problem boundaries, so that the bytes in flight per SM do not
// depend on registers or on the unroll depth of a load loop (the __ldg version reached 50-60 % of
// the HBM peak on 100 k x 1024 points).  Lanes read consecutive 16-byte pixels: conflict-free.  The
// pattern (24 KB for 1024 points) is read through L1 instead of taking shared memory from the ring.
// Requires all landmarks (no selection) and rows that are a multiple of 16 bytes.
// ------------------------------------------------------------------------------------------
// Sum v[k] over the 32 lanes of a warp so that lane k ends up with the total of v[k] in v[0] (k < N; N <= 32 values, the rest
// structurally zero): five halving steps -- at offset h a lane keeps the half of the index range that contains its own index
// and receives the partner's partial sums of that half -- 31 shuffled values and 31 additions instead of the 32 x 5 of a
// butterfly that leaves every sum in every lane.
template <typename T, int N>
PNP_DEV void warp_reduce_scatter(T (&v)[32], int lane)
{
#pragma unroll
    for (int h = 16; h >= 1; h >>= 1) {
        const bool hi = (lane & h) != 0;
#pragma unroll
        for (int i = 0; i < h; ++i) {
            if (h < 16 || i + h < N) {
                const T send = hi ? v[i] : v[i + h];
                const T keep = hi ? v[i + h] : v[i];
                v[i] = keep + __shfl_xor_sync(0xffffffffu, send, h);
            } else {
                v[i] += __shfl_xor_sync(0xffffffffu, v[i], h);   // the upper half does not exist: only the lower lanes' sums matter
            }
        }
    }
}

// Fixed shape.  (Other shapes were tried on 100 k x 1024 points, tools/build_variant.py: 3 slots x 128 points 0.57 ms, 16 warps
// per CTA 0.39 ms against 0.42 ms for this one.  2 x 256, 4 x 128 and 6 x 128 faulted with an illegal address on about half of
// the FIRST launches of a process and never on a later one, in the round-1 form of this kernel as well.  Bisected on the GPU,
// profiles/r02u_ring_fault_bisect.md: the fault survives staging with plain loads instead of TMA, dropping the pattern reads or
// the moment stores, moving or invalidating the barriers, zero-filling the slots, a block-wide barrier after the initialisation,
// eager module loading and a maximal shared-memory carve-out; it disappears when ANY 256-thread kernel of this translation
// unit has run before.  No access of the kernel is out of range under its own logic, so the cause is not in this source; this
// shape ran 100 of 100 first launches (tools/first_launch_soak.py) and every test / bench / soak process clean; the others are not offered.)
constexpr int kRingSlots = 3;
constexpr int kRingPoints = 256;          // 4 KB per slot in FP64: 8 points per lane between two barrier waits
constexpr int kRingWarps = 8;

template <typename T, int METHOD, int PASS>
__global__ void __launch_bounds__(kRingWarps * 32) k_stream_warp_tma(const __grid_constant__ MomArgs<T> a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    typedef typename Vec2<T>::type V2;
    T* sRing = reinterpret_cast<T*>(smem_raw);                                 // [warp][slot][kRingPoints][2]
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + (size_t)kRingWarps * kRingSlots * kRingPoints * 2 * sizeof(T));
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const T* __restrict__ gP = a.pattern;
    T* ring = sRing + (size_t)warp * kRingSlots * kRingPoints * 2;
    uint64_t* bar = bars + warp * kRingSlots;
    if (lane == 0)
        for (int k = 0; k < kRingSlots; ++k) mbar_init(bar + k, 1);
    __syncwarp();
    const T k00 = (T)a.kinv[0], k01 = (T)a.kinv[1], k02 = (T)a.kinv[2];
    const T k10 = (T)a.kinv[3], k11 = (T)a.kinv[4], k12 = (T)a.kinv[5];
    const int n = a.n, cpp = (n + kRingPoints - 1) / kRingPoints;            // chunks per problem
    const long long w0 = (long long)blockIdx.x * kRingWarps + warp, wstride = (long long)gridDim.x * kRingWarps;
    const long long my_problems = (w0 < a.B) ? (a.B - w0 + wstride - 1) / wstride : 0;
    const long long total = my_problems * cpp;                                // chunks this warp will consume
    // The copy stream runs kRingSlots - 1 chunks ahead of the arithmetic, straight across problem boundaries: chunk g of
    // this warp = chunk (g % cpp) of problem w0 + (g / cpp) * wstride, kept as running (row pointer, chunk, slot) instead
    // of 64-bit divisions per chunk.
    const T* irow = a.uv + (size_t)w0 * n * 2;                               // row of the problem whose chunks are being issued
    const size_t irow_step = (size_t)wstride * n * 2;
    int ic = 0, islot = 0;
    long long issued = 0;
    auto issue_next = [&]() {
        if (lane == 0) {
            const int cnt = (n - ic * kRingPoints < kRingPoints) ? (n - ic * kRingPoints) : kRingPoints;
            const uint32_t bytes = (uint32_t)cnt * 2u * (uint32_t)sizeof(T);
            mbar_expect_tx(bar + islot, bytes);
            bulk_copy_g2s(ring + (size_t)islot * kRingPoints * 2, irow + (size_t)ic * kRingPoints * 2, bytes, bar + islot);
        }
        ++issued;
        if (++ic == cpp) { ic = 0; irow += irow_step; }
        if (++islot == kRingSlots) islot = 0;
    };
    for (int k = 0; k < kRingSlots - 1 && issued < total; ++k) issue_next();
    uint32_t phase = 0;                                                      // bit s = parity to wait for on slot s
    int slot = 0;
    for (long long p = 0; p < my_problems; ++p) {
        const long long b = w0 + p * wstride;
        Moments<T> mom;
        T st[PNP_NTAIL];
        LmResidualState<T> lr;
        T acc0 = T(0), acc1 = T(0);
        if (PASS == 0) mom.zero();
        else {
#pragma unroll
            for (int k = 0; k < PNP_NTAIL; ++k) st[k] = a.tail[(size_t)k * a.ld + b];
            if (method_lm_residual(METHOD)) lr.load(st);
        }
        for (int c = 0; c < cpp; ++c) {
            // refill the slot that was consumed one step ago, then wait for this one
            if (issued < total) {
                __syncwarp();
                fence_proxy_async();
                issue_next();
            }
            mbar_wait(bar + slot, (phase >> slot) & 1u);
            phase ^= (1u << slot);
            const V2* row = reinterpret_cast<const V2*>(ring + (size_t)slot * kRingPoints * 2) + lane;
            const int cnt = (n - c * kRingPoints < kRingPoints) ? (n - c * kRingPoints) : kRingPoints;
            const T* __restrict__ gPl = gP + 3 * (c * kRingPoints + lane);
            // a full slot is kRingPoints / 32 points per lane at compile-time offsets (no loop counter, no bounds test)
            const int per_lane = (cnt == kRingPoints) ? kRingPoints / 32 : (cnt - lane + 31) / 32;
            auto point = [&](int j) {
                const V2 px = row[32 * j];
                T bx, by;                                                     // nu = K^-1 [u, v, 1]^T (:3305)
                normalise_px<T>(px.x, px.y, k00, k01, k02, k10, k11, k12, bx, by);
                const T th[3] = { __ldg(gPl + 96 * j), __ldg(gPl + 96 * j + 1), __ldg(gPl + 96 * j + 2) };
                if (PASS == 0) {
                    mom.template add<method_with_w(METHOD), method_with_s(METHOD)>(th, bx, by);
                } else if (method_lm_residual(METHOD)) {
                    lr.add(th, bx, by, acc0);                                 // z - hx (:3750, :2679)
                } else {
                    const T db = T(1) + (th[0] * st[0] + th[1] * st[1] + th[2] * st[2]);
                    const T dx = th[0] * st[3] + th[1] * st[4] + th[2] * st[5] + st[6];
                    const T dy = th[0] * st[7] + th[1] * st[8] + th[2] * st[9] + st[10];
                    const T ex = bx * db - dx, ey = by * db - dy;
                    acc0 = t_fma(ex, ex, acc0); acc1 = t_fma(ey, ey, acc1);
                }
            };
            if (cnt == kRingPoints) {
#pragma unroll
                for (int j = 0; j < kRingPoints / 32; ++j) point(j);
            } else {
                for (int j = 0; j < per_lane; ++j) point(j);
            }
            if (++slot == kRingSlots) slot = 0;
        }
        if (PASS == 0) {
            T v[32];                                                          // lane k leaves with the total of moment k
#pragma unroll
            for (int k = 0; k < 32; ++k) v[k] = (k < method_nmom(METHOD)) ? mom.at(k) : T(0);
            warp_reduce_scatter<T, method_nmom(METHOD)>(v, lane);
            if (lane < method_nmom(METHOD)) a.mom[(size_t)lane * a.ld + b] = v[0];
        } else {
            acc0 = group_sum<32>(acc0); acc1 = group_sum<32>(acc1);
            if (lane == 0 && a.res) {
                if (method_lm_residual(METHOD)) a.res[b] = t_sqrt(acc0);   // :2681
                else { const T nx = t_sqrt(acc0), ny = t_sqrt(acc1); a.res[b] = t_sqrt(nx * nx + ny * ny); }   // :3374
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// Fix-up pass of the filters' moment mapping.  k_iterate takes the early-exit decisions of QEIF / EIF2 from the moment form of
// the residual and certifies each of them against the rounding error of that form (exit_decision_uncertain); a problem with a
// decision it cannot certify leaves k_iterate marked (iters = -1).  These kernels re-solve the marked problems with the direct
// mappings' arithmetic -- residual point by point in every iteration, the reference's decisions exactly -- and overwrite their
// pose, iteration count and the state the residual pass (or the fused report) evaluates res_norm at.  A tile / warp whose
// problems are all unmarked reads 32 / 1 flags and leaves.
// ------------------------------------------------------------------------------------------
template <typename T> __device__ __forceinline__ void write_pose(const MomArgs<T>& a, long long b, const Result<T>& out);
constexpr int kWarpsPerFixup = 8;                             // k_fixup_warp: 256 threads

template <typename T, int METHOD, int LPP, typename Pts>
PNP_DEV void run_filter_with_tail(const Pts& pts, const T* sP, const T* sC, int n, int sub, const SolverPrm<T>& prm, T (&xt)[12],
                                  Result<T>& out)
{
    if (METHOD == PNP_METHOD_QEIF_HYBRID) solve_qeif_with_tail<T, LPP, Pts>(pts, sP, sC, n, sub, prm, xt, out);
    else                                  solve_eif2_with_tail<T, LPP, Pts>(pts, sP, sC, n, sub, prm, xt, out);
}

// MASKED: each lane solves on its problem's visible landmarks with its own constants
template <typename T, int METHOD, bool MASKED = false>
__global__ void __launch_bounds__(32) k_fixup_thread(const __grid_constant__ MomArgs<T> a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    T* sRows = reinterpret_cast<T*>(smem_raw);
    T* sP = sRows + (size_t)kTileProblems * a.row_pitch;
    T* sC = sP + (size_t)a.n * 3;
    int32_t* sIdx = reinterpret_cast<int32_t*>(sC + (MASKED ? kTileProblems : 1) * PNP_PATC);
    const int lane = threadIdx.x;
    const int32_t* sel = selection_of(a);
    const int n_marked = a.fix_list[0];                       // (complete: k_iterate has finished)
    if (n_marked <= a.fix_warp_max) return;                   // few marked tiles: k_fixup_warp takes them
    bool staged = false;
    RowTile<T> tile_buf;
    for (int i = blockIdx.x; i < n_marked; i += gridDim.x) {
        const long long tile = a.fix_list[1 + i];
        const long long b = tile * kTileProblems + lane;
        const bool marked = (b < a.B) && (a.iters[b] < 0);
        if (!staged) {                                        // first marked tile of this CTA: pattern, constants, barrier
            tile_buf.init(sRows, carve_bar<T>(smem_raw, sIdx + (sel ? a.n : 0)), a.uv, a.B, a.n_total, a.row_pitch, a.use_tma, a.kinv, lane);
            load_pattern<T>(a.pattern, sel, a.n_total, a.n, 1, sP, sIdx, lane, 32);
            if (!MASKED) pattern_constants<T>(sP, a.n, sC, lane);
            __syncwarp();
            staged = true;
        } else {
            tile_buf.release();
        }
        const int valid = tile_buf.issue(tile, lane);
        PtsRow<T> pts;
        pts.row = tile_buf.acquire(lane, valid);
        pts.idx = sel ? sIdx : nullptr;
        Result<T> out;
        T xt[12];
        if constexpr (MASKED) {
            PtsMasked<PtsRow<T> > pm;
            static_cast<PtsRow<T>&>(pm) = pts;
            pm.words = a.vis + (size_t)(tile * kTileProblems + (lane < valid ? lane : valid - 1)) * a.vis_words;
            pm.nvis = count_visible(pm.words, pm.idx, a.n);
            T* myC = sC + (size_t)lane * PNP_PATC;
            pattern_constants_masked<T, 1>(pm, sP, a.n, myC, 0);
            run_filter_with_tail<T, METHOD, 1, PtsMasked<PtsRow<T> > >(pm, sP, myC, a.n, 0, a.prm, xt, out);
        } else {
            run_filter_with_tail<T, METHOD, 1, PtsRow<T> >(pts, sP, sC, a.n, 0, a.prm, xt, out);
        }
        if (marked) {
#pragma unroll
            for (int k = 0; k < PNP_NTAIL; ++k) a.tail[(size_t)k * a.ld + b] = xt[k];
            write_pose<T>(a, b, out);
        }
    }
}

// MASKED: each warp solves on its problem's visible landmarks with the problem's constants
template <typename T, int METHOD, bool MASKED = false>
__global__ void __launch_bounds__(256) k_fixup_warp(const __grid_constant__ MomArgs<T> a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    T* sP = reinterpret_cast<T*>(smem_raw);
    T* sC = sP + (size_t)a.n * 3;
    int32_t* sIdx = reinterpret_cast<int32_t*>(sC + (MASKED ? kWarpsPerFixup : 1) * PNP_PATC);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int32_t* sel = selection_of(a);
    const int n_marked = a.fix_list[0];                       // marked tiles (complete: k_iterate has finished)
    if ((int)blockIdx.x >= n_marked || n_marked > a.fix_warp_max) return;   // CTA i takes the marked tiles i, i + gridDim.x, ...; many: k_fixup_thread
    load_pattern<T>(a.pattern, sel, a.n_total, a.n, 1, sP, sIdx, threadIdx.x, blockDim.x);
    if (!MASKED && warp == 0) pattern_constants<T>(sP, a.n, sC, lane);
    __syncthreads();
    PtsGlobal<T> pts;
    pts.idx = sel ? sIdx : nullptr;
    pts.k00 = (T)a.kinv[0]; pts.k01 = (T)a.kinv[1]; pts.k02 = (T)a.kinv[2];
    pts.k10 = (T)a.kinv[3]; pts.k11 = (T)a.kinv[4]; pts.k12 = (T)a.kinv[5];
    for (long long w = (long long)blockIdx.x * kTileProblems + warp; w < (long long)n_marked * kTileProblems;
         w = ((w % kTileProblems) + nwarps < kTileProblems) ? w + nwarps : (w / kTileProblems + gridDim.x) * kTileProblems + warp) {
        // warp-item w = problem (w % 32) of the marked tile (w / 32): a CTA takes whole tiles, its warps the problems of each
        const long long b = (long long)a.fix_list[1 + (int)(w / kTileProblems)] * kTileProblems + (w % kTileProblems);
        if (b >= a.B || a.iters[b] >= 0) continue;
        pts.row = a.uv + (size_t)b * a.n_total * 2;
        Result<T> out;
        T xt[12];
        if constexpr (MASKED) {
            PtsMasked<PtsGlobal<T> > pm;
            static_cast<PtsGlobal<T>&>(pm) = pts;
            pm.words = a.vis + (size_t)b * a.vis_words;
            pm.nvis = count_visible(pm.words, pm.idx, a.n);
            T* myC = sC + (size_t)warp * PNP_PATC;
            pattern_constants_masked<T, 32>(pm, sP, a.n, myC, lane);
            __syncwarp();
            run_filter_with_tail<T, METHOD, 32, PtsMasked<PtsGlobal<T> > >(pm, sP, myC, a.n, lane, a.prm, xt, out);
            __syncwarp();                                     // the next problem's constants replace these
        } else {
            run_filter_with_tail<T, METHOD, 32, PtsGlobal<T> >(pts, sP, sC, a.n, lane, a.prm, xt, out);
        }
        if (lane == 0) {
#pragma unroll
            for (int k = 0; k < PNP_NTAIL; ++k) a.tail[(size_t)k * a.ld + b] = xt[k];
            write_pose<T>(a, b, out);
        }
    }
}

// The O(1)-per-iteration part of the moment mapping for one problem per thread: moments parked in shared
// memory ([PNP_NMOM][stride] columns, this thread's column at sMomCol) -> pose `out` and the 12 numbers the
// residual pass needs (LM: the state before the last update; F2: its tail).
template <typename T, int METHOD>
__device__ __forceinline__ void iterate_core(T* sMomCol, int stride, const T* sC, const SolverPrm<T>& prm,
                                             T (&st)[PNP_NTAIL], Result<T>& out)
{
    MomentsRef<T> mom;
    mom.base = sMomCol;
    mom.stride = stride;
    mom.core = sMomCol + PNP_NMOM * stride;               // [PNP_NCORE][stride] behind the moments (LM only)
    if (METHOD == PNPB200_METHOD_LM) {
        T xp[12];
        solve_lm_from_moments<T, MomentsRef<T> >(mom, sC, prm, xp, out);
#pragma unroll
        for (int k = 0; k < 12; ++k) st[k] = xp[k];
    } else if (METHOD == PNP_METHOD_LM_TRUEJAC) {
        T xp[12];
        solve_lm_from_moments<T, MomentsRef<T>, true>(mom, sC, prm, xp, out);
#pragma unroll
        for (int k = 0; k < 12; ++k) st[k] = xp[k];
    } else if (METHOD == PNP_METHOD_QEIF_HYBRID) {
        Moments<T> mr;                                        // 6 x 6 system: the moments fit in registers next to it
#pragma unroll
        for (int k = 0; k < PNP_NMOM; ++k) mr.at(k) = sMomCol[k * stride];
        T xt[12];
        solve_qeif_from_moments<T>(mr, sC, prm, xt, out);
#pragma unroll
        for (int k = 0; k < 12; ++k) st[k] = xt[k];
    } else if (METHOD == PNPB200_METHOD_EIF2) {
        T xt[12];
        solve_eif2_from_moments<T, MomentsRef<T> >(mom, sC, prm, xt, out);   // 12 x 12 system: moments stay in shared memory
#pragma unroll
        for (int k = 0; k < 12; ++k) st[k] = xt[k];
    } else if (METHOD == PNPB200_METHOD_LM_PLUS) {
        Moments<T> mr;
#pragma unroll
        for (int k = 0; k < PNP_NMOM_LM; ++k) mr.at(k) = sMomCol[k * stride];
        mr.sw0 = T(0);
        T xf[12];
        solve_lm_plus_from_moments<T, MomentsRef<T> >(mom, mr, sC, prm, xf, out);
#pragma unroll
        for (int k = 0; k < 12; ++k) st[k] = xf[k];
    } else {
        Moments<T> mr;
#pragma unroll
        for (int k = 0; k < PNP_NMOM_LM; ++k) mr.at(k) = sMomCol[k * stride];
        mr.sw0 = T(0);
        F2Tail<T> f;
        solve_f2_from_moments<T>(mr, sC, prm, f, out);
#pragma unroll
        for (int k = 0; k < 3; ++k) st[k] = f.phi3[k];
#pragma unroll
        for (int k = 0; k < 4; ++k) { st[3 + k] = f.pxn[k]; st[7 + k] = f.pyn[k]; }
        st[11] = T(0);
    }
}

template <typename T>
__device__ __forceinline__ void write_pose(const MomArgs<T>& a, long long b, const Result<T>& out)
{
    if (a.R) {
#pragma unroll
        for (int e = 0; e < 9; ++e) a.R[b * 9 + e] = out.R[e];
    }
    if (a.t) {
#pragma unroll
        for (int e = 0; e < 3; ++e) a.t[b * 3 + e] = out.t[e];
    }
    if (a.euler) {
        double Rd[9], e3[3];
#pragma unroll
        for (int e = 0; e < 9; ++e) Rd[e] = (double)out.R[e];
        euler_from_R(Rd, true, e3);
#pragma unroll
        for (int e = 0; e < 3; ++e) a.euler[b * 3 + e] = (T)e3[e];
    }
    if (a.iters) a.iters[b] = out.iters;
    if (a.best) a.best[b] = 0;
}

// MASKED: every thread builds its problem's constants from the pattern moments of the workspace (a.pmom)
template <typename T, int METHOD, int BLOCK, bool MASKED = false>
__device__ __forceinline__ void iterate_body(const MomArgs<T>& a)
{
    constexpr int kIterBlock = BLOCK;
    __shared__ T sC[PNP_PATC];
    constexpr int kRows = PNP_NMOM + (method_has_core(METHOD) ? PNP_NCORE : 0);
    __shared__ T sMom[kRows * kIterBlock];                // [moment | constant LM blocks][thread]: conflict-free columns
    if (!MASKED && threadIdx.x < PNP_PATC) sC[threadIdx.x] = a.patc[threadIdx.x];
    long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool ok = b < a.B;
    if (!ok) b = a.B - 1;
#pragma unroll
    for (int k = 0; k < method_nmom(METHOD); ++k) sMom[k * kIterBlock + threadIdx.x] = a.mom[(size_t)k * a.ld + b];
    const T* myC = sC;
    int nvis = 0;
    if constexpr (MASKED) {
        __shared__ T sCm[PNP_PATC * kIterBlock];          // [thread][constant]
        double pm[kPatternMoments];
#pragma unroll
        for (int k = 0; k < kPatternMoments; ++k) pm[k] = (double)a.pmom[(size_t)k * a.ld + b];
        constants_from_pattern_moments<T>(pm, sCm + threadIdx.x * PNP_PATC);
        myC = sCm + threadIdx.x * PNP_PATC;
        nvis = (int)pm[9];
    }
    __syncthreads();
    Result<T> out;
    T st[PNP_NTAIL];
    iterate_core<T, METHOD>(sMom + threadIdx.x, kIterBlock, myC, a.prm, st, out);
    if constexpr (MASKED) {
        if (nvis < kMinVisible) {                             // not solved: NaN pose, NaN state (so NaN res_norm), 0 iterations, unmarked
            int unused;
            too_few_landmarks<T>(out, unused);
#pragma unroll
            for (int k = 0; k < PNP_NTAIL; ++k) st[k] = out.res;
        }
    }
    if (method_with_s(METHOD) && BLOCK == 32 && a.fix_list) {    // a block is one 32-problem tile: list it if any of its problems is marked
        const bool marked = ok && out.iters < 0;
        if (__any_sync(0xffffffffu, marked) && threadIdx.x == 0) a.fix_list[1 + atomicAdd(a.fix_list, 1)] = (int32_t)blockIdx.x;
    }
    if (!ok) return;
#pragma unroll
    for (int k = 0; k < PNP_NTAIL; ++k) a.tail[(size_t)k * a.ld + b] = st[k];
    write_pose<T>(a, b, out);
}

// Register budget per thread given directly.  Warps live on one of the four sub-partitions of an SM, each with
// 16 Ki registers: 2 warps per sub-partition from 169 to 255 registers, 3 at <= 168 (FP64 LM wants ~214 and spills
// ~26 doubles at 168).  Measured for 1 Mi x 68 LM FP64 on B200 (final step): 0.886 ms at 224, 0.904 at 255 (240 used),
// 0.912 at 184, 0.905 at 168, 0.931 at 160 -- the third warp does not pay for its spills.
template <typename T, int METHOD, int BLOCK, int MAXREG, bool MASKED = false>
__global__ void __launch_bounds__(BLOCK) __maxnreg__(MAXREG) k_iterate(const __grid_constant__ MomArgs<T> a)
{
    iterate_body<T, METHOD, BLOCK, MASKED>(a);
}

template <typename T, int METHOD, int BLOCK, int MAXREG, bool MASKED = false>
static void launch_iterate_as(const MomArgs<T>& m, cudaStream_t stream)
{
    k_iterate<T, METHOD, BLOCK, MAXREG, MASKED><<<(unsigned)((m.B + BLOCK - 1) / BLOCK), BLOCK, 0, stream>>>(m); count_kernel_launches(1);
}

template <typename T, int METHOD>
static void launch_iterate(const MomArgs<T>& m, int tune, cudaStream_t stream)
{
    if (m.vis) {
        launch_iterate_as<T, METHOD, 32, (METHOD == PNPB200_METHOD_EIF2 || METHOD == PNP_METHOD_QEIF_HYBRID) ? 255 : 224, true>(m, stream);
        return;
    }
    switch (tune) {
#if PNP_TUNE_VARIANTS
    case 2:  launch_iterate_as<T, METHOD, 32, 255>(m, stream); break;    // no cap
    case 30: launch_iterate_as<T, METHOD, 64, 200>(m, stream); break;    // 10 warps / SM
    case 31: launch_iterate_as<T, METHOD, 32, 184>(m, stream); break;    // 11 warps / SM
    case 32: launch_iterate_as<T, METHOD, 32, 168>(m, stream); break;    // 3 warps per sub-partition
    case 33: launch_iterate_as<T, METHOD, 32, 160>(m, stream); break;
#endif
    default:
        // LM: 224 registers (2 warps per sub-partition, no spills); EIF2 carries a 12 x 12 matrix (156 registers) and QEIF's
        // moment form of H^T H a hundred temporaries: no cap (any cap below 255 spills: 684 bytes at 168, 1164 at 128)
        launch_iterate_as<T, METHOD, 32, (METHOD == PNPB200_METHOD_EIF2 || METHOD == PNP_METHOD_QEIF_HYBRID) ? 255 : 224>(m, stream);
        break;
    }
}

// ------------------------------------------------------------------------------------------
// one problem per warp (large n)
// ------------------------------------------------------------------------------------------
constexpr int kWarpsPerBlock = 8;

// MASKED: problem b sees only its visible landmarks (a.vis); every warp computes its problem's constants
template <typename T, int METHOD, bool MASKED = false>
__global__ void __launch_bounds__(kWarpsPerBlock * 32) k_solve_warp(const __grid_constant__ SolveArgs<T> a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    T* sP = reinterpret_cast<T*>(smem_raw);
    T* sC = sP + (size_t)a.n_patterns * a.n * 3;
    int32_t* sIdx = reinterpret_cast<int32_t*>(sC + (MASKED ? kWarpsPerBlock : 1) * a.n_patterns * PNP_PATC);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    const int32_t* sel = selection_of(a);
    load_pattern<T>(a.pattern, sel, a.n_total, a.n, a.n_patterns, sP, sIdx, threadIdx.x, blockDim.x);
    if (!MASKED && method_uses_patc(METHOD)) {
        for (int p = warp; p < a.n_patterns; p += kWarpsPerBlock)
            pattern_constants<T>(sP + (size_t)p * a.n * 3, a.n, sC + p * PNP_PATC, lane);
        __syncthreads();
    }
    PtsGlobal<T> pts;
    pts.idx = sel ? sIdx : nullptr;
    pts.k00 = (T)a.kinv[0]; pts.k01 = (T)a.kinv[1]; pts.k02 = (T)a.kinv[2];
    pts.k10 = (T)a.kinv[3]; pts.k11 = (T)a.kinv[4]; pts.k12 = (T)a.kinv[5];
    for (long long b = (long long)blockIdx.x * kWarpsPerBlock + warp; b < a.B; b += (long long)gridDim.x * kWarpsPerBlock) {
        pts.row = a.uv + (size_t)b * a.n_total * 2;
        Result<T> best;
        int best_p;
        if constexpr (MASKED) {
            PtsMasked<PtsGlobal<T> > pm;
            static_cast<PtsGlobal<T>&>(pm) = pts;
            pm.words = a.vis + (size_t)b * a.vis_words;
            pm.nvis = count_visible(pm.words, pm.idx, a.n);
            T* myC = sC + (size_t)warp * a.n_patterns * PNP_PATC;
            if (method_uses_patc(METHOD)) {
                for (int p = 0; p < a.n_patterns; ++p)
                    pattern_constants_masked<T, 32>(pm, sP + (size_t)p * a.n * 3, a.n, myC + p * PNP_PATC, lane);
                __syncwarp();
            }
            solve_all_patterns<T, METHOD, 32, PtsMasked<PtsGlobal<T> > >(pm, sP, myC, a.n, a.n_patterns, lane, a.prm, best, best_p);
            if (pm.nvis < kMinVisible) too_few_landmarks<T>(best, best_p);
            __syncwarp();                                     // the next problem's constants replace these
        } else {
            solve_all_patterns<T, METHOD, 32, PtsGlobal<T> >(pts, sP, sC, a.n, a.n_patterns, lane, a.prm, best, best_p);
        }
        if (lane == 0) write_result<T>(a, b, best, best_p);
    }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
template <typename T>
static SolverPrm<T> make_prm(const pnpb200_params& p)
{
    SolverPrm<T> s;
    s.max_it = p.max_it;
    s.linear_it = p.linear_it;
    s.lm_lambda = (T)p.lm_lambda;
    s.exit_tol = (T)p.exit_tol;
    // eif_Q_diag = sigma^2 / f^2; eif_Q_pinv = 1 / eif_Q_diag (:2844-2852)
    s.meas_w = (T)(1.0 / ((p.meas_sigma_px * p.meas_sigma_px) / (p.f_weight * p.f_weight)));
    s.proc_q = (T)p.proc_q;
    s.proc_d = (T)p.proc_d;
    s.sigma0 = (T)(1.0 / p.omega0);
    s.res_old0 = (T)p.res_old0;
    return s;
}

static long long persistent_grid(long long work_items, int sm_count, int per_sm)
{
    if (per_sm < 1) per_sm = 1;
    const long long cap = (long long)sm_count * per_sm;      // a multiple of the SM count
    return work_items < cap ? (work_items < 1 ? 1 : work_items) : cap;
}

// one of the three passes over the problems [b0, b0 + nb) of the batch
template <typename T, int METHOD>
static int launch_moment_pass(int pass, const MomArgs<T>& full, long long b0, long long nb, int shape, const StreamGeom& sg,
                              size_t smem, int per_sm, const DeviceProps& dp, int tune, cudaStream_t stream)
{
    MomArgs<T> m = full;
    m.B = nb;
    m.uv = full.uv + (size_t)b0 * full.n_total * 2;
    m.mom = full.mom + b0; m.tail = full.tail + b0;
    if (full.pmom) m.pmom = full.pmom + b0;
    if (full.vis) m.vis = full.vis + (size_t)b0 * full.vis_words;
    if (full.R) m.R = full.R + b0 * 9;
    if (full.t) m.t = full.t + b0 * 3;
    if (full.euler) m.euler = full.euler + b0 * 3;
    if (full.res) m.res = full.res + b0;
    if (full.iters) m.iters = full.iters + b0;
    if (full.best) m.best = full.best + b0;
    if (pass == 1) { launch_iterate<T, METHOD>(m, tune, stream); return PNPB200_OK; }
    const long long n_tiles = (nb + kTileProblems - 1) / kTileProblems;
    const unsigned tile_grid = (unsigned)(n_tiles < 0x7fffffffLL ? n_tiles : 0x7fffffffLL);
    const bool masked = m.vis != nullptr;
    if (shape == 0) {                                         // chunked row streaming
        m.row_pitch = sg.pitch;
        m.use_tma = sg.chunk;                                 // RowStream: points per chunk
        m.use_tmap = (sg.pitch == sg.chunk * 2) ? make_row_tensor_map(&m.tmap, m.uv, (int)sizeof(T), nb, m.n_total, sg.chunk) : 0;
        if (masked) {
            if (pass == 0) k_stream_chunk<T, METHOD, 0, true><<<tile_grid, 32, smem, stream>>>(m);
            else           k_stream_chunk<T, METHOD, 1, true><<<tile_grid, 32, smem, stream>>>(m);
        } else if (pass == 0) k_stream_chunk<T, METHOD, 0><<<tile_grid, 32, smem, stream>>>(m);
        else           k_stream_chunk<T, METHOD, 1><<<tile_grid, 32, smem, stream>>>(m);
        count_kernel_launches(1);
    } else if (shape == 1) {                                  // whole-row tiles
        if (masked) {
            if (pass == 0) k_stream_thread<T, METHOD, 0, true><<<tile_grid, 32, smem, stream>>>(m);
            else           k_stream_thread<T, METHOD, 1, true><<<tile_grid, 32, smem, stream>>>(m);
        } else if (pass == 0) k_stream_thread<T, METHOD, 0><<<tile_grid, 32, smem, stream>>>(m);
        else           k_stream_thread<T, METHOD, 1><<<tile_grid, 32, smem, stream>>>(m);
        count_kernel_launches(1);
    } else if (shape == 3) {                                  // one problem per warp, rows through a TMA ring
        const unsigned grid = (unsigned)persistent_grid((nb + kRingWarps - 1) / kRingWarps, dp.sm_count, per_sm);
        if (pass == 0) k_stream_warp_tma<T, METHOD, 0><<<grid, kRingWarps * 32, smem, stream>>>(m);
        else           k_stream_warp_tma<T, METHOD, 1><<<grid, kRingWarps * 32, smem, stream>>>(m);
        count_kernel_launches(1);
    } else {                                                  // one problem per warp, coalesced loads
        const unsigned grid = (unsigned)persistent_grid((nb + 7) / 8, dp.sm_count, per_sm);
        if (masked) {
            if (pass == 0) k_stream_warp<T, METHOD, 0, true><<<grid, 256, smem, stream>>>(m);
            else           k_stream_warp<T, METHOD, 1, true><<<grid, 256, smem, stream>>>(m);
        } else if (pass == 0) k_stream_warp<T, METHOD, 0><<<grid, 256, smem, stream>>>(m);
        else           k_stream_warp<T, METHOD, 1><<<grid, 256, smem, stream>>>(m);
        count_kernel_launches(1);
    }
    return PNPB200_OK;
}

// A handful of marked tiles (the normal case on detected pixels) is latency: one problem per warp finishes them in a few
// microseconds; thousands of them (noise-free pixels) is throughput: one problem per thread.  Both kernels read the count and
// exactly one of them acts (rows too long for a tile: always per warp).
template <typename T, int METHOD, bool MASKED>
static int launch_filter_fixup_as(const MomArgs<T>& m, const RowGeom& g, bool by_thread, size_t thread_smem, size_t warp_smem,
                                  const DeviceProps& dp, cudaStream_t stream)
{
    MomArgs<T> f = m;
    const long long n_tiles = (m.B + kTileProblems - 1) / kTileProblems;
    f.fix_warp_max = by_thread ? dp.sm_count : 0x7fffffff;
    {
        const size_t smem = warp_smem + (MASKED ? kWarpsPerFixup : 1) * PNP_PATC * sizeof(T);   // masked: constants per warp
        PNP_CUDA_OK(set_dynamic_smem((const void*)k_fixup_warp<T, METHOD, MASKED>, smem));
        int per_sm = 1;
        PNP_CUDA_OK(blocks_per_sm(&per_sm, (const void*)k_fixup_warp<T, METHOD, MASKED>, 256, smem));
        const unsigned grid = (unsigned)persistent_grid(n_tiles, dp.sm_count, per_sm);   // CTAs beyond the number of marked tiles leave at once
        k_fixup_warp<T, METHOD, MASKED><<<grid, 256, smem, stream>>>(f);
        count_kernel_launches(1);
    }
    if (by_thread) {
        f.row_pitch = g.row_pitch; f.use_tma = g.use_tma;
        const size_t smem = thread_smem + (MASKED ? kTileProblems : 1) * PNP_PATC * sizeof(T);   // masked: constants per lane
        PNP_CUDA_OK(set_dynamic_smem((const void*)k_fixup_thread<T, METHOD, MASKED>, smem));
        int per_sm = 1;
        PNP_CUDA_OK(blocks_per_sm(&per_sm, (const void*)k_fixup_thread<T, METHOD, MASKED>, 32, smem));
        const unsigned grid = (unsigned)persistent_grid(n_tiles, dp.sm_count, per_sm);
        k_fixup_thread<T, METHOD, MASKED><<<grid, 32, smem, stream>>>(f);
        count_kernel_launches(1);
    }
    return PNPB200_OK;
}

template <typename T, int METHOD>
static int launch_filter_fixup(const MomArgs<T>& m, const RowGeom& g, bool by_thread, size_t thread_smem, size_t warp_smem,
                               const DeviceProps& dp, cudaStream_t stream)
{
    if (m.vis) return launch_filter_fixup_as<T, METHOD, true>(m, g, by_thread, thread_smem, warp_smem, dp, stream);
    return launch_filter_fixup_as<T, METHOD, false>(m, g, by_thread, thread_smem, warp_smem, dp, stream);
}

// LM / linear F2 with one pattern: moments -> iterate -> residual (see the kernels' header).
// (Measured and rejected: (1) cutting the batch into slices that flow through the three passes on
// different streams -- the kernels do overlap, but k_iterate fills the register file, so the
// streaming blocks displace iterate blocks instead of adding warps: same total time; (2) the three
// passes in one kernel per 32-problem tile, second stream issued before the iterations: 1.479 ms
// against 1.460 ms -- with 8 warps per SM the warps that stream are simply missing from the FP64
// pipe; (3) warp-specialised producer / consumer CTAs do not fit: setmaxnreg works per 128-thread
// warpgroup, and 4 compute warps at 224 registers + 4 streaming warps already fill half an SM.)
template <typename T, int METHOD>
static int launch_moment(const SolveArgs<T>& a, const DeviceProps& dp, cudaStream_t stream)
{
    const RowGeom g = row_geometry<T>(a.n_total);
    const size_t idx_bytes = a.idx_mode ? (size_t)a.n * sizeof(int32_t) : 0;
    const size_t pat_bytes = (size_t)a.n * 3 * sizeof(T);
    const size_t thread_smem = g.tile_bytes + pat_bytes + idx_bytes + 16;
    const size_t warp_smem = pat_bytes + idx_bytes;
    const bool by_thread = g.tile_bytes <= 48 * 1024 && thread_smem <= (size_t)dp.max_smem_optin;
    if (!by_thread && warp_smem > (size_t)dp.max_smem_optin) return PNPB200_ETOOLARGE;

    const bool masked = a.vis != nullptr;
    T* ws = nullptr;
    // masked: the per-problem pattern moments ride behind the moments ([kPatternMoments][B])
    const size_t ws_elems = (size_t)(PNP_NMOM + (masked ? kPatternMoments : 0) + PNP_NTAIL) * (size_t)a.B + PNP_PATC;
    const bool own_ws = !(a.ws && a.ws_bytes >= ws_elems * sizeof(T));
    if (own_ws) PNP_CUDA_OK(cudaMallocAsync((void**)&ws, ws_elems * sizeof(T), stream));
    else ws = (T*)a.ws;
    struct WsGuard {                                          // every return below hands the scratch back to the pool
        void* p; cudaStream_t st;
        ~WsGuard() { if (p) cudaFreeAsync(p, st); }
    } ws_guard = { own_ws ? (void*)ws : nullptr, stream };
    MomArgs<T> m;
    m.uv = a.uv; m.pattern = a.pattern; m.idx = a.idx; m.idx_mode = a.idx_mode;
    for (int e = 0; e < PNP_MAX_INLINE_IDX; ++e) m.idx_inline[e] = a.idx_inline[e];
    m.B = a.B; m.ld = a.B; m.n_total = a.n_total; m.n = a.n;
    m.row_pitch = g.row_pitch; m.use_tma = g.use_tma;
    for (int e = 0; e < 6; ++e) m.kinv[e] = a.kinv[e];
    m.prm = a.prm;
    m.mom = ws; m.tail = ws + (size_t)PNP_NMOM * a.B; m.patc = m.tail + (size_t)PNP_NTAIL * a.B;
    m.vis = a.vis; m.vis_words = a.vis_words; m.pmom = nullptr;
    if (masked) { m.pmom = ws + (size_t)PNP_NMOM * a.B; m.tail = m.pmom + (size_t)kPatternMoments * a.B; m.patc = m.tail + (size_t)PNP_NTAIL * a.B; }
    m.R = a.R; m.t = a.t; m.euler = a.euler; m.res = a.res; m.iters = a.iters; m.best = a.best;
    m.use_tmap = 0;
    struct ItersGuard { void* p; cudaStream_t st; ~ItersGuard() { if (p) cudaFreeAsync(p, st); } } iters_guard = { nullptr, stream }, list_guard = { nullptr, stream };
    m.fix_list = nullptr; m.fix_warp_max = 0;
    if (method_with_s(METHOD)) {
        if (!m.iters) {                                       // the marks of the fix-up pass travel in the iteration counts
            PNP_CUDA_OK(cudaMallocAsync((void**)&m.iters, sizeof(int32_t) * (size_t)a.B, stream));
            iters_guard.p = m.iters;
        }
        const size_t n_tiles = ((size_t)a.B + kTileProblems - 1) / kTileProblems;
        PNP_CUDA_OK(cudaMallocAsync((void**)&m.fix_list, sizeof(int32_t) * (n_tiles + 1), stream));
        list_guard.p = m.fix_list;
        PNP_CUDA_OK(cudaMemsetAsync(m.fix_list, 0, sizeof(int32_t), stream));
    }

    // kernel shape of the two streaming passes
    const StreamGeom sg = stream_geometry<T>(a.n_total);
    int shape, per_sm = 1;
    size_t smem;
    if (by_thread && !a.idx_mode && sg.use_stream && a.tune != 9) {
        shape = 0; smem = 2 * sg.buf_bytes + pat_bytes + 32;
        PNP_CUDA_OK(set_dynamic_smem(masked ? (const void*)k_stream_chunk<T, METHOD, 0, true> : (const void*)k_stream_chunk<T, METHOD, 0>, smem));
        PNP_CUDA_OK(set_dynamic_smem(masked ? (const void*)k_stream_chunk<T, METHOD, 1, true> : (const void*)k_stream_chunk<T, METHOD, 1>, smem));
    } else if (by_thread) {
        shape = 1; smem = thread_smem;
        PNP_CUDA_OK(set_dynamic_smem(masked ? (const void*)k_stream_thread<T, METHOD, 0, true> : (const void*)k_stream_thread<T, METHOD, 0>, smem));
        PNP_CUDA_OK(set_dynamic_smem(masked ? (const void*)k_stream_thread<T, METHOD, 1, true> : (const void*)k_stream_thread<T, METHOD, 1>, smem));
    } else if (!masked && !a.idx_mode && ((size_t)a.n_total * 2 * sizeof(T)) % 16 == 0 && a.tune != 9 &&
               a.n_total >= kRingPoints) {                // (no masked ring kernel: masked rows take the per-warp shape below)
        shape = 3;
        smem = (size_t)kRingWarps * kRingSlots * (kRingPoints * 2 * sizeof(T) + 8);
        PNP_CUDA_OK(set_dynamic_smem((const void*)k_stream_warp_tma<T, METHOD, 0>, smem));
        PNP_CUDA_OK(set_dynamic_smem((const void*)k_stream_warp_tma<T, METHOD, 1>, smem));
        PNP_CUDA_OK(blocks_per_sm(&per_sm, (const void*)k_stream_warp_tma<T, METHOD, 0>, kRingWarps * 32, smem));
    } else {
        shape = 2; smem = warp_smem;
        const void* k0 = masked ? (const void*)k_stream_warp<T, METHOD, 0, true> : (const void*)k_stream_warp<T, METHOD, 0>;
        PNP_CUDA_OK(set_dynamic_smem(k0, smem));
        PNP_CUDA_OK(set_dynamic_smem(masked ? (const void*)k_stream_warp<T, METHOD, 1, true> : (const void*)k_stream_warp<T, METHOD, 1>, smem));
        PNP_CUDA_OK(blocks_per_sm(&per_sm, k0, 256, smem));
    }

    // -DPNP_DEBUG_SYNC (tools/build_variant.py): synchronise after every launch and name the kernel a fault belongs to
#ifdef PNP_DEBUG_SYNC
#define PNP_DEBUG_CHECK(what) do { cudaError_t e_ = cudaStreamSynchronize(stream); if (e_ != cudaSuccess) { \
        fprintf(stderr, "[pnpb200 debug] after %s (shape %d, smem %zu, per_sm %d): %s\n", what, shape, smem, per_sm, cudaGetErrorString(e_)); return PNPB200_ECUDA; } } while (0)
#else
#define PNP_DEBUG_CHECK(what) do { } while (0)
#endif
    if (!masked) {                                            // (masked: per problem, from the moments pass)
        k_pattern_constants<T><<<1, 32, 0, stream>>>(m); count_kernel_launches(1);
        PNP_DEBUG_CHECK("k_pattern_constants");
    }
    const int slot = a.profile ? g_prof.begin() : -1;
    g_prof.mark(slot, stream);
    launch_moment_pass<T, METHOD>(0, m, 0, a.B, shape, sg, smem, per_sm, dp, a.tune, stream);
    PNP_DEBUG_CHECK("moments pass");
    g_prof.mark(slot, stream);
    launch_moment_pass<T, METHOD>(1, m, 0, a.B, shape, sg, smem, per_sm, dp, a.tune, stream);
    PNP_DEBUG_CHECK("k_iterate");
    if (method_with_s(METHOD)) {                              // filters: re-solve what k_iterate could not certify (see k_fixup_*)
        const int rc = launch_filter_fixup<T, METHOD>(m, g, by_thread, thread_smem, warp_smem, dp, stream);
        if (rc != PNPB200_OK) return rc;
    }
    g_prof.mark(slot, stream);
    if (a.res && !a.skip_residual) launch_moment_pass<T, METHOD>(2, m, 0, a.B, shape, sg, smem, per_sm, dp, a.tune, stream);
    if (!a.skip_residual) g_prof.mark(slot, stream);      // (the fused report + residual pass is marked by its launcher)
    PNP_CUDA_OK(cudaGetLastError());
    return PNPB200_OK;
}

// solve_pnp's arg-min over patterns (:166-199) for the moment mapping, which solves one pattern per pass: the candidate of
// pattern p replaces the best so far where its res_norm is strictly smaller (first wins; a NaN never wins, as `<` in the reference)
template <typename T>
__global__ void __launch_bounds__(256) k_merge_best(long long B, int p, const T* __restrict__ cR, const T* __restrict__ ct,
                                                    const T* __restrict__ ce, const T* __restrict__ cres, const int32_t* __restrict__ cit,
                                                    T* R, T* t, T* e, T* res, int32_t* it, int32_t* best, T* best_res)
{
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const T r = cres[b];
    if (!(r < best_res[b])) return;
    best_res[b] = r;
    if (res) res[b] = r;
    if (R) {
#pragma unroll
        for (int k = 0; k < 9; ++k) R[b * 9 + k] = cR[b * 9 + k];
    }
    if (t) {
#pragma unroll
        for (int k = 0; k < 3; ++k) t[b * 3 + k] = ct[b * 3 + k];
    }
    if (e) {
#pragma unroll
        for (int k = 0; k < 3; ++k) e[b * 3 + k] = ce[b * 3 + k];
    }
    if (it) it[b] = cit[b];
    if (best) best[b] = p;
}

// LM / linear F2 over several stored patterns: one moment-mapping solve per pattern, arg-min on res_norm in between
template <typename T, int METHOD>
static int launch_moment_patterns(const SolveArgs<T>& a, const DeviceProps& dp, cudaStream_t stream)
{
    const size_t B = (size_t)a.B;
    // candidate outputs of patterns 1.., and the running minimum when the caller did not ask for res_norm
    const size_t elems = B * (9 + 3 + 3 + 1 + 1);
    T* buf = nullptr;
    PNP_CUDA_OK(cudaMallocAsync((void**)&buf, elems * sizeof(T) + B * sizeof(int32_t), stream));
    struct Guard { void* p; cudaStream_t st; ~Guard() { cudaFreeAsync(p, st); } } guard = { buf, stream };
    T *cR = buf, *ct = cR + B * 9, *ce = ct + B * 3, *cres = ce + B * 3, *own_res = cres + B;
    int32_t* cit = reinterpret_cast<int32_t*>(own_res + B);
    for (int p = 0; p < a.n_patterns; ++p) {
        SolveArgs<T> one = a;
        one.n_patterns = 1;
        one.pattern = a.pattern + (size_t)p * a.n_total * 3;
        if (p == 0) {
            one.res = a.res ? a.res : own_res;
        } else {
            one.R = cR; one.t = ct; one.euler = a.euler ? ce : nullptr; one.res = cres; one.iters = cit; one.best = nullptr;
        }
        const int rc = launch_moment<T, METHOD>(one, dp, stream);
        if (rc != PNPB200_OK) return rc;
        if (p > 0) {
            k_merge_best<T><<<(unsigned)((a.B + 255) / 256), 256, 0, stream>>>(a.B, p, cR, ct, ce, cres, cit, a.R, a.t, a.euler, a.res, a.iters,
                                                                               a.best, a.res ? a.res : own_res);
            count_kernel_launches(1);
        }
    }
    PNP_CUDA_OK(cudaGetLastError());
    return PNPB200_OK;
}

template <typename T, int METHOD>
static int launch_solve(const SolveArgs<T>& a, int mapping, cudaStream_t stream)
{
    DeviceProps dp;
    int rc = get_device_props(&dp);
    if (rc != PNPB200_OK) return rc;
    // (the filters' exit test from the moments needs FP64: in FP32 the moment-form residual is noise at res / |z| ~ 1e-3)
    constexpr bool has_moment_form = (METHOD == PNPB200_METHOD_LM || METHOD == PNPB200_METHOD_LINEAR_F2 || METHOD == PNPB200_METHOD_LM_PLUS ||
                                      METHOD == PNP_METHOD_LM_TRUEJAC ||
                                      ((METHOD == PNP_METHOD_QEIF_HYBRID || METHOD == PNPB200_METHOD_EIF2) && sizeof(T) == 8));
    // a visibility mask (a.vis) takes the same mapping as the call without it; its kernels keep the pattern constants per
    // problem.  (LM_TRUEJAC exists in the moment mapping only: no direct kernels, masked or not, are launched for it.)
    constexpr bool can_mask = METHOD != PNP_METHOD_LM_TRUEJAC;
    const bool masked = a.vis != nullptr;
    const RowGeom g = row_geometry<T>(a.n_total);
    const size_t pat_bytes = ((size_t)a.n_patterns * a.n * 3 + (size_t)a.n_patterns * PNP_PATC) * sizeof(T);
    const size_t idx_bytes = a.idx_mode ? (size_t)a.n * sizeof(int32_t) : 0;
    const size_t patc_bytes = (size_t)a.n_patterns * PNP_PATC * sizeof(T);
    const size_t thread_smem = g.tile_bytes + pat_bytes + idx_bytes + 16 + (masked ? (kTileProblems - 1) * patc_bytes : 0);
    const size_t warp_smem = pat_bytes + idx_bytes + (masked ? (kWarpsPerBlock - 1) * patc_bytes : 0);
    const int direct = (g.tile_bytes <= 48 * 1024 && thread_smem <= (size_t)dp.max_smem_optin) ? PNPB200_MAP_THREAD : PNPB200_MAP_WARP;
    if (mapping == PNPB200_MAP_AUTO) mapping = has_moment_form ? PNPB200_MAP_MOMENT : direct;
    if (mapping == PNPB200_MAP_MOMENT) {
        if (!has_moment_form) return PNPB200_EINVAL;
        if (a.n_patterns == 1) return launch_moment<T, has_moment_form ? METHOD : PNPB200_METHOD_LM>(a, dp, stream);
        return launch_moment_patterns<T, has_moment_form ? METHOD : PNPB200_METHOD_LM>(a, dp, stream);
    }
    if ((mapping == PNPB200_MAP_THREAD || mapping == PNPB200_MAP_WARP) && masked && !can_mask) return PNPB200_EINVAL;
    if (mapping == PNPB200_MAP_THREAD) {
        if (thread_smem > (size_t)dp.max_smem_optin) return PNPB200_ETOOLARGE;
        if constexpr (can_mask) {
            if (masked) PNP_CUDA_OK(set_dynamic_smem((const void*)k_solve_thread<T, METHOD, true>, thread_smem));
        }
        if (!masked) PNP_CUDA_OK(set_dynamic_smem((const void*)k_solve_thread<T, METHOD>, thread_smem));
        SolveArgs<T> at = a;
        at.row_pitch = g.row_pitch;
        at.use_tma = g.use_tma;
        const long long n_tiles = (a.B + kTileProblems - 1) / kTileProblems;
        const long long grid = n_tiles < 0x7fffffffLL ? n_tiles : 0x7fffffffLL;
        const int slot = a.profile ? g_prof.begin() : -1;
        g_prof.mark(slot, stream);
        if constexpr (can_mask) {
            if (masked) k_solve_thread<T, METHOD, true><<<(unsigned)grid, 32, thread_smem, stream>>>(at);
        }
        if (!masked) k_solve_thread<T, METHOD><<<(unsigned)grid, 32, thread_smem, stream>>>(at);
        count_kernel_launches(1);
        g_prof.mark(slot, stream);
    } else if (mapping == PNPB200_MAP_WARP) {
        if (warp_smem > (size_t)dp.max_smem_optin) return PNPB200_ETOOLARGE;
        const void* kfn = (const void*)k_solve_warp<T, METHOD>;
        if constexpr (can_mask) {
            if (masked) kfn = (const void*)k_solve_warp<T, METHOD, true>;
        }
        PNP_CUDA_OK(set_dynamic_smem(kfn, warp_smem));
        int per_sm = 1;
        PNP_CUDA_OK(blocks_per_sm(&per_sm, kfn, kWarpsPerBlock * 32, warp_smem));
        const long long grid = persistent_grid((a.B + kWarpsPerBlock - 1) / kWarpsPerBlock, dp.sm_count, per_sm);
        const int slot = a.profile ? g_prof.begin() : -1;
        g_prof.mark(slot, stream);
        if constexpr (can_mask) {
            if (masked) k_solve_warp<T, METHOD, true><<<(unsigned)grid, kWarpsPerBlock * 32, warp_smem, stream>>>(a);
        }
        if (!masked) k_solve_warp<T, METHOD><<<(unsigned)grid, kWarpsPerBlock * 32, warp_smem, stream>>>(a);
        count_kernel_launches(1);
        g_prof.mark(slot, stream);
    } else {
        return PNPB200_EINVAL;
    }
    PNP_CUDA_OK(cudaGetLastError());
    return PNPB200_OK;
}

template <typename T>
static int solve_typed(int method, long long B, int n_total, int n, const void* uv, const void* pattern,
                       int n_patterns, const int32_t* idx_host, const int32_t* idx_dev, const double* K, const pnpb200_params& prm,
                       void* R, void* t, void* euler, void* res, int32_t* iters, int32_t* best, cudaStream_t stream,
                       const uint32_t* vis)
{
    SolveArgs<T> a;
    a.uv = (const T*)uv; a.pattern = (const T*)pattern; a.idx = idx_dev;
    a.idx_mode = idx_host ? (idx_dev ? 2 : 1) : 0;
    for (int e = 0; e < PNP_MAX_INLINE_IDX; ++e) a.idx_inline[e] = (idx_host && !idx_dev && e < n) ? idx_host[e] : 0;
    a.B = B; a.n_total = n_total; a.n = n; a.n_patterns = n_patterns;
    a.row_pitch = 0; a.use_tma = 0;
    double Kinv[9];
    host_inv3(K, Kinv);
    for (int e = 0; e < 9; ++e)
        if (!(Kinv[e] - Kinv[e] == 0.0)) return PNPB200_EINVAL;   // singular or non-finite camera matrix (np.linalg.inv raises there)
    for (int e = 0; e < 6; ++e) a.kinv[e] = Kinv[e];
    a.prm = make_prm<T>(prm);
    a.R = (T*)R; a.t = (T*)t; a.euler = (T*)euler; a.res = (T*)res; a.iters = iters; a.best = best;
    a.profile = (prm.flags & PNPB200_FLAG_PROFILE) ? 1 : 0;
    a.skip_residual = (prm.flags & PNP_FLAG_INTERNAL_NO_RESIDUAL) ? 1 : 0;
    a.tune = (prm.flags >> 8) & 0xff;                     // undocumented tuning knob (register budget of k_iterate, slice size)
    a.ws = prm.workspace; a.ws_bytes = (prm.workspace && prm.workspace_bytes > 0) ? (size_t)prm.workspace_bytes : 0;
    a.vis = vis; a.vis_words = (n_total + 31) / 32;
    switch (method) {
#if PNP_GROUP == 0
    case PNPB200_METHOD_QEIF:
        if (n >= PNP_QEIF_HYBRID_MIN_N && !(prm.flags & PNPB200_FLAG_QEIF_DIRECT)) return launch_solve<T, PNP_METHOD_QEIF_HYBRID>(a, prm.mapping, stream);
        return launch_solve<T, PNPB200_METHOD_QEIF>(a, prm.mapping, stream);
    case PNPB200_METHOD_LINEAR_F1: return launch_solve<T, PNPB200_METHOD_LINEAR_F1>(a, prm.mapping, stream);
#elif PNP_GROUP == 1
    case PNPB200_METHOD_LM:
        if (prm.flags & PNPB200_FLAG_LM_TRUE_JACOBIAN) {     // non-parity extra: exists in the moment mapping only
            if (prm.mapping != PNPB200_MAP_AUTO && prm.mapping != PNPB200_MAP_MOMENT) return PNPB200_EINVAL;
            return launch_solve<T, PNP_METHOD_LM_TRUEJAC>(a, PNPB200_MAP_MOMENT, stream);
        }
        return launch_solve<T, PNPB200_METHOD_LM>(a, prm.mapping, stream);
    case PNPB200_METHOD_LM_PLUS: {
        // non-parity extra: exists in the moment mapping only
        if (prm.mapping != PNPB200_MAP_AUTO && prm.mapping != PNPB200_MAP_MOMENT) return PNPB200_EINVAL;
        DeviceProps dp;
        int rc = get_device_props(&dp);
        if (rc != PNPB200_OK) return rc;
        if (n_patterns > 1) return launch_moment_patterns<T, PNPB200_METHOD_LM_PLUS>(a, dp, stream);
        return launch_moment<T, PNPB200_METHOD_LM_PLUS>(a, dp, stream);
    }
#elif PNP_GROUP == 2
    case PNPB200_METHOD_LINEAR_F2: return launch_solve<T, PNPB200_METHOD_LINEAR_F2>(a, prm.mapping, stream);
#else
    case PNPB200_METHOD_EIF2:      return launch_solve<T, PNPB200_METHOD_EIF2>(a, prm.mapping, stream);
#endif
    default: return PNPB200_EINVAL;
    }
}

#define PNP_CAT3_(a, b, c) a##b##c
#define PNP_CAT3(a, b, c) PNP_CAT3_(a, b, c)
#if PNP_F64
#define PNP_PART_NAME PNP_CAT3(solve_part_f64_g, PNP_GROUP, )
typedef double part_scalar;
#else
#define PNP_PART_NAME PNP_CAT3(solve_part_f32_g, PNP_GROUP, )
typedef float part_scalar;
#endif

int PNP_PART_NAME(PNP_SOLVE_PART_ARGS)
{
    return solve_typed<part_scalar>(method, B, n_total, n, uv, pattern, n_patterns, idx_host, idx_dev, K, prm, R, t, euler, res,
                                    iters, best, stream, vis);
}

}  // namespace pnpb200
