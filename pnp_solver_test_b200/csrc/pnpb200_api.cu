// pnpb200_api.cu -- the C ABI of the solve path (include/pnpb200.h): argument checks, dispatch to the
// per-(dtype, method group) objects of pnpb200_kernels.cu, per-kernel profiling, and the
// host-buffer pipeline.
#include <atomic>
#include <map>
#include <mutex>
#include <string.h>
#include <thread>
#include <vector>

#include "pnpb200_common.cuh"

namespace pnpb200 {

// ------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------
static thread_local char g_last_error[512] = "";

void set_last_error(const char* where, cudaError_t e)
{
    snprintf(g_last_error, sizeof(g_last_error), "%s: %s (%s)", where, cudaGetErrorName(e), cudaGetErrorString(e));
}

int get_device_props(DeviceProps* out)
{
    static std::mutex mu;
    static std::vector<DeviceProps> cache;
    int dev = 0;
    PNP_CUDA_OK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(mu);
    for (const DeviceProps& p : cache)
        if (p.device == dev) { *out = p; return PNPB200_OK; }
    DeviceProps p;
    p.device = dev;
    PNP_CUDA_OK(cudaDeviceGetAttribute(&p.sm_count, cudaDevAttrMultiProcessorCount, dev));
    PNP_CUDA_OK(cudaDeviceGetAttribute(&p.cc_major, cudaDevAttrComputeCapabilityMajor, dev));
    PNP_CUDA_OK(cudaDeviceGetAttribute(&p.cc_minor, cudaDevAttrComputeCapabilityMinor, dev));
    PNP_CUDA_OK(cudaDeviceGetAttribute(&p.max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    size_t free_b = 0;
    PNP_CUDA_OK(cudaMemGetInfo(&free_b, &p.total_mem));
    {   // keep stream-ordered scratch cached in the device's default pool instead of returning it
        // to the driver at every synchronisation (a moment-mapping call would re-map it each time)
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
            unsigned long long thr = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
        }
        cudaGetLastError();
    }
    cache.push_back(p);
    *out = p;
    return PNPB200_OK;
}


thread_local ProfileRing g_prof;

static std::atomic<long long> g_launches{0};
void count_kernel_launches(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

namespace {
struct KernelKey {
    int dev; const void* fn; int block; size_t smem;
    bool operator<(const KernelKey& o) const
    {
        if (dev != o.dev) return dev < o.dev;
        if (fn != o.fn) return fn < o.fn;
        if (block != o.block) return block < o.block;
        return smem < o.smem;
    }
};
}  // namespace

int make_row_tensor_map(CUtensorMap* out, const void* uv, int elem_bytes, long long B, int n_total, int chunk_points)
{
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static const EncodeFn encode = []() -> EncodeFn {
        if (getenv("PNPB200_NO_TENSOR_MAP")) return nullptr;                  // tuning / A-B comparisons only
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess) { cudaGetLastError(); return nullptr; }
        return (EncodeFn)fn;
    }();
    const unsigned long long row_bytes = (unsigned long long)n_total * 2ull * (unsigned long long)elem_bytes;
    if (!encode || B < 1 || B > 0x7fffffffLL || chunk_points < 1 || chunk_points * 2 > 256 || (row_bytes & 15ull) ||
        ((unsigned long long)chunk_points * 2ull * elem_bytes & 15ull) || ((uintptr_t)uv & 15u))
        return 0;
    const cuuint64_t dims[2] = { (cuuint64_t)n_total * 2u, (cuuint64_t)B };
    const cuuint64_t strides[1] = { (cuuint64_t)row_bytes };
    const cuuint32_t box[2] = { (cuuint32_t)chunk_points * 2u, 32u };
    const cuuint32_t estr[2] = { 1u, 1u };
    const CUresult r = encode(out, elem_bytes == 8 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                              const_cast<void*>(uv), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 1 : 0;
}

cudaError_t set_dynamic_smem(const void* kernel, size_t bytes)
{
    static std::mutex mu;
    static std::map<KernelKey, size_t> done;               // largest size set so far
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lk(mu);
    size_t& cur = done[KernelKey{ dev, kernel, 0, 0 }];
    if (cur >= bytes && cur != 0) return cudaSuccess;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) cur = bytes;
    return e;
}

cudaError_t blocks_per_sm(int* out, const void* kernel, int block_threads, size_t smem_bytes)
{
    static std::mutex mu;
    static std::map<KernelKey, int> cache;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lk(mu);
    const KernelKey key{ dev, kernel, block_threads, smem_bytes };
    auto it = cache.find(key);
    if (it != cache.end()) { *out = it->second; return cudaSuccess; }
    int n = 1;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, block_threads, smem_bytes);
    if (e == cudaSuccess) { cache[key] = n; *out = n; }
    return e;
}

void fill_default_params(pnpb200_params* p)
{
    p->max_it = 14; p->linear_it = 3;
    p->lm_lambda = 1e-5; p->exit_tol = 1e-2;
    p->f_weight = 225.68; p->meas_sigma_px = 3.0;
    p->proc_q = 1e-1; p->proc_d = 1e-2; p->omega0 = 1e-5; p->res_old0 = 1e-7;
    p->mapping = PNPB200_MAP_AUTO; p->flags = 0;
    p->workspace = nullptr; p->workspace_bytes = 0;
}


}  // namespace pnpb200

using namespace pnpb200;

extern "C" {

int pnpb200_version(void) { return PNPB200_VERSION; }
int64_t pnpb200_launch_count(void) { return (int64_t)g_launches.load(std::memory_order_relaxed); }
const char* pnpb200_last_error(void) { return g_last_error; }

int pnpb200_default_params(pnpb200_params* p)
{
    if (!p) return PNPB200_EINVAL;
    fill_default_params(p);
    return PNPB200_OK;
}

int pnpb200_device_info(int* sm_count, int* cc_major, int* cc_minor, int64_t* hbm_bytes)
{
    DeviceProps dp;
    int rc = get_device_props(&dp);
    if (rc != PNPB200_OK) return rc;
    if (sm_count) *sm_count = dp.sm_count;
    if (cc_major) *cc_major = dp.cc_major;
    if (cc_minor) *cc_minor = dp.cc_minor;
    if (hbm_bytes) *hbm_bytes = (int64_t)dp.total_mem;
    return PNPB200_OK;
}

int pnpb200_profile_reset(void)
{
    g_prof.next = 0; g_prof.count = 0;
    if (g_prof.created)
        for (int s = 0; s < ProfileRing::kSlots; ++s) g_prof.used[s] = 0;
    return PNPB200_OK;
}

int pnpb200_profile_read(float* ms, int* n_calls)
{
    if (!ms) return PNPB200_EINVAL;
    double acc[3] = { 0, 0, 0 };
    int calls = 0;
    for (int s = 0; s < g_prof.count && g_prof.created; ++s) {
        const int u = g_prof.used[s];
        if (u < 2) continue;
        PNP_CUDA_OK(cudaEventSynchronize(g_prof.ev[s][u - 1]));
        for (int k = 0; k + 1 < u; ++k) {
            float t = 0.f;
            PNP_CUDA_OK(cudaEventElapsedTime(&t, g_prof.ev[s][k], g_prof.ev[s][k + 1]));
            acc[k] += t;
        }
        ++calls;
    }
    for (int k = 0; k < 3; ++k) ms[k] = calls ? (float)(acc[k] / calls) : 0.f;
    if (n_calls) *n_calls = calls;
    return PNPB200_OK;
}

int64_t pnpb200_workspace_bytes(int method, int dtype, int64_t B, int n_patterns, int mapping)
{
    (void)n_patterns;                                       // several patterns are solved one after the other with the same scratch
    const bool moment_form = (method == PNPB200_METHOD_LM || method == PNPB200_METHOD_LINEAR_F2 || method == PNPB200_METHOD_LM_PLUS ||
                              ((method == PNPB200_METHOD_EIF2 || method == PNPB200_METHOD_QEIF) && dtype == PNPB200_DTYPE_F64));   // (QEIF: from 12 landmarks on)
    if (B <= 0 || !moment_form || (mapping != PNPB200_MAP_AUTO && mapping != PNPB200_MAP_MOMENT)) return 0;
    const int64_t esz = (dtype == PNPB200_DTYPE_F32) ? 4 : 8;
    return ((int64_t)(PNP_NMOM + PNP_NTAIL) * B + PNP_PATC) * esz;
}

int64_t pnpb200_workspace_bytes_masked(int method, int dtype, int64_t B, int n_patterns, int mapping)
{
    // the moment mapping keeps 10 pattern moments (sum theta theta^T, sum theta, count) per problem beside the moments
    const int64_t plain = pnpb200_workspace_bytes(method, dtype, B, n_patterns, mapping);
    return plain > 0 ? plain + (int64_t)PNP_NPMOM * B * ((dtype == PNPB200_DTYPE_F32) ? 4 : 8) : 0;
}

int64_t pnpb200_workspace_bytes_weighted(int method, int dtype, int64_t B, int n_patterns, int mapping)
{
    // the weighted pattern moments (sum w theta theta^T, sum w theta, sum w) and the count of landmarks taking part
    const int64_t plain = pnpb200_workspace_bytes(method, dtype, B, n_patterns, mapping);
    return plain > 0 ? plain + (int64_t)PNP_NPMOM_W * B * ((dtype == PNPB200_DTYPE_F32) ? 4 : 8) : 0;
}

}  // extern "C"

namespace pnpb200 {
// vis: [B, ceil(n_total / 32)] per-problem visibility bits (device), or nullptr for every landmark
// wts: [B, n_total] float32 per-landmark weights (device), or nullptr for weight 1 (at most one of vis, wts)
int solve_batch_impl(int method, int dtype, int64_t B, int n_total, int n, const void* uv, const void* pattern,
                     int n_patterns, const int32_t* point_index, const double* K, const pnpb200_params& prm,
                     void* R, void* t, void* euler_deg, void* res_norm, int32_t* iters, int32_t* best_pattern,
                     cudaStream_t st, const uint32_t* vis, const float* wts)
{
    if (B < 0 || n_total < 1 || n < 1 || (!point_index && n != n_total) || !uv || !pattern || !K) return PNPB200_EINVAL;
    if (vis && !vis_aligned(vis)) return PNPB200_EINVAL;
    if ((wts && ((uintptr_t)wts & 3u) != 0) || (vis && wts)) return PNPB200_EINVAL;
    if (((uintptr_t)uv & 15u) != 0) return PNPB200_EINVAL;   // rows are staged with 16-byte bulk copies / vector loads
    if (n_patterns < 1 || n_patterns > PNPB200_MAX_PATTERNS) return PNPB200_EINVAL;
    if (method < 0 || method > 5 || (dtype != PNPB200_DTYPE_F64 && dtype != PNPB200_DTYPE_F32)) return PNPB200_EINVAL;
    if (B == 0) return PNPB200_OK;
    int32_t* idx_dev = nullptr;
    if (point_index) {
        for (int i = 0; i < n; ++i)
            if (point_index[i] < 0 || point_index[i] >= n_total) return PNPB200_EINVAL;
        if (n > PNP_MAX_INLINE_IDX) {   // large selections go through device memory; small ones ride in the kernel arguments
            PNP_CUDA_OK(cudaMallocAsync((void**)&idx_dev, sizeof(int32_t) * (size_t)n, st));
            PNP_CUDA_OK(cudaMemcpyAsync(idx_dev, point_index, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, st));
        }
    }
    const int group = (method == PNPB200_METHOD_QEIF || method == PNPB200_METHOD_LINEAR_F1) ? 0
                      : (method == PNPB200_METHOD_LINEAR_F2 ? 2 : (method == PNPB200_METHOD_EIF2 ? 3 : 1));
    typedef int (*part_fn)(PNP_SOLVE_PART_ARGS);
    static const part_fn parts[2][4] = { { solve_part_f64_g0, solve_part_f64_g1, solve_part_f64_g2, solve_part_f64_g3 },
                                         { solve_part_f32_g0, solve_part_f32_g1, solve_part_f32_g2, solve_part_f32_g3 } };
    const int rc = parts[dtype == PNPB200_DTYPE_F64 ? 0 : 1][group](method, B, n_total, n, uv, pattern, n_patterns, point_index,
                                                                   idx_dev, K, prm, R, t, euler_deg, res_norm, iters,
                                                                   best_pattern, st, vis, wts);
    if (idx_dev) cudaFreeAsync(idx_dev, st);
    return rc;
}
}  // namespace pnpb200

extern "C" {

int pnpb200_solve_batch(int method, int dtype, int64_t B, int n_total, int n, const void* uv, const void* pattern,
                        int n_patterns, const int32_t* point_index, const double* K, const pnpb200_params* params,
                        void* R, void* t, void* euler_deg, void* res_norm, int32_t* iters, int32_t* best_pattern,
                        void* stream)
{
    pnpb200_params prm;
    if (params) prm = *params; else fill_default_params(&prm);
    prm.flags &= ~PNP_FLAG_INTERNAL_NO_RESIDUAL;
    return solve_batch_impl(method, dtype, B, n_total, n, uv, pattern, n_patterns, point_index, K, prm, R, t, euler_deg, res_norm,
                            iters, best_pattern, (cudaStream_t)stream);
}

int pnpb200_solve_batch_masked(int method, int dtype, int64_t B, int n_total, int n, const void* uv, const void* pattern,
                               int n_patterns, const int32_t* point_index, const double* K, const pnpb200_params* params,
                               void* R, void* t, void* euler_deg, void* res_norm, int32_t* iters, int32_t* best_pattern,
                               const uint32_t* visible, void* stream)
{
    if (!visible) return PNPB200_EINVAL;
    pnpb200_params prm;
    if (params) prm = *params; else fill_default_params(&prm);
    prm.flags &= ~PNP_FLAG_INTERNAL_NO_RESIDUAL;
    return solve_batch_impl(method, dtype, B, n_total, n, uv, pattern, n_patterns, point_index, K, prm, R, t, euler_deg, res_norm,
                            iters, best_pattern, (cudaStream_t)stream, visible);
}

int pnpb200_solve_batch_weighted(int method, int dtype, int64_t B, int n_total, int n, const void* uv, const void* pattern,
                                 int n_patterns, const int32_t* point_index, const double* K, const pnpb200_params* params,
                                 void* R, void* t, void* euler_deg, void* res_norm, int32_t* iters, int32_t* best_pattern,
                                 const float* weights, void* stream)
{
    if (!weights || ((uintptr_t)weights & 3u) != 0) return PNPB200_EINVAL;
    pnpb200_params prm;
    if (params) prm = *params; else fill_default_params(&prm);
    prm.flags &= ~PNP_FLAG_INTERNAL_NO_RESIDUAL;
    return solve_batch_impl(method, dtype, B, n_total, n, uv, pattern, n_patterns, point_index, K, prm, R, t, euler_deg, res_norm,
                            iters, best_pattern, (cudaStream_t)stream, nullptr, weights);
}

static int solve_report_impl(int method, int dtype, int64_t B, int n_total, int n, const void* uv, const void* pattern,
                             const int32_t* point_index, const double* K, const pnpb200_params* params,
                             void* R, void* t, void* euler_deg, void* res_norm, int32_t* iters,
                             const double* gt, const double* bounds, double* report, int64_t report_stride_problem,
                             int64_t report_stride_column, int32_t* flags, int32_t* max_idx, void* stream, const uint32_t* vis)
{
    if (!R || !t || !euler_deg || !gt || !report) return PNPB200_EINVAL;          // the report reads the pose
    pnpb200_params prm;
    if (params) prm = *params; else fill_default_params(&prm);
    prm.flags &= ~PNP_FLAG_INTERNAL_NO_RESIDUAL;
    cudaStream_t st = (cudaStream_t)stream;
    // One pass over the pixel rows for res_norm AND the report when the solve runs as the moment mapping over all
    // landmarks with chunk-streamed rows; every other shape is the two calls back to back.
    const bool moment = (method == PNPB200_METHOD_LM || method == PNPB200_METHOD_LINEAR_F2 || method == PNPB200_METHOD_LM_PLUS ||
                         (dtype == PNPB200_DTYPE_F64 && (method == PNPB200_METHOD_EIF2 ||
                          (method == PNPB200_METHOD_QEIF && n >= PNP_QEIF_HYBRID_MIN_N && !(prm.flags & PNPB200_FLAG_QEIF_DIRECT))))) &&
                        (prm.mapping == PNPB200_MAP_AUTO || prm.mapping == PNPB200_MAP_MOMENT);
    const bool fuse = !vis && moment && !point_index && n == n_total && res_norm && B > 0 && ((prm.flags >> 8) & 0xff) != 9 &&
                      (dtype == PNPB200_DTYPE_F64 || dtype == PNPB200_DTYPE_F32) && report_can_fuse(dtype, n_total);
    if (!fuse) {
        const int rc = solve_batch_impl(method, dtype, B, n_total, n, uv, pattern, 1, point_index, K, prm, R, t, euler_deg, res_norm,
                                        iters, nullptr, st, vis);
        if (rc != PNPB200_OK) return rc;
        return report_launch(dtype, B, n_total, pattern, uv, K, R, t, euler_deg, gt, bounds, report, report_stride_problem,
                             report_stride_column, flags, max_idx, nullptr, st, vis);
    }
    const size_t esz = (dtype == PNPB200_DTYPE_F64) ? 8 : 4;
    const size_t ws_bytes = (size_t)pnpb200_workspace_bytes(method, dtype, B, 1, PNPB200_MAP_MOMENT);
    void* ws = nullptr;
    const bool own_ws = !(prm.workspace && prm.workspace_bytes >= (int64_t)ws_bytes);
    if (own_ws) {
        PNP_CUDA_OK(cudaMallocAsync(&ws, ws_bytes, st));
        prm.workspace = ws; prm.workspace_bytes = (int64_t)ws_bytes;
    }
    prm.flags |= PNP_FLAG_INTERNAL_NO_RESIDUAL;
    int rc = solve_batch_impl(method, dtype, B, n_total, n, uv, pattern, 1, nullptr, K, prm, R, t, euler_deg, res_norm, iters,
                              nullptr, st);
    if (rc == PNPB200_OK) {
        ReportFuse f;
        f.res_mode = (method == PNPB200_METHOD_LINEAR_F2) ? 2 : 1;
        f.tail = (const char*)prm.workspace + (size_t)PNP_NMOM * (size_t)B * esz;
        f.ld = B;
        f.res = res_norm;
        double Kinv[9];
        host_inv3(K, Kinv);
        for (int e = 0; e < 6; ++e) f.kinv[e] = Kinv[e];
        const int slot = (prm.flags & PNPB200_FLAG_PROFILE) ? g_prof.last() : -1;
        rc = report_launch(dtype, B, n_total, pattern, uv, K, R, t, euler_deg, gt, bounds, report, report_stride_problem,
                           report_stride_column, flags, max_idx, &f, st);
        g_prof.mark(slot, st);                            // third interval of the call's profile slot: the fused report + residual
    }
    if (own_ws) cudaFreeAsync(ws, st);
    return rc;
}

int pnpb200_solve_report_batch(int method, int dtype, int64_t B, int n_total, int n, const void* uv, const void* pattern,
                               const int32_t* point_index, const double* K, const pnpb200_params* params,
                               void* R, void* t, void* euler_deg, void* res_norm, int32_t* iters,
                               const double* gt, const double* bounds, double* report, int64_t report_stride_problem,
                               int64_t report_stride_column, int32_t* flags, int32_t* max_idx, void* stream)
{
    return solve_report_impl(method, dtype, B, n_total, n, uv, pattern, point_index, K, params, R, t, euler_deg, res_norm, iters, gt,
                             bounds, report, report_stride_problem, report_stride_column, flags, max_idx, stream, nullptr);
}

int pnpb200_solve_report_batch_masked(int method, int dtype, int64_t B, int n_total, int n, const void* uv, const void* pattern,
                                      const int32_t* point_index, const double* K, const pnpb200_params* params,
                                      void* R, void* t, void* euler_deg, void* res_norm, int32_t* iters,
                                      const double* gt, const double* bounds, double* report, int64_t report_stride_problem,
                                      int64_t report_stride_column, int32_t* flags, int32_t* max_idx, const uint32_t* visible,
                                      void* stream)
{
    if (!visible) return PNPB200_EINVAL;
    return solve_report_impl(method, dtype, B, n_total, n, uv, pattern, point_index, K, params, R, t, euler_deg, res_norm, iters, gt,
                             bounds, report, report_stride_problem, report_stride_column, flags, max_idx, stream, visible);
}

// ------------------------------------------------------------------------------------------
// host-buffer entry point: chunked, multi-stream H2D -> solve -> D2H pipeline
// ------------------------------------------------------------------------------------------
// One slot = a stream with every device buffer a chunk needs.  Slots [0, n_streams) carry chunks as they
// are; the pack slots behind them carry chunks whose pixels went over PCIe as int16 (pnpb200_pack.cpp).
struct PipeSlot {
    cudaStream_t stream = nullptr;
    void *d_uv = nullptr, *d_R = nullptr, *d_t = nullptr, *d_e = nullptr, *d_res = nullptr, *d_ws = nullptr;
    int32_t *d_it = nullptr, *d_best = nullptr;
    int16_t *h_pack = nullptr, *d_pack = nullptr;        // pinned staging / device copy of the packed pixels
    void* d_narrow = nullptr;                             // device copy of a chunk of int16 / uint16 / float32 pixels (solve_batch_host_px)
    int32_t* d_status = nullptr;                          // outputs of the solution check (solve_check_batch_host), from its first call
    void* d_reproj = nullptr;
    uint32_t* d_vis = nullptr;                            // visibility words of a chunk (solve_batch_host_masked), from its first call
    uint32_t* h_vis = nullptr;                            // ... staged in pinned memory so that their copy is asynchronous
    cudaEvent_t vis_free = nullptr;                       // the H2D copy out of h_vis has finished
    cudaEvent_t pack_free = nullptr;                      // the H2D copy out of h_pack has finished
    cudaEvent_t h2d_done = nullptr;                       // the slot's last pixel copy has finished (back-pressure)
    cudaEvent_t piece_done[2] = { nullptr, nullptr };     // parts of a plain chunk's pixel copy, two in flight (submit_chunk)
};

struct pnpb200_pipeline {
    int dtype, n_total, n_patterns, n_streams, device;
    int pack_threads;                                     // 0: packed transfer off
    int64_t chunk;
    size_t esz;
    std::vector<PipeSlot> slots;                          // n_streams plain slots, then the pack slots
    size_t ws_bytes;
    void* d_pattern;
    int64_t last_packed, last_chunks;                     // chunks of the last call that travelled packed / all of them
};

constexpr int kPackSlots = 4;
#ifndef PNP_PLAIN_PIECES
#define PNP_PLAIN_PIECES 8
#endif
constexpr int kPlainPieces = PNP_PLAIN_PIECES;   // parts of a plain chunk's pixel copy beside the packing thread (submit_chunk)

static int alloc_slot(pnpb200_pipeline* p, PipeSlot& sl, bool pack)
{
    const size_t c = (size_t)p->chunk, esz = p->esz;
    PNP_CUDA_OK(cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking));
    PNP_CUDA_OK(cudaMalloc(&sl.d_uv, esz * c * p->n_total * 2));
    PNP_CUDA_OK(cudaMalloc(&sl.d_R, esz * c * 9));
    PNP_CUDA_OK(cudaMalloc(&sl.d_t, esz * c * 3));
    PNP_CUDA_OK(cudaMalloc(&sl.d_e, esz * c * 3));
    PNP_CUDA_OK(cudaMalloc(&sl.d_res, esz * c));
    PNP_CUDA_OK(cudaMalloc((void**)&sl.d_it, sizeof(int32_t) * c));
    PNP_CUDA_OK(cudaMalloc((void**)&sl.d_best, sizeof(int32_t) * c));
    PNP_CUDA_OK(cudaMalloc(&sl.d_ws, p->ws_bytes));
    PNP_CUDA_OK(cudaEventCreateWithFlags(&sl.h2d_done, cudaEventDisableTiming));
    for (cudaEvent_t& e : sl.piece_done) PNP_CUDA_OK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    if (pack) {
        const size_t pb = sizeof(int16_t) * (c * p->n_total * 2 + 8);
        PNP_CUDA_OK(cudaMallocHost((void**)&sl.h_pack, pb));
        PNP_CUDA_OK(cudaMalloc((void**)&sl.d_pack, pb));
        PNP_CUDA_OK(cudaEventCreateWithFlags(&sl.pack_free, cudaEventDisableTiming));
    }
    return PNPB200_OK;
}

static void free_slot(PipeSlot& sl)
{
    if (sl.stream) { cudaStreamSynchronize(sl.stream); cudaStreamDestroy(sl.stream); }
    cudaFree(sl.d_uv); cudaFree(sl.d_R); cudaFree(sl.d_t); cudaFree(sl.d_e); cudaFree(sl.d_res); cudaFree(sl.d_ws);
    cudaFree(sl.d_it); cudaFree(sl.d_best); cudaFree(sl.d_pack); cudaFree(sl.d_narrow); cudaFree(sl.d_status); cudaFree(sl.d_reproj); cudaFree(sl.d_vis);
    if (sl.h_pack) cudaFreeHost(sl.h_pack);
    if (sl.h_vis) cudaFreeHost(sl.h_vis);
    if (sl.vis_free) cudaEventDestroy(sl.vis_free);
    if (sl.pack_free) cudaEventDestroy(sl.pack_free);
    if (sl.h2d_done) cudaEventDestroy(sl.h2d_done);
    for (cudaEvent_t e : sl.piece_done) if (e) cudaEventDestroy(e);
    sl = PipeSlot();
}

int pnpb200_pipeline_create(pnpb200_pipeline** out, int dtype, int64_t chunk_problems, int n_total, int n_patterns,
                            int n_streams)
{
    if (!out || chunk_problems < 1 || n_total < 1 || n_patterns < 1 || n_patterns > PNPB200_MAX_PATTERNS) return PNPB200_EINVAL;
    if (dtype != PNPB200_DTYPE_F64 && dtype != PNPB200_DTYPE_F32) return PNPB200_EINVAL;
    if (n_streams < 1) n_streams = 3;
    pnpb200_pipeline* p = new pnpb200_pipeline();
    p->dtype = dtype; p->n_total = n_total; p->n_patterns = n_patterns; p->n_streams = n_streams;
    p->chunk = chunk_problems;
    p->esz = (dtype == PNPB200_DTYPE_F64) ? 8 : 4;
    p->d_pattern = nullptr;
    p->pack_threads = 0; p->last_packed = 0; p->last_chunks = 0;
    p->ws_bytes = (size_t)pnpb200_workspace_bytes(PNPB200_METHOD_LM, dtype, chunk_problems, 1, PNPB200_MAP_MOMENT);
    *out = p;
    PNP_CUDA_OK(cudaGetDevice(&p->device));
    PNP_CUDA_OK(cudaMalloc(&p->d_pattern, p->esz * (size_t)n_patterns * n_total * 3));
    p->slots.resize((size_t)n_streams);
    for (int s = 0; s < n_streams; ++s) {
        const int rc = alloc_slot(p, p->slots[(size_t)s], false);
        if (rc != PNPB200_OK) return rc;
    }
    return PNPB200_OK;
}

int pnpb200_pipeline_set_packing(pnpb200_pipeline* p, int n_threads)
{
    if (!p || n_threads < 0 || n_threads > 256) return PNPB200_EINVAL;
    if (n_threads > 0 && p->slots.size() == (size_t)p->n_streams) {       // first use: the pack slots
        p->slots.resize((size_t)p->n_streams + kPackSlots);
        for (size_t s = (size_t)p->n_streams; s < p->slots.size(); ++s) {
            const int rc = alloc_slot(p, p->slots[s], true);
            if (rc != PNPB200_OK) return rc;
        }
    }
    p->pack_threads = n_threads;
    return PNPB200_OK;
}

int pnpb200_pipeline_last_packed(const pnpb200_pipeline* p, int64_t* packed_chunks, int64_t* chunks)
{
    if (!p) return PNPB200_EINVAL;
    if (packed_chunks) *packed_chunks = p->last_packed;
    if (chunks) *chunks = p->last_chunks;
    return PNPB200_OK;
}

int pnpb200_host_alloc(void** out, int64_t bytes, int write_combined)
{
    if (!out || bytes < 0) return PNPB200_EINVAL;
    *out = nullptr;
    PNP_CUDA_OK(cudaHostAlloc(out, (size_t)(bytes > 0 ? bytes : 1), write_combined ? cudaHostAllocWriteCombined : cudaHostAllocDefault));
    return PNPB200_OK;
}

int pnpb200_host_free(void* ptr)
{
    if (ptr) PNP_CUDA_OK(cudaFreeHost(ptr));
    return PNPB200_OK;
}

int pnpb200_pipeline_destroy(pnpb200_pipeline* p)
{
    if (!p) return PNPB200_EINVAL;
    for (PipeSlot& sl : p->slots) free_slot(sl);
    if (p->d_pattern) cudaFree(p->d_pattern);
    delete p;
    return PNPB200_OK;
}

namespace {
size_t pixel_bytes(int pixel_type) { return pixel_type == PNPB200_PIXEL_F32 ? 4 : 2; }

struct HostCall {
    pnpb200_pipeline* p;
    int method, n, pixel_type;
    int64_t B;
    const void* uv_host;
    const int32_t* point_index;
    const double* K;
    const pnpb200_params* params;
    void *R, *t, *euler_deg, *res_norm;
    int32_t *iters, *best_pattern;
    int32_t* status;                                      // non-NULL: the solution check runs after each chunk's solve
    void* reproj;
    double reproj_limit_px;
    const uint32_t* vis;                                  // [B, ceil(n_total / 32)] host visibility words, or NULL
};

// queue one chunk on a slot: pixels host -> device (packed if `packed`), solve, results device -> host.
// pieces > 1 (plain FP64 / FP32 pixels beside a packing thread): the pixel copy goes out in that many parts and each
// part only when the one before has left the host, so that this thread never holds more than one part's worth of the
// host-to-device engine ahead of a packed chunk.
int submit_chunk(const HostCall& c, PipeSlot& sl, int64_t done, int64_t nb, bool packed, int pieces = 1)
{
    pnpb200_pipeline* p = c.p;
    const size_t esz = p->esz;
    cudaStream_t st = sl.stream;
    const size_t values = (size_t)nb * p->n_total * 2;
    if (packed) {
        PNP_CUDA_OK(cudaMemcpyAsync(sl.d_pack, sl.h_pack, sizeof(int16_t) * values, cudaMemcpyHostToDevice, st));
        PNP_CUDA_OK(cudaEventRecord(sl.pack_free, st));
        const int rc = widen_launch(PNPB200_PIXEL_I16, p->dtype, (long long)values, sl.d_pack, sl.d_uv, st);
        if (rc != PNPB200_OK) return rc;
    } else if (c.pixel_type != PNPB200_PIXEL_NATIVE) {
        // narrow detections as the caller holds them: a half / a quarter of the bytes cross PCIe, widened on the device
        const size_t psz = pixel_bytes(c.pixel_type);
        const char* src = (const char*)c.uv_host + psz * (size_t)done * p->n_total * 2;
        PNP_CUDA_OK(cudaMemcpyAsync(sl.d_narrow, src, psz * values, cudaMemcpyHostToDevice, st));
        PNP_CUDA_OK(cudaEventRecord(sl.h2d_done, st));
        const int rc = widen_launch(c.pixel_type, p->dtype, (long long)values, sl.d_narrow, sl.d_uv, st);
        if (rc != PNPB200_OK) return rc;
    } else {
        const char* src = (const char*)c.uv_host + esz * (size_t)done * p->n_total * 2;
        const int64_t per = (nb + pieces - 1) / pieces;
        int k = 0;
        for (int64_t b0 = 0; b0 < nb; b0 += per, ++k) {
            const int64_t pn = (nb - b0 < per) ? (nb - b0) : per;
            const size_t off = esz * (size_t)b0 * p->n_total * 2;
            if (k >= 2) PNP_CUDA_OK(cudaEventSynchronize(sl.piece_done[k & 1]));      // part k - 2 has left the host
            PNP_CUDA_OK(cudaMemcpyAsync((char*)sl.d_uv + off, src + off, esz * (size_t)pn * p->n_total * 2, cudaMemcpyHostToDevice, st));
            if (pieces > 1) PNP_CUDA_OK(cudaEventRecord(sl.piece_done[k & 1], st));
        }
        PNP_CUDA_OK(cudaEventRecord(sl.h2d_done, st));
    }
    const uint32_t* vis = nullptr;
    if (c.vis) {                                          // the chunk's mask travels with its pixels, on the same stream
        const size_t W = ((size_t)p->n_total + 31) / 32;
        PNP_CUDA_OK(cudaEventSynchronize(sl.vis_free));     // the slot's previous mask copy has left the staging buffer
        memcpy(sl.h_vis, c.vis + (size_t)done * W, sizeof(uint32_t) * W * (size_t)nb);
        PNP_CUDA_OK(cudaMemcpyAsync(sl.d_vis, sl.h_vis, sizeof(uint32_t) * W * (size_t)nb, cudaMemcpyHostToDevice, st));
        PNP_CUDA_OK(cudaEventRecord(sl.vis_free, st));
        vis = sl.d_vis;
    }
    pnpb200_params prm;
    if (c.params) prm = *c.params; else fill_default_params(&prm);
    prm.flags &= ~PNP_FLAG_INTERNAL_NO_RESIDUAL;
    // always the slot's own scratch: chunks run concurrently on several streams, one caller workspace would be shared by them
    prm.workspace = sl.d_ws; prm.workspace_bytes = (int64_t)p->ws_bytes;
    // the check reads the pose and the winning pattern whether or not the caller asked for them
    const bool chk = c.status != nullptr, want_best = c.best_pattern || (chk && p->n_patterns > 1);
    int rc = solve_batch_impl(c.method, p->dtype, nb, p->n_total, c.n, sl.d_uv, p->d_pattern, p->n_patterns,
                              c.point_index, c.K, prm, (c.R || chk) ? sl.d_R : nullptr, (c.t || chk) ? sl.d_t : nullptr,
                              c.euler_deg ? sl.d_e : nullptr, c.res_norm ? sl.d_res : nullptr,
                              c.iters ? sl.d_it : nullptr, want_best ? sl.d_best : nullptr, st, vis);
    if (rc != PNPB200_OK) return rc;
    if (chk) {
        rc = check_launch(p->dtype, nb, p->n_total, p->d_pattern, p->n_patterns, sl.d_uv, c.K, sl.d_R, sl.d_t,
                          c.res_norm ? sl.d_res : nullptr, p->n_patterns > 1 ? sl.d_best : nullptr, c.reproj_limit_px,
                          sl.d_status, c.reproj ? sl.d_reproj : nullptr, st, vis);
        if (rc != PNPB200_OK) return rc;
        PNP_CUDA_OK(cudaMemcpyAsync(c.status + done, sl.d_status, sizeof(int32_t) * (size_t)nb, cudaMemcpyDeviceToHost, st));
        if (c.reproj)
            PNP_CUDA_OK(cudaMemcpyAsync((char*)c.reproj + esz * (size_t)done * 2, sl.d_reproj, esz * (size_t)nb * 2, cudaMemcpyDeviceToHost, st));
    }
    if (c.R) PNP_CUDA_OK(cudaMemcpyAsync((char*)c.R + esz * (size_t)done * 9, sl.d_R, esz * (size_t)nb * 9, cudaMemcpyDeviceToHost, st));
    if (c.t) PNP_CUDA_OK(cudaMemcpyAsync((char*)c.t + esz * (size_t)done * 3, sl.d_t, esz * (size_t)nb * 3, cudaMemcpyDeviceToHost, st));
    if (c.euler_deg) PNP_CUDA_OK(cudaMemcpyAsync((char*)c.euler_deg + esz * (size_t)done * 3, sl.d_e, esz * (size_t)nb * 3, cudaMemcpyDeviceToHost, st));
    if (c.res_norm) PNP_CUDA_OK(cudaMemcpyAsync((char*)c.res_norm + esz * (size_t)done, sl.d_res, esz * (size_t)nb, cudaMemcpyDeviceToHost, st));
    if (c.iters) PNP_CUDA_OK(cudaMemcpyAsync(c.iters + done, sl.d_it, sizeof(int32_t) * (size_t)nb, cudaMemcpyDeviceToHost, st));
    if (c.best_pattern) PNP_CUDA_OK(cudaMemcpyAsync(c.best_pattern + done, sl.d_best, sizeof(int32_t) * (size_t)nb, cudaMemcpyDeviceToHost, st));
    return PNPB200_OK;
}
}  // namespace

int pnpb200_solve_batch_host(pnpb200_pipeline* p, int method, int64_t B, int n, const void* uv_host,
                             const void* pattern_host, const int32_t* point_index, const double* K,
                             const pnpb200_params* params, void* R, void* t, void* euler_deg, void* res_norm,
                             int32_t* iters, int32_t* best_pattern)
{
    return pnpb200_solve_batch_host_px(p, method, B, n, PNPB200_PIXEL_NATIVE, uv_host, pattern_host, point_index, K, params, R, t,
                                       euler_deg, res_norm, iters, best_pattern);
}

namespace {
int solve_host(pnpb200_pipeline* p, int method, int64_t B, int n, int pixel_type, const void* uv_host, const void* pattern_host,
               const int32_t* point_index, const double* K, const pnpb200_params* params, void* R, void* t, void* euler_deg,
               void* res_norm, int32_t* iters, int32_t* best_pattern, int32_t* status, void* reproj, double reproj_limit_px,
               const uint32_t* vis)
{
    if (!p || !uv_host || !pattern_host || !K || B < 0) return PNPB200_EINVAL;
    if (n < 1 || n > p->n_total || (!point_index && n != p->n_total)) return PNPB200_EINVAL;
    if (pixel_type == PNPB200_PIXEL_F32 && p->dtype == PNPB200_DTYPE_F32) pixel_type = PNPB200_PIXEL_NATIVE;
    if (pixel_type != PNPB200_PIXEL_NATIVE && pixel_type != PNPB200_PIXEL_I16 && pixel_type != PNPB200_PIXEL_U16 &&
        pixel_type != PNPB200_PIXEL_F32)
        return PNPB200_EINVAL;
    if (params && params->workspace) return PNPB200_EINVAL;   // the pipeline owns one scratch per stream
    const size_t esz = p->esz;
    if (pixel_type != PNPB200_PIXEL_NATIVE) {                  // first narrow call: the per-slot staging buffers
        for (int s = 0; s < p->n_streams; ++s) {
            PipeSlot& sl = p->slots[(size_t)s];
            if (!sl.d_narrow) PNP_CUDA_OK(cudaMalloc(&sl.d_narrow, 4 * ((size_t)p->chunk * p->n_total * 2 + 8)));
        }
    }
    if (status) {                                             // first checked call: the per-slot check outputs
        for (PipeSlot& sl : p->slots) {
            if (!sl.d_status) PNP_CUDA_OK(cudaMalloc((void**)&sl.d_status, sizeof(int32_t) * (size_t)p->chunk));
            if (!sl.d_reproj) PNP_CUDA_OK(cudaMalloc(&sl.d_reproj, esz * (size_t)p->chunk * 2));
        }
    }
    if (vis) {                                                // first masked call: the per-slot mask buffers, the larger scratch
        if (!vis_aligned(vis)) return PNPB200_EINVAL;
        const size_t W = ((size_t)p->n_total + 31) / 32;
        const size_t ws = (size_t)pnpb200_workspace_bytes_masked(PNPB200_METHOD_LM, p->dtype, p->chunk, 1, PNPB200_MAP_MOMENT);
        for (PipeSlot& sl : p->slots) {
            if (!sl.d_vis) {
                PNP_CUDA_OK(cudaMalloc((void**)&sl.d_vis, sizeof(uint32_t) * (size_t)p->chunk * W));
                PNP_CUDA_OK(cudaMallocHost((void**)&sl.h_vis, sizeof(uint32_t) * (size_t)p->chunk * W));
                PNP_CUDA_OK(cudaEventCreateWithFlags(&sl.vis_free, cudaEventDisableTiming));
            }
            if (p->ws_bytes < ws) {
                PNP_CUDA_OK(cudaStreamSynchronize(sl.stream));
                PNP_CUDA_OK(cudaFree(sl.d_ws));
                sl.d_ws = nullptr;
                PNP_CUDA_OK(cudaMalloc(&sl.d_ws, ws));
            }
        }
        if (p->ws_bytes < ws) p->ws_bytes = ws;
    }
    PNP_CUDA_OK(cudaMemcpyAsync(p->d_pattern, pattern_host, esz * (size_t)p->n_patterns * p->n_total * 3,
                                cudaMemcpyHostToDevice, p->slots[0].stream));
    PNP_CUDA_OK(cudaStreamSynchronize(p->slots[0].stream));
    const HostCall call = { p, method, n, pixel_type, B, uv_host, point_index, K, params, R, t, euler_deg, res_norm, iters, best_pattern,
                            status, reproj, reproj_limit_px, vis };
    const int64_t n_chunks = (B + p->chunk - 1) / p->chunk;
    p->last_chunks = n_chunks; p->last_packed = 0;
    // Chunks are handed out from both ends of the batch: this thread sends chunks as they are from the front
    // (PCIe-bound), a second thread packs chunks from the back with the pack threads (CPU-bound) and sends
    // those as int16; whichever is faster takes more of them, and they meet somewhere in the middle.
    std::mutex mu;
    int64_t lo = 0, hi = n_chunks - 1;
    auto claim = [&](bool from_back) -> int64_t {
        std::lock_guard<std::mutex> lk(mu);
        if (lo > hi) return -1;
        return from_back ? hi-- : lo++;
    };
    std::atomic<int> rc_pack{PNPB200_OK};
    std::atomic<long long> n_packed{0};
    char packer_error[sizeof(g_last_error)] = "";          // the packing thread's pnpb200_last_error(), handed to the caller
    std::thread packer;
    // narrow pixels are already as small as the packed transfer makes them: nothing to pack
    const bool packing = p->pack_threads > 0 && p->slots.size() > (size_t)p->n_streams && n_chunks >= 2 && pixel_type == PNPB200_PIXEL_NATIVE;
    if (packing) {
        const int64_t first = claim(true);                 // the last chunk is the packing thread's whatever the timing
        packer = std::thread([&, first]() {
            if (cudaSetDevice(p->device) != cudaSuccess) { rc_pack = PNPB200_ECUDA; return; }
            size_t s = (size_t)p->n_streams;
            for (int64_t c = first; c >= 0; c = claim(true)) {
                PipeSlot& sl = p->slots[s];
                const int64_t done = c * p->chunk, nb = (B - done < p->chunk) ? (B - done) : p->chunk;
                if (cudaEventSynchronize(sl.pack_free) != cudaSuccess) { rc_pack = PNPB200_ECUDA; break; }   // staging buffer free again
                const char* src = (const char*)uv_host + esz * (size_t)done * p->n_total * 2;
                const int exact = pnpb200_pack_i16(p->dtype, src, nb * p->n_total * 2, sl.h_pack, p->pack_threads);
                if (exact < 0) { rc_pack = exact; break; }
                const int rc = submit_chunk(call, sl, done, nb, exact == 1);
                if (rc != PNPB200_OK) { rc_pack = rc; break; }
                if (exact == 1) n_packed.fetch_add(1);
                s = (s + 1 < p->slots.size()) ? s + 1 : (size_t)p->n_streams;
            }
            if (rc_pack.load() != PNPB200_OK) memcpy(packer_error, g_last_error, sizeof(packer_error));   // thread-local there
        });
    }
    int rc_main = PNPB200_OK;
    int s = 0;
    // back-pressure: take the next chunk only when the pixel copy `depth` chunks back has left the host.  Copies of
    // all streams share the host-to-device engine in submission order, so with packing on only one plain copy is
    // kept queued -- a packed copy then waits for one chunk at most, and the rest of the batch stays open to the
    // packing thread; without packing a slot is simply reused when its turn comes.
    const int depth = packing ? 1 : p->n_streams;
    for (;;) {
        const int wait_slot = (s + p->n_streams - (depth % p->n_streams)) % p->n_streams;    // the slot used `depth` chunks ago
        if (cudaEventSynchronize(p->slots[(size_t)wait_slot].h2d_done) != cudaSuccess) { rc_main = PNPB200_ECUDA; break; }
        const int64_t c = claim(false);
        if (c < 0) break;
        const int64_t done = c * p->chunk, nb = (B - done < p->chunk) ? (B - done) : p->chunk;
        rc_main = submit_chunk(call, p->slots[(size_t)s], done, nb, false, packing ? kPlainPieces : 1);
        if (rc_main != PNPB200_OK) break;
        s = (s + 1) % p->n_streams;
        // a slot's buffers are reused n_streams chunks later; stream order protects them
    }
    if (rc_main != PNPB200_OK) { std::lock_guard<std::mutex> lk(mu); lo = hi + 1; }    // stop the packer
    if (packer.joinable()) packer.join();
    p->last_packed = n_packed.load();
    for (PipeSlot& sl : p->slots) PNP_CUDA_OK(cudaStreamSynchronize(sl.stream));
    if (rc_main != PNPB200_OK) return rc_main;
    if (rc_pack.load() != PNPB200_OK) memcpy(g_last_error, packer_error, sizeof(g_last_error));
    return rc_pack.load();
}
}  // namespace

int pnpb200_solve_batch_host_px(pnpb200_pipeline* p, int method, int64_t B, int n, int pixel_type, const void* uv_host,
                                const void* pattern_host, const int32_t* point_index, const double* K,
                                const pnpb200_params* params, void* R, void* t, void* euler_deg, void* res_norm,
                                int32_t* iters, int32_t* best_pattern)
{
    return solve_host(p, method, B, n, pixel_type, uv_host, pattern_host, point_index, K, params, R, t, euler_deg, res_norm, iters,
                      best_pattern, nullptr, nullptr, 0.0, nullptr);
}

int pnpb200_solve_check_batch_host(pnpb200_pipeline* p, int method, int64_t B, int n, int pixel_type, const void* uv_host,
                                   const void* pattern_host, const int32_t* point_index, const double* K,
                                   const pnpb200_params* params, void* R, void* t, void* euler_deg, void* res_norm,
                                   int32_t* iters, int32_t* best_pattern, double reproj_limit_px, int32_t* status, void* reproj)
{
    if (!status) return PNPB200_EINVAL;
    return solve_host(p, method, B, n, pixel_type, uv_host, pattern_host, point_index, K, params, R, t, euler_deg, res_norm, iters,
                      best_pattern, status, reproj, reproj_limit_px, nullptr);
}

int pnpb200_solve_batch_host_masked(pnpb200_pipeline* p, int method, int64_t B, int n, int pixel_type, const void* uv_host,
                                    const void* pattern_host, const int32_t* point_index, const double* K,
                                    const pnpb200_params* params, void* R, void* t, void* euler_deg, void* res_norm,
                                    int32_t* iters, int32_t* best_pattern, const uint32_t* visible, double reproj_limit_px,
                                    int32_t* status, void* reproj)
{
    if (!visible || (reproj && !status)) return PNPB200_EINVAL;
    return solve_host(p, method, B, n, pixel_type, uv_host, pattern_host, point_index, K, params, R, t, euler_deg, res_norm, iters,
                      best_pattern, status, reproj, reproj_limit_px, visible);
}

}  // extern "C"
