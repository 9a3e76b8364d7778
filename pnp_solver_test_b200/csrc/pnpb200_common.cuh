// pnpb200_common.cuh -- error plumbing and host helpers shared by the translation units.
#pragma once
#include <cuda.h>            // CUtensorMap (types only: the encoder is fetched through the runtime, no libcuda link)
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/pnpb200.h"

// workspace layout of the moment mapping: [PNP_NMOM][B] moments, [PNP_NTAIL][B] state before the last
// update (or the F2 tail), PNP_PATC pattern constants (see pnpb200_solvers.cuh)
#define PNP_NMOM 30        // rows of the moment workspace: the 29 moments LM / linear F2 use + sum (bx^2 + by^2) (filters' residual)
#define PNP_NMOM_LM 29     // ... of which LM, LM+ and linear F2 read and write the first 29
#define PNP_NCORE 33        // constants of the LM system kept next to the moments by k_iterate (S33 6, S13 9, S23 9, c 9)
#define PNP_NTAIL 12
#define PNP_PATC 20
#define PNP_NPMOM 10       // masked moment mapping: per-problem pattern moments (sum theta theta^T 6, sum theta 3, count) behind the moments
// landmark selections up to this size travel inside the kernel arguments; larger ones through device memory
#define PNP_MAX_INLINE_IDX 96
// QEIF takes H^T H, H^T v (and, in the moment mapping, the residual of its exit test) from the moments from this many landmarks on
#define PNP_QEIF_HYBRID_MIN_N 12
// internal bit of pnpb200_params.flags (masked off at the C ABI): the moment mapping skips its residual pass
#define PNP_FLAG_INTERNAL_NO_RESIDUAL (1 << 30)

namespace pnpb200 {

void set_last_error(const char* where, cudaError_t e);   // defined in pnpb200_api.cu

#define PNP_CUDA_OK(call)                                                   \
    do {                                                                    \
        cudaError_t _e = (call);                                            \
        if (_e != cudaSuccess) {                                            \
            ::pnpb200::set_last_error(#call, _e);                           \
            return (_e == cudaErrorNoDevice || _e == cudaErrorInsufficientDriver) ? PNPB200_ENODEVICE \
                                                                                  : PNPB200_ECUDA;   \
        }                                                                   \
    } while (0)

// np.linalg.inv(K) for the 3x3 camera matrix (PNP_SOLVER_LIB.py:2596, :2811), on the host.
inline void host_inv3(const double* M, double* out)
{
    const double d = M[0] * (M[4] * M[8] - M[5] * M[7]) - M[1] * (M[3] * M[8] - M[5] * M[6]) +
                     M[2] * (M[3] * M[7] - M[4] * M[6]);
    const double id = 1.0 / d;
    out[0] = (M[4] * M[8] - M[5] * M[7]) * id; out[1] = (M[2] * M[7] - M[1] * M[8]) * id; out[2] = (M[1] * M[5] - M[2] * M[4]) * id;
    out[3] = (M[5] * M[6] - M[3] * M[8]) * id; out[4] = (M[0] * M[8] - M[2] * M[6]) * id; out[5] = (M[2] * M[3] - M[0] * M[5]) * id;
    out[6] = (M[3] * M[7] - M[4] * M[6]) * id; out[7] = (M[1] * M[6] - M[0] * M[7]) * id; out[8] = (M[0] * M[4] - M[1] * M[3]) * id;
}

struct DeviceProps {
    int device, sm_count, cc_major, cc_minor, max_smem_optin;
    size_t total_mem;
};
int get_device_props(DeviceProps* out);   // cached per device; defined in pnpb200_api.cu

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) and the occupancy query, remembered per (device, kernel): both cost
// tens of microseconds on the host, which is visible when a call is only a few hundred microseconds of kernels
void count_kernel_launches(int n);   // kernels this library has launched (pnpb200_launch_count); defined in pnpb200_api.cu
// 2-D tensor map over the pixel rows uv[B][n_total][2]: box = (chunk_points x 32 problems); returns 0 when
// the driver entry point is missing or the shape does not qualify (callers keep the per-row copies).  pnpb200_api.cu
int make_row_tensor_map(CUtensorMap* out, const void* uv, int elem_bytes, long long B, int n_total, int chunk_points);
// narrow pixels (PNPB200_PIXEL_I16 / U16 / F32) -> the arithmetic type, on the device; pnpb200_aux.cu
int widen_launch(int pixel_type, int dtype, long long n_values, const void* in, void* out, cudaStream_t stream);
// error report (pnpb200_aux.cu); with `fuse` the streaming report kernel also evaluates res_norm of the moment mapping
struct ReportFuse { int res_mode; /* 1: LM, 2: linear F2 */ const void* tail; long long ld; void* res; double kinv[6]; };
bool report_can_fuse(int dtype, int n);
int report_launch(int dtype, int64_t B, int n, const void* pattern, const void* uv, const double* K, const void* R, const void* t,
                  const void* euler_deg, const double* gt, const double* bounds, double* report, int64_t report_stride_problem,
                  int64_t report_stride_column, int32_t* flags, int32_t* max_idx, const ReportFuse* fuse, cudaStream_t st,
                  const uint32_t* vis = nullptr);
// a visibility mask [B, ceil(n_total / 32)] uint32 must be 4-byte aligned
inline bool vis_aligned(const uint32_t* vis) { return ((uintptr_t)vis & 3u) == 0; }
// solution check (pnpb200_check_batch), pnpb200_aux.cu
int check_launch(int dtype, int64_t B, int n, const void* pattern, int n_patterns, const void* uv, const double* K,
                 const void* R, const void* t, const void* res_norm, const int32_t* best_pattern, double limit,
                 int32_t* status, void* reproj, cudaStream_t st, const uint32_t* vis = nullptr);
// pnpb200_solve_batch(_masked) without the entry's parameter copy (pnpb200_api.cu); vis = nullptr: every landmark
int solve_batch_impl(int method, int dtype, int64_t B, int n_total, int n, const void* uv, const void* pattern, int n_patterns,
                     const int32_t* point_index, const double* K, const pnpb200_params& prm, void* R, void* t, void* euler_deg,
                     void* res_norm, int32_t* iters, int32_t* best_pattern, cudaStream_t st, const uint32_t* vis = nullptr);
// the hypothesis stage (pnpb200_hypothesize_batch) with its parameters given, and their checks; pnpb200_ransac.cu
bool hypothesis_params_ok(const pnpb200_hypothesis_params& h);
void fill_default_hypothesis(pnpb200_hypothesis_params* h);
int hypothesize_impl(int dtype, int64_t B, int n_total, int n, const void* uv, const void* pattern, int n_patterns,
                     const int32_t* point_index, const double* K, const uint32_t* visible, const pnpb200_hypothesis_params& hp,
                     void* R, void* t, int32_t* best_pattern, uint32_t* consensus_mask, int32_t* consensus, int32_t* drawn,
                     cudaStream_t st);
cudaError_t set_dynamic_smem(const void* kernel, size_t bytes);                                   // defined in pnpb200_api.cu
cudaError_t blocks_per_sm(int* out, const void* kernel, int block_threads, size_t smem_bytes);   // defined in pnpb200_api.cu

// ------------------------------------------------------------------------------------------
// optional per-kernel timing (PNPB200_FLAG_PROFILE): a ring of event quadruples per host thread
// ------------------------------------------------------------------------------------------
struct ProfileRing {
    static constexpr int kSlots = 64;
    cudaEvent_t ev[kSlots][4];
    int used[kSlots];     // number of events recorded in the slot (0 = empty)
    bool created = false;
    int next = 0, count = 0;
    int begin()
    {
        if (!created) {
            for (int s = 0; s < kSlots; ++s) {
                for (int e = 0; e < 4; ++e) cudaEventCreate(&ev[s][e]);
                used[s] = 0;
            }
            created = true;
        }
        const int s = next;
        next = (next + 1) % kSlots;
        if (count < kSlots) ++count;
        used[s] = 0;
        return s;
    }
    int last() const { return count ? (next + kSlots - 1) % kSlots : -1; }   // the slot of the most recent begin()
    // Inside a stream capture the record becomes an event-record NODE of the graph (cudaEventRecordExternal): every
    // replay of the graph re-records the event, so the times read afterwards are those of the last replay.
    void mark(int slot, cudaStream_t st)
    {
        if (slot < 0 || used[slot] >= 4) return;
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(st, &cs) != cudaSuccess) { cudaGetLastError(); cs = cudaStreamCaptureStatusNone; }
        cudaEventRecordWithFlags(ev[slot][used[slot]++], st,
                                 cs == cudaStreamCaptureStatusActive ? cudaEventRecordExternal : cudaEventRecordDefault);
    }
};
extern thread_local ProfileRing g_prof;            // defined in pnpb200_api.cu

// ------------------------------------------------------------------------------------------
// The templated solve path (pnpb200_kernels.cu) is compiled once per (scalar type, method group)
// so that the objects build in parallel; pnpb200_api.cu dispatches to these entry points.
//   group 0: QEIF, linear F1      group 1: LM, LM+      group 2: linear F2      group 3: EIF2
// ------------------------------------------------------------------------------------------
#define PNP_SOLVE_PART_ARGS                                                                                          \
    int method, long long B, int n_total, int n, const void *uv, const void *pattern, int n_patterns,                 \
        const int32_t *idx_host, const int32_t *idx_dev, const double *K, const pnpb200_params &prm, void *R, void *t, \
        void *euler, void *res, int32_t *iters, int32_t *best, cudaStream_t stream, const uint32_t *vis
int solve_part_f64_g0(PNP_SOLVE_PART_ARGS);
int solve_part_f64_g1(PNP_SOLVE_PART_ARGS);
int solve_part_f64_g2(PNP_SOLVE_PART_ARGS);
int solve_part_f64_g3(PNP_SOLVE_PART_ARGS);
int solve_part_f32_g0(PNP_SOLVE_PART_ARGS);
int solve_part_f32_g1(PNP_SOLVE_PART_ARGS);
int solve_part_f32_g2(PNP_SOLVE_PART_ARGS);
int solve_part_f32_g3(PNP_SOLVE_PART_ARGS);
void fill_default_params(pnpb200_params* p);          // defined in pnpb200_api.cu

}  // namespace pnpb200
