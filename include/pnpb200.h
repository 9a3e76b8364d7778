/*
 * pnpb200.h -- C ABI of the B200-native batched PnP solver (libpnpb200.so).
 *
 * The reference (Benson516/pnp_solver_test) is pure Python and has no FFI boundary: its
 * boundary is the class PNP_SOLVER in scripts/PNP_SOLVER_LIB.py.  Every entry point below
 * names the reference interface it replaces (file:line, relative to the reference root).
 * The Python mirror of that class (pnp_solver_test_b200/solver.py) binds these symbols with
 * ctypes; INTEGRATION.md shows the stub a maintainer of the reference would add.
 *
 * Conventions
 *  - extern "C", plain pointers and sizes.  No torch types.
 *  - Pointers marked [device] are CUDA device pointers owned by the caller, 16-byte aligned;
 *    [host] are ordinary host pointers read during the call.
 *  - Every call is asynchronous on `stream` (a cudaStream_t passed as void*; NULL = default
 *    stream) unless stated otherwise.  The library allocates nothing persistent except inside
 *    a pnpb200_pipeline (host entry point), which the caller creates and destroys.
 *  - Return value: 0 on success, a negative PNPB200_E* code otherwise.  Like the reference,
 *    the numeric path never raises: a diverged solve returns garbage R/t and a large res_norm.
 *  - dtype selects BOTH the I/O element type of the float arrays and the arithmetic type.
 *    FP64 is the parity mode (the reference is float64 only).
 */
#ifndef PNPB200_H
#define PNPB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PNPB200_VERSION 100

/* method: which single-pattern solver of the reference to run */
#define PNPB200_METHOD_QEIF       0  /* solve_pnp_QEIF_single_pattern,          PNP_SOLVER_LIB.py:2771-3025 (what solve_pnp() dispatches to, :179) */
#define PNPB200_METHOD_LM         1  /* solve_pnp_LM_single_pattern,            PNP_SOLVER_LIB.py:2567-2769 */
#define PNPB200_METHOD_LINEAR_F2  2  /* solve_pnp_formulation_2_single_pattern, PNP_SOLVER_LIB.py:693-953   */
#define PNPB200_METHOD_LINEAR_F1  3  /* solve_pnp_single_pattern,               PNP_SOLVER_LIB.py:205-430   */
#define PNPB200_METHOD_LM_PLUS    4  /* NOT in the reference (non-parity extra): linear F2 initial pose, then LM's 12-state
                                        damped Gauss-Newton with the true constraint gradients and a convergence test
                                        (max |dx| <= 1e-10); res_norm at the returned state; moment mapping only */
#define PNPB200_METHOD_EIF2       5  /* solve_pnp_EIF2_single_pattern,          PNP_SOLVER_LIB.py:2001-2276: iterated information filter
                                        on LM's 12-state model with EKF2_get_process_covariance_R (:3668-3716) and QEIF's early exit */

#define PNPB200_DTYPE_F64 0
#define PNPB200_DTYPE_F32 1

/* execution shape (0 = let the library choose from n) */
#define PNPB200_MAP_AUTO    0
#define PNPB200_MAP_THREAD  1   /* one problem per thread, correspondences staged in shared memory */
#define PNPB200_MAP_MOMENT  2   /* moments -> O(1) iterations -> point-wise residual, as three      */
                                /* streaming kernels: LM, LM+, linear F2 and, in FP64, EIF2 and     */
                                /* QEIF from 12 landmarks on (their exit decisions certified, the   */
                                /* rest re-solved point-wise by a fix-up pass).  The default there; */
                                /* several patterns: one such solve per pattern, arg-min in between */
#define PNPB200_MAP_WARP    32  /* one problem per warp, shuffle-reduced normal equations          */

#define PNPB200_OK          0
#define PNPB200_EINVAL     -1   /* bad argument (null pointer, n < 1, unknown method/dtype, ...)   */
#define PNPB200_ECUDA      -2   /* a CUDA runtime call failed; see pnpb200_last_error()            */
#define PNPB200_ENODEVICE  -3   /* no usable CUDA device                                           */
#define PNPB200_ETOOLARGE  -4   /* n exceeds what the selected mapping can hold                    */

#define PNPB200_FLAG_PROFILE 1  /* record CUDA events around each kernel of the call (pnpb200_profile_read) */
#define PNPB200_FLAG_QEIF_DIRECT 2 /* QEIF in the direct mappings: accumulate H^T H point by point even for n >= 12 (default there: from
                                      the moments); with PNPB200_MAP_AUTO it also keeps QEIF out of the moment mapping */
#define PNPB200_FLAG_LM_TRUE_JACOBIAN 4 /* method LM only, NOT a parity mode: the reference's loop (identity start, max_it iterations,
                                           constant lambda) with the true gradients of its nine constraint rows (2u for the quadratic rows,
                                           u/|u| for the norm rows) in place of the halved ones it uses (PNP_SOLVER_LIB.py:3787-3823);
                                           moment mapping only */

#define PNPB200_MAX_PATTERNS 8
#define PNPB200_REPORT_WIDTH 16

/* Solver constants.  The reference hard-codes these inline; defaults reproduce it. */
typedef struct pnpb200_params {
    int32_t max_it;        /* 14      PNP_SOLVER_LIB.py:2635 (LM), :2857 (QEIF)                   */
    int32_t linear_it;     /* 3       :223 (F1), :762 (F2)                                         */
    double  lm_lambda;     /* 1e-5    :2631  constant damping                                      */
    double  exit_tol;      /* 1e-2    :2952  QEIF early exit on |d res / res|                      */
    double  f_weight;      /* 225.68  :2845  focal length used in the measurement weight (NOT K)   */
    double  meas_sigma_px; /* 3.0     :2846                                                        */
    double  proc_q;        /* 1e-1    :2792  process noise, quaternion states                      */
    double  proc_d;        /* 1e-2    :2793  process noise, delta states                           */
    double  omega0;        /* 1e-5    :2836  initial information                                   */
    double  res_old0;      /* 1e-7    :2863                                                        */
    int32_t mapping;       /* PNPB200_MAP_*                                                        */
    int32_t flags;         /* PNPB200_FLAG_*                                                       */
    void*   workspace;     /* [device] optional scratch of workspace_bytes (pnpb200_workspace_bytes);  */
    int64_t workspace_bytes; /* NULL/0: the call takes it from the stream-ordered CUDA memory pool   */
} pnpb200_params;

/* Synthetic workload description (random_stress_test.py:246-258, LM_noise_test.py:141-189). */
typedef struct pnpb200_synth {
    uint64_t seed;            /* Philox4x32-10 key; the counter is the GLOBAL problem index        */
    double   angle_range_deg; /* 45    roll, pitch, yaw ~ U(-a, a)                                 */
    double   depth_min_m;     /* 0.20                                                              */
    double   depth_max_m;     /* 2.25                                                              */
    double   fov_max_deg;     /* 45    t = depth * [tan U(-f,f), tan U(-f,f), 1]                   */
    int32_t  is_quantized;    /* round pixels to multiples of quantize_q (np.around)               */
    int32_t  reserved;
    double   quantize_q;      /* 1.0                                                               */
    double   noise_sigma_px;  /* 0 = none; Gaussian pixel noise added after quantisation           */
    double   roll_center_deg; /* 0    angles are centre + U(-angle_range, angle_range); a fixed    */
    double   pitch_center_deg;/* 0    pose (LM_noise_test.py:180-182, :262) is range 0 + centres   */
    double   yaw_center_deg;  /* 0                                                                 */
} pnpb200_synth;

int pnpb200_version(void);
int64_t pnpb200_launch_count(void);             /* kernels launched by this library since it was loaded (all threads) */
const char* pnpb200_last_error(void);          /* text of the last CUDA error seen by this thread */
int pnpb200_default_params(pnpb200_params* p);
int pnpb200_default_synth(pnpb200_synth* s);
int pnpb200_device_info(int* sm_count, int* cc_major, int* cc_minor, int64_t* hbm_bytes);
/* scratch bytes pnpb200_solve_batch needs for this call shape (0 for the direct mappings; QEIF: sized for the
   moment mapping, which it uses from 12 landmarks on) */
int64_t pnpb200_workspace_bytes(int method, int dtype, int64_t B, int n_patterns, int mapping);

/*
 * The hot path.  Replaces the per-problem loop around PNP_SOLVER.solve_pnp
 * (PNP_SOLVER_LIB.py:144-203; callers random_stress_test.py:322, LM_noise_test.py:312,
 * face_variation_test.py:431) and the solve_pnp_*_single_pattern methods it dispatches to.
 * One launch does, per problem: correspondence packing and K^-1 normalisation
 * (f2_get_P :3260, f2_get_B_xy :3291), the selected solver for each of the n_patterns patterns,
 * the arg-min over patterns on res_norm (strict <, first wins; :185), (R, t) reconstruction
 * (:3500 / :3542 / :4158) and Euler extraction (:4474).
 *
 *   uv        [device] [B, n_total, 2] pixels (u, v); the homogeneous coordinate is 1
 *   pattern   [device] [n_patterns, n_total, 3] metres, shared by all problems
 *   point_index [host] n indices into 0..n_total-1 selecting (and ordering) the landmarks the
 *             solver sees -- the LM_key_list of PNP_SOLVER_LIB.py:156 -- or NULL for all n_total
 *   K         [host] [3,3] row-major camera matrix (np_K_camera_est)
 *   params    [host] or NULL for defaults
 *   R [B,9]  t [B,3]  euler_deg [B,3] = (roll, yaw, pitch)  res_norm [B]      [device], dtype
 *   iters [B]  best_pattern [B]                                           [device], int32
 *             (any output pointer may be NULL to skip it)
 */
int pnpb200_solve_batch(int method, int dtype, int64_t B, int n_total, int n,
                        const void* uv, const void* pattern, int n_patterns,
                        const int32_t* point_index, const double* K,
                        const pnpb200_params* params,
                        void* R, void* t, void* euler_deg, void* res_norm,
                        int32_t* iters, int32_t* best_pattern, void* stream);

/*
 * Image points whose homogeneous coordinate is not 1.  The reference's packing stage multiplies the (3,1) vector it is
 * given by K^-1 without looking at its third entry (f2_get_B_xy, PNP_SOLVER_LIB.py:3305-3307), and its own projection
 * emits w = -1 for points behind the camera (perspective_projection :4548).  This entry computes that product for
 * n_points points, uvw [n_points, 3] -> uv_normalised [n_points, 2] = rows 0, 1 of K^-1 [u, v, w]^T (both device, dtype);
 * pnpb200_solve_batch is then called on uv_normalised with K = identity.  (Pixels with w = 1 need none of this.)
 */
int pnpb200_normalise_uvw(int dtype, int64_t n_points, const void* uvw, const double* K, void* uv_normalised, void* stream);

/*
 * Per-kernel device times of the pnpb200_solve_batch calls made by this thread with
 * PNPB200_FLAG_PROFILE since the last reset, measured with CUDA events on the call's stream.
 * ms[3] = average duration of (moments | direct solve kernel, iterate, residual); kernels a
 * mapping does not launch report 0.  pnpb200_profile_read synchronises with the recorded events.
 */
int pnpb200_profile_reset(void);
int pnpb200_profile_read(float* ms, int* n_calls);

/*
 * Same, from HOST buffers (pageable or pinned), chunked and double-buffered through a
 * caller-created pipeline so that H2D copies, the solve kernel and D2H copies overlap.
 * This is the call the drop-in PNP_SOLVER.solve_pnp_batch_host() makes for NumPy inputs and what
 * bench.py times as `e2e`.  Blocks until the results are in the host buffers.
 */
typedef struct pnpb200_pipeline pnpb200_pipeline;
int pnpb200_pipeline_create(pnpb200_pipeline** out, int dtype, int64_t chunk_problems, int n_total,
                            int n_patterns, int n_streams);
int pnpb200_pipeline_destroy(pnpb200_pipeline* p);

/*
 * Packed pixel transfer for pnpb200_solve_batch_host.  Detected landmarks are whole pixels
 * (random_stress_test.py projects with is_quantized=True, PNP_SOLVER_LIB.py:4549-4552) that the
 * reference carries as float64.  With n_threads > 0 a second host thread takes chunks from the far end
 * of the batch, converts each to int16 with n_threads workers (pnpb200_pack_i16) and, if that was exact
 * for every value of the chunk, ships the int16 copy (a quarter of the PCIe bytes) and widens it on the
 * device -- the solver sees the same values; chunks that are not whole numbers travel as they are.
 * The calling thread keeps sending chunks unchanged from the near end (in eighths, two in flight, so that a
 * packed copy never queues behind a whole plain chunk), so PCIe and the CPU work at the same time and share
 * the batch by their speeds.  n_threads = 0 switches it off (the default).
 * pnpb200_pipeline_last_packed: how many chunks of the last call travelled packed, of how many.
 */
int pnpb200_pipeline_set_packing(pnpb200_pipeline* p, int n_threads);
int pnpb200_pipeline_last_packed(const pnpb200_pipeline* p, int64_t* packed_chunks, int64_t* chunks);

/*
 * Host helper of the packed transfer: dst[i] = (int16) src[i] for n_values FP64 / FP32 values (dtype),
 * on n_threads threads (the calling thread and n_threads - 1 workers that stay alive, asleep, between calls;
 * concurrent calls take turns).  Returns 1 if every value was a whole number in [-32768, 32767] (the packing is
 * lossless; -0.0 counts as 0), 0 if not (dst is then not to be used), < 0 on a bad argument.
 */
int pnpb200_pack_i16(int dtype, const void* src, int64_t n_values, int16_t* dst, int n_threads);
/* params->workspace must be NULL here (EINVAL otherwise): the chunks run concurrently and the pipeline owns one scratch per stream */
int pnpb200_solve_batch_host(pnpb200_pipeline* p, int method, int64_t B, int n,
                             const void* uv_host, const void* pattern_host,
                             const int32_t* point_index, const double* K,
                             const pnpb200_params* params,
                             void* R, void* t, void* euler_deg, void* res_norm,
                             int32_t* iters, int32_t* best_pattern);

/*
 * The same for callers that hold their detections in a narrow type.  Landmark detectors deliver whole pixels
 * (the reference rounds them itself: is_quantized=True, PNP_SOLVER_LIB.py:4549-4552, random_stress_test.py:290)
 * and only the reference's dict-of-float64 convention makes them 16 bytes per landmark.  uv_host is
 * [B, n_total, 2] of pixel_type; a half (float32) or a quarter (int16 / uint16) of the bytes cross PCIe and the
 * values are widened on the device to the pipeline's arithmetic type -- exactly, so the results are bit-identical
 * to those of the same values handed over in the pipeline's dtype.  PNPB200_PIXEL_NATIVE = pnpb200_solve_batch_host.
 * No host pass, no packing thread: nothing on this path touches the pixels on the CPU.
 */
#define PNPB200_PIXEL_NATIVE 0   /* the pipeline's dtype */
#define PNPB200_PIXEL_I16    1
#define PNPB200_PIXEL_U16    2
#define PNPB200_PIXEL_F32    3   /* float32 pixels, arithmetic in the pipeline's dtype */
int pnpb200_solve_batch_host_px(pnpb200_pipeline* p, int method, int64_t B, int n, int pixel_type,
                                const void* uv_host, const void* pattern_host,
                                const int32_t* point_index, const double* K,
                                const pnpb200_params* params,
                                void* R, void* t, void* euler_deg, void* res_norm,
                                int32_t* iters, int32_t* best_pattern);

/*
 * pnpb200_solve_batch_host_px with the solution check (pnpb200_check_batch) of every chunk on the chunk's stream,
 * right after its solve, on the pixels in the pipeline's dtype (after widening) and the solve's best_pattern: the
 * per-problem loop of random_stress_test.py:322 with a verdict per pose, for callers without ground truth.
 * status [B] int32 (required) and reproj [B, 2] (pipeline dtype, may be NULL) are host buffers filled like the others;
 * res_norm enters the NONFINITE bit only where it is requested.  Every other output is that of
 * pnpb200_solve_batch_host_px.  The pipeline allocates the device buffers of the two outputs on its first checked call.
 */
int pnpb200_solve_check_batch_host(pnpb200_pipeline* p, int method, int64_t B, int n, int pixel_type,
                                   const void* uv_host, const void* pattern_host,
                                   const int32_t* point_index, const double* K,
                                   const pnpb200_params* params,
                                   void* R, void* t, void* euler_deg, void* res_norm,
                                   int32_t* iters, int32_t* best_pattern,
                                   double reproj_limit_px, int32_t* status, void* reproj);

/*
 * Page-locked host memory for the buffers of the two calls above (cudaHostAlloc): copies from / to pinned memory
 * run asynchronously at full PCIe rate, pageable buffers are staged by the driver and block the submitting thread.
 * write_combined = 1 for buffers the CPU only WRITES (the pixels): not snooped, faster for the device to read,
 * very slow for the CPU to read back -- do not use it for the result buffers or with the packed transfer.
 */
int pnpb200_host_alloc(void** out, int64_t bytes, int write_combined);
int pnpb200_host_free(void* ptr);

/*
 * Euler <-> R, batched on the device.
 * Replaces get_rotation_matrix_from_Euler (PNP_SOLVER_LIB.py:4442-4472) and
 * get_Euler_from_rotation_matrix (:4474-4517).  euler = (roll, yaw, pitch).
 */
int pnpb200_R_from_euler(int dtype, int64_t B, const void* euler, int is_degree, void* R, void* stream);
int pnpb200_euler_from_R(int dtype, int64_t B, const void* R, int is_degree, void* euler, void* stream);

/*
 * Pinhole projection of a pattern, batched.  Replaces perspective_projection (:4532-4557) and
 * perspective_projection_golden_landmarks (:4586-4621): K (R theta + t) / |z|, optional
 * rounding to a grid (np.around = half to even).  uvw: [B, n, 3] homogeneous pixels.
 */
int pnpb200_project(int dtype, int64_t B, int n, const void* pattern, const double* K,
                    const void* R, const void* t, int is_quantized, double quantize_q,
                    void* uvw, void* stream);

/*
 * Synthetic workload generator, FP64 internally.  Problems b0 .. b0+B-1 of a global
 * counter-based stream, so a shard reproduces exactly the slice of the unsharded run.
 *   uv [B,n,2] (dtype)   gt [B,4] = (distance m, roll, pitch, yaw deg) (f64)
 *   R_gt [B,9], t_gt [B,3] (f64, may be NULL)
 * Workload definition: random_stress_test.py:246-290 (+ LM_noise_test.py noise).
 */
int pnpb200_synth_batch(int dtype, int64_t b0, int64_t B, int n, const void* pattern_f64,
                        const double* K, const pnpb200_synth* cfg,
                        void* uv, double* gt, double* R_gt, double* t_gt, void* stream);

/*
 * The workload of face_variation_test.py (:296-356): the same pose stream, but the pixels are the
 * projection of a PERTURBED pattern -- a random direction of the 3 (n - 1) coordinates of all
 * landmarks but `fixed_index` ("eye_c_51", :318; -1 = none fixed), scaled to perturb_radius_m
 * (0.02, :319) -- while the solver keeps the golden pattern.  perturb [B,n,3] (f64, may be NULL)
 * receives np_pattern_perturbation_dict of each problem, the input of pnpb200_fragility_accumulate.
 */
int pnpb200_synth_face_variation(int dtype, int64_t b0, int64_t B, int n, const void* pattern_f64,
                                 const double* K, const pnpb200_synth* cfg, double perturb_radius_m,
                                 int fixed_index, void* uv, double* gt, double* R_gt, double* t_gt,
                                 double* perturb, void* stream);

/*
 * Error reporting per problem.  Replaces check_if_the_sample_passed (TEST_TOOLBOX.py:55-62),
 * cal_LM_error_distances (:252-286), the error fields of compare_result_and_generate_result_dict
 * (:396-463) and the glue at random_stress_test.py:353-377.  Always FP64 outputs.
 *   report [B,16]: 0 depth_err(m) 1 roll_err 2 pitch_err 3 yaw_err (deg)
 *                  4,5 LM_GT avg,max  6,7 predict_LM avg,max  8,9 predict_GT avg,max (x distance_GT)
 *                  10 t3_est 11 distance_GT 12 roll_est 13 pitch_est 14 yaw_est 15 reserved
 *   flags [B,4] = depth, roll, pitch, yaw passed;  max_idx [B,3] = landmark index of each max
 *   bounds [host] 4 doubles (10 cm, 10, 10, 10 deg in the reference; NULL = 10 each)
 * The depth flag is |t3 * 100 - distance_GT * 100| < bounds[0] with both products rounded to FP64 before the difference,
 * as the reference evaluates it; the angle flags are |est - GT| < bound; a NaN fails.  A landmark distance whose square is
 * not finite (a projection at depth exactly 0, a non-finite pixel) is NaN, as in the solution check: the mean is then NaN
 * and that landmark is never the maximum (strict >, the first landmark wins ties, -1 when no distance is > 0).  The
 * prediction-vs-GT difference is taken through the pixel, (prediction - pixel) + (pixel - GT), so a non-finite visible
 * pixel makes all three distances of its landmark NaN; hide such pixels with the masked entry.
 */
int pnpb200_report_batch(int dtype, int64_t B, int n, const void* pattern, const void* uv,
                         const double* K, const void* R, const void* t, const void* euler_deg,
                         const double* gt, const double* bounds,
                         double* report, int32_t* flags, int32_t* max_idx, void* stream);

/*
 * The solve and the error report of the same problems in one call: pnpb200_solve_batch (one pattern) followed by
 * pnpb200_report_batch_strided over all n_total landmarks -- the body of the loop of random_stress_test.py:322-377
 * (solve_pnp, then compare_result_and_generate_result_dict on its result).  When the solve runs as the moment
 * mapping (LM / linear F2 / LM+, all landmarks) its last pass -- res_norm at the stored state, point by point -- is
 * folded into the report kernel, so the pixel rows are read twice per problem (moments; residual + report) instead
 * of three times; the results are those of the two separate calls.  Every other method / mapping runs the two calls
 * back to back.  R, t, euler_deg, gt and report are required; res_norm, iters, flags, max_idx may be NULL.
 */
int pnpb200_solve_report_batch(int method, int dtype, int64_t B, int n_total, int n,
                               const void* uv, const void* pattern, const int32_t* point_index, const double* K,
                               const pnpb200_params* params,
                               void* R, void* t, void* euler_deg, void* res_norm, int32_t* iters,
                               const double* gt, const double* bounds,
                               double* report, int64_t report_stride_problem, int64_t report_stride_column,
                               int32_t* flags, int32_t* max_idx, void* stream);

/*
 * The same report into a strided array: value k of problem b goes to
 * report[b * report_stride_problem + k * report_stride_column] (elements).  (16, 1) is the row layout
 * of pnpb200_report_batch; (1, B) is the column layout the Python wrapper uses: the kernels' writes
 * and the statistics' reads of one quantity are then contiguous.
 */
int pnpb200_report_batch_strided(int dtype, int64_t B, int n, const void* pattern, const void* uv,
                                 const double* K, const void* R, const void* t, const void* euler_deg,
                                 const double* gt, const double* bounds,
                                 double* report, int64_t report_stride_problem, int64_t report_stride_column,
                                 int32_t* flags, int32_t* max_idx, void* stream);

/*
 * Per-problem solution check WITHOUT ground truth.  Not a reference function: the reference returns a diverged pose
 * without any signal (see the conventions above), and its res_norm, taken at the state before the last update, does not
 * tell the failures apart.  This is the ground-truth-free counterpart of pnpb200_report_batch, for any pose (not only
 * this library's), and it never changes R, t.  Like the report it uses ALL n_total landmarks of each row; there is no
 * landmark subset.  Inputs and arithmetic as pnpb200_report_batch (FP32 inputs are widened and computed in FP64).
 *   pattern      [device] [n_patterns, n_total, 3]; problem b is checked against pattern best_pattern[b]
 *   best_pattern [device] [B] int32 (as pnpb200_solve_batch returns it), or NULL for pattern 0.  An entry outside
 *                [0, n_patterns) gives reproj = NaN and PNPB200_CHECK_NONFINITE.
 *   res_norm     [device] [B] dtype or NULL; only its finiteness is looked at
 *   status       [device] [B] int32, a set of PNPB200_CHECK_* bits, 0 = nothing found
 *   reproj       [device] [B, 2] dtype or NULL: (mean, max) over the landmarks of the prediction-vs-landmark distance of
 *                cal_LM_error_distances (TEST_TOOLBOX.py:252-286), in pixels: report columns 6, 7 with distance_GT = 1
 *                (bit for bit where the report runs its streaming kernel)
 *   reproj_limit_px  PNPB200_CHECK_REPROJ is set where the mean exceeds it; <= 0 or NaN disables that bit
 * What the bits find (C oracle, random_stress_test.py pose distribution, quantised noise-free pixels, seed 42, 8 192
 * problems, against the 10 cm / 10 deg test of random_stress_test.py; "flagged" = BEHIND or REPROJ at 1 px):
 *   LM, 68 landmarks: 30.6 % fail.  BEHIND is set on 12.5 % of the problems and every one of them fails; 36.4 % are
 *   flagged, which catches 85 % of the failures, and 7.1 % of the unflagged problems fail.
 *   LM, 15 landmarks (Alexander): 35.9 % fail; BEHIND 18.7 %, all failing; 32.6 % flagged, 80 % of the failures caught,
 *   10.9 % of the unflagged fail.  LM+, 68: 1.05 % fail, all flagged, none of the unflagged fail.
 *   EIF2, 15: 2.0 % fail and reproject well -- the check does NOT find the failures of EIF2.
 *   (Multiplying the mean by the ground-truth distance, as report column 6 does, would separate LM-68 better -- 96 % of
 *   the failures caught, 2.0 % of the unflagged failing -- but needs the ground truth this check does without.)
 *   1 px assumes whole-pixel, noise-free detections: with pixel noise of sigma px scale the limit with sigma.
 * Returns PNPB200_ETOOLARGE when the streaming kernel cannot hold every pattern in shared memory.
 */
#define PNPB200_CHECK_NONFINITE 1   /* R, t, res_norm (if given) or the reprojection is not finite                     */
#define PNPB200_CHECK_DEPTH     2   /* t3 <= 0: the pattern is not in front of the camera                               */
#define PNPB200_CHECK_BEHIND    4   /* a landmark projects with homogeneous coordinate -1 (behind the camera); the      */
                                    /* reference's projection (perspective_projection :4548) turns it into plausible pixels */
#define PNPB200_CHECK_REPROJ    8   /* mean reprojection distance > reproj_limit_px                                     */
int pnpb200_check_batch(int dtype, int64_t B, int n_total, const void* pattern, int n_patterns, const void* uv,
                        const double* K, const void* R, const void* t, const void* res_norm,
                        const int32_t* best_pattern, double reproj_limit_px, int32_t* status, void* reproj,
                        void* stream);

/*
 * Per-problem landmark visibility.  A detector does not find every landmark: self-occlusion, leaving the image or a
 * confidence threshold hide a different set in every frame.  The _masked entries below are the entries above plus
 *   visible  [device] (host for pnpb200_solve_batch_host_masked) [B, W] uint32, W = ceil(n_total / 32), row-major,
 *            4-byte aligned: bit i % 32 of word i / 32 (least significant bit first) = landmark i is visible; bits at and
 *            beyond n_total are ignored.  NULL or a misaligned pointer is PNPB200_EINVAL (the unmasked entries are the
 *            call without a mask).
 * The rule, for every output: problem b is solved, reported and checked as the problem made of its visible landmarks
 * alone -- with point_index, the visible landmarks of point_index in point_index order -- which is the reference's
 * result with the pattern dict and the image-point dict both restricted to those keys (f2_get_P :3260, f2_get_B_xy
 * :3291, LM_key_list :156).
 *  - The pixels of a hidden landmark are never used in arithmetic: NaN, +-Inf or any other value there changes no
 *    output bit, so "missing = NaN" works as is.
 *  - Fewer than 4 visible selected landmarks: the problem is not solved.  R, t, euler_deg, res_norm are NaN, iters 0,
 *    best_pattern 0; the check reports PNPB200_CHECK_NONFINITE with reproj NaN; report columns 4-9 are NaN and max_idx
 *    is -1 (with the unsolved NaN pose every column but 11 and 15 is NaN and every pass flag false).  Its neighbours in
 *    the batch are unaffected.
 *  - Linear F1 / F2 (and so the start of LM+) need visible landmarks that are not coplanar.  On a coplanar set (e.g. 6 of
 *    the 15 golden landmarks, 10 of which lie in z = 0) the reference's pinv solves a rank-deficient system; the device's
 *    LDL^T / SPD solves have no rank-deficient branch and return NaN there.  LM, QEIF and EIF2 are not affected.
 *  - Report: means and maxima of columns 4-9 run over the visible landmarks; max_idx is in the 0..n_total-1 numbering.
 *    Check: reproj (mean, max) and the BEHIND bit run over the visible landmarks.  Several patterns: the arg-min is
 *    taken on the masked res_norm.
 * A masked solve takes the mapping the same call without a mask takes, every method and flag included (LM+ and
 * PNPB200_FLAG_LM_TRUE_JACOBIAN too); its kernels keep the pattern constants (M0, m0, n, G) per problem: the moment
 * mapping's moments pass stores sum theta theta^T, sum theta and the count of each problem beside its moments, and
 * k_iterate builds the constants per thread.  Rows of 256 landmarks and more take the per-warp streaming shape (there is
 * no masked TMA ring).  pnpb200_solve_report_batch_masked is the masked solve followed by the masked report (never the
 * fused pass).  pnpb200_workspace_bytes_masked is the scratch of a masked solve: that of pnpb200_workspace_bytes plus
 * 10 values per problem where that is not 0.
 * pnpb200_solve_batch_host_masked is pnpb200_solve_batch_host_px with the chunk's mask words copied beside its pixels;
 * with non-NULL status it also runs the check of pnpb200_solve_check_batch_host (reproj may then be NULL).
 * How much visibility the methods tolerate (C oracle, random_stress_test.py pose distribution, quantised noise-free pixels,
 * seed 42, 8 192 problems, 68 landmarks of which a uniformly drawn 100 / 75 / 50 % per problem are visible; share passing
 * the 10 cm / 10 deg test of random_stress_test.py; tests/visibility_accuracy.py):
 *            100 %    75 %    50 %
 *   LM       69.4 %  68.3 %  67.0 %
 *   LM+      99.0 %  98.8 %  98.7 %
 *   EIF2     99.2 %  98.9 %  98.6 %
 *   QEIF    100.0 % 100.0 % 100.0 %   (all 68 landmarks, not solve_pnp's 6)
 * Half the landmarks cost the filters well under a point of pass rate on noise-free pixels.
 */
int pnpb200_solve_batch_masked(int method, int dtype, int64_t B, int n_total, int n,
                               const void* uv, const void* pattern, int n_patterns,
                               const int32_t* point_index, const double* K,
                               const pnpb200_params* params,
                               void* R, void* t, void* euler_deg, void* res_norm,
                               int32_t* iters, int32_t* best_pattern, const uint32_t* visible, void* stream);
int pnpb200_solve_report_batch_masked(int method, int dtype, int64_t B, int n_total, int n,
                                      const void* uv, const void* pattern, const int32_t* point_index, const double* K,
                                      const pnpb200_params* params,
                                      void* R, void* t, void* euler_deg, void* res_norm, int32_t* iters,
                                      const double* gt, const double* bounds,
                                      double* report, int64_t report_stride_problem, int64_t report_stride_column,
                                      int32_t* flags, int32_t* max_idx, const uint32_t* visible, void* stream);
int pnpb200_report_batch_strided_masked(int dtype, int64_t B, int n, const void* pattern, const void* uv,
                                        const double* K, const void* R, const void* t, const void* euler_deg,
                                        const double* gt, const double* bounds,
                                        double* report, int64_t report_stride_problem, int64_t report_stride_column,
                                        int32_t* flags, int32_t* max_idx, const uint32_t* visible, void* stream);
int pnpb200_check_batch_masked(int dtype, int64_t B, int n_total, const void* pattern, int n_patterns, const void* uv,
                               const double* K, const void* R, const void* t, const void* res_norm,
                               const int32_t* best_pattern, double reproj_limit_px, int32_t* status, void* reproj,
                               const uint32_t* visible, void* stream);
int64_t pnpb200_workspace_bytes_masked(int method, int dtype, int64_t B, int n_patterns, int mapping);
int pnpb200_solve_batch_host_masked(pnpb200_pipeline* p, int method, int64_t B, int n, int pixel_type,
                                    const void* uv_host, const void* pattern_host,
                                    const int32_t* point_index, const double* K,
                                    const pnpb200_params* params,
                                    void* R, void* t, void* euler_deg, void* res_norm,
                                    int32_t* iters, int32_t* best_pattern, const uint32_t* visible,
                                    double reproj_limit_px, int32_t* status, void* reproj);

/*
 * Outlier-robust solve.  Not a reference function.  A detector also misplaces landmarks (a mouth corner on the lip, an eye
 * corner on the brow), and one such landmark ruins the pose of every method.  This entry rejects landmarks by their
 * reprojection distance and re-solves each problem on its inliers, with the masked solve above.  Per problem b:
 *  - Candidates C = the landmarks the solver sees (point_index, or all n_total) that are visible (all when visible is NULL).
 *  - Round 0 solves on M0 = C.  After the solve on M_r, d_i (i in C) is the check's prediction-vs-landmark distance of landmark
 *    i (pnpb200_check_batch: pose_r, pattern best_pattern_r, FP64, the same arithmetic); med = the lower median of {d_i}, the
 *    element of rank floor((|C| - 1) / 2) in ascending order with NaN last; tau = max(floor_px, k_median * med), floor_px
 *    where k_median * med is not finite; M_{r+1} = {i in C : d_i <= tau} (a NaN distance is an outlier).  d_i is never
 *    infinite: where its square is not finite (depth exactly 0, a non-finite pixel, an overflow) it is NaN, so even
 *    floor_px = +Inf drops such a landmark.
 *  - M_{r+1} = M_r: converged, the result is pose_r on M_r.  Else |M_{r+1}| < min_inliers: pose_r and M_r are kept with
 *    PNPB200_ROBUST_TOO_FEW.  Else, if r + 1 < max_rounds, the problem is solved on M_{r+1} and classified again; if
 *    r + 1 = max_rounds, pose_r and M_r are kept with PNPB200_ROBUST_NOT_CONVERGED.
 * Contract: every output of problem b (R, t, euler_deg, res_norm, iters, best_pattern) is, bit for bit, what
 * pnpb200_solve_batch_masked returns for b with visible = the returned inlier mask; so the pose inherits the masked solve's
 * contract (fewer than 4 landmarks: NaN pose; hidden pixels are never read).  A non-finite VISIBLE pixel gives a NaN round-0
 * pose, every distance NaN and TOO_FEW: hide such pixels in `visible`.  Re-solved problems are solved as a compacted batch
 * (cub::DeviceSelect::Flagged, gather, masked solve, scatter); a masked solve's result does not depend on the batch around
 * it, with one exception: QEIF and EIF2 in FP64 re-solve the exit decisions the moment mapping cannot certify point by point,
 * per warp when at most 148 tiles of 32 problems need it and per thread above, and the two agree to rounding only.  On
 * whole-pixel detections a few problems per million need it; on noise-free unrounded pixels most do.
 *   arguments   those of pnpb200_solve_batch_masked, but `visible` may be NULL (every landmark visible); R and t are required,
 *               and best_pattern too when n_patterns > 1
 *   robust      [host] or NULL for pnpb200_default_robust_params; PNPB200_EINVAL, before any launch, unless max_rounds >= 1,
 *               min_inliers >= 4, k_median finite and >= 0, floor_px >= 0 (+Inf keeps every finite distance)
 *   inliers     [device] [B, W] uint32 (the format of `visible`): the mask the returned pose was solved on, 0 outside C
 *   rounds      [device] [B] int32: the number of solves of problem b (1 .. max_rounds)
 *   robust_status [device] [B] int32: PNPB200_ROBUST_* bits, 0 = converged
 *   params->workspace: NULL, or pnpb200_robust_workspace_bytes of scratch (the masked solve's and the compacted batch's);
 *               with less the call takes its scratch from the stream-ordered pool.
 * The call synchronises `stream` once per round to read the number of re-solved problems (one int32 through a pinned word
 * kept per calling thread), so it cannot be captured into a CUDA graph.
 * Defaults (k_median 3, floor_px 2 px, min_inliers 6, max_rounds 4) are those of the probe that motivated the entry, kept.
 * Pass rate on the 10 cm / 10 deg test (C oracle, random_stress_test.py pose distribution, seed 42, 8 192 problems, 68 landmarks,
 * whole-pixel detections of which a random f % per problem are moved by U(a, b) px in a random direction and rounded again;
 * plain -> robust, defaults; tests/outlier_accuracy.py):
 *   moved by    f      LM+             QEIF            EIF2
 *   -           0 %    99.0 ->  99.1  100.0 -> 100.0   99.2 ->  99.2
 *   5-30 px    10 %    48.8 ->  98.3   50.1 -> 100.0    9.8 ->  21.9
 *   5-30 px    30 %    26.8 ->  97.5   28.1 -> 100.0    3.4 ->   4.3
 *   30-150 px  10 %     2.3 ->  87.2    3.2 -> 100.0    0.1 ->   3.0
 *   30-150 px  30 %     0.1 ->  43.8    0.4 ->  99.5    0.0 ->   0.0
 * A tenth of the landmarks misplaced halves every method's pass rate; the rule restores QEIF (all 68 landmarks) and, but for
 * 30 % far outliers, LM+.
 * EIF2's pose under outliers is too far off for its distances to single the outliers out: the rule does not rescue it (as
 * the check does not find EIF2's failures).  Neither does it rescue LM+ at 30 % far outliers: that needs minimal-sample
 * hypotheses (RANSAC), which pnpb200_solve_ransac_batch below draws before it runs this loop.
 */
#define PNPB200_ROBUST_TOO_FEW       1   /* M_{r+1} held fewer than min_inliers landmarks: pose_r on M_r kept               */
#define PNPB200_ROBUST_NOT_CONVERGED 2   /* max_rounds solves without a fixed point: the last pose and its mask kept         */
typedef struct pnpb200_robust_params {
    int32_t max_rounds;    /* 4    solves at most                                                                     */
    double  k_median;      /* 3.0  tau = max(floor_px, k_median * median distance)                                     */
    double  floor_px;      /* 2.0                                                                                      */
    int32_t min_inliers;   /* 6    (>= 4)                                                                              */
} pnpb200_robust_params;
int pnpb200_default_robust_params(pnpb200_robust_params* p);
int64_t pnpb200_robust_workspace_bytes(int method, int dtype, int64_t B, int n_total, int n_patterns, int mapping);
int pnpb200_solve_robust_batch(int method, int dtype, int64_t B, int n_total, int n,
                               const void* uv, const void* pattern, int n_patterns,
                               const int32_t* point_index, const double* K,
                               const pnpb200_params* params,
                               void* R, void* t, void* euler_deg, void* res_norm,
                               int32_t* iters, int32_t* best_pattern, const uint32_t* visible,
                               const pnpb200_robust_params* robust, uint32_t* inliers, int32_t* rounds,
                               int32_t* robust_status, void* stream);

/*
 * Minimal-sample hypotheses (RANSAC, Fischler & Bolles 1981).  Not a reference function.  The robust solve above starts from
 * the pose solved on all candidates, so a contaminated first pose decides which landmarks it rejects.  This stage finds each
 * problem's largest consensus set from minimal samples instead.  Per problem b, with C = its candidates (the landmarks of
 * point_index, in solver order, that are visible) and c = |C|:
 *  - Sample s (s = 0, 1, ...): u = Philox4x32-10 with counter (g lo, g hi, s, 4) and key seed, g = idx0 + b;
 *    j_k = u_k mod (c - k), k = 0..3; the k-th sample landmark is the j_k-th candidate not yet chosen, in candidate order.
 *  - Hypothesis: a P3P pose (Lambda Twist, FP64) of the first three sample landmarks, for every pattern; bearings are
 *    K^-1 [u, v, 1] normalised.  Among its 0..4 roots the one whose distance d (below) at the 4th landmark is smallest wins
 *    (strict <, the first root wins ties; a NaN distance never wins); the pattern's hypothesis survives where that distance
 *    is <= consensus_px.  A sample none of whose patterns survives is not scored.
 *  - Consensus of a surviving hypothesis: the number of candidates i with d_i <= consensus_px, d_i the check's
 *    prediction-vs-landmark distance (pnpb200_check_batch's arithmetic, FP64 for both dtypes; NaN is an outlier).  A sample's
 *    consensus is the maximum over its patterns (ties to the lower pattern); the winner has the largest consensus (ties to
 *    the lower s).
 *  - Stop after sample s when (1 - w^4)^(s + 1) <= 1 - confidence, w = best consensus / c (evaluated as
 *    ((c^4 - best^4) / c^4)^(s + 1), one division and binary powering), and after max_samples samples in any case.  On clean
 *    data the first good sample ends the search.
 *   arguments   as pnpb200_solve_batch_masked (visible may be NULL: every landmark visible); n <= 1024 and n_total <= 65536,
 *               else PNPB200_ETOOLARGE
 *   hyp         [host] or NULL for pnpb200_default_hypothesis_params; PNPB200_EINVAL, before any launch, unless
 *               max_samples >= 0, consensus_px >= 0 (not NaN) and 0 < confidence <= 1
 *   R, t        [device] [B,3,3], [B,3] (dtype): the winner's pose; best_pattern [device] [B] int32 (may be NULL for one pattern)
 *   consensus_mask [device] [B, W] uint32 (the format of `visible`): the winner's consensus set, a subset of C
 *   consensus   [device] [B] int32: its size;  drawn [device] [B] int32 or NULL: the number of samples taken
 * Speed (1 Mi x 68, B200 at 1000 W, tools/time_ransac.py): 9.6 ms on clean data, 17.8 ms with 30 % far outliers (DESIGN.md 6).
 * c < 4, or no sample survives: consensus 0, mask 0, NaN pose, best_pattern 0.  The candidates' pixels sit in shared memory
 * (one warp per problem, 18 bytes per candidate), so every n up to 1024 fits.  The result of problem b depends on idx0 + b
 * and its own row only: a shard called with idx0 = its first global index returns, bit for bit, its slice of the
 * unsharded call.  The entry does not synchronise and allocates nothing, so it can be captured into a CUDA graph.
 */
typedef struct pnpb200_hypothesis_params {
    int32_t  max_samples;   /* 128                                                                                    */
    double   consensus_px;  /* 4.0  px: the 4th-landmark test and the consensus threshold                             */
    double   confidence;    /* 0.999                                                                                  */
    uint64_t seed;          /* 0                                                                                      */
    int64_t  idx0;          /* 0    global index of problem 0 of the call                                             */
} pnpb200_hypothesis_params;
int pnpb200_default_hypothesis_params(pnpb200_hypothesis_params* p);
int pnpb200_hypothesize_batch(int dtype, int64_t B, int n_total, int n, const void* uv, const void* pattern, int n_patterns,
                              const int32_t* point_index, const double* K, const uint32_t* visible,
                              const pnpb200_hypothesis_params* hyp, void* R, void* t, int32_t* best_pattern,
                              uint32_t* consensus_mask, int32_t* consensus, int32_t* drawn, void* stream);

/*
 * RANSAC solve: the hypothesis stage above, then the robust loop of pnpb200_solve_robust_batch started from its consensus set.
 * M0 = the winner's consensus set where consensus >= min_inliers, else C; then exactly the loop of the robust entry from M0
 * instead of C (solve on M_r, the median rule on C, compacted re-solves, the same rounds and robust_status).
 * Contract: that of the robust entry, unchanged.  Every output of problem b (R, t, euler_deg, res_norm, iters, best_pattern)
 * is bit for bit pnpb200_solve_batch_masked's on the returned inlier mask, with the same QEIF / EIF2 FP64 fix-up exception.
 * With max_samples = 0 every output, mask, round count and status word is bit-identical to pnpb200_solve_robust_batch.
 *   arguments   those of pnpb200_solve_robust_batch, plus hyp (as pnpb200_hypothesize_batch), consensus [device] [B] int32
 *               (the hypothesis stage's) and drawn [device] [B] int32 or NULL
 *   params->workspace: NULL, or pnpb200_ransac_workspace_bytes of scratch (the robust entry's plus the hypothesis stage's)
 * The call synchronises `stream` once per round, as the robust entry does.
 * Pass rate on the 10 cm / 10 deg test, on the problems of the robust entry's table plus a 50 % row (C oracle,
 * tests/ransac_accuracy.py), plain -> robust -> RANSAC, defaults:
 *   moved by    f      LM+                QEIF               EIF2
 *   -           0 %    99.0  99.1  99.1  100.0 100.0 100.0   99.2  99.2  99.2
 *   5-30 px    10 %    48.8  98.3  99.2   50.1 100.0 100.0    9.8  21.9  99.0
 *   5-30 px    30 %    26.8  97.5  99.0   28.1 100.0 100.0    3.4   4.3  98.7
 *   30-150 px  10 %     2.3  87.2  99.0    3.2 100.0 100.0    0.1   3.0  99.1
 *   30-150 px  30 %     0.1  43.8  99.0    0.4  99.5 100.0    0.0   0.0  98.7
 *   30-150 px  50 %     0.0   0.1  98.6    0.1   2.9  99.9    0.0   0.0  98.2
 * The minimal samples rescue every method, EIF2 included: its pose is as good on the consensus set as on clean data.
 * consensus_px: the RANSAC pass rate per method on clean data, 30 % and 50 % moved by 30-150 px:
 *     2 px           99.1  99.0  98.5   100.0 100.0  99.8    99.2  98.7  98.1
 *     4 px           99.1  99.0  98.6   100.0 100.0  99.9    99.2  98.7  98.2
 *     8 px           99.1  99.0  98.6   100.0 100.0  99.9    99.2  98.7  98.2
 * 4 px is the default: the smallest threshold within 0.1 point of the best everywhere (a tighter one keeps near outliers,
 * the 5-30 px rows, out of the consensus set; 2 px loses samples to the whole-pixel rounding of the detections).
 */
int64_t pnpb200_ransac_workspace_bytes(int method, int dtype, int64_t B, int n_total, int n_patterns, int mapping);
int pnpb200_solve_ransac_batch(int method, int dtype, int64_t B, int n_total, int n,
                               const void* uv, const void* pattern, int n_patterns,
                               const int32_t* point_index, const double* K,
                               const pnpb200_params* params,
                               void* R, void* t, void* euler_deg, void* res_norm,
                               int32_t* iters, int32_t* best_pattern, const uint32_t* visible,
                               const pnpb200_robust_params* robust, uint32_t* inliers, int32_t* rounds,
                               int32_t* robust_status, const pnpb200_hypothesis_params* hyp, int32_t* consensus,
                               int32_t* drawn, void* stream);

/*
 * Error statistics, two passes so that shards can be combined with two small all-reduce phases
 * (TEST_TOOLBOX.get_statistic_of_result, TEST_TOOLBOX.py:892-937), for nq <= 4 quantities at once
 * (depth, roll, pitch, yaw in TEST_TOOLBOX.data_analysis_and_saving, :1070-1112), per class and,
 * in the extra LAST row, over all problems.
 *   est[q], gt[q]: FP64 device vectors with element strides est_stride[q], gt_stride[q]
 *                  (gt or gt[q] may be NULL: statistics of the value itself);  arrays of nq [host]
 *   class_id: [B] int32 device or NULL (every problem in class 0); n_class <= 64 classes
 *   pass 1 -> sums1 [nq, n_class+1, 4] = n, sum(est/gt), sum(e), 0                  (SUM-reducible)
 *   pass 2, given the (all-reduced) sums1 from which it derives the means itself
 *          -> sums2 [nq, n_class+1, 4] = sum((e-m)^2), sum|e|, sum|e-m|, 0           (SUM-reducible)
 *             max2  [nq, n_class+1]    = max|e-m|                                    (MAX-reducible)
 */
int pnpb200_stats_pass1(int64_t B, int nq, const double* const* est, const int64_t* est_stride,
                        const double* const* gt, const int64_t* gt_stride,
                        const int32_t* class_id, int n_class, double* sums1, void* stream);
int pnpb200_stats_pass2(int64_t B, int nq, const double* const* est, const int64_t* est_stride,
                        const double* const* gt, const int64_t* gt_stride,
                        const int32_t* class_id, int n_class, const double* sums1, double* sums2,
                        double* max2, void* stream);

/*
 * Ground-truth classification, np.digitize(value, bins) (TEST_TOOLBOX.classify_drpy,
 * TEST_TOOLBOX.py:239-247): class = number of bins b with b <= value.  values: FP64 device,
 * element stride in doubles; bins [host], ascending, n_bins <= 32; class_id [B] int32 device.
 */
int pnpb200_classify(int64_t B, const double* values, int64_t stride, double scale,
                     const double* bins, int n_bins, int32_t* class_id, void* stream);

/*
 * The analysis stage of face_variation_test.py (:631-759) for up to 4 error quantities at once.
 *
 * Selection of the top k problems by |value| -- what the script does by popping k items off heaps of
 * (-|err|, idx) tuples (:631-653), so ties go to the SMALLER index -- as an exact radix select on the
 * 96-bit key (bits of |value|, then ~global index), 12 digits of 8 bits, most significant first.
 * pnpb200_topk_histogram counts, per quantity, the problems whose key starts with the
 * n_digits_decided digits of (prefix_hi, prefix_lo), by their next digit: hist [nq, 256] (device,
 * uint64).  The caller (workload.fragility_analysis) walks the histogram from 255 down to pick the
 * next digit; across GPUs the histograms are summed, nothing else is exchanged.  idx0 = global index
 * of this shard's first problem.  values[q]: device doubles with element stride[q].
 */
int pnpb200_topk_histogram(int64_t B, int64_t idx0, int nq, const double* const* values, const int64_t* stride,
                           const uint64_t* prefix_hi, const uint32_t* prefix_lo, int n_digits_decided,
                           uint64_t* hist, void* stream);

/*
 * get_most_fragile_point_and_perturbation_direction (face_variation_test.py:658-728) over the
 * problems whose key is >= (threshold_hi, threshold_lo): per quantity, n_selected, the sum and the
 * maximum of |value| (top_value_mean, value_max), count [nq, n] = how often each landmark carried
 * the largest perturbation norm (strict >, first landmark wins), and gram [nq, 3n, 3n] = sum of
 * v v^T over the selected perturbation vectors (upper 16 x 16 tiles only; mirror it), whose
 * eigen-decomposition is the script's SVD of the m x 3n perturbation matrix (singular values =
 * sqrt of the eigenvalues, right singular vectors = eigenvectors).  perturb [B, n, 3] from
 * pnpb200_synth_face_variation; list [nq, list_capacity] receives the selected local indices.
 * All outputs are device memory and are zeroed by the call.
 */
int pnpb200_fragility_accumulate(int64_t B, int64_t idx0, int nq, const double* const* values, const int64_t* stride,
                                 const uint64_t* threshold_hi, const uint32_t* threshold_lo, const double* perturb,
                                 int n, int64_t list_capacity, int64_t* list, uint64_t* n_selected, uint64_t* count,
                                 double* value_sum, double* value_max, double* gram, void* stream);

/*
 * Host-side result table (no GPU): the CSV that TEST_TOOLBOX.write_result_to_csv (TEST_TOOLBOX.py:693-708)
 * writes from the list of result dicts of compare_result_and_generate_result_dict (:396-463), straight
 * from the arrays pnpb200_report_batch returns, copied to the host (pinned or not).  Same column names
 * and order for every scalar / string / tuple / dict field (the six ndarray fields are left out), same
 * csv dialect (QUOTE_MINIMAL, "\r\n"), floats as Python's repr(float), bools as True / False.
 *   report [B,16], flags [B,4], max_idx [B,3], res_norm [B], gt [B,4]        (host)
 *   key_names [n_keys]: landmark names in pattern order (the *_error_max_key columns)
 *   bins[q] / n_bins[q] / labels[q], q = depth (cm), roll, pitch, yaw: classify_drpy (:239-247),
 *   n_bins[q] + 1 labels each; they give the `class` and `file_name` columns (random_stress_test.py:300-306)
 *   append = 0: truncate and write the header; 1: append rows (shards / chunks in order); idx0 = first idx
 * pnpb200_format_repr exposes the float formatter for the tests (out_size >= 32).
 */
int pnpb200_write_result_csv(const char* path, int append, int64_t B, int64_t idx0, const double* report,
                             const int32_t* flags, const int32_t* max_idx, const double* res_norm, const double* gt,
                             const char* const* key_names, int n_keys, const double* const* bins, const int32_t* n_bins,
                             const char* const* const* labels, int n_threads);
int pnpb200_format_repr(double v, char* out, int out_size);

/*
 * Combined class of the four ground-truth quantities (TEST_TOOLBOX.get_all_class_seperated_result,
 * :975-1030): id = ((cd * nr + cr) * np + cp) * ny + cy, each c = np.digitize(gt[:, q] * scale[q], bins[q])
 * in the order distance, roll, pitch, yaw; gt [B,4] device; bins / n_bins / scale host arrays of 4.
 * pnpb200_stats_pass1/2 accept the resulting n_class = nd*nr*np*ny (up to 2^20): beyond 64 classes
 * they add straight into the global table.
 */
int pnpb200_classify_drpy(int64_t B, const double* gt, const double* const* bins, const int32_t* n_bins,
                          const double* scale, int32_t* class_id, void* stream);

/*
 * FMA-pipe microbenchmark used by bench.py for the roofline denominator (MEASURED_PEAKS.json
 * has no FP64/FP32 FMA figure).  Runs `iters` dependent-chain-free FMAs per thread on a full
 * grid and returns the device-timed rate in FLOP/s (2 per FMA).  Synchronous.
 */
int pnpb200_fma_peak(int dtype, int iters, double* flops_per_s);

/*
 * Test hook: the branch-free FP64 reciprocal, reciprocal square root and square root that the
 * solvers use for pivots and norms (csrc/pnpb200_math.cuh), element-wise on n device doubles
 * (positive, normal).  No reference counterpart; tests/test_gpu_parity.py bounds their error.
 */
int pnpb200_selftest_math(int64_t n, const double* in, double* rcp, double* rsqrt, double* sqrt_out, void* stream);

/*
 * Test hook: the branch-free sine / cosine of bounded angles (radians, |x| < 1e4) that the report
 * kernels build the ground-truth rotation with (csrc/pnpb200_math.cuh, sincos_bounded).
 */
int pnpb200_selftest_sincos(int64_t n, const double* in, double* sin_out, double* cos_out, void* stream);

/*
 * Test hook: the P3P solver of the hypothesis stage (csrc/pnpb200_p3p.cuh), on m device triples: pattern points X [m,3,3]
 * (metres) and unit bearings f [m,3,3].  R [m,4,9], t [m,4,3]: the valid roots first, NaN after; n_sol [m]: their number.
 */
int pnpb200_selftest_p3p(int64_t m, const double* X, const double* f, double* R, double* t, int32_t* n_sol, void* stream);

/*
 * Test hook: one inlier classification pass of the robust loop (pnpb200_solve_robust_batch above: d_i over C, the lower median
 * with NaN last, tau, M' and the decision) on poses the caller supplies, in one of its two kernel shapes.
 *   dtype, B, n_total, n, uv, pattern, n_patterns, point_index, K, visible, robust: as in pnpb200_solve_robust_batch
 *   R, t        [device] [B,3,3], [B,3] (dtype); best_pattern [device] [B] int32 or NULL (pattern 0)
 *   idx         [device] [B] int32 or NULL (the identity): batch entry k reads row k of uv, R, t and best_pattern, and problem
 *               idx[k]'s rows of visible, inliers, rounds and robust_status (the compacted batch of rounds >= 1)
 *   last_round  nonzero: a mask that would change is kept with NOT_CONVERGED
 *   inliers, rounds, robust_status [device], in / out: M and its problem's state, updated as the robust loop updates them
 *   flag        [device] [B] uint8: 1 where batch entry k is to be solved again;  tau [device] [B] double or NULL: its threshold
 *   shape       0 the kernel the robust loop picks, 1 the streaming kernel (PNPB200_EINVAL where it cannot run), 2 one warp
 *               per problem (PNPB200_ETOOLARGE where its shared memory does not fit)
 * Argument errors return PNPB200_EINVAL before any CUDA call.
 */
int pnpb200_selftest_inliers(int dtype, int64_t B, int n_total, int n, const void* uv, const void* pattern, int n_patterns,
                             const int32_t* point_index, const double* K, const uint32_t* visible,
                             const pnpb200_robust_params* robust, const void* R, const void* t, const int32_t* best_pattern,
                             const int32_t* idx, int last_round, uint32_t* inliers, int32_t* rounds, int32_t* robust_status,
                             uint8_t* flag, double* tau, int shape, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PNPB200_H */
