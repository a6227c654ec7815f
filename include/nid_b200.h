/*
 * nid_b200.h — C-ABI of the B200-native NID cost + Jacobian path.
 *
 * Drop-in boundary for the three CUDA host entry points of arpg/NID-Pose-Estimation and the
 * g2o-side NID edge. Citations are file:line in the upstream tree.
 *
 *   reference interface                                             replaced by
 *   ------------------------------------------------------------    ----------------------------------
 *   Calculate3Dpoint            CudaPoints3d.cuh:6                  nid_set_pair / nid_set_pairs_u16 + nid_get_points3d
 *   CudaComputeHref             CudaComputeHref.cuh:6               nid_prepare / nid_prepare_pairs + nid_get_ref_weights
 *   g2o::CudaComputeH           g2o/g2o/core/computeH.cuh:8         nid_eval / nid_eval_jobs
 *   Edge::computeError          types_six_dof_expmap.h:220-228      nid_eval_gn (err[])
 *   Edge::linearizeOplus        types_six_dof_expmap.cpp:381-541    nid_eval_gn (J[])
 *   constructQuadraticForm+Huber base_unary_edge.hpp:43-72          nid_eval_gn (H36, b6, chi2)
 *   LM::solve / optimize(10)    optimization_algorithm_levenberg.cpp:61-225,
 *                               sparse_optimizer.cpp:356-450        nid_solve / nid_solve_jobs
 *   NID::ComputeHref/ComputeH   NID_standard_property.cpp:342-485   nid_hard_eval_jobs
 *   CalculateProKernel, per-pixel part (warp, bounds, sample, gradient)
 *                               computeH.cu:137-176                 nid_warp_sample / nid_warp_sample_jobs
 *   (no counterpart: a new target frame against a resident reference) nid_set_target
 *
 * The exact-signature C++ shims (`Calculate3Dpoint`, `CudaComputeHref`, `g2o::CudaComputeH`) live in
 * the same shared library (csrc/ref_shims.cu) and forward to these entry points.
 *
 * Conventions (identical to the reference):
 *   - all matrices are column-major 4x4 doubles (Eigen `.data()`), T_cw1 maps world -> camera 1
 *   - intr = {fx, fy, cx, cy, depth_factor}          (NID_pose_estimation.cpp:232-233)
 *   - cell index c = ci*cell + cj, row-major; remainder rows/cols are dropped
 *   - an inactive cell (fewer than 300 in-bounds points at the prepare pose) reports NaN in
 *     Href / Htarget / Hjoint / der  (computeH.cu:271-275, 313-322)
 *   - der = d(err)/d(xi), xi = (omega, upsilon), update T <- exp(xi) * T  (types_six_dof_expmap.h:74-77)
 *   - Jacobian bounds test follows the CPU edge (`u+3 <= cols-1`, types_six_dof_expmap.cpp:433)
 *
 * Every function returns 0 on success, a negative nid_status otherwise; nid_last_error() describes
 * the most recent failure on the calling thread. There is no CPU fallback: without a CUDA device
 * nid_create fails.
 */
#ifndef NID_B200_H
#define NID_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct nid_ctx nid_ctx;

enum nid_status {
  NID_OK = 0,
  NID_ERR_CUDA = -1,
  NID_ERR_ARG = -2,
  NID_ERR_STATE = -3,
  NID_ERR_UNSUPPORTED = -4
};

#define NID_MIN_CELL_POINTS 300 /* computeH.cu:271, types_six_dof_expmap.cpp:609,710 */

const char* nid_last_error(void);
int nid_version(void);

/* A context owns device storage for `n_pairs` frame pairs of one geometry and for `max_jobs`
 * simultaneous evaluations ("jobs": one pose applied to one pair). degree must be 3. */
int nid_create(nid_ctx** ctx, int device, int rows, int cols, int cell, int bins, int degree,
               int n_pairs, int max_jobs);
int nid_destroy(nid_ctx* ctx);
int nid_sync(nid_ctx* ctx);

/* a1 (CudaPoints3d.cu:5-74): upload one pair and back-project its reference depth to world points.
 * depth: rows*cols metres (host). im0/im1: 8-bit gray (host). T_wc0: camera-0-to-world. */
int nid_set_pair(nid_ctx* ctx, int pair, const double* depth, const uint8_t* im0, const uint8_t* im1,
                 const double T_wc0[16], const double intr[5]);
/* The same for n consecutive pair slots [pair0, pair0 + n) in one submission (a tracking sequence, BASELINE config 4),
 * from the dataset's own formats: raw 16-bit depth (metres = raw * intr[4], the driver's
 * `depth.convertTo(CV_64F, depth_factor)`, NID_pose_estimation.cpp:105-106, config_eth_cvg.yaml:13) and 8-bit gray.
 * depth_raw/im0/im1: [n][rows*cols]; T_wc0: [n][16]; intr: [n][5]. ASYNCHRONOUS: copies and kernels are queued on the
 * context stream and the call returns; from pinned host memory nothing blocks. The host buffers must stay untouched
 * until nid_sync or the next blocking call on this context (nid_prepare_pairs is one). */
int nid_set_pairs_u16(nid_ctx* ctx, int pair0, int n, const uint16_t* depth_raw, const uint8_t* im0, const uint8_t* im1,
                      const double* T_wc0, const double* intr);
/* Coarse levels for coarse-to-fine solves. Fill pair slots [dst_pair0, dst_pair0 + n) of dst with the 2x2-downsampled pairs
 * [src_pair0, src_pair0 + n) of src, device to device. Destination pixel (i, j) covers source pixels (2i..2i+1, 2j..2j+1);
 * an odd last source row or column is dropped. Images: (a+b+c+d+2)>>2. Depth: the mean of the valid samples (0.01 <= z
 * <= 100; NaN and Inf are invalid), summed in row-major order of the 2x2 block, 0 (invalid) when none is valid. Intrinsics
 * fx/2, fy/2, (cx-0.5)/2, (cy-0.5)/2 (a coarse pixel centre sits at fine coordinate 2j + 0.5); T_wc0 is copied; the
 * destination holds fp64 depth. dst must have rows == src rows / 2 and cols == src cols / 2 (cell and bins are free) and
 * live on the same device; levels chain (level 2 from level 1 from level 0).
 * ASYNCHRONOUS on dst's stream, ordered after all work queued on src so far; later work on src (a refill of the source
 * slots by nid_set_pairs_u16, say) is ordered after it. The slots must be prepared (nid_prepare*) before they are evaluated
 * or solved. NID_ERR_ARG: geometry, ranges, devices, NULL; NID_ERR_STATE: a source pair not set, or either context
 * holding caller-supplied world points (nid_set_pair_points). */
int nid_set_pairs_downsampled(nid_ctx* dst, int dst_pair0, const nid_ctx* src, int src_pair0, int n);
/* Reference-frame reuse (tracking against a key frame): replace only the target image of a pair that has been
 * set; depth, reference image and world points stay on the device. The pair must be prepared again
 * (nid_prepare at the new initial pose: the in-bounds set, n_c and H_ref depend on it, CudaComputeHref.cu:33-135). */
int nid_set_target(nid_ctx* ctx, int pair, const uint8_t* im1);
/* same, from the reference's double-valued images; values must be integral after the reference's
 * clamp to [0,255) else NID_ERR_UNSUPPORTED. Either image may be NULL to keep the current one. */
int nid_set_pair_f64(nid_ctx* ctx, int pair, const double* depth, const double* im0, const double* im1,
                     const double T_wc0[16], const double intr[5]);
/* Upload a pair whose world points were produced elsewhere (the reference keeps them in a managed
 * buffer between its three entry points): points_3d is 3*rows*cols doubles, AoS, NaN = invalid.
 * im0/im1 as in nid_set_pair_f64 (either may be NULL to keep the current one). */
int nid_set_pair_points(nid_ctx* ctx, int pair, const double* points_3d, const double* im0, const double* im1,
                        const double intr[5]);
/* Adopt a prepare computed elsewhere (the reference's bs_value/bs_index/bs_counter/Href arrays):
 * in-bounds flags are taken from !isnan(bs_value[4i]), n_c from bs_counter, H_ref from Href. */
int nid_import_prepare(nid_ctx* ctx, int pair, const double* bs_value, const int* bs_counter, const double* Href);
/* in-bounds-at-prepare flags, one byte per pixel (host buffer of rows*cols) */
int nid_get_inbounds(nid_ctx* ctx, int pair, uint8_t* flags);
/* points_3d: 3*rows*cols doubles, AoS, NaN triple for invalid depth; host/managed/device memory */
int nid_get_points3d(nid_ctx* ctx, int pair, double* points_3d);

/* a2 (CudaComputeHref.cu:33-223 == computeHref, types_six_dof_expmap.cpp:655-725) at the initial pose.
 * bs_counter[cell^2] = n_c, Href[cell^2] is OVERWRITTEN (NaN when n_c < 300). Either may be NULL. */
int nid_prepare(nid_ctx* ctx, int pair, const double T_cw1_init[16], int* bs_counter, double* Href);
/* a2 for the n consecutive pairs [pair0, pair0 + n) in a handful of launches: T_cw1_init [n][16]; bs_counter and Href
 * [n][cell^2] (either may be NULL). The task / slice tables of the regrouped pixel store are built on the device.
 * Blocking (one synchronisation for the whole range). */
int nid_prepare_pairs(nid_ctx* ctx, int pair0, int n, const double* T_cw1_init, int* bs_counter, double* Href);
/* per-pixel reference spline data in the reference's layout: bs_value[4*N], bs_index[N];
 * pixels without a valid in-bounds sample at the prepare pose get NaN weights / index 0. */
int nid_get_ref_weights(nid_ctx* ctx, int pair, double* bs_value, int* bs_index);

/* a9 (computeH.cu:373-502): one evaluation of pair `pair` at T_cw1. Htarget/Hjoint[cell^2] and, when
 * want_jac, der[6*cell^2] are OVERWRITTEN; der is not touched when want_jac == 0. Blocking. */
int nid_eval(nid_ctx* ctx, int pair, const double T_cw1[16], int want_jac, double* Htarget,
             double* Hjoint, double* der);
/* n_jobs evaluations in one submission: job j applies poses[16*j..] to pair job_pair[j]
 * (job_pair == NULL means pair 0 for every job). Outputs are [n_jobs][cell^2] (der: [..][6]). */
int nid_eval_jobs(nid_ctx* ctx, int n_jobs, const int* job_pair, const double* poses, int want_jac,
                  double* Htarget, double* Hjoint, double* der);

/* Device-resident flavour: stage jobs once, evaluate asynchronously on the context stream,
 * read results back when wanted. nid_eval_staged does no host<->device copy and no sync. */
int nid_stage_jobs(nid_ctx* ctx, int n_jobs, const int* job_pair, const double* poses);
int nid_eval_staged(nid_ctx* ctx, int n_jobs, int want_jac);
int nid_fetch_results(nid_ctx* ctx, int n_jobs, int want_jac, double* Htarget, double* Hjoint, double* der);

/* a10 + a11: per-cell error e_c = (2Hj - Href - Ht)/Hj, Jacobian J_c[6], and the Huber-weighted
 * Gauss-Newton block over the active cells: chi2 = sum rho0(e^2), H += rho1 J^T J, b -= rho1 J^T e.
 * err[cell^2], J[6*cell^2] (NaN for inactive cells), H36 row-major. Any output may be NULL. */
int nid_eval_gn(nid_ctx* ctx, int pair, const double T_cw1[16], double huber_delta, double* chi2,
                double* H36, double* b6, double* err, double* J);

/* One pose solve == SparseOptimizer::optimize(max_iters) with the reference's LM schedule.
 * pose7 = {tx,ty,tz,qx,qy,qz,qw} of T_cw1, in/out. trace (may be NULL): 10 doubles per outer
 * iteration {chi2, lambda, lm_trials, pose7}. stats (may be NULL): {outer_iters, jac_evals, cost_evals}.
 * The pair must have been prepared (the reference prepares at the initial pose). */
int nid_solve(nid_ctx* ctx, int pair, double pose7[7], int max_iters, double huber_delta, double* trace,
              int* stats);
/* n independent solves in lockstep, pair job_pair[j] (NULL: pair j), poses7 [n][7] in/out, stats [n][3]. */
int nid_solve_jobs(nid_ctx* ctx, int n, const int* job_pair, double* poses7, int max_iters,
                   double huber_delta, int* stats);
/* Joint solves: n_groups independent problems; group g has group_size[g] >= 1 jobs (pairs) that share ONE unknown pose
 * (a rig of cameras on one body, or several reference keyframes of one target frame). Jobs are listed group after group;
 * job i uses pair job_pair[i] (NULL: pair i); the same pair may appear in several jobs. poses7 [n_groups][7] in/out is the
 * group's pose T_bw as {t, q}. Job i is evaluated at T_cw1 = T_cb[i] * T_bw; T_cb [n_jobs][16] is column-major rigid
 * camera-from-body (NULL: identity for every job, i.e. several pairs observed from one camera pose). One optimize(max_iters)
 * per group over the cell edges of all its jobs: chi2, H and b are the sums over the jobs in job order, each job's Jacobian
 * taken w.r.t. the body update T_bw <- exp(xi) * T_bw (J_body = J_cam * Ad(T_cb)). stats [n_groups][3] as in nid_solve,
 * counting evaluations of the whole group; trace (may be NULL) [n_groups][max_iters][10] as in nid_solve (rows past a
 * group's outer iterations are not written). Every job's pair must be prepared, at T_cb[i] * (initial T_bw) for the
 * reference's semantics. sum(group_size) <= max_jobs. Runs in latency mode (see "lm_speculate") when there are at most 4
 * groups and room for 2 trial poses of every job. A group of one job with T_cb NULL is exactly nid_solve_jobs of that job.
 * Validated before any work; poses7, stats and trace are written only on success. NID_ERR_ARG: n_groups < 1, a group size
 * < 1, more jobs than max_jobs, NULL poses7 or group_size, a job_pair out of range, a T_cb that is not rigid (bottom row
 * not exactly (0,0,0,1), or R^T R != I to 1e-9, or det R < 0). NID_ERR_STATE: a job's pair not prepared.
 * A group whose jobs have no active cell has chi2 == 0 and a zero system: it reports {1, 1, 1} and keeps its pose. */
int nid_solve_groups(nid_ctx* ctx, int n_groups, const int* group_size, const int* job_pair, const double* T_cb,
                     double* poses7, int max_iters, double huber_delta, int* stats, double* trace);
/* Coarse-to-fine optimize(): levels[0] is the finest context, levels[n_levels-1] the coarsest (1 <= n_levels <= 8; build the
 * coarse levels with nid_set_pairs_downsampled). For l = n_levels-1 .. 0: prepare pairs job_pair[j] of levels[l] at the
 * current poses (nid_prepare_pairs), then nid_solve_jobs(levels[l], ..., max_iters[l], ...) and hand the poses down. Job pairs
 * must be distinct (a pair is prepared at one pose); NULL means pair j. A level with max_iters[l] == 0 is skipped (its stats
 * are 0). n_levels == 1 is exactly nid_prepare_pairs + nid_solve_jobs. stats (may be NULL): [n][n_levels][3] as in nid_solve.
 * poses7 and stats are written only on success. Validated before any work: every level non-NULL, n <= max_jobs and every
 * job's pair set at every level (NID_ERR_STATE if not), pairs distinct.
 * A job without an active cell at a level (every cell under NID_MIN_CELL_POINTS in-bounds points at the prepare pose, as on
 * a level too coarse for its cell grid) has chi2 == 0 and a zero Gauss-Newton system there: the LM schedule rejects its
 * first trial (no decrease) and stops, so that level reports {1, 1, 1} and hands the pose down unchanged. */
int nid_solve_pyramid_jobs(nid_ctx* const* levels, int n_levels, int n, const int* job_pair, double* poses7,
                           const int* max_iters, double huber_delta, int* stats);

/* a12: hard-binned NID of NID_standard_property (no B-spline, normaliser = in-bounds count of this
 * pose). total[n_jobs] = sqrt(sum_c nid_c^2); nid_cells [n_jobs][cell^2] may be NULL. */
int nid_hard_eval_jobs(nid_ctx* ctx, int n_jobs, const int* job_pair, const double* poses, double* total,
                       double* nid_cells);

/* Kernel-1 output for parity / roofline: per pixel {I_c, g_x, g_y, valid} as float4
 * (valid: 0 invalid, 1 cost only, 3 cost+Jacobian). out: host buffer of 4*rows*cols floats, or NULL
 * to leave the result on the device (timing). */
int nid_warp_sample(nid_ctx* ctx, int pair, const double T_cw1[16], float* out);
/* The same kernel-1 record for n_jobs (pair, pose) jobs in one launch, from the pairs' depth planes (fast composed
 * warp with the exact fallbacks of the evaluation path). out: host buffer of n_jobs*4*rows*cols floats, or NULL to
 * leave the result on the device (bench.py's HBM-roofline probe). Depth pairs only (nid_set_pair). */
int nid_warp_sample_jobs(nid_ctx* ctx, int n_jobs, const int* job_pair, const double* poses, float* out);
/* fp64 per-pixel record for strict parity: out[8*N] = {u,v,I_c,g_x,g_y,valid_cost,valid_jac,p_z} */
int nid_warp_sample_f64(nid_ctx* ctx, int pair, const double T_cw1[16], double* out);

/* introspection for tests: normalised histograms of job `job` of the last evaluation */
int nid_debug_hist(nid_ctx* ctx, int job, int cell_index, double* P_t, double* P_j);
/* number of kernels launched by this context so far */
long long nid_launch_count(nid_ctx* ctx);
/* number of CUDA resources (device and pinned buffers, streams, events, arrays, textures, graphs) held by all
 * contexts of the process: a context releases every one of them in nid_destroy, and a failed nid_create holds none */
long long nid_live_resources(void);
/* accumulated device time (ms) and launch count per kernel since "time_kernels" was set:
 * [0] pass-1 histogram kernel, [1] pass-2 Jacobian kernel, [2] Jacobian tail, [3] entropy tail */
int nid_kernel_times(nid_ctx* ctx, double ms[4], long long calls[4]);
/* the CUDA stream (cudaStream_t) every call of this context is issued on */
void* nid_stream(nid_ctx* ctx);
/* CUDA-event stopwatch on the context stream: record slot 0 (start) / 1 (stop), then read the elapsed
 * device time between them (synchronises on the stop event). */
int nid_event_record(nid_ctx* ctx, int slot);
int nid_event_elapsed_ms(nid_ctx* ctx, float* ms);
/* options: "path" (0 automatic, 1 natural-order kernels, 2 sorted kernels); "keep_hist" (1: keep the
 * normalised histograms of every evaluation for nid_debug_hist);
 * "force_strips" (natural path: CTAs per cell and job; 0 = automatic); "time_kernels" (1: bracket every kernel
 * of nid_eval_staged / nid_eval_jobs with CUDA events and accumulate per-kernel device time; resets);
 * "task_px" (sorted path: pixels per task, a multiple of 4 in [8, 256]; default by geometry, 32 for cells of 2560
 * pixels or more and 16 below; set before nid_prepare*. Latency-bound callers -- one pair, one solve at a time, the
 * reference's own use -- should set 16: more and shorter slices, 1.68 -> 1.37 ms per 640x480 solve; throughput-bound
 * callers keep the default. Results for different task lengths agree to rounding, not bit for bit);
 * "lm_reuse" (1, default: nid_solve_jobs linearises at an accepted trial pose without recomputing its histograms);
 * "lm_speculate" (0..8, default 4: up to four problems per nid_solve_jobs call run in latency mode, every round
 * evaluates this many trial poses of the LM schedule at once; 0/1: plain state machine);
 * "lm_graph" (1, default: a round of the latency mode is one CUDA-graph launch);
 * launch shapes, for tests and A/B timing only -- none of them changes a result: "stage_bulk" (-1 by geometry, 0 / 1: pass 2
 * stages the cell's log tables by a bulk copy), "asm_wide" (1 default: the 1024-thread assembly where it pays, 0 never, 2 always) */
int nid_set_option(nid_ctx* ctx, const char* key, int value);

#ifdef __cplusplus
}
#endif
#endif
