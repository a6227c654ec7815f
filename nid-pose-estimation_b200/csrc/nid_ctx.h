// Internal context layout shared by the kernels TU, the C-ABI TU and the LM driver.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <memory>
#include <string>
#include <vector>

#include "../../include/nid_b200.h"
#include "nid_handles.h"

#define NID_NCLS 257  /* reference-intensity classes 0..255 + 256 = valid point without reference sample */
#define NID_SORTED_MIN_BINS 6  /* the two 3x3 end blocks of the basis fold must not overlap */
#define NID_SORTED_MAX_BINS 40 /* k_assemble keeps 5*B^2 + 257*B doubles in shared memory */
#define NID_STAGE_RING 4
#define NID_MIN_JOB_SLOTS 8
#define NID_TASK_PX_MAX 256 /* upper bound of the pixels per task of the sorted path (option "task_px") */

namespace nid {

// Everything the evaluation kernels need; passed by value (fits the 4 KB parameter space easily).
struct EvalParams {
  int rows, cols, cell, bins, rb, cb, N, ncell;  // ncell = cell*cell
  int job0;        // first job handled by this launch (index into job_list when that is set)
  const int* job_list;  // optional indirection: the i-th job of the launch is job_list[job0 + i] (LM driver: fixed slots)
  int S;           // strips per cell (CTAs per cell and job)
  int strip_rows;  // rows of a cell handled by one strip
  int hist_stride; // bins*bins + bins
  // per pair [n_pairs][...]
  const double* pwx;
  const double* pwy;
  const double* pwz;
  const uint8_t* im0;
  const uint8_t* im1;
  const uint8_t* inb0;
  const int* n_c;       // [n_pairs][ncell]
  const double* href;   // [n_pairs][ncell]
  const double* cam;    // [n_pairs][4]
  // reference-intensity lookup (depends on bins only)
  const double* lut_w;  // [256][4]
  const int* lut_k;     // [256]
  // per job
  const double* poses;  // [jobs][16]
  const int* job_pair;  // [jobs]
  double* part;         // [jobs][ncell][S][hist_stride]
  double* jpart;        // [jobs][ncell][S][6]
  double* hist;         // [jobs][ncell][hist_stride] normalised P_j | P_t of the last eval
  double* ht;           // [jobs][ncell]
  double* hj;
  double* err;
  double* der;          // [jobs][ncell][6]
  double* gn;           // [jobs][44] : chi2, H[36], b[6], n_active
  double huber_delta;
  double huber_dsqr;
  // sorted path: sliced-ELL pixel store, see nid_sorted.cu
  const double* sd0;    // [n_pairs][sell_cap] depth z (depth form) or world x (point form)
  const double* sd1;    // point form only: world y
  const double* sd2;    // point form only: world z
  const unsigned* sid;  // [n_pairs][sell_cap] (row << 16) | col, 0xFFFFFFFF = padding
  int stage_bulk;       // pass 2 stages the cell's log tables by a bulk copy (small cells: short slices)
  const int* sl_off;    // [n_pairs][max_slices+1] first pixel slot of every slice (multiples of 128)
  const int* sl_task;   // [n_pairs][max_slices*32] task of every lane, -1 = none
  const int* sl_desc;   // [n_pairs][max_slices*32] that task's descriptor (tasks[].y: count | cls<<9 | cell<<18), 0 = none
  const unsigned short* task_cls;  // [n_pairs][max_tasks] class of every task (the warp assembly reads two bytes per row)
  const int* sl_cell;   // [n_pairs][max_slices] cell of every slice
  const int* nslices;   // [n_pairs]
  size_t sell_cap;      // pixel slots per pair
  int max_slices;
  const double* Twc0;   // [n_pairs][16]
  const int2* tasks;    // [n_pairs][max_tasks] {rank of first pixel in its class segment, count | cls<<9 | cell<<18}
  const int* ntasks;    // [n_pairs]
  const int* cell_task_start;  // [n_pairs][ncell+1]
  const int* cell_slice_start; // [n_pairs][ncell+1] first slice of every cell (slices never mix cells)
  const int* cls_task_start;   // [n_pairs][ncell][NID_NCLS+1] first task of every class
  const int* span_start;       // [bins-2] first class whose k_r is >= k (classes of span k: [k], [k+1])
  double* wv;                  // [jobs][ncell][bins*bins+bins] scaled log tables (assemble -> pass 2)
  int max_tasks;        // task-table stride per pair
  int g_stride;         // partial-buffer stride per job (tasks)
  double* G;            // [jobs][g_stride][bins]
  const unsigned* fp1;              // [n_pairs][N] footprint-packed target image (pass 1), see k_pack_fp
  const cudaTextureObject_t* tex2;  // [n_pairs] packed I | Gx | Gy 32-bit texture (k_pack_tex)
  const cudaTextureObject_t* k1tex; // [n_pairs] kernel 1: fp16 planes I, Gx/2, Gy/2 stacked (k_pack_k1); built on first use
};

}  // namespace nid

namespace nid {
struct LatencyGraph;
struct LatencyGraphDelete { void operator()(LatencyGraph* g) const; };  // (nid_sorted.cu)
}  // namespace nid
// A context owns every handle it holds (nid_handles.h). The evaluation launchers take the stream and the job table they
// work on from their JobSet argument, so nothing here is repointed while a call runs.
struct nid_ctx {
  int device = 0;
  int rows = 0, cols = 0, cell = 0, bins = 0, degree = 3;
  int N = 0, ncell = 0, rb = 0, cb = 0;
  int n_pairs = 0, max_jobs = 0;
  int job_cap = 0;             // job slots actually allocated: max(max_jobs, NID_MIN_JOB_SLOTS) (speculative LM trials need a few)
  int sm_count = 148;
  nid::Stream stream;     // the context stream
  nid::Stream lm_stream;  // the second half of the lock-step LM driver (nid_solve_jobs), created on first use
  nid::DeviceBuffer<int> chunk_cnt;    // [setup_batch][ncell][chunks of 256 px][NID_NCLS] scratch of the regrouping scatter
  // batched pair set-up (nid_set_pairs_u16 / nid_prepare_pairs): up to setup_batch pairs per launch
  int setup_batch = 1;
  nid::DeviceBuffer<int> lay_tot;     // [setup_batch][ncell][3] tasks, slices, pixel slots of every cell
  nid::DeviceBuffer<int> lay_base;    // [setup_batch][ncell][3] their exclusive scans over the cells of a pair
  nid::DeviceBuffer<double> prep_poses;  // [setup_batch][16] initial poses of the batch
  nid::DeviceBuffer<uint16_t> depth16; // [n_pairs][N] raw 16-bit depth (allocated by the first nid_set_pairs_u16)
  nid::DeviceBuffer<double> depth_factor;  // [n_pairs]
  std::vector<char> pair_u16;  // the pair's depth16 plane is valid
  nid::PinnedBuffer<char> h_arena;    // pinned bump arena for the small per-pair arrays of the asynchronous set-up calls
  size_t h_arena_cap = 0, h_arena_used = 0;
  nid::PinnedBuffer<char> h_res;      // pinned results of nid_prepare_pairs (n_c, H_ref, task and slice counts)
  size_t h_res_cap = 0;
  long long launches = 0;

  // per pair
  nid::DeviceBuffer<double> pwx, pwy, pwz;
  nid::DeviceBuffer<uint8_t> im0, im1, inb0;
  nid::DeviceBuffer<int> n_c;
  nid::DeviceBuffer<double> href, cam;
  nid::DeviceBuffer<double> Twc0;     // [n_pairs][16]
  nid::DeviceBuffer<unsigned int> cnt; // [n_pairs][ncell][NID_NCLS] pixel counts per reference class at prepare
  // sorted path, per pair
  nid::DeviceBuffer<double> depth;    // [n_pairs][N] reference depth as uploaded (depth form)
  nid::DeviceBuffer<double> sd0, sd1, sd2;
  nid::DeviceBuffer<unsigned> sid;
  size_t sell_cap = 0;
  nid::DeviceBuffer<int> sl_desc;
  nid::DeviceBuffer<unsigned short> task_cls;
  nid::DeviceBuffer<int> sl_off, sl_task, sl_cell, nslices, task_pos;
  int max_slices = 0;
  std::vector<int> h_nslices;
  int max_nslices_prepared = 0;
  int task_px = 32;            // L: pixels per task
  bool sell_points = false;    // pairs carry caller-supplied world points (nid_set_pair_points)
  nid::DeviceBuffer<int2> tasks;
  nid::DeviceBuffer<int> ntasks, cell_task_start, cell_slice_start, cls_task_start, span_start;
  nid::DeviceBuffer<double> wv;
  int max_tasks = 0;
  std::vector<int> h_ntasks;
  int max_ntasks_prepared = 0;
  // sorted path, per job (grown on demand)
  nid::DeviceBuffer<double> G, jpart_s;
  std::vector<nid::GatherTexture> tex2;  // [n_pairs] packed target textures
  nid::DeviceBuffer<cudaTextureObject_t> d_tex2;
  // kernel 1 (nid_warp_sample_jobs): fp16 target planes, created and filled on first use per pair
  std::vector<nid::GatherTexture> k1tex;
  nid::DeviceBuffer<cudaTextureObject_t> d_k1tex;
  std::vector<char> k1_ready;
  nid::DeviceBuffer<unsigned short> d_k1pack;  // [3N] scratch
  nid::DeviceBuffer<unsigned> fp1;    // [n_pairs][N]
  std::vector<double> h_Twc0, h_cam;  // host copies per pair (geometry tables are built on the host)
  nid::DeviceBuffer<unsigned> d_pack;  // [setup_batch][N] scratch for the packed textures
  size_t g_stride = 0;
  int opt_path = 0;            // 0 auto, 1 natural-order atomics (v1), 2 sorted
  int opt_keep_hist = 0;
  std::vector<char> pair_set, pair_prepared, pair_sorted;
  // staging
  nid::DeviceBuffer<double> d_depth;  // [N] scratch
  nid::DeviceBuffer<double> d_img64;  // [N] scratch for the f64 image entry point
  nid::DeviceBuffer<int> d_flag;
  nid::DeviceBuffer<double> d_pix;    // [8N] scratch for nid_warp_sample_f64
  nid::DeviceBuffer<float> d_pix4;    // [4N] scratch for nid_warp_sample
  nid::DeviceBuffer<float> d_pix4_jobs;  // [max_jobs][4N] output of nid_warp_sample_jobs (allocated on first use)
  nid::DeviceBuffer<double> d_bsv;    // [4N] scratch for nid_get_ref_weights
  nid::DeviceBuffer<int> d_bsi;       // [N]
  // luts
  nid::DeviceBuffer<double> lut_w;
  nid::DeviceBuffer<int> lut_k;
  // per job
  nid::DeviceBuffer<double> pose_buf;  // [job_cap][16] the staged poses
  nid::DeviceBuffer<int> job_pair;
  nid::DeviceBuffer<double> part, jpart, hist;
  nid::DeviceBuffer<double> ht, hj, err, der, gn;
  nid::DeviceBuffer<double> hard;     // [jobs][ncell+1]
  size_t part_slots = 0;       // capacity in (job,strip) units
  // pinned host mirrors of the staged jobs: a ring of NID_STAGE_RING slots, each guarded by an event recorded after
  // the slot's H2D copies, so that a slot is never rewritten while a copy from it is still pending (the staged
  // API is asynchronous: stage, eval, stage, eval ... without a synchronisation in between). The lock-step LM driver
  // takes its pinned job table from the ring the same way.
  nid::PinnedBuffer<double> h_poses_ring;  // [NID_STAGE_RING][job_cap][16]
  nid::PinnedBuffer<int> h_job_pair_ring;  // [NID_STAGE_RING][job_cap]
  nid::Event stage_ev[NID_STAGE_RING];
  int stage_slot = 0;             // the slot taken last: the host mirror of the staged jobs
  int staged_jobs = 0;            // jobs of the last nid_stage_jobs (nid_eval_staged refuses more)
  // nid_prepare / nid_warp_sample* take their pose through their own scratch (both calls are blocking), so that
  // they never disturb staged jobs
  nid::PinnedBuffer<double> h_aux_pose;  // [16]
  nid::DeviceBuffer<double> aux_pose;    // [16]
  nid::PinnedBuffer<double> h_out;    // [max_jobs][ncell*8 + 44]
  int opt_force_strips = 0;
  // LM driver: per half-batch job lists (pinned mirror + device copy), [2 halves][2 lists][max_jobs]
  nid::PinnedBuffer<int> h_lm_lists;
  nid::DeviceBuffer<int> d_lm_lists;
  nid::PinnedBuffer<char> h_lm_stage;  // latency mode: poses + slot list of a round, pinned / device
  nid::PinnedBuffer<int> h_lm_pair;    // latency mode: the slot -> pair mirror [job_cap]
  nid::DeviceBuffer<char> d_lm_stage;
  std::unique_ptr<nid::LatencyGraph, nid::LatencyGraphDelete> lm_graph;  // latency mode: the captured round
  const void* last_hist_func = nullptr;     // the pixel-kernel instantiations the last launch used (graph node lookup)
  const void* last_jac_func = nullptr;
  int opt_lm_graph = 1;
  int opt_stage_bulk = -1;  // pass 2 table staging by cp.async.bulk: -1 by geometry (cells under 2048 pixels), 0 never, 1 always
  int opt_asm_wide = 1;  // 1024-thread assembly when there are fewer (cell, job) units than SMs
  int opt_lm_spec = 4;         // latency mode of nid_solve_jobs (few problems): trial poses evaluated per round and problem
  int opt_lm_reuse = 1;        // a cost+Jacobian job at the pose of the accepted trial reuses that trial's histograms and tables
  nid::Event ev[2];
  // nid_set_pairs_downsampled into this context: [0] recorded on the source's stream before the kernel, [1] on this
  // context's stream after it (created on first use)
  nid::Event ds_ev[2];
  int opt_time_kernels = 0;
  nid::Event kev[5];
  double kernel_ms[4] = {0, 0, 0, 0};  // k_hist, k_jac, k_jac_final, k_entropy
  long long kernel_calls[4] = {0, 0, 0, 0};

  // the members release their handles after the streams have drained
  ~nid_ctx() {
    cudaSetDevice(device);
    for (cudaStream_t s : {stream.get(), lm_stream.get()})
      if (s) cudaStreamSynchronize(s);
  }
};

namespace nid {
// the i-th job of a launch
// up to this many bins pass 2 stages the cell's log tables per warp and k_assemble the reference weight table in shared memory;
// beyond, the staging areas would cost a resident CTA per SM and the tables are read through L1
#define NID_FEW_BINS(bins) ((bins) <= 20)
// cells of fewer pixels than this are "small": 16-pixel tasks, bulk-copy staging and one-warp CTAs in pass 2.
// Measured at 640x480 (evaluations/s as small / as large): 16x16 cells of 1200 pixels 90.6k / 72.5k, 12x12 cells of 2120
// pixels 107.8k / 102.1k, 8x8 cells of 4800 pixels 109.7k / 119.1k.
#ifndef NID_SMALL_CELL_PX
#define NID_SMALL_CELL_PX 2560
#endif
// Layout of the scaled log tables W | V of one (job, cell), written by the assembly and read by pass 2: B rows of W at a
// stride of wv_row(B) doubles -- B + 1 where pass 2 stages the block in shared memory (its lanes then read four rows
// each without bank conflicts, and the block is staged by ONE bulk copy, byte for byte) -- then the B entries of V;
// the block is padded to an even number of doubles (bulk copies move 16-byte units).
__host__ __device__ inline int wv_row(int B) { return NID_FEW_BINS(B) ? B + 1 : B; }
__host__ __device__ inline int wv_stride(int B) { return (B * wv_row(B) + B + 1) & ~1; }
__host__ __device__ inline int job_at(const EvalParams& p, int i) { return p.job_list ? p.job_list[p.job0 + i] : p.job0 + i; }
// The Huber threshold delta^2 as the reference keeps it: `float dsqr` (robust_kernel_impl.h:84). Every launcher that fills
// EvalParams::huber_dsqr takes it from here, so that all Gauss-Newton kernels classify a cell by the same rounded value.
inline double huber_dsqr(double delta) { return (double)(float)(delta * delta); }
#ifdef __CUDACC__
// a11: the Huber-weighted Gauss-Newton block of a job, summed over its active cells in cell order
// (base_unary_edge.hpp:43-72, robust_kernel_impl.cpp:78-90, sparse_optimizer.cpp:102-116):
// entry 0 chi2, 1..36 H (row-major), 37..42 b, 43 the number of active cells.
// huber_weights: rho(e^2) and rho'(e^2) of one cell (robust_kernel_impl.cpp:78-90 with its `float dsqr`).
// gn_accumulate adds the cells [0, n) of the staged arrays (error, the two weights, six Jacobian entries per cell) to
// entry `ent`, in cell order.
__device__ __forceinline__ void huber_weights(double ec, double dsqr, double delta, double& rho0, double& rho1) {
  const double chi = ec * ec;
  if (chi <= dsqr) { rho0 = chi; rho1 = 1.0; }
  else { const double sq = sqrt(chi); rho0 = 2 * sq * delta - dsqr; rho1 = delta / sq; }
}
// (staged arrays: inactive cells -- NaN error -- hold zeros everywhere, so the loops need no branch: adding +0.0 changes nothing)
__device__ __forceinline__ void gn_accumulate(double& acc, const double* e, const double* r0, const double* r1, const double* act,
                                              const double* J, int n, int ent) {
  if (ent == 0) {
    for (int c = 0; c < n; c++) acc += r0[c];
  } else if (ent <= 36) {
    const int i = (ent - 1) / 6, j = (ent - 1) % 6;
    for (int c = 0; c < n; c++) acc += J[6 * c + i] * r1[c] * J[6 * c + j];
  } else if (ent <= 42) {
    const int i = ent - 37;
    for (int c = 0; c < n; c++) acc -= r1[c] * J[6 * c + i] * e[c];
  } else {
    for (int c = 0; c < n; c++) acc += act[c];
  }
}
// The block of one job by one CTA of at least 128 threads: the job's errors and Jacobians are staged in shared memory 256
// cells at a time by all threads (coalesced, independent loads) and every thread computes the Huber weights of its cells
// -- an fp64 square root and a division each -- then 44 threads walk the staged cells in order, one entry each: the sum is
// the sequential one. The entries are dealt to the warps by kind (H: threads 0..35, b: 64..69, chi2: 96, count: 97) so
// that no warp diverges inside its loop. Before: one thread per entry looping over global memory with the weights inline,
// 256 times in a row at the reference's default geometry (256 cells): 49-68 us per launch, a third of a latency-mode round.
// out: 44 doubles per job (device or pinned host memory). want_jac == 0: chi2 and the active count only.
#define NID_GN_CHUNK 256
__device__ __forceinline__ void gn_block(const EvalParams& p, int job, int want_jac, double* __restrict__ out) {
  __shared__ double s_e[NID_GN_CHUNK], s_r0[NID_GN_CHUNK], s_r1[NID_GN_CHUNK], s_act[NID_GN_CHUNK];
  __shared__ double s_J[6 * NID_GN_CHUNK];
  const double* e = p.err + (size_t)job * p.ncell;
  const double* J = p.der + (size_t)job * p.ncell * 6;
  const int t = threadIdx.x;
  const int ent = t < 36 ? t + 1 : (t >= 64 && t < 70) ? t - 64 + 37 : t == 96 ? 0 : t == 97 ? 43 : -1;
  const bool mine = ent >= 0 && (want_jac || ent == 0 || ent == 43);
  double acc = 0.0;
  for (int c0 = 0; c0 < p.ncell; c0 += NID_GN_CHUNK) {
    const int n = min(NID_GN_CHUNK, p.ncell - c0);
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const double ec = e[c0 + i];
      const bool active = !isnan(ec);
      double rho0 = 0.0, rho1 = 0.0;
      if (active) huber_weights(ec, p.huber_dsqr, p.huber_delta, rho0, rho1);
      s_e[i] = active ? ec : 0.0; s_r0[i] = rho0; s_r1[i] = rho1; s_act[i] = active ? 1.0 : 0.0;
    }
    if (want_jac)
      for (int i = threadIdx.x; i < 6 * n; i += blockDim.x) {
        const double v = J[6 * c0 + i];
        s_J[i] = isnan(e[c0 + i / 6]) ? 0.0 : v;  // (inactive cells carry NaN Jacobians)
      }
    __syncthreads();
    if (mine) gn_accumulate(acc, s_e, s_r0, s_r1, s_act, s_J, n, ent);
    __syncthreads();
  }
  if (mine) out[job * 44 + ent] = acc;
}
#endif
void set_error(const std::string& s);
int check_cuda(cudaError_t e, const char* what);
EvalParams make_params(nid_ctx* c, int n_jobs);  // (set-up launchers: no pose table)

// optional per-kernel stopwatch (option "time_kernels"): events between the launches of one evaluation
inline void ktime_mark(nid_ctx* c, cudaStream_t stream, int i) {
  if (!c->opt_time_kernels) return;
  if (!c->kev[i]) c->kev[i].create(cudaEventDefault, "cudaEventCreate (kernel timer)");
  cudaEventRecord(c->kev[i], stream);
}
// adds the interval between marks i and i + 1 to the bucket slot[i] (-1: no kernel ran in it)
inline void ktime_collect(nid_ctx* c, int n, const int* slot) {
  if (!c->opt_time_kernels) return;
  cudaEventSynchronize(c->kev[n]);
  for (int i = 0; i < n; i++) {
    if (slot[i] < 0) continue;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, c->kev[i], c->kev[i + 1]);
    c->kernel_ms[slot[i]] += ms;
    c->kernel_calls[slot[i]]++;
  }
}
bool use_sorted(const nid_ctx* c);
int ensure_job_buffers(nid_ctx* c);

// The evaluation, on either kernel family (use_sorted picks it), of a set of job slots: d_list[first .. first + n)
// (h_list: the host copy of d_list), or the slots first .. first + n - 1 when d_list is null. `slots` is the number of
// slots the set addresses (first + n for a range, the solve's slot count in the LM); pass 1 and pass 2 of the same jobs
// must be given the same value (see strips_for). The launches go on `stream`. Slot s is evaluated at the pose
// d_poses[s] for the pair c->job_pair[s]; h_poses and h_pair are their host mirrors, which the geometry tables are
// built from.
struct JobSet {
  const int* d_list; const int* h_list; int first, n; int slots;
  cudaStream_t stream;
  double* d_poses;  // [slots][16] (the latency round copies its staging block here)
  const double* h_poses; const int* h_pair;
};
EvalParams make_params(nid_ctx* c, const JobSet& js);
// Will pass 2 run on none, some or all of the jobs of a pass 1? Sorted: unless none, the assembly also writes the scaled
// log tables pass 2 reads. Natural: with all, k_jac writes the cost and pass 1 skips k_entropy.
enum class Pass2 { none, some, all };
// nid_sorted.cu: pass 1 writes the histograms and the cost (ht, hj, err) between timer marks 0, 1, 2; pass 2 the Jacobian
// (der) of jobs whose pass 1 has run, up to marks 3, 4. nid_kernels.cu: the Gauss-Newton block (gn), chi2 after pass 1,
// with want_jac also H and b after pass 2.
int launch_pass1(nid_ctx* c, const JobSet& js, Pass2 p2);
int launch_pass2(nid_ctx* c, const JobSet& js);
int launch_gn(nid_ctx* c, const JobSet& js, double delta, int want_jac);

// sorted path (nid_sorted.cu)
int sorted_init(nid_ctx* c);
int launch_count_classes(nid_ctx* c, int pair);
int launch_layout_and_scatter(nid_ctx* c, int pair0, int n);
int launch_pack(nid_ctx* c, int pair0, int n);
int launch_pack_k1(nid_ctx* c, int pair, unsigned short* d_out);
int launch_sorted_tail_gn(nid_ctx* c, const JobSet& js, double delta, double* gn_out);
int launch_latency_round(nid_ctx* c, const JobSet& js, size_t h2d_bytes, double delta, double* gn_out);
int launch_href(nid_ctx* c, int pair0, int n);

// kernel launchers (nid_kernels.cu)
int launch_build_lut(nid_ctx* c);
int launch_points(nid_ctx* c, int pair0, int n, bool u16);
int launch_downsample2(nid_ctx* dst, int dst_pair0, const nid_ctx* src, int src_pair0, int n);
int launch_prepare(nid_ctx* c, int pair0, int n, const double* d_poses16);
int launch_ref_weights(nid_ctx* c, int pair);
int launch_points_aos(nid_ctx* c, int pair, double* d_out);
int launch_hard(nid_ctx* c, const JobSet& js);
int launch_warp_sample(nid_ctx* c, int pair, const double* d_pose16, int f64);
int launch_warp_sample_jobs(nid_ctx* c, const JobSet& js, float4* d_out, bool u16);
int launch_check_integral(nid_ctx* c, const double* d_src, uint8_t* d_dst, int is_ref);
int launch_points_soa(nid_ctx* c, int pair, const double* d_in);
int launch_import_flags(nid_ctx* c, int pair, const double* d_bsv);
}  // namespace nid
