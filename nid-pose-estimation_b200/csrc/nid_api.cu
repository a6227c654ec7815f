// C-ABI of the B200-native NID path (include/nid_b200.h): context, staging, and the host-side
// Levenberg-Marquardt driver (the only CPU arithmetic is the 6x6 solve and the pose update, as in the
// reference: optimization_algorithm_levenberg.cpp:61-225).
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <limits>
#include <string>
#include <chrono>
#include <vector>

#include "../host/nid_host_math.hpp"
#include "nid_ctx.h"

namespace nid {

static thread_local std::string g_err;
void set_error(const std::string& s) { g_err = s; }
int check_cuda(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return NID_OK;
  g_err = std::string(what) + ": " + cudaGetErrorString(e);
  return NID_ERR_CUDA;
}

#define CU(call, what)                                   \
  do {                                                   \
    cudaError_t e_ = (call);                             \
    if (e_ != cudaSuccess) return check_cuda(e_, what);  \
  } while (0)
#define OKR(call)               \
  do {                          \
    int r_ = (call);            \
    if (r_ != NID_OK) return r_; \
  } while (0)

static int strips_for(const nid_ctx* c, int n_jobs) {
  int S;
  if (c->opt_force_strips > 0) S = std::min(c->opt_force_strips, c->rb);
  else {
    long long want = 2LL * c->sm_count;
    long long per = (long long)c->ncell * n_jobs;
    S = (int)((want + per - 1) / per);
    S = std::max(1, std::min(S, std::min(c->rb, 32)));
  }
  // the natural-order kernels write n_jobs * S (job, strip) partials: never more than the buffers hold. They index them
  // by (slot * ncell + cell) * S + strip, so pass 1 and pass 2 of the same slots must use the same S: n_jobs is the
  // number of slots a job set addresses (JobSet::slots), not the length of its list.
  if (c->part_slots > 0 && n_jobs > 0) S = (int)std::max<size_t>(1, std::min<size_t>((size_t)S, c->part_slots / (size_t)n_jobs));
  return S;
}

EvalParams make_params(nid_ctx* c, int n_jobs) {
  EvalParams p;
  memset(&p, 0, sizeof(p));
  p.rows = c->rows; p.cols = c->cols; p.cell = c->cell; p.bins = c->bins;
  p.rb = c->rb; p.cb = c->cb; p.N = c->N; p.ncell = c->ncell;
  p.S = strips_for(c, n_jobs);
  p.strip_rows = (c->rb + p.S - 1) / p.S;
  p.hist_stride = c->bins * c->bins + c->bins;
  p.pwx = c->pwx; p.pwy = c->pwy; p.pwz = c->pwz;
  p.im0 = c->im0; p.im1 = c->im1; p.inb0 = c->inb0;
  p.n_c = c->n_c; p.href = c->href; p.cam = c->cam;
  p.lut_w = c->lut_w; p.lut_k = c->lut_k;
  p.poses = c->poses; p.job_pair = c->job_pair;
  const bool sorted = use_sorted(c);
  p.part = c->part; p.jpart = sorted ? c->jpart_s : c->jpart; p.hist = c->opt_keep_hist ? c->hist.get() : nullptr;
  p.ht = c->ht; p.hj = c->hj; p.err = c->err; p.der = c->der; p.gn = c->gn;
  p.sd0 = c->sd0; p.sd1 = c->sd1; p.sd2 = c->sd2; p.sid = c->sid;
  p.stage_bulk = (c->opt_stage_bulk < 0 ? (long long)c->rb * c->cb < NID_SMALL_CELL_PX : c->opt_stage_bulk) ? 1 : 0;
  p.sl_off = c->sl_off; p.sl_task = c->sl_task; p.sl_desc = c->sl_desc; p.task_cls = c->task_cls; p.sl_cell = c->sl_cell; p.nslices = c->nslices;
  p.sell_cap = c->sell_cap; p.max_slices = c->max_slices; p.Twc0 = c->Twc0;
  p.tasks = c->tasks; p.ntasks = c->ntasks; p.cell_task_start = c->cell_task_start; p.cell_slice_start = c->cell_slice_start;
  p.cls_task_start = c->cls_task_start; p.span_start = c->span_start; p.wv = c->wv;
  p.max_tasks = c->max_tasks; p.g_stride = (int)c->g_stride;
  p.G = c->G; p.fp1 = c->fp1; p.tex2 = c->d_tex2; p.k1tex = c->d_k1tex;
  return p;
}

// Path selection. The sorted path (no floating-point atomics) wins wherever it is available: measured on B200 at
// 640x480, cost+Jacobian: 4x4 cells/16 bins 77k vs 9k evals/s, the reference's default 16x16 cells/10 bins 29k vs 9k
// (tools/time_config.py). The natural-order kernels remain for bin counts outside [6, 40] and as a second,
// independently written implementation the parity tests hold to the same bar.
bool use_sorted(const nid_ctx* c) {
  // the assembly tables must fit in shared memory; the end-block fold needs the two 3x3 blocks disjoint (B >= 6, the
  // reference's smallest knot table, computeH.cu:100)
  if (c->bins > NID_SORTED_MAX_BINS || c->bins < NID_SORTED_MIN_BINS) return false;
  if (c->opt_path == 1) return false;
  return true;
}

std::atomic<long long> live_handles{0};

// Replaces a buffer by one of n elements. The old buffer is released only after the context stream has drained: work
// queued on it may still read the buffer.
template <typename B>
static int regrow(nid_ctx* c, B& buf, size_t n, const char* sync_what, const char* what) {
  CU(cudaStreamSynchronize(c->stream), sync_what);
  return buf.alloc(n, what);
}

// per-job scratch of the active path, allocated on first use / grown when a pair with more tasks is prepared
int ensure_job_buffers(nid_ctx* c) {
  const size_t J = c->job_cap, NC = c->ncell;
  const size_t hs = (size_t)c->bins * c->bins + c->bins;
  if (c->opt_keep_hist && !c->hist) OKR(c->hist.alloc(J * NC * hs, "hist"));
  if (use_sorted(c)) {
    const size_t need = (size_t)std::max(c->max_ntasks_prepared, 1);
    if (c->g_stride < need) {
      c->g_stride = 0;
      OKR(regrow(c, c->G, J * need * c->bins, "sync before growing job buffers", "G"));
      c->g_stride = need;
    }
    if (!c->jpart_s) OKR(c->jpart_s.alloc(J * (size_t)c->max_slices * 6, "jpart_s"));  // one partial per slice
    if (!c->wv) {
      OKR(c->wv.alloc(J * NC * (size_t)nid::wv_stride(c->bins), "wv"));
      CU(cudaMemset(c->wv, 0, sizeof(double) * J * NC * (size_t)nid::wv_stride(c->bins)), "memset wv");  // (the padding is copied, never used)
    }
  } else if (!c->part) {
    c->part_slots = J + 2 * (size_t)c->sm_count + 64;
    OKR(c->part.alloc(c->part_slots * NC * hs, "part"));
    OKR(c->jpart.alloc(c->part_slots * NC * 6, "jpart"));
  }
  return NID_OK;
}

// footprint-packed plane and gather texture of the targets of pairs [pair0, pair0 + n)
static int update_textures(nid_ctx* c, int pair0, int n) {
  for (int i = 0; i < n; i++) c->k1_ready[pair0 + i] = 0;  // kernel 1's planes follow the target image (rebuilt on next use)
  for (int p0 = pair0; p0 < pair0 + n; p0 += c->setup_batch) {
    const int nb = std::min(c->setup_batch, pair0 + n - p0);
    OKR(launch_pack(c, p0, nb));
    for (int i = 0; i < nb; i++)
      CU(cudaMemcpy2DToArrayAsync(c->tex2[p0 + i].array, 0, 0, c->d_pack + (size_t)i * c->N, sizeof(unsigned) * c->cols,
                                  sizeof(unsigned) * c->cols, c->rows, cudaMemcpyDeviceToDevice, c->stream), "packed im1 -> texture array");
  }
  return NID_OK;
}
static int update_texture(nid_ctx* c, int pair) { return update_textures(c, pair, 1); }

// Pinned bump arena for the small per-pair arrays (poses, intrinsics) that the asynchronous set-up calls copy to the
// device: a region is only handed out again after the stream was synchronised.
static int arena_take(nid_ctx* c, size_t bytes, void** out) {
  bytes = (bytes + 63) & ~(size_t)63;
  if (bytes > c->h_arena_cap) {
    const size_t cap = std::max(bytes * 4, (size_t)1 << 20);
    c->h_arena_cap = 0; c->h_arena_used = 0;
    OKR(regrow(c, c->h_arena, cap, "sync before growing the staging arena", "pinned staging arena"));
    c->h_arena_cap = cap;
  }
  if (c->h_arena_used + bytes > c->h_arena_cap) {
    CU(cudaStreamSynchronize(c->stream), "sync to recycle the staging arena");
    c->h_arena_used = 0;
  }
  *out = c->h_arena + c->h_arena_used;
  c->h_arena_used += bytes;
  return NID_OK;
}

// Staging of n_jobs (pair, pose) jobs: the next slot of the pinned ring is taken (waiting, if need be, for the copies
// that last read it), filled, and copied to the device asynchronously on the context stream.
// mode 0: pairs must be prepared (evaluation); 1: pairs must be set (hard-binned NID, kernel 1).
static int stage_jobs(nid_ctx* c, int n_jobs, const int* job_pair, const double* poses, int mode = 0) {
  if (n_jobs < 1 || n_jobs > c->max_jobs) { set_error("n_jobs out of range"); return NID_ERR_ARG; }
  for (int j = 0; j < n_jobs; j++) {
    int pr = job_pair ? job_pair[j] : 0;
    if (pr < 0 || pr >= c->n_pairs) { set_error("job_pair out of range"); return NID_ERR_ARG; }
    if (mode == 1) {
      if (!c->pair_set[pr]) { set_error("job_pair invalid or pair not set"); return NID_ERR_ARG; }
      continue;
    }
    if (!c->pair_prepared[pr]) { set_error("pair not prepared (call nid_prepare)"); return NID_ERR_STATE; }
    if (use_sorted(c) && !c->pair_sorted[pr]) {
      set_error("pair not prepared for the sorted path (call nid_prepare after selecting the path)");
      return NID_ERR_STATE;
    }
  }
  const int slot = (c->stage_slot + 1) % NID_STAGE_RING;
  CU(cudaEventSynchronize(c->stage_ev[slot]), "wait for the staging slot");  // (returns at once for an unrecorded event)
  c->stage_slot = slot;
  c->h_poses = c->h_poses_ring + (size_t)slot * 16 * c->job_cap;
  c->h_job_pair = c->h_job_pair_ring + (size_t)slot * c->job_cap;
  for (int j = 0; j < n_jobs; j++) c->h_job_pair[j] = job_pair ? job_pair[j] : 0;
  memcpy(c->h_poses, poses, sizeof(double) * 16 * n_jobs);
  CU(cudaMemcpyAsync(c->poses, c->h_poses, sizeof(double) * 16 * n_jobs, cudaMemcpyHostToDevice, c->stream), "H2D poses");
  CU(cudaMemcpyAsync(c->job_pair, c->h_job_pair, sizeof(int) * n_jobs, cudaMemcpyHostToDevice, c->stream), "H2D job_pair");
  CU(cudaEventRecord(c->stage_ev[slot], c->stream), "record staging event");
  c->staged_jobs = n_jobs;
  return NID_OK;
}

static int fetch(nid_ctx* c, int n_jobs, int want_jac, double* Ht, double* Hj, double* der) {
  const size_t nc = (size_t)n_jobs * c->ncell;
  double* h = c->h_out;
  if (Ht) CU(cudaMemcpyAsync(h, c->ht, sizeof(double) * nc, cudaMemcpyDeviceToHost, c->stream), "D2H ht");
  if (Hj) CU(cudaMemcpyAsync(h + nc, c->hj, sizeof(double) * nc, cudaMemcpyDeviceToHost, c->stream), "D2H hj");
  if (want_jac && der) CU(cudaMemcpyAsync(h + 2 * nc, c->der, sizeof(double) * 6 * nc, cudaMemcpyDeviceToHost, c->stream), "D2H der");
  CU(cudaStreamSynchronize(c->stream), "sync");
  if (Ht) memcpy(Ht, h, sizeof(double) * nc);
  if (Hj) memcpy(Hj, h + nc, sizeof(double) * nc);
  if (want_jac && der) memcpy(der, h + 2 * nc, sizeof(double) * 6 * nc);
  return NID_OK;
}

}  // namespace nid

using namespace nid;

extern "C" {

const char* nid_last_error(void) { return g_err.c_str(); }
int nid_version(void) { return 100; }

int nid_create(nid_ctx** out, int device, int rows, int cols, int cell, int bins, int degree, int n_pairs, int max_jobs) {
  cudaGetLastError();  // a stale error of another library in this process must not fail our first launch check
  if (!out) { set_error("ctx out pointer is NULL"); return NID_ERR_ARG; }
  *out = nullptr;
  if (degree != 3) { set_error("only bs_degree == 3 (order-4 B-splines) is supported, as in the reference"); return NID_ERR_UNSUPPORTED; }
  if (rows > 65535 || cols > 65535) { set_error("rows, cols must be < 65536"); return NID_ERR_ARG; }
  if (cell > 90) { set_error("cell must be <= 90 (the task descriptors keep the cell index in 13 bits)"); return NID_ERR_ARG; }
  if (rows < 8 || cols < 8 || cell < 1 || bins < 6 || bins > 64 || n_pairs < 1 || max_jobs < 1 || cell > rows || cell > cols) {
    set_error("bad geometry (need rows,cols>=8, 1<=cell<=min(rows,cols), 6<=bins<=64, n_pairs,max_jobs>=1)");
    return NID_ERR_ARG;
  }
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    set_error(std::string("no CUDA device: ") + cudaGetErrorString(e) + " (this library has no CPU path)");
    return NID_ERR_CUDA;
  }
  if (device < 0 || device >= ndev) { set_error("device index out of range"); return NID_ERR_ARG; }
  CU(cudaSetDevice(device), "cudaSetDevice");
  auto c = std::make_unique<nid_ctx>();  // (released on every error return: the members free what was allocated)
  c->device = device; c->rows = rows; c->cols = cols; c->cell = cell; c->bins = bins; c->degree = degree;
  c->N = rows * cols; c->ncell = cell * cell; c->rb = rows / cell; c->cb = cols / cell;
  c->n_pairs = n_pairs; c->max_jobs = max_jobs;
  c->job_cap = std::max(max_jobs, NID_MIN_JOB_SLOTS);
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device), "cudaGetDeviceProperties");
  c->sm_count = prop.multiProcessorCount;
  OKR(c->streams[0].create("cudaStreamCreate"));
  c->stream = c->streams[0];
  const size_t N = c->N, P = n_pairs, J = c->job_cap, NC = c->ncell;
  const size_t hs = (size_t)bins * bins + bins;
  OKR(c->pwx.alloc(P * N, "pwx")); OKR(c->pwy.alloc(P * N, "pwy")); OKR(c->pwz.alloc(P * N, "pwz"));
  OKR(c->im0.alloc(P * N, "im0")); OKR(c->im1.alloc(P * N, "im1")); OKR(c->inb0.alloc(P * N, "inb0"));
  OKR(c->n_c.alloc(P * NC, "n_c")); OKR(c->href.alloc(P * NC, "href"));
  OKR(c->cam.alloc(P * 4, "cam")); OKR(c->Twc0.alloc(P * 16, "Twc0"));
  OKR(c->cnt.alloc(P * NC * NID_NCLS, "cnt"));
  // pixels per task, by geometry only (never by the capacity of the context: a shard of a job must compute the same
  // bits as the whole job). Measured at 640x480, 96 evaluations in flight: 4x4 cells 144k evaluations/s with 32-pixel
  // tasks, 137k with 24, 126k with 16 (twice the task rows to assemble); 8x8 cells 112k / 110k / 103k; the reference's
  // default 16x16 cells (1200 pixels, ~5 per reference intensity) 72.5k with 32, 78.7k with 16 or 20, 77k with 12 (before
  // the other small-cell choices of NID_SMALL_CELL_PX): their
  // tasks are short anyway and a slice is as long as its longest task. Shorter tasks also cut the latency of a lone
  // solve (more, shorter slices: 1.68 -> 1.37 ms at 4x4 cells with 16): option "task_px" for latency-bound callers.
  c->task_px = (long long)c->rb * c->cb < NID_SMALL_CELL_PX ? 16 : 32;
  const int min_task_px = 8;
  c->max_tasks = (int)(N / min_task_px + NC * NID_NCLS + 1);
  c->max_slices = c->max_tasks / 32 + (int)NC + 1;
  // pixel slots per pair: every task is padded to a multiple of 4 and every cell's slices to their longest task
  c->sell_cap = (N + 3 * (size_t)c->max_tasks + NC * 32 * (size_t)(NID_TASK_PX_MAX + 4) + 255) / 128 * 128;
  OKR(c->depth.alloc(P * N, "depth"));
  OKR(c->sl_off.alloc(P * ((size_t)c->max_slices + 1), "sl_off"));
  OKR(c->sl_task.alloc(P * (size_t)c->max_slices * 32, "sl_task"));
  OKR(c->sl_desc.alloc(P * (size_t)c->max_slices * 32, "sl_desc"));
  OKR(c->task_cls.alloc(P * (size_t)c->max_tasks, "task_cls"));
  OKR(c->sl_cell.alloc(P * (size_t)c->max_slices, "sl_cell"));
  OKR(c->task_pos.alloc(P * (size_t)c->max_tasks, "task_pos"));
  OKR(c->nslices.alloc(P, "nslices"));
  CU(cudaMemset(c->nslices, 0, sizeof(int) * P), "memset nslices");
  c->h_nslices.assign(P, 0);
  OKR(c->tasks.alloc(P * (size_t)c->max_tasks, "tasks"));
  OKR(c->ntasks.alloc(P, "ntasks"));
  CU(cudaMemset(c->ntasks, 0, sizeof(int) * P), "memset ntasks");
  OKR(c->cell_task_start.alloc(P * (NC + 1), "cell_task_start"));
  OKR(c->cell_slice_start.alloc(P * (NC + 1), "cell_slice_start"));
  OKR(c->cls_task_start.alloc(P * NC * (NID_NCLS + 1), "cls_task_start"));
  {
    // first class of every span: k_r(v) = floor(v' (B-3)/255), v' = 254.999 for v = 255, is monotone in v
    const int NS = bins - 3;
    std::vector<int> ss(NS + 1, 256);
    auto kr = [bins](int v) { double o = v >= 255 ? 254.999 : (double)v; return (int)std::floor(o * (bins - 3) / 255.0); };
    for (int v = 255; v >= 0; v--)
      for (int k = 0; k <= kr(v) && k <= NS; k++) ss[k] = v;
    ss[NS] = 256;
    OKR(c->span_start.alloc(ss.size(), "span_start"));
    CU(cudaMemcpy(c->span_start, ss.data(), sizeof(int) * ss.size(), cudaMemcpyHostToDevice), "H2D span_start");
  }
  c->h_ntasks.assign(P, 0);
  // packed target images as gather-able textures (tex2Dgather needs a CUDA array created with cudaArrayTextureGather)
  {
    // packed I | Gx | Gy texels, 32 bit
    c->tex2.resize(P);
    std::vector<cudaTextureObject_t> h_tex2(P);
    for (size_t i = 0; i < P; i++) {
      if (c->tex2[i].create(cudaCreateChannelDesc<unsigned int>(), cols, rows, "packed target") != NID_OK) {
        cudaGetLastError();
        set_error("could not create the packed gather textures for the target images");
        return NID_ERR_CUDA;
      }
      h_tex2[i] = c->tex2[i].tex;
    }
    OKR(c->d_tex2.alloc(P, "d_tex2"));
    OKR(c->d_k1tex.alloc(P, "d_k1tex"));
    CU(cudaMemset(c->d_k1tex, 0, sizeof(cudaTextureObject_t) * P), "memset k1tex");
    c->k1tex.resize(P);
    c->k1_ready.assign(P, 0);
    CU(cudaMemcpy(c->d_tex2, h_tex2.data(), sizeof(cudaTextureObject_t) * P, cudaMemcpyHostToDevice), "H2D tex2 handles");
    c->setup_batch = (int)std::min<size_t>(P, 32);
    OKR(c->d_pack.alloc(N * (size_t)c->setup_batch, "d_pack"));
    OKR(c->lay_tot.alloc((size_t)c->setup_batch * NC * 3, "lay_tot"));
    OKR(c->lay_base.alloc((size_t)c->setup_batch * NC * 3, "lay_base"));
    OKR(c->prep_poses.alloc((size_t)c->setup_batch * 16, "prep_poses"));
    OKR(c->depth_factor.alloc(P, "depth_factor"));
    c->pair_u16.assign(P, 0);
    OKR(c->fp1.alloc(P * N, "fp1"));
    c->h_Twc0.assign(P * 16, 0.0);
    c->h_cam.assign(P * 4, 1.0);
  }
  OKR(c->d_depth.alloc(N, "d_depth")); OKR(c->d_img64.alloc(N, "d_img64")); OKR(c->d_flag.alloc(2, "d_flag"));
  CU(cudaMemset(c->d_flag, 0, sizeof(int) * 2), "memset flag");
  OKR(c->lut_w.alloc(256 * 4, "lut_w")); OKR(c->lut_k.alloc(256, "lut_k"));
  OKR(c->pose_buf.alloc(J * 16, "poses")); OKR(c->job_pair.alloc(J, "job_pair"));
  c->poses = c->pose_buf;
  CU(cudaMemset(c->job_pair, 0, sizeof(int) * J), "memset job_pair");
  CU(cudaMemset(c->poses, 0, sizeof(double) * 16 * J), "memset poses");
  OKR(c->aux_pose.alloc(16, "aux_pose"));
  (void)hs;
  OKR(c->ht.alloc(J * NC, "ht")); OKR(c->hj.alloc(J * NC, "hj")); OKR(c->err.alloc(J * NC, "err"));
  OKR(c->der.alloc(J * NC * 6, "der")); OKR(c->gn.alloc(J * 44, "gn"));
  OKR(c->hard.alloc(J * (NC + 1), "hard"));
  OKR(c->h_poses_ring.alloc(16 * J * NID_STAGE_RING, "pinned poses"));
  OKR(c->h_job_pair_ring.alloc(J * NID_STAGE_RING, "pinned job_pair"));
  memset(c->h_poses_ring, 0, sizeof(double) * 16 * J * NID_STAGE_RING);
  memset(c->h_job_pair_ring, 0, sizeof(int) * J * NID_STAGE_RING);
  c->h_poses = c->h_poses_ring;
  c->h_job_pair = c->h_job_pair_ring;
  for (auto& e : c->stage_ev) OKR(e.create(cudaEventDisableTiming, "cudaEventCreate (staging)"));
  OKR(c->h_aux_pose.alloc(16, "pinned aux pose"));
  OKR(c->h_out.alloc(J * (NC * 8 + 44), "pinned out"));
  c->pair_set.assign(P, 0);
  c->pair_prepared.assign(P, 0);
  c->pair_sorted.assign(P, 0);
  OKR(launch_build_lut(c.get()));
  OKR(sorted_init(c.get()));
  CU(cudaStreamSynchronize(c->stream), "sync after lut");
  *out = c.release();
  return NID_OK;
}

int nid_destroy(nid_ctx* c) {
  delete c;
  return NID_OK;
}

int nid_sync(nid_ctx* c) {
  if (!c) { set_error("NULL ctx"); return NID_ERR_ARG; }
  CU(cudaSetDevice(c->device), "cudaSetDevice");
  CU(cudaStreamSynchronize(c->stream), "nid_sync");
  c->h_arena_used = 0;
  return NID_OK;
}

// Geometry of pairs [pair0, pair0 + n): T_wc0 [n][16] and intr [n][5] go through the pinned arena (the device keeps
// fx fy cx cy and the depth factor in separate tables), then the world points. depth64 / depth16: [n][N], one of them.
static int set_pairs_geometry(nid_ctx* c, int pair0, int n, const double* depth64, const uint16_t* depth16, const double* T_wc0,
                              const double* intr) {
  if (pair0 < 0 || n < 1 || pair0 + n > c->n_pairs) { set_error("pair range out of bounds"); return NID_ERR_ARG; }
  if ((!depth64 && !depth16) || !T_wc0 || !intr) { set_error("NULL argument"); return NID_ERR_ARG; }
  CU(cudaSetDevice(c->device), "cudaSetDevice");
  const size_t N = c->N;
  if (depth16) {
    if (!c->depth16) OKR(c->depth16.alloc((size_t)c->n_pairs * N, "depth16"));
    CU(cudaMemcpyAsync(c->depth16 + (size_t)pair0 * N, depth16, sizeof(uint16_t) * N * n, cudaMemcpyDefault, c->stream), "H2D depth (u16)");
  } else {
    CU(cudaMemcpyAsync(c->depth + (size_t)pair0 * N, depth64, sizeof(double) * N * n, cudaMemcpyDefault, c->stream), "H2D depth");
  }
  double* a = nullptr;
  OKR(arena_take(c, sizeof(double) * 21 * n, (void**)&a));
  double *aT = a, *acam = a + 16 * (size_t)n, *afac = a + 20 * (size_t)n;
  memcpy(aT, T_wc0, sizeof(double) * 16 * n);
  for (int i = 0; i < n; i++) {
    memcpy(acam + 4 * i, intr + 5 * (size_t)i, sizeof(double) * 4);
    afac[i] = intr[5 * (size_t)i + 4];
  }
  CU(cudaMemcpyAsync(c->Twc0 + 16 * (size_t)pair0, aT, sizeof(double) * 16 * n, cudaMemcpyHostToDevice, c->stream), "H2D Twc0");
  CU(cudaMemcpyAsync(c->cam + 4 * (size_t)pair0, acam, sizeof(double) * 4 * n, cudaMemcpyHostToDevice, c->stream), "H2D intr");
  CU(cudaMemcpyAsync(c->depth_factor + pair0, afac, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream), "H2D depth factor");
  memcpy(c->h_Twc0.data() + 16 * (size_t)pair0, aT, sizeof(double) * 16 * n);
  memcpy(c->h_cam.data() + 4 * (size_t)pair0, acam, sizeof(double) * 4 * n);
  OKR(launch_points(c, pair0, n, depth16 != nullptr));
  for (int i = 0; i < n; i++) { c->pair_prepared[pair0 + i] = 0; c->pair_u16[pair0 + i] = depth16 ? 1 : 0; }
  return NID_OK;
}
static int set_pair_common(nid_ctx* c, int pair, const double* depth, const double T_wc0[16], const double intr[5]) {
  if (pair < 0 || pair >= c->n_pairs) { set_error("pair index out of range"); return NID_ERR_ARG; }
  return set_pairs_geometry(c, pair, 1, depth, nullptr, T_wc0, intr);
}

int nid_set_pair(nid_ctx* c, int pair, const double* depth, const uint8_t* im0, const uint8_t* im1, const double T_wc0[16],
                 const double intr[5]) {
  if (!c) { set_error("NULL ctx"); return NID_ERR_ARG; }
  if (!im0 || !im1) { set_error("NULL image"); return NID_ERR_ARG; }
  OKR(set_pair_common(c, pair, depth, T_wc0, intr));
  CU(cudaMemcpyAsync(c->im0 + (size_t)pair * c->N, im0, c->N, cudaMemcpyDefault, c->stream), "H2D im0");
  CU(cudaMemcpyAsync(c->im1 + (size_t)pair * c->N, im1, c->N, cudaMemcpyDefault, c->stream), "H2D im1");
  OKR(update_texture(c, pair));
  CU(cudaStreamSynchronize(c->stream), "sync set_pair");
  c->pair_set[pair] = 1;
  return NID_OK;
}

int nid_set_pairs_u16(nid_ctx* c, int pair0, int n, const uint16_t* depth_raw, const uint8_t* im0, const uint8_t* im1,
                      const double* T_wc0, const double* intr) {
  if (!c) { set_error("NULL ctx"); return NID_ERR_ARG; }
  if (!im0 || !im1 || !depth_raw) { set_error("NULL image"); return NID_ERR_ARG; }
  if (c->sell_points) { set_error("this context holds caller-supplied world points (nid_set_pair_points)"); return NID_ERR_STATE; }
  OKR(set_pairs_geometry(c, pair0, n, nullptr, depth_raw, T_wc0, intr));
  const size_t N = c->N;
  CU(cudaMemcpyAsync(c->im0 + (size_t)pair0 * N, im0, N * n, cudaMemcpyDefault, c->stream), "H2D im0");
  CU(cudaMemcpyAsync(c->im1 + (size_t)pair0 * N, im1, N * n, cudaMemcpyDefault, c->stream), "H2D im1");
  OKR(update_textures(c, pair0, n));
  for (int i = 0; i < n; i++) c->pair_set[pair0 + i] = 1;
  return NID_OK;  // (asynchronous: see the header)
}

// A coarser level of pairs that already live on the device: k_downsample2 writes depth and images, the intrinsics are
// derived on the host from the source's mirror, T_wc0 is copied device to device; then the ordinary world points and
// target textures. dst's stream waits for the source's queued work, and the source's stream waits for the kernel, so a
// refill of the source slot issued right after this call cannot overwrite what is being read.
int nid_set_pairs_downsampled(nid_ctx* dst, int dst_pair0, const nid_ctx* src, int src_pair0, int n) {
  if (!dst || !src) { set_error("NULL context"); return NID_ERR_ARG; }
  if (dst->rows != src->rows / 2 || dst->cols != src->cols / 2) {
    set_error("destination geometry must be (source rows / 2, source cols / 2)");
    return NID_ERR_ARG;
  }
  if (n < 1 || n > dst->n_pairs || n > src->n_pairs || dst_pair0 < 0 || src_pair0 < 0 || dst_pair0 > dst->n_pairs - n ||
      src_pair0 > src->n_pairs - n) {
    set_error("pair range out of bounds");
    return NID_ERR_ARG;
  }
  if (dst->device != src->device) { set_error("source and destination contexts live on different devices"); return NID_ERR_ARG; }
  if (src->sell_points || dst->sell_points) {
    set_error("downsampling needs depth pairs on both sides, not caller-supplied world points (nid_set_pair_points)");
    return NID_ERR_STATE;
  }
  for (int i = 0; i < n; i++)
    if (!src->pair_set[src_pair0 + i]) { set_error("source pair not set"); return NID_ERR_STATE; }
  CU(cudaSetDevice(dst->device), "cudaSetDevice");
  for (int i = 0; i < 2; i++)
    if (!dst->ds_ev[i]) OKR(dst->ds_ev[i].create(cudaEventDisableTiming, "cudaEventCreate (downsample)"));
  double* a = nullptr;
  OKR(arena_take(dst, sizeof(double) * 5 * n, (void**)&a));
  double *acam = a, *afac = a + 4 * (size_t)n;
  for (int i = 0; i < n; i++) {
    // a coarse pixel centre j sits at fine coordinate 2j + 0.5 (the reference samples pixel j at u = j)
    const double* k = src->h_cam.data() + 4 * (size_t)(src_pair0 + i);
    acam[4 * i] = k[0] * 0.5; acam[4 * i + 1] = k[1] * 0.5;
    acam[4 * i + 2] = (k[2] - 0.5) * 0.5; acam[4 * i + 3] = (k[3] - 0.5) * 0.5;
    afac[i] = 1.0;  // (unused: the destination holds fp64 depth)
  }
  CU(cudaEventRecord(dst->ds_ev[0], src->stream), "record source event");
  CU(cudaStreamWaitEvent(dst->stream, dst->ds_ev[0], 0), "wait for the source");
  CU(cudaMemcpyAsync(dst->cam + 4 * (size_t)dst_pair0, acam, sizeof(double) * 4 * n, cudaMemcpyHostToDevice, dst->stream), "H2D intr");
  CU(cudaMemcpyAsync(dst->depth_factor + dst_pair0, afac, sizeof(double) * n, cudaMemcpyHostToDevice, dst->stream), "H2D depth factor");
  CU(cudaMemcpyAsync(dst->Twc0 + 16 * (size_t)dst_pair0, src->Twc0 + 16 * (size_t)src_pair0, sizeof(double) * 16 * n,
                     cudaMemcpyDeviceToDevice, dst->stream), "D2D Twc0");
  memcpy(dst->h_cam.data() + 4 * (size_t)dst_pair0, acam, sizeof(double) * 4 * n);
  memcpy(dst->h_Twc0.data() + 16 * (size_t)dst_pair0, src->h_Twc0.data() + 16 * (size_t)src_pair0, sizeof(double) * 16 * n);
  OKR(launch_downsample2(dst, dst_pair0, src, src_pair0, n));
  OKR(launch_points(dst, dst_pair0, n, false));
  OKR(update_textures(dst, dst_pair0, n));
  CU(cudaEventRecord(dst->ds_ev[1], dst->stream), "record destination event");
  CU(cudaStreamWaitEvent(src->stream, dst->ds_ev[1], 0), "order the source after the kernel");
  for (int i = 0; i < n; i++) {
    dst->pair_set[dst_pair0 + i] = 1;
    dst->pair_prepared[dst_pair0 + i] = 0;
    dst->pair_u16[dst_pair0 + i] = 0;
  }
  return NID_OK;  // (asynchronous: see the header)
}

int nid_set_target(nid_ctx* c, int pair, const uint8_t* im1) {
  if (!c || !im1) { set_error("bad argument"); return NID_ERR_ARG; }
  if (pair < 0 || pair >= c->n_pairs) { set_error("pair index out of range"); return NID_ERR_ARG; }
  if (!c->pair_set[pair]) { set_error("pair not set (nid_set_target replaces the target of an existing pair)"); return NID_ERR_STATE; }
  CU(cudaSetDevice(c->device), "cudaSetDevice");
  CU(cudaMemcpyAsync(c->im1 + (size_t)pair * c->N, im1, c->N, cudaMemcpyDefault, c->stream), "H2D im1");
  OKR(update_texture(c, pair));
  CU(cudaStreamSynchronize(c->stream), "sync set_target");
  c->pair_prepared[pair] = 0;
  return NID_OK;
}

static int upload_images_f64(nid_ctx* c, int pair, const double* im0, const double* im1);
static int build_sorted_layout(nid_ctx* c, int pair0, int n);
static int finish_sorted_layout(nid_ctx* c, int pair0, int n, int* bs_counter, double* Href);

int nid_set_pair_f64(nid_ctx* c, int pair, const double* depth, const double* im0, const double* im1,
                     const double T_wc0[16], const double intr[5]) {
  if (!c) { set_error("NULL ctx"); return NID_ERR_ARG; }
  OKR(set_pair_common(c, pair, depth, T_wc0, intr));
  OKR(upload_images_f64(c, pair, im0, im1));
  c->pair_set[pair] = 1;
  return NID_OK;
}

static int upload_images_f64(nid_ctx* c, int pair, const double* im0, const double* im1) {
  CU(cudaMemsetAsync(c->d_flag, 0, sizeof(int), c->stream), "memset flag");
  if (im0) {
    CU(cudaMemcpyAsync(c->d_img64, im0, sizeof(double) * c->N, cudaMemcpyDefault, c->stream), "H2D im0 f64");
    OKR(launch_check_integral(c, c->d_img64, c->im0 + (size_t)pair * c->N, 1));
  }
  if (im1) {
    CU(cudaMemcpyAsync(c->d_img64, im1, sizeof(double) * c->N, cudaMemcpyDefault, c->stream), "H2D im1 f64");
    OKR(launch_check_integral(c, c->d_img64, c->im1 + (size_t)pair * c->N, 0));
    OKR(update_texture(c, pair));
  }
  int flag = 0;
  CU(cudaMemcpyAsync(&flag, c->d_flag, sizeof(int), cudaMemcpyDeviceToHost, c->stream), "D2H flag");
  CU(cudaStreamSynchronize(c->stream), "sync upload images");
  if (flag) {
    set_error("image holds non-8-bit values (non-integral or outside [0,255]); only 8-bit gray is supported");
    return NID_ERR_UNSUPPORTED;
  }
  return NID_OK;
}

int nid_set_pair_points(nid_ctx* c, int pair, const double* points_3d, const double* im0, const double* im1,
                        const double intr[5]) {
  if (!c || pair < 0 || pair >= c->n_pairs) { set_error("bad argument"); return NID_ERR_ARG; }
  CU(cudaSetDevice(c->device), "cudaSetDevice");
  if (points_3d) {
    if (!intr) { set_error("intr required with points"); return NID_ERR_ARG; }
    if (!c->d_pix) OKR(c->d_pix.alloc((size_t)8 * c->N, "d_pix"));
    CU(cudaMemcpyAsync(c->d_pix, points_3d, sizeof(double) * 3 * c->N, cudaMemcpyDefault, c->stream), "H2D points3d");
    CU(cudaMemcpyAsync(c->cam + 4 * pair, intr, sizeof(double) * 4, cudaMemcpyDefault, c->stream), "H2D intr");
    memcpy(c->h_cam.data() + 4 * (size_t)pair, intr, sizeof(double) * 4);
    OKR(launch_points_soa(c, pair, c->d_pix));
    c->pair_prepared[pair] = 0;
    if (!c->sell_points) {
      // caller-supplied world points cannot be rebuilt from (depth, pixel): the sorted store keeps the points
      CU(cudaStreamSynchronize(c->stream), "sync before switching to the point form");
      c->sell_points = true;
      std::fill(c->pair_prepared.begin(), c->pair_prepared.end(), 0);
    }
  }
  OKR(upload_images_f64(c, pair, im0, im1));
  c->pair_set[pair] = 1;
  return NID_OK;
}

int nid_import_prepare(nid_ctx* c, int pair, const double* bs_value, const int* bs_counter, const double* Href) {
  if (!c || pair < 0 || pair >= c->n_pairs || !bs_value || !bs_counter || !Href) { set_error("bad argument"); return NID_ERR_ARG; }
  if (!c->pair_set[pair]) { set_error("pair not set"); return NID_ERR_STATE; }
  CU(cudaSetDevice(c->device), "cudaSetDevice");
  if (!c->d_bsv) { OKR(c->d_bsv.alloc((size_t)4 * c->N, "d_bsv")); OKR(c->d_bsi.alloc((size_t)c->N, "d_bsi")); }
  CU(cudaMemcpyAsync(c->d_bsv, bs_value, sizeof(double) * 4 * c->N, cudaMemcpyDefault, c->stream), "H2D bs_value");
  OKR(launch_import_flags(c, pair, c->d_bsv));
  CU(cudaMemcpyAsync(c->n_c + pair * c->ncell, bs_counter, sizeof(int) * c->ncell, cudaMemcpyDefault, c->stream), "H2D n_c");
  CU(cudaMemcpyAsync(c->href + pair * c->ncell, Href, sizeof(double) * c->ncell, cudaMemcpyDefault, c->stream), "H2D href");
  CU(cudaMemsetAsync(c->cnt + (size_t)pair * c->ncell * NID_NCLS, 0, sizeof(unsigned int) * c->ncell * NID_NCLS, c->stream), "memset cnt");
  OKR(launch_count_classes(c, pair));
  OKR(build_sorted_layout(c, pair, 1));
  OKR(finish_sorted_layout(c, pair, 1, nullptr, nullptr));
  c->pair_prepared[pair] = 1;
  return NID_OK;
}

int nid_get_inbounds(nid_ctx* c, int pair, uint8_t* flags) {
  if (!c || pair < 0 || pair >= c->n_pairs || !flags) { set_error("bad argument"); return NID_ERR_ARG; }
  if (!c->pair_prepared[pair]) { set_error("pair not prepared"); return NID_ERR_STATE; }
  CU(cudaSetDevice(c->device), "cudaSetDevice");
  CU(cudaMemcpyAsync(flags, c->inb0 + (size_t)pair * c->N, c->N, cudaMemcpyDefault, c->stream), "D2H inb0");
  CU(cudaStreamSynchronize(c->stream), "sync inb0");
  return NID_OK;
}

int nid_get_points3d(nid_ctx* c, int pair, double* points_3d) {
  if (!c || pair < 0 || pair >= c->n_pairs || !points_3d) { set_error("bad argument"); return NID_ERR_ARG; }
  if (!c->pair_set[pair]) { set_error("pair not set"); return NID_ERR_STATE; }
  CU(cudaSetDevice(c->device), "cudaSetDevice");
  if (!c->d_pix) OKR(c->d_pix.alloc((size_t)8 * c->N, "d_pix"));
  OKR(launch_points_aos(c, pair, c->d_pix));
  CU(cudaMemcpyAsync(points_3d, c->d_pix, sizeof(double) * 3 * c->N, cudaMemcpyDefault, c->stream), "copy points3d");
  CU(cudaStreamSynchronize(c->stream), "sync points3d");
  return NID_OK;
}

// Regroup the valid pixels of pairs [pair0, pair0 + n) by (cell, reference class), cut the segments into tasks of at most
// task_px pixels, order the tasks by length and pack them 32 to a slice (nid_sorted.cu). Everything happens on the
// device, from the class counts k_prepare left there: table kernels, then the regrouping scatter. Asynchronous.
static int build_sorted_layout(nid_ctx* c, int pair0, int n) {
  for (int i = 0; i < n; i++) c->pair_sorted[pair0 + i] = 0;
  if (!use_sorted(c)) return NID_OK;  // the natural-order kernels need none of this
  if (!c->sd0) {
    OKR(c->sd0.alloc((size_t)c->n_pairs * c->sell_cap, "sd0"));
    OKR(c->sid.alloc((size_t)c->n_pairs * c->sell_cap, "sid"));
  }
  if (c->sell_points && !c->sd1) {
    OKR(c->sd1.alloc((size_t)c->n_pairs * c->sell_cap, "sd1"));
    OKR(c->sd2.alloc((size_t)c->n_pairs * c->sell_cap, "sd2"));
  }
  if (!c->chunk_cnt) {
    const size_t nchunks = ((size_t)c->rb * c->cb + 255) / 256;
    OKR(c->chunk_cnt.alloc((size_t)c->setup_batch * c->ncell * nchunks * NID_NCLS, "chunk_cnt"));
  }
  for (int p0 = pair0; p0 < pair0 + n; p0 += c->setup_batch)
    OKR(launch_layout_and_scatter(c, p0, std::min(c->setup_batch, pair0 + n - p0)));
  return NID_OK;
}

// One synchronisation for the whole range: n_c and H_ref for the caller, task and slice counts for the launch geometry.
static int finish_sorted_layout(nid_ctx* c, int pair0, int n, int* bs_counter, double* Href) {
  const size_t NC = c->ncell;
  const size_t bytes = (size_t)n * (NC * (sizeof(double) + sizeof(int)) + 2 * sizeof(int)) + sizeof(int) + 64;
  if (c->h_res_cap < bytes) {
    c->h_res_cap = 0;
    OKR(regrow(c, c->h_res, bytes * 2, "sync before growing the result buffer", "pinned prepare results"));
    c->h_res_cap = bytes * 2;
  }
  double* h_href = (double*)c->h_res.get();
  int* h_nc = (int*)(h_href + (size_t)n * NC);
  int* h_nt = h_nc + (size_t)n * NC;
  int* h_ns = h_nt + n;
  int* h_ovf = h_ns + n;
  CU(cudaMemcpyAsync(h_nc, c->n_c + (size_t)pair0 * NC, sizeof(int) * NC * n, cudaMemcpyDeviceToHost, c->stream), "D2H n_c");
  CU(cudaMemcpyAsync(h_href, c->href + (size_t)pair0 * NC, sizeof(double) * NC * n, cudaMemcpyDeviceToHost, c->stream), "D2H href");
  const bool sorted = use_sorted(c);
  if (sorted) {
    CU(cudaMemcpyAsync(h_nt, c->ntasks + pair0, sizeof(int) * n, cudaMemcpyDeviceToHost, c->stream), "D2H ntasks");
    CU(cudaMemcpyAsync(h_ns, c->nslices + pair0, sizeof(int) * n, cudaMemcpyDeviceToHost, c->stream), "D2H nslices");
    CU(cudaMemcpyAsync(h_ovf, c->d_flag + 1, sizeof(int), cudaMemcpyDeviceToHost, c->stream), "D2H overflow flag");
  }
  CU(cudaStreamSynchronize(c->stream), "sync prepare");
  c->h_arena_used = 0;
  if (sorted) {
    if (*h_ovf) { set_error("sliced pixel store overflow"); return NID_ERR_STATE; }
    for (int i = 0; i < n; i++) {
      c->h_ntasks[pair0 + i] = h_nt[i];
      c->h_nslices[pair0 + i] = h_ns[i];
      c->pair_sorted[pair0 + i] = 1;
    }
    c->max_ntasks_prepared = 0;
    for (int v : c->h_ntasks) c->max_ntasks_prepared = std::max(c->max_ntasks_prepared, v);
    c->max_nslices_prepared = 0;
    for (int v : c->h_nslices) c->max_nslices_prepared = std::max(c->max_nslices_prepared, v);
  }
  if (bs_counter) memcpy(bs_counter, h_nc, sizeof(int) * NC * n);
  if (Href) memcpy(Href, h_href, sizeof(double) * NC * n);
  return NID_OK;
}

int nid_prepare_pairs(nid_ctx* c, int pair0, int n, const double* T_cw1, int* bs_counter, double* Href) {
  if (!c || !T_cw1 || n < 1 || pair0 < 0 || pair0 + n > c->n_pairs) { set_error("bad argument"); return NID_ERR_ARG; }
  for (int i = 0; i < n; i++)
    if (!c->pair_set[pair0 + i]) { set_error("pair not set"); return NID_ERR_STATE; }
  CU(cudaSetDevice(c->device), "cudaSetDevice");
  for (int p0 = pair0; p0 < pair0 + n; p0 += c->setup_batch) {
    const int nb = std::min(c->setup_batch, pair0 + n - p0);
    double* a = nullptr;
    OKR(arena_take(c, sizeof(double) * 16 * nb, (void**)&a));
    memcpy(a, T_cw1 + 16 * (size_t)(p0 - pair0), sizeof(double) * 16 * nb);
    CU(cudaMemcpyAsync(c->prep_poses, a, sizeof(double) * 16 * nb, cudaMemcpyHostToDevice, c->stream), "H2D initial poses");
    OKR(launch_prepare(c, p0, nb, c->prep_poses));
    OKR(launch_href(c, p0, nb));
    OKR(build_sorted_layout(c, p0, nb));
  }
  OKR(finish_sorted_layout(c, pair0, n, bs_counter, Href));
  for (int i = 0; i < n; i++) c->pair_prepared[pair0 + i] = 1;
  return NID_OK;
}

int nid_prepare(nid_ctx* c, int pair, const double T_cw1[16], int* bs_counter, double* Href) {
  if (!c || pair < 0 || pair >= c->n_pairs || !T_cw1) { set_error("bad argument"); return NID_ERR_ARG; }
  return nid_prepare_pairs(c, pair, 1, T_cw1, bs_counter, Href);
}

int nid_get_ref_weights(nid_ctx* c, int pair, double* bs_value, int* bs_index) {
  if (!c || pair < 0 || pair >= c->n_pairs) { set_error("bad argument"); return NID_ERR_ARG; }
  if (!c->pair_prepared[pair]) { set_error("pair not prepared"); return NID_ERR_STATE; }
  CU(cudaSetDevice(c->device), "cudaSetDevice");
  if (!c->d_bsv) { OKR(c->d_bsv.alloc((size_t)4 * c->N, "d_bsv")); OKR(c->d_bsi.alloc((size_t)c->N, "d_bsi")); }
  OKR(launch_ref_weights(c, pair));
  if (bs_value) CU(cudaMemcpyAsync(bs_value, c->d_bsv, sizeof(double) * 4 * c->N, cudaMemcpyDefault, c->stream), "D2H bs_value");
  if (bs_index) CU(cudaMemcpyAsync(bs_index, c->d_bsi, sizeof(int) * c->N, cudaMemcpyDefault, c->stream), "D2H bs_index");
  CU(cudaStreamSynchronize(c->stream), "sync ref_weights");
  return NID_OK;
}

int nid_stage_jobs(nid_ctx* c, int n_jobs, const int* job_pair, const double* poses) {
  if (!c || !poses) { set_error("bad argument"); return NID_ERR_ARG; }
  CU(cudaSetDevice(c->device), "cudaSetDevice");
  return stage_jobs(c, n_jobs, job_pair, poses);
}

// cost (+ Jacobian) of the staged jobs 0 .. n - 1
static int eval_range(nid_ctx* c, int n, int want_jac) {
  OKR(ensure_job_buffers(c));
  const JobSet js{nullptr, nullptr, 0, n, n};
  OKR(launch_pass1(c, js, want_jac ? Pass2::all : Pass2::none));
  if (!want_jac) {
    const int slot[2] = {0, 3};
    ktime_collect(c, 2, slot);
    return NID_OK;
  }
  OKR(launch_pass2(c, js));
  const int sorted_slot[4] = {0, 3, 1, 2}, natural_slot[4] = {0, -1, 1, 2};  // (natural: no cost tail between marks 1 and 2)
  ktime_collect(c, 4, use_sorted(c) ? sorted_slot : natural_slot);
  return NID_OK;
}

int nid_eval_staged(nid_ctx* c, int n_jobs, int want_jac) {
  if (!c || n_jobs < 1 || n_jobs > c->max_jobs) { set_error("bad argument"); return NID_ERR_ARG; }
  if (n_jobs > c->staged_jobs) { set_error("nid_eval_staged: more jobs than the last nid_stage_jobs staged"); return NID_ERR_STATE; }
  CU(cudaSetDevice(c->device), "cudaSetDevice");
  return eval_range(c, n_jobs, want_jac);
}

int nid_fetch_results(nid_ctx* c, int n_jobs, int want_jac, double* Ht, double* Hj, double* der) {
  if (!c || n_jobs < 1 || n_jobs > c->max_jobs) { set_error("bad argument"); return NID_ERR_ARG; }
  CU(cudaSetDevice(c->device), "cudaSetDevice");
  return fetch(c, n_jobs, want_jac, Ht, Hj, der);
}

int nid_eval_jobs(nid_ctx* c, int n_jobs, const int* job_pair, const double* poses, int want_jac, double* Ht, double* Hj,
                  double* der) {
  if (!c || !poses) { set_error("bad argument"); return NID_ERR_ARG; }
  CU(cudaSetDevice(c->device), "cudaSetDevice");
  OKR(stage_jobs(c, n_jobs, job_pair, poses));
  OKR(eval_range(c, n_jobs, want_jac));
  return fetch(c, n_jobs, want_jac, Ht, Hj, der);
}

int nid_eval(nid_ctx* c, int pair, const double T_cw1[16], int want_jac, double* Ht, double* Hj, double* der) {
  return nid_eval_jobs(c, 1, &pair, T_cw1, want_jac, Ht, Hj, der);
}

int nid_eval_gn(nid_ctx* c, int pair, const double T_cw1[16], double delta, double* chi2, double* H36, double* b6,
                double* err, double* J) {
  if (!c || !T_cw1) { set_error("bad argument"); return NID_ERR_ARG; }
  CU(cudaSetDevice(c->device), "cudaSetDevice");
  OKR(stage_jobs(c, 1, &pair, T_cw1));
  OKR(eval_range(c, 1, 1));
  OKR(launch_gn(c, JobSet{nullptr, nullptr, 0, 1, 1}, delta, 1));
  double* h = c->h_out;
  const size_t nc = c->ncell;
  CU(cudaMemcpyAsync(h, c->gn, sizeof(double) * 44, cudaMemcpyDeviceToHost, c->stream), "D2H gn");
  CU(cudaMemcpyAsync(h + 44, c->err, sizeof(double) * nc, cudaMemcpyDeviceToHost, c->stream), "D2H err");
  CU(cudaMemcpyAsync(h + 44 + nc, c->der, sizeof(double) * 6 * nc, cudaMemcpyDeviceToHost, c->stream), "D2H der");
  CU(cudaStreamSynchronize(c->stream), "sync gn");
  if (chi2) *chi2 = h[0];
  if (H36) memcpy(H36, h + 1, sizeof(double) * 36);
  if (b6) memcpy(b6, h + 37, sizeof(double) * 6);
  if (err) memcpy(err, h + 44, sizeof(double) * nc);
  if (J) memcpy(J, h + 44 + nc, sizeof(double) * 6 * nc);
  return NID_OK;
}

// ---------------------------------------------------------------------------------------------- LM
namespace {
// One LM problem: one unknown pose `est` shared by the problem's jobs (a pair each). nid_solve_jobs gives every problem one
// job; nid_solve_groups several, whose Gauss-Newton blocks are summed into the problem's one block before every step.
struct LM {
  nidhost::Pose7 est, backup;
  double lambda = -1., ni = 2.;
  int nBad = 0, it = 0, qmax = 0;
  double currentChi = 0, iniChi = 0, rho = 0;
  double H[36], b[6], x[6] = {0, 0, 0, 0, 0, 0};
  bool ok2 = true;
  int phase = 0;  // 0 need jac, 1 need trial, 2 done
  int jac_evals = 0, cost_evals = 0;
  int slot0 = 0, nj = 1;        // the jobs: lock-step job slots [slot0, slot0 + nj), latency mode see solve_speculative
  const int* pairs = nullptr;   // [nj]
  const double* T_cb = nullptr; // [nj][16] camera-from-body per job, or null: every job is evaluated at est itself
  const double* Ad = nullptr;   // [nj][36] their adjoints (set with T_cb)
  double* trace = nullptr;      // [max_iters][10] or null
  bool slot_holds_est = false;  // the problem's job slots hold the evaluations (histograms, err, tables) of `est`
};

void lm_start_trial(LM& s) {
  s.backup = s.est;  // push
  double Hl[36];
  memcpy(Hl, s.H, sizeof(Hl));
  for (int j = 0; j < 6; j++) Hl[7 * j] += s.lambda;  // setLambda (block_solver.hpp:573-599)
  s.ok2 = nidhost::ldlt6_solve(Hl, s.b, s.x);
  s.est = nidhost::pose_mul(nidhost::pose_exp(s.x), s.est);  // oplusImpl
  s.phase = 1;
}

// the pose matrix job g of problem s is evaluated at when the problem's pose is P
void stage_pose(const LM& s, const nidhost::Pose7& P, int g, double* out16) {
  if (!s.T_cb) { nidhost::pose_to_mat16(P, out16); return; }
  double M[16];
  nidhost::pose_to_mat16(P, M);
  nidhost::mat16_mul(s.T_cb + 16 * (size_t)g, M, out16);
}
}  // namespace

// One LM step of problem s from the 44 doubles {chi2, H[36], b[6], -} of its jobs combined
// (optimization_algorithm_levenberg.cpp:98-141 after a cost+Jacobian job, :173-202 after a trial-pose cost job).
static void lm_absorb(LM& s, const double* g, int max_iters) {
  const int maxTrials = 10;
  const double tau = 1e-5, goodUp = 2. / 3., goodLo = 1. / 3.;
  if (s.phase == 0) {
    s.jac_evals++;
    s.currentChi = g[0];
    s.iniChi = s.currentChi;
    memcpy(s.H, g + 1, sizeof(double) * 36);
    memcpy(s.b, g + 37, sizeof(double) * 6);
    if (s.it == 0) {
      double md = 0.;
      for (int j = 0; j < 6; j++) md = std::max(std::fabs(s.H[7 * j]), md);
      s.lambda = tau * md;
      s.ni = 2;
      s.nBad = 0;
    }
    s.rho = 0;
    s.qmax = 0;
    lm_start_trial(s);
    return;
  }
  s.cost_evals++;
  double tempChi = g[0];
  if (!s.ok2) tempChi = std::numeric_limits<double>::max();
  double rho = s.currentChi - tempChi;
  double scale = 0.;
  for (int j = 0; j < 6; j++) scale += s.x[j] * (s.lambda * s.x[j] + s.b[j]);
  scale += 1e-3;
  rho /= scale;
  if (rho > 0 && std::isfinite(tempChi)) {
    double alpha = 1. - std::pow((2 * rho - 1), 3);
    alpha = std::min(alpha, goodUp);
    double sf = std::max(goodLo, alpha);
    s.lambda *= sf;
    s.ni = 2;
    s.currentChi = tempChi;
  } else {
    s.lambda *= s.ni;
    s.ni *= 2;
    s.est = s.backup;  // pop
    s.slot_holds_est = false;
  }
  s.rho = rho;
  s.qmax++;
  if (rho < 0 && s.qmax < maxTrials) {
    lm_start_trial(s);
    return;
  }
  bool terminate = (s.qmax == maxTrials || rho == 0);
  if (!terminate) {
    if ((s.iniChi - s.currentChi) * 1e3 < s.iniChi) s.nBad++;
    else s.nBad = 0;
    if (s.nBad >= 3) terminate = true;
  }
  s.it++;
  s.phase = (!terminate && s.it < max_iters) ? 0 : 2;
  if (s.trace) {
    double* t = s.trace + 10 * (s.it - 1);
    t[0] = s.currentChi; t[1] = s.lambda; t[2] = s.qmax;
    memcpy(t + 3, s.est.t, sizeof(double) * 3);
    memcpy(t + 6, s.est.q, sizeof(double) * 4);
  }
}

// Latency mode of the LM driver (a handful of problems, the reference's own use: one pair per process,
// NID_pose_estimation.cpp:350). With one job in flight the device is nearly idle and a solve is a chain of ~34
// dependent rounds (10 linearisations + ~24 trial poses), each a few small kernels and a host round trip. The trial
// poses of an outer iteration are known in advance: after a rejection the schedule retries with lambda * ni, ni * 2
// (optimization_algorithm_levenberg.cpp:186-199). So every round evaluates, per problem, the next K trial poses of that
// sequence at once and completely (histograms, err, chi2 AND Jacobian / Gauss-Newton block); the host then walks the
// unchanged state machine over the cached results: the first accepted trial ends the iteration and its Gauss-Newton
// block is already there for the next one. Same decisions, same numbers (the kernels are deterministic), about one
// round per outer iteration instead of three and a half.
// Slots: job g of trial k of problem j is slot slot0_j * K + k * nj_j + g; the cache holds the combined block of every
// (problem, trial), made as in lock-step.
static int solve_speculative(nid_ctx* c, std::vector<LM>& st, int n, int n_jobs, int max_iters, double delta, int K) {
  struct Cand { nidhost::Pose7 pose; double gn[44]; bool valid; };
  std::vector<Cand> cache((size_t)n * K);
  for (auto& q : cache) q.valid = false;
  // one staging block per round: the poses of all n_jobs * K slots, then the list of the slots in use (one H2D copy); the
  // kernels read both from there for the duration of the solve
  const int nslots = n_jobs * K;
  const size_t stage_bytes = sizeof(double) * 16 * (size_t)c->job_cap + sizeof(int) * (size_t)c->job_cap;
  if (!c->d_lm_stage) {
    OKR(c->h_lm_stage.alloc(stage_bytes, "pinned LM staging"));
    OKR(c->d_lm_stage.alloc(stage_bytes, "LM staging"));
  }
  struct Swap {  // restores the context's pose buffers on every way out
    nid_ctx* c; double* poses; double* h_poses;
    ~Swap() { c->poses = poses; c->h_poses = h_poses; }
  } swap{c, c->poses, c->h_poses};
  c->poses = reinterpret_cast<double*>(c->d_lm_stage.get());
  c->h_poses = reinterpret_cast<double*>(c->h_lm_stage.get());
  int* const list = reinterpret_cast<int*>(c->h_poses + 16 * (size_t)nslots);
  int* const d_list = reinterpret_cast<int*>(c->poses + 16 * (size_t)nslots);
  auto slot_of = [&](int j, int k, int g) { return st[j].slot0 * K + k * st[j].nj + g; };
  for (int j = 0; j < n; j++)
    for (int k = 0; k < K; k++)
      for (int g = 0; g < st[j].nj; g++) c->h_job_pair[slot_of(j, k, g)] = st[j].pairs[g];
  CU(cudaMemcpyAsync(c->job_pair, c->h_job_pair, sizeof(int) * nslots, cudaMemcpyHostToDevice, c->stream), "H2D job_pair");
  CU(cudaStreamSynchronize(c->stream), "sync before LM");
  auto same_pose = [](const nidhost::Pose7& a, const nidhost::Pose7& b) {
    return memcmp(a.t, b.t, sizeof(a.t)) == 0 && memcmp(a.q, b.q, sizeof(a.q)) == 0;
  };
  const bool tt_on = getenv("NID_LM_TIMES") != nullptr;
  double tt[4] = {0, 0, 0, 0};
  int tt_rounds = 0;
  auto now = [] { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  for (;;) {
    const double t0 = now();
    // 1. let every problem consume what the cache already holds
    bool progress = true;
    while (progress) {
      progress = false;
      for (int j = 0; j < n; j++) {
        LM& s = st[j];
        if (s.phase == 2) continue;
        for (int k = 0; k < K; k++) {
          Cand& q = cache[(size_t)j * K + k];
          if (q.valid && same_pose(q.pose, s.est)) {
            lm_absorb(s, q.gn, max_iters);  // phase 0 reads chi2/H/b, phase 1 reads chi2: both are in the block
            progress = true;
            break;
          }
        }
      }
    }
    // 2. the next round: per unfinished problem the pose it waits for and the trials that would follow rejections
    int nround = 0;
    for (int j = 0; j < n; j++) {
      LM& s = st[j];
      for (int k = 0; k < K; k++) cache[(size_t)j * K + k].valid = false;
      if (s.phase == 2) continue;
      LM sim = s;
      for (int k = 0; k < K; k++) {
        Cand& q = cache[(size_t)j * K + k];
        q.pose = sim.est;
        q.valid = true;
        for (int g = 0; g < s.nj; g++) stage_pose(s, sim.est, g, c->h_poses + 16 * (size_t)slot_of(j, k, g));
        nround++;
        if (sim.phase != 1 || sim.qmax + 1 >= 10) break;  // only trial poses have successors; maxTrials = 10
        // the trial after a rejection of this one (lm_absorb's else branch, then lm_start_trial)
        sim.lambda *= sim.ni;
        sim.ni *= 2;
        sim.est = sim.backup;
        sim.qmax++;
        lm_start_trial(sim);
      }
    }
    if (nround == 0) break;
    const double t1 = now();
    // every slot is evaluated every round (one fixed chain: see launch_latency_round); the slots this round has no use
    // for repeat their problem's first pose and their results are ignored
    for (int j = 0; j < n; j++) {
      for (int k = 0; k < K; k++) {
        if (cache[(size_t)j * K + k].valid) continue;
        for (int g = 0; g < st[j].nj; g++) {
          double* m = c->h_poses + 16 * (size_t)slot_of(j, k, g);
          if (k > 0) memcpy(m, c->h_poses + 16 * (size_t)slot_of(j, 0, g), sizeof(double) * 16);
          else stage_pose(st[j], st[j].est, g, m);
        }
      }
    }
    for (int i = 0; i < nslots; i++) list[i] = i;
    OKR(launch_latency_round(c, nslots, d_list, list, sizeof(double) * 16 * nslots + sizeof(int) * nslots, delta, c->h_out));
    const double t2 = now();
    CU(cudaStreamSynchronize(c->stream), "sync lm");
    const double t3 = now();
    for (int j = 0; j < n; j++)
      for (int k = 0; k < K; k++) {
        Cand& q = cache[(size_t)j * K + k];
        if (q.valid) nidhost::gn_combine(st[j].nj, c->h_out + 44 * (size_t)slot_of(j, k, 0), st[j].Ad, q.gn);
      }
    tt[0] += t1 - t0; tt[1] += t2 - t1; tt[2] += t3 - t2; tt[3] += now() - t3; tt_rounds++;
  }
  if (tt_on) fprintf(stderr, "lm rounds %d: host %.1f issue %.1f wait %.1f copy %.1f us per round\n", tt_rounds, tt[0] / tt_rounds, tt[1] / tt_rounds, tt[2] / tt_rounds, tt[3] / tt_rounds);
  return NID_OK;
}

// Lock-step LM over n problems. The problems are cut into two halves that ping-pong: while the device evaluates the
// jobs of one half (its own stream and its own range of job slots), the host absorbs the results of the other half,
// solves the 6x6 systems and stages the next poses. Each problem sees exactly the schedule of a solo solve.
//
// Every job keeps ONE job slot for the whole solve, the jobs of a problem consecutive, and every round hands the kernels
// two lists of slots: list 1 gets pass 1 + assembly (histograms, entropies, err, chi2 and the scaled log tables), list 2
// gets pass 2 + the Gauss-Newton block. All jobs of a problem go on the same lists in the same round. A trial pose is on
// list 1 only. A cost+Jacobian job is on list 2 and -- this is the point -- on list 1 only when its slot does not already
// hold the evaluation of that very pose: after an accepted trial the next outer iteration linearises at the pose the
// trial was evaluated at (optimization_algorithm_levenberg.cpp:173-199 then :98), and the sorted kernels are
// deterministic, so the histograms, err and tables in the slot are bit for bit what a recomputation would produce. The
// reference evaluates them again (CudaComputeH(true) repeats the cost half); skipping that repeats nothing observable and
// saves a third of the device work of a solve (option "lm_reuse").
// The natural-order kernels sum with shared-memory atomics, so their histograms are not bit-reproducible: there every
// active job is on list 1.
static int solve_lockstep(nid_ctx* c, std::vector<LM>& st, int n, int n_jobs, int max_iters, double delta) {
  const bool sorted = use_sorted(c);
  const bool reuse = sorted && c->opt_lm_reuse;
  // (the natural-order kernels index their partial buffers by (slot, cell, strip): two halves in flight would need the
  // same strip count S)
  const int nh = (n >= 8 && sorted) ? 2 : 1;
  if (nh == 2 && !c->streams[1]) OKR(c->streams[1].create("cudaStreamCreate (LM)"));
  if (!c->d_lm_lists) {
    OKR(c->h_lm_lists.alloc(2 * (size_t)c->job_cap, "pinned LM lists"));
    OKR(c->d_lm_lists.alloc(2 * (size_t)c->job_cap, "LM lists"));
  }
  CU(cudaStreamSynchronize(c->stream), "sync before LM");
  // half h owns the problems [p0, p1), their slots [lo, hi) and the list storage [2 lo, 2 hi): list 1 then list 2
  struct Half { int p0, p1, lo, hi, n1, n2, na; cudaStream_t stream; };
  auto half = [&](int p0, int p1, cudaStream_t stream) {
    return Half{p0, p1, st[p0].slot0, p1 > p0 ? st[p1 - 1].slot0 + st[p1 - 1].nj : st[p0].slot0, 0, 0, 0, stream};
  };
  Half H[2];
  H[0] = half(0, nh == 2 ? n / 2 : n, c->stream);
  H[1] = half(n / 2, n, c->streams[1]);
  cudaStream_t const main_stream = c->stream;
  for (int j = 0; j < n; j++)
    for (int g = 0; g < st[j].nj; g++) c->h_job_pair[st[j].slot0 + g] = st[j].pairs[g];
  CU(cudaMemcpyAsync(c->job_pair, c->h_job_pair, sizeof(int) * n_jobs, cudaMemcpyHostToDevice, main_stream), "H2D job_pair");
  CU(cudaStreamSynchronize(main_stream), "sync job_pair");
  int rc = NID_OK;
  auto issue = [&](Half& h) -> int {
    int* l1 = c->h_lm_lists + 2 * (size_t)h.lo;
    int* l2 = l1 + (h.hi - h.lo);
    h.n1 = h.n2 = h.na = 0;
    for (int j = h.p0; j < h.p1; j++) {
      LM& s = st[j];
      if (s.phase == 2) continue;
      h.na++;
      for (int g = 0; g < s.nj; g++) stage_pose(s, s.est, g, c->h_poses + 16 * (size_t)(s.slot0 + g));
      const bool full = s.phase == 0;
      const bool pass1 = !full || !(reuse && s.slot_holds_est);
      for (int g = 0; g < s.nj; g++) {
        if (full) l2[h.n2++] = s.slot0 + g;
        if (pass1) l1[h.n1++] = s.slot0 + g;
      }
      s.slot_holds_est = true;  // after this round the slots hold the evaluations of s.est (a rejection resets it)
    }
    if (h.na == 0) return NID_OK;
    const int cnt = h.hi - h.lo;
    CU(cudaMemcpyAsync(c->poses + 16 * (size_t)h.lo, c->h_poses + 16 * (size_t)h.lo, sizeof(double) * 16 * cnt, cudaMemcpyHostToDevice, h.stream),
       "H2D poses");
    int* d1 = c->d_lm_lists + 2 * (size_t)h.lo;
    int* d2 = d1 + cnt;
    CU(cudaMemcpyAsync(d1, l1, sizeof(int) * 2 * cnt, cudaMemcpyHostToDevice, h.stream), "H2D job lists");
    c->stream = h.stream;  // the launchers issue on the context's current stream
    const JobSet js1{d1, l1, 0, h.n1, n_jobs}, js2{d2, l2, 0, h.n2, n_jobs};  // (slots: the solve's, the same in every round)
    int r = NID_OK;
    if (h.n1 > 0) r = launch_pass1(c, js1, Pass2::some);
    if (r == NID_OK && h.n2 > 0) r = launch_pass2(c, js2);
    if (r == NID_OK && h.n2 > 0) r = launch_gn(c, js2, delta, 1);
    if (r == NID_OK && h.n1 > 0) r = launch_gn(c, js1, delta, 0);  // chi2 of the trial poses (and, harmlessly, again of full jobs)
    c->stream = main_stream;
    if (r != NID_OK) return r;
    CU(cudaMemcpyAsync(c->h_out + 44 * (size_t)h.lo, c->gn + 44 * (size_t)h.lo, sizeof(double) * 44 * cnt, cudaMemcpyDeviceToHost, h.stream),
       "D2H gn");
    return NID_OK;
  };
  for (int i = 0; i < nh && rc == NID_OK; i++) rc = issue(H[i]);
  while (rc == NID_OK && (H[0].na > 0 || (nh == 2 && H[1].na > 0))) {
    for (int i = 0; i < nh && rc == NID_OK; i++) {
      Half& h = H[i];
      if (h.na == 0) continue;
      if (cudaStreamSynchronize(h.stream) != cudaSuccess) { rc = check_cuda(cudaGetLastError(), "sync lm"); break; }
      for (int j = h.p0; j < h.p1; j++) {
        LM& s = st[j];
        if (s.phase == 2) continue;
        double g[44];
        nidhost::gn_combine(s.nj, c->h_out + 44 * (size_t)s.slot0, s.Ad, g);
        lm_absorb(s, g, max_iters);
      }
      rc = issue(h);
    }
  }
  c->stream = main_stream;
  if (nh == 2) cudaStreamSynchronize(c->streams[1]);
  cudaStreamSynchronize(main_stream);
  return rc;
}

// The LM solve behind nid_solve, nid_solve_jobs and nid_solve_groups: n_groups problems, group j owning the next
// group_size[j] jobs. Everything is validated before any work; poses7, stats and trace are written only on success.
static int solve_groups(nid_ctx* c, int n_groups, const int* group_size, const int* job_pair, const double* T_cb, double* poses7,
                        int max_iters, double delta, int* stats, double* trace) {
  if (!c || n_groups < 1 || !group_size || !poses7) { set_error("bad argument"); return NID_ERR_ARG; }
  long long total = 0;
  for (int j = 0; j < n_groups; j++) {
    if (group_size[j] < 1) { set_error("group size must be >= 1"); return NID_ERR_ARG; }
    total += group_size[j];
  }
  if (total > c->max_jobs) { set_error("more jobs than max_jobs"); return NID_ERR_ARG; }
  const int n_jobs = (int)total;
  if (T_cb)
    for (int i = 0; i < n_jobs; i++)
      if (!nidhost::is_rigid(T_cb + 16 * (size_t)i)) { set_error("T_cb is not a rigid transform"); return NID_ERR_ARG; }
  std::vector<int> pairs(n_jobs);
  for (int i = 0; i < n_jobs; i++) {
    const int p = job_pair ? job_pair[i] : i;
    if (p < 0 || p >= c->n_pairs) { set_error("job_pair out of range"); return NID_ERR_ARG; }
    if (!c->pair_prepared[p] || (use_sorted(c) && !c->pair_sorted[p])) { set_error("pair not prepared"); return NID_ERR_STATE; }
    pairs[i] = p;
  }
  CU(cudaSetDevice(c->device), "cudaSetDevice");
  std::vector<double> Ad(T_cb ? 36 * (size_t)n_jobs : 0);
  for (int i = 0; T_cb && i < n_jobs; i++) nidhost::adjoint6(T_cb + 16 * (size_t)i, &Ad[36 * (size_t)i]);
  const int tr = std::max(max_iters, 0);
  std::vector<double> tbuf(trace ? 10 * (size_t)tr * n_groups : 0);
  std::vector<LM> st(n_groups);
  for (int j = 0, i0 = 0; j < n_groups; i0 += group_size[j++]) {
    LM& s = st[j];
    s.slot0 = i0;
    s.nj = group_size[j];
    s.pairs = &pairs[i0];
    if (T_cb) { s.T_cb = T_cb + 16 * (size_t)i0; s.Ad = Ad.data() + 36 * (size_t)i0; }
    if (trace) s.trace = tbuf.data() + 10 * (size_t)tr * j;
    memcpy(s.est.t, poses7 + 7 * j, sizeof(double) * 3);
    memcpy(s.est.q, poses7 + 7 * j + 3, sizeof(double) * 4);
    s.phase = max_iters > 0 ? 0 : 2;
  }
  OKR(ensure_job_buffers(c));
  c->staged_jobs = 0;  // the solver rewrites the staged poses and job table
  const int K = std::min(c->opt_lm_spec, c->job_cap / n_jobs);
  if (use_sorted(c) && n_groups <= 4 && K >= 2) OKR(solve_speculative(c, st, n_groups, n_jobs, max_iters, delta, K));
  else OKR(solve_lockstep(c, st, n_groups, n_jobs, max_iters, delta));
  for (int j = 0; j < n_groups; j++) {
    memcpy(poses7 + 7 * j, st[j].est.t, sizeof(double) * 3);
    memcpy(poses7 + 7 * j + 3, st[j].est.q, sizeof(double) * 4);
    if (stats) { stats[3 * j] = st[j].it; stats[3 * j + 1] = st[j].jac_evals; stats[3 * j + 2] = st[j].cost_evals; }
    if (trace && st[j].it > 0) memcpy(trace + 10 * (size_t)tr * j, st[j].trace, sizeof(double) * 10 * st[j].it);
  }
  return NID_OK;
}

int nid_solve_groups(nid_ctx* c, int n_groups, const int* group_size, const int* job_pair, const double* T_cb, double* poses7,
                     int max_iters, double delta, int* stats, double* trace) {
  return solve_groups(c, n_groups, group_size, job_pair, T_cb, poses7, max_iters, delta, stats, trace);
}

int nid_solve_jobs(nid_ctx* c, int n, const int* job_pair, double* poses7, int max_iters, double delta, int* stats) {
  if (!c || n < 1 || n > c->max_jobs || !poses7) { set_error("bad argument"); return NID_ERR_ARG; }
  const std::vector<int> ones(n, 1);
  return solve_groups(c, n, ones.data(), job_pair, nullptr, poses7, max_iters, delta, stats, nullptr);
}

int nid_solve(nid_ctx* c, int pair, double pose7[7], int max_iters, double delta, double* trace, int* stats) {
  if (!c) { set_error("NULL ctx"); return NID_ERR_ARG; }
  const int one = 1;
  return solve_groups(c, 1, &one, &pair, nullptr, pose7, max_iters, delta, stats, trace);
}

// Coarse-to-fine: every level is prepared at the poses the coarser level handed down (the in-bounds set and n_c depend on
// the prepare pose), then solved. The pairs of a run of consecutive job pairs are prepared in one nid_prepare_pairs call.
int nid_solve_pyramid_jobs(nid_ctx* const* levels, int n_levels, int n, const int* job_pair, double* poses7, const int* max_iters,
                           double delta, int* stats) {
  if (!levels || n_levels < 1 || n_levels > 8 || n < 1 || !poses7 || !max_iters) { set_error("bad argument"); return NID_ERR_ARG; }
  std::vector<int> jp(n);
  for (int j = 0; j < n; j++) jp[j] = job_pair ? job_pair[j] : j;
  for (int l = 0; l < n_levels; l++) {
    const nid_ctx* c = levels[l];
    if (!c) { set_error("NULL level context"); return NID_ERR_ARG; }
    if (max_iters[l] < 0) { set_error("max_iters must be >= 0"); return NID_ERR_ARG; }
    if (n > c->max_jobs) { set_error("more jobs than a level's max_jobs"); return NID_ERR_ARG; }
    for (int j = 0; j < n; j++) {
      if (jp[j] < 0 || jp[j] >= c->n_pairs) { set_error("job_pair out of range"); return NID_ERR_ARG; }
      if (!c->pair_set[jp[j]]) { set_error("job pair not set at every level"); return NID_ERR_STATE; }
    }
  }
  {
    std::vector<int> s = jp;
    std::sort(s.begin(), s.end());
    if (std::adjacent_find(s.begin(), s.end()) != s.end()) {
      set_error("job pairs must be distinct (a pair is prepared at one pose)");
      return NID_ERR_ARG;
    }
  }
  std::vector<double> cur(poses7, poses7 + 7 * (size_t)n), T(16 * (size_t)n);
  std::vector<int> st(3 * (size_t)n), all(3 * (size_t)n * n_levels, 0);
  for (int l = n_levels - 1; l >= 0; l--) {
    if (max_iters[l] == 0) continue;
    nid_ctx* c = levels[l];
    for (int j = 0; j < n; j++) {
      nidhost::Pose7 p;
      memcpy(p.t, &cur[7 * (size_t)j], sizeof(double) * 3);
      memcpy(p.q, &cur[7 * (size_t)j + 3], sizeof(double) * 4);
      nidhost::pose_to_mat16(p, &T[16 * (size_t)j]);
    }
    for (int j0 = 0, j1; j0 < n; j0 = j1) {
      for (j1 = j0 + 1; j1 < n && jp[j1] == jp[j1 - 1] + 1; j1++) {}
      OKR(nid_prepare_pairs(c, jp[j0], j1 - j0, &T[16 * (size_t)j0], nullptr, nullptr));
    }
    OKR(nid_solve_jobs(c, n, jp.data(), cur.data(), max_iters[l], delta, st.data()));
    for (int j = 0; j < n; j++)
      for (int k = 0; k < 3; k++) all[((size_t)j * n_levels + l) * 3 + k] = st[3 * (size_t)j + k];
  }
  memcpy(poses7, cur.data(), sizeof(double) * 7 * (size_t)n);
  if (stats) memcpy(stats, all.data(), sizeof(int) * all.size());
  return NID_OK;
}

int nid_hard_eval_jobs(nid_ctx* c, int n_jobs, const int* job_pair, const double* poses, double* total, double* nid_cells) {
  if (!c || !poses) { set_error("bad argument"); return NID_ERR_ARG; }
  CU(cudaSetDevice(c->device), "cudaSetDevice");
  OKR(stage_jobs(c, n_jobs, job_pair, poses, 1));
  c->staged_jobs = 0;  // (not evaluation jobs: the pairs need not be prepared)
  OKR(launch_hard(c, n_jobs));
  const size_t w = c->ncell + 1;
  CU(cudaMemcpyAsync(c->h_out, c->hard, sizeof(double) * w * n_jobs, cudaMemcpyDeviceToHost, c->stream), "D2H hard");
  CU(cudaStreamSynchronize(c->stream), "sync hard");
  for (int j = 0; j < n_jobs; j++) {
    if (total) total[j] = c->h_out[j * w + c->ncell];
    if (nid_cells) memcpy(nid_cells + (size_t)j * c->ncell, c->h_out + j * w, sizeof(double) * c->ncell);
  }
  return NID_OK;
}

static int warp_sample_common(nid_ctx* c, int pair, const double T_cw1[16], int f64) {
  if (!c || pair < 0 || pair >= c->n_pairs || !T_cw1) { set_error("bad argument"); return NID_ERR_ARG; }
  if (!c->pair_set[pair]) { set_error("pair not set"); return NID_ERR_STATE; }
  CU(cudaSetDevice(c->device), "cudaSetDevice");
  if (f64 && !c->d_pix) OKR(c->d_pix.alloc((size_t)8 * c->N, "d_pix"));
  if (!f64 && !c->d_pix4) OKR(c->d_pix4.alloc((size_t)4 * c->N, "d_pix4"));
  memcpy(c->h_aux_pose, T_cw1, sizeof(double) * 16);  // (both callers synchronise before returning)
  CU(cudaMemcpyAsync(c->aux_pose, c->h_aux_pose, sizeof(double) * 16, cudaMemcpyHostToDevice, c->stream), "H2D pose");
  return launch_warp_sample(c, pair, c->aux_pose, f64);
}

int nid_warp_sample(nid_ctx* c, int pair, const double T_cw1[16], float* out) {
  OKR(warp_sample_common(c, pair, T_cw1, 0));
  if (out) CU(cudaMemcpyAsync(out, c->d_pix4, sizeof(float) * 4 * c->N, cudaMemcpyDefault, c->stream), "D2H pix4");
  CU(cudaStreamSynchronize(c->stream), "sync warp_sample");
  return NID_OK;
}

// Kernel 1's target texture of one pair: three stacked fp16 planes (I, Gx/2, Gy/2) in a gather-able CUDA array, created
// and filled the first time the pair is used by nid_warp_sample_jobs after its target image changed.
static int ensure_k1_texture(nid_ctx* c, int pair) {
  if (c->k1_ready[pair]) return NID_OK;
  nid::GatherTexture& t = c->k1tex[pair];
  if (!t.tex) {
    OKR(t.create(cudaCreateChannelDescHalf(), c->cols, 3 * c->rows, "kernel-1 planes"));
    CU(cudaMemcpyAsync(c->d_k1tex + pair, t.tex.handle_address(), sizeof(cudaTextureObject_t), cudaMemcpyHostToDevice, c->stream),
       "H2D k1 texture handle");
  }
  if (!c->d_k1pack) OKR(c->d_k1pack.alloc((size_t)3 * c->N, "d_k1pack"));
  OKR(launch_pack_k1(c, pair, c->d_k1pack));
  CU(cudaMemcpy2DToArrayAsync(t.array, 0, 0, c->d_k1pack, sizeof(unsigned short) * c->cols, sizeof(unsigned short) * c->cols,
                              3 * c->rows, cudaMemcpyDeviceToDevice, c->stream), "fp16 planes -> texture array");
  c->k1_ready[pair] = 1;
  return NID_OK;
}

int nid_warp_sample_jobs(nid_ctx* c, int n_jobs, const int* job_pair, const double* poses, float* out) {
  if (!c || !poses) { set_error("bad argument"); return NID_ERR_ARG; }
  CU(cudaSetDevice(c->device), "cudaSetDevice");
  if (n_jobs < 1 || n_jobs > c->max_jobs) { set_error("n_jobs out of range"); return NID_ERR_ARG; }
  if (c->sell_points) { set_error("nid_warp_sample_jobs needs depth pairs (nid_set_pair), not caller-supplied points"); return NID_ERR_UNSUPPORTED; }
  if (!c->d_pix4_jobs) OKR(c->d_pix4_jobs.alloc((size_t)4 * c->N * c->max_jobs, "d_pix4_jobs"));
  OKR(stage_jobs(c, n_jobs, job_pair, poses, 1));
  c->staged_jobs = 0;  // (not evaluation jobs: the pairs need not be prepared)
  // pairs uploaded as raw 16-bit depth are read as such (2 B/px); a mixed batch falls back to the fp64 planes, which
  // every pair has
  bool u16 = true;
  for (int j = 0; j < n_jobs; j++) {
    u16 = u16 && c->pair_u16[c->h_job_pair[j]];
    OKR(ensure_k1_texture(c, c->h_job_pair[j]));
  }
  OKR(launch_warp_sample_jobs(c, n_jobs, (float4*)c->d_pix4_jobs.get(), u16));
  if (out) CU(cudaMemcpyAsync(out, c->d_pix4_jobs, sizeof(float) * 4 * c->N * (size_t)n_jobs, cudaMemcpyDefault, c->stream), "D2H pix4 jobs");
  CU(cudaStreamSynchronize(c->stream), "sync warp_sample_jobs");
  return NID_OK;
}

int nid_warp_sample_f64(nid_ctx* c, int pair, const double T_cw1[16], double* out) {
  OKR(warp_sample_common(c, pair, T_cw1, 1));
  if (out) CU(cudaMemcpyAsync(out, c->d_pix, sizeof(double) * 8 * c->N, cudaMemcpyDefault, c->stream), "D2H pix8");
  CU(cudaStreamSynchronize(c->stream), "sync warp_sample_f64");
  return NID_OK;
}

int nid_debug_hist(nid_ctx* c, int job, int cell_index, double* P_t, double* P_j) {
  if (!c || job < 0 || job >= c->max_jobs || cell_index < 0 || cell_index >= c->ncell) { set_error("bad argument"); return NID_ERR_ARG; }
  const size_t hs = (size_t)c->bins * c->bins + c->bins;
  if (!c->hist) { set_error("set option keep_hist=1 before the evaluation"); return NID_ERR_STATE; }
  const double* src = c->hist + ((size_t)job * c->ncell + cell_index) * hs;
  CU(cudaSetDevice(c->device), "cudaSetDevice");
  CU(cudaStreamSynchronize(c->stream), "sync");
  if (P_j) CU(cudaMemcpy(P_j, src, sizeof(double) * c->bins * c->bins, cudaMemcpyDeviceToHost), "D2H P_j");
  if (P_t) CU(cudaMemcpy(P_t, src + c->bins * c->bins, sizeof(double) * c->bins, cudaMemcpyDeviceToHost), "D2H P_t");
  return NID_OK;
}

long long nid_launch_count(nid_ctx* c) { return c ? c->launches : 0; }

long long nid_live_resources(void) { return live_handles.load(); }

int nid_kernel_times(nid_ctx* c, double ms[4], long long calls[4]) {
  if (!c || !ms || !calls) { set_error("bad argument"); return NID_ERR_ARG; }
  for (int i = 0; i < 4; i++) { ms[i] = c->kernel_ms[i]; calls[i] = c->kernel_calls[i]; }
  return NID_OK;
}

void* nid_stream(nid_ctx* c) { return c ? (void*)c->stream : nullptr; }

int nid_event_record(nid_ctx* c, int slot) {
  if (!c || slot < 0 || slot > 1) { set_error("bad argument"); return NID_ERR_ARG; }
  CU(cudaSetDevice(c->device), "cudaSetDevice");
  if (!c->ev[slot]) OKR(c->ev[slot].create(cudaEventDefault, "cudaEventCreate"));
  CU(cudaEventRecord(c->ev[slot], c->stream), "cudaEventRecord");
  return NID_OK;
}

int nid_event_elapsed_ms(nid_ctx* c, float* ms) {
  if (!c || !ms || !c->ev[0] || !c->ev[1]) { set_error("bad argument or events not recorded"); return NID_ERR_ARG; }
  CU(cudaEventSynchronize(c->ev[1]), "cudaEventSynchronize");
  CU(cudaEventElapsedTime(ms, c->ev[0], c->ev[1]), "cudaEventElapsedTime");
  return NID_OK;
}

int nid_set_option(nid_ctx* c, const char* key, int value) {
  if (!c || !key) { set_error("bad argument"); return NID_ERR_ARG; }
  if (!strcmp(key, "force_strips")) {
    if (value < 0) { set_error("force_strips must be >= 0 (0 = automatic)"); return NID_ERR_ARG; }
    c->opt_force_strips = value;
    return NID_OK;
  }
  if (!strcmp(key, "path")) {
    if (value < 0 || value > 2) { set_error("path must be 0 (auto), 1 (natural) or 2 (sorted)"); return NID_ERR_ARG; }
    if (value == 2 && (c->bins > NID_SORTED_MAX_BINS || c->bins < NID_SORTED_MIN_BINS)) { set_error("the sorted path supports 6 to 40 bins"); return NID_ERR_UNSUPPORTED; }
    c->opt_path = value;
    return NID_OK;
  }
  if (!strcmp(key, "keep_hist")) { c->opt_keep_hist = value; return NID_OK; }
  if (!strcmp(key, "lm_reuse")) { c->opt_lm_reuse = value ? 1 : 0; return NID_OK; }
  if (!strcmp(key, "lm_graph")) { c->opt_lm_graph = value ? 1 : 0; return NID_OK; }
  if (!strcmp(key, "asm_wide")) { c->opt_asm_wide = value < 0 ? 0 : std::min(value, 2); return NID_OK; }
  if (!strcmp(key, "stage_bulk")) { c->opt_stage_bulk = value < 0 ? -1 : (value ? 1 : 0); return NID_OK; }
  if (!strcmp(key, "lm_speculate")) {
    if (value < 0 || value > 8) { set_error("lm_speculate must be 0 (off) .. 8 trial poses per round"); return NID_ERR_ARG; }
    c->opt_lm_spec = value;
    return NID_OK;
  }
  if (!strcmp(key, "task_px")) {
    if (value < 8 || value > NID_TASK_PX_MAX || (value & 3)) { set_error("task_px must be a multiple of 4 in [8, 256]"); return NID_ERR_ARG; }
    if (value != c->task_px) {
      c->task_px = value;
      std::fill(c->pair_prepared.begin(), c->pair_prepared.end(), 0);  // the pixel store is laid out per task
    }
    return NID_OK;
  }
  if (!strcmp(key, "time_kernels")) {
    c->opt_time_kernels = value;
    for (int i = 0; i < 4; i++) { c->kernel_ms[i] = 0; c->kernel_calls[i] = 0; }
    return NID_OK;
  }
  set_error(std::string("unknown option ") + key);
  return NID_ERR_ARG;
}

}  // extern "C"
