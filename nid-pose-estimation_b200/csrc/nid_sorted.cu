// "Sorted" evaluation path (the production path for cells of a few thousand pixels and more).
//
// Idea 1 -- class factorisation. The reference image never changes between the evaluations of one pair,
// and a pixel's four reference spline weights depend only on its 8-bit reference intensity v.
// nid_prepare therefore regroups the valid pixels of every cell by v (257 classes: 0..255, plus 256 =
// "no reference sample": valid depth but out of bounds at the prepare pose, which the CPU edge still
// counts in the target marginal, types_six_dof_expmap.cpp:593-602 with zero bs_value_ref_ rows). For a
// class the joint histogram update  P_j[k_r+m][k_t+n] += w_ref[m] * w_t[n]
// (types_six_dof_expmap.cpp:598-601) factors into  w_ref[m] * ( sum_i w_t,i[n] ): one *un-weighted* soft
// histogram h_v[B] per class, 4 accumulations per pixel instead of 20, and
//     P_j[r][t] = sum_v w_ref,v[r - k_r(v)] * h_v[t],      P_t[t] = sum_v h_v[t].
// The same factorisation turns the Jacobian's 16-term table lookup into a 4-term one against a per-class table.
//
// Idea 2 -- one lane per task, sliced-ELL storage. A "task" is up to L consecutive pixels of one
// (cell, class) segment. 64-bit shared-memory atomics are CAS loops on sm_100
// (profiles/r01_atom_bench_microbenchmark.txt), so nothing is shared: ONE THREAD owns a task, walks its
// pixels sequentially and accumulates into a private shared-memory row (pass 1) or registers (pass 2).
// Tasks are ordered by length and packed 32 to a "slice" (one warp); the pixels of a slice are stored
// interleaved -- group g of lane l at slice_off + (g*32 + l)*4 -- so every warp load is a fully coalesced
// 128-bit access and the lanes of a warp run out of work together (SELL-C-sigma, as in sparse mat-vec).
// Each task writes one partial; partials are combined per cell in task order => no floating-point
// atomics anywhere and bit-reproducible results.
//
// Idea 3 -- a fast path that cannot change a decision. Per pixel only the depth z and the pixel index are
// stored (12 B); the camera-frame point is z * (M0 cxn + M1 cyn + M2) + M3 with M = T_cw1 * T_wc0 composed
// once per job, and one reciprocal serves the projection and the Jacobian. That differs from the
// reference's operation order (CudaPoints3d.cu:20-28, computeH.cu:152-158) by a few ulp, which is harmless
// everywhere except at the reference's discontinuities: the in-bounds tests, the (int) truncation of
// (u, v) and the `>= 255 -> 254.999` clamp on saturated plateaus. A pixel whose (u, v) lands within 2^-24
// of an integer, or whose four taps are all 255, is therefore re-evaluated with the reference's exact
// sequence (exact_uv), so every decision is bit-identical to the reference's and everything else agrees
// to ~1e-13.
//
// Idea 4 -- the uniform spline basis with an exact end-block fold instead of per-span polynomials (see
// bspline4_uniform below): one branch-free weight formula per pixel in both passes.
//
// Memory-system details that were measured to matter (DESIGN.md 6a): the pixel store is read with evict-first
// loads and prefetched into L2 two groups ahead, so that L1 stays with the target-image gathers; CTAs are small
// (pass 1: one warp, register budget for 18-20 resident warps; pass 2: two warps at 16 resident warps); the
// shared-memory carve-out is requested per kernel. Also in this file: the device-side construction of the task and
// slice tables (k_layout_*), the warp-per-cell assembly for small cells, and kernel 1 on its own (k_warp_sample_jobs).
#include <cuda_fp16.h>
#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "nid_ctx.h"
#include "nid_device.cuh"

namespace nid {

#define NID_LAUNCH_CHECK(c, what)                         \
  do {                                                    \
    (c)->launches++;                                      \
    cudaError_t e__ = cudaGetLastError();                 \
    if (e__ != cudaSuccess) return check_cuda(e__, what); \
  } while (0)

#define NID_PAD_ID 0xFFFFFFFFu
// grid of the pixel kernels: the job index is the fast dimension (chunk-of-slices fast was measured 6 % slower)
#define NID_BLK_JOB blockIdx.x
#define NID_BLK_CHUNK blockIdx.y
#define NID_GRID(jobs, chunks) dim3(jobs, chunks)
#ifndef NID_PREFETCH_L2
#define NID_PREFETCH_L2 2  // groups beyond the register prefetch that the pixel kernels pull into L2 (0: off)
#endif

// counts per (cell, class) from existing in-bounds flags (nid_import_prepare path)
__global__ void k_count_classes(EvalParams p, int pair, unsigned int* __restrict__ cnt) {
  const size_t base = (size_t)pair * p.N;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < p.N; i += gridDim.x * blockDim.x) {
    int row = i / p.cols, col = i % p.cols;
    if (isnan(p.pwx[base + i]) || row >= p.rb * p.cell || col >= p.cb * p.cell) continue;
    int c = (row / p.rb) * p.cell + (col / p.cb);
    int key = p.inb0[base + i] ? (int)p.im0[base + i] : 256;
    atomicAdd(&cnt[((size_t)pair * p.ncell + c) * NID_NCLS + key], 1u);
  }
}

// ------------------------------------------------------------------------------------------------
// prepare: stable counting-sort scatter of every cell's valid pixels into the sliced-ELL layout, in three launches
// over (chunk, cell) with chunks of 256 consecutive pixels of the cell (row-major): per-chunk class counts, an exclusive
// scan of the counts along the chunks of a cell, then the scatter proper. key: 0..255 reference intensity (in
// bounds at the prepare pose), 256 valid but out of bounds, -1 invalid depth. The r-th pixel (row-major order) of
// class `key` goes to pixel o = r % L of task cls_task_start[key] + r / L, i.e. to  task_pos[task] + (o/4)*128 + o%4.
// PTS: store the world point (pairs set from caller-supplied points); else the depth z only.
__device__ __forceinline__ int sell_key(const EvalParams& p, size_t base, int c, int t, int& row, int& col) {
  const int npx = p.rb * p.cb;
  if (t >= npx) return -1;
  row = (c / p.cell) * p.rb + t / p.cb;
  col = (c % p.cell) * p.cb + t % p.cb;
  const size_t i = base + (size_t)row * p.cols + col;
  if (isnan(p.pwx[i])) return -1;
  return p.inb0[i] ? (int)p.im0[i] : 256;
}

__global__ void __launch_bounds__(256) k_chunk_count(EvalParams p, int pair0, int* __restrict__ chunk_cnt_all) {
  __shared__ int s_cnt[NID_NCLS];
  const int chunk = blockIdx.x, c = blockIdx.y, pair = pair0 + blockIdx.z;
  int* chunk_cnt = chunk_cnt_all + (size_t)blockIdx.z * p.ncell * gridDim.x * NID_NCLS;
  for (int k = threadIdx.x; k < NID_NCLS; k += blockDim.x) s_cnt[k] = 0;
  __syncthreads();
  int row, col;
  const int key = sell_key(p, (size_t)pair * p.N, c, chunk * 256 + threadIdx.x, row, col);
  if (key >= 0) atomicAdd(&s_cnt[key], 1);  // integer counts: order does not matter
  __syncthreads();
  int* out = chunk_cnt + ((size_t)c * gridDim.x + chunk) * NID_NCLS;
  for (int k = threadIdx.x; k < NID_NCLS; k += blockDim.x) out[k] = s_cnt[k];
}

// in place: chunk_cnt[cell][chunk][class] -> number of pixels of that class in the earlier chunks of the cell
__global__ void __launch_bounds__(256) k_chunk_scan(int ncell, int nchunks, int* __restrict__ chunk_cnt_all) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ncell * NID_NCLS) return;
  int* chunk_cnt = chunk_cnt_all + (size_t)blockIdx.y * ncell * nchunks * NID_NCLS;
  const int c = i / NID_NCLS, k = i - c * NID_NCLS;
  int* q = chunk_cnt + (size_t)c * nchunks * NID_NCLS + k;
  int run = 0, j = 0;
  for (; j + 16 <= nchunks; j += 16) {  // sixteen independent loads in flight per thread
    int v[16];
#pragma unroll
    for (int u = 0; u < 16; u++) v[u] = q[(size_t)(j + u) * NID_NCLS];
#pragma unroll
    for (int u = 0; u < 16; u++) { q[(size_t)(j + u) * NID_NCLS] = run; run += v[u]; }
  }
  for (; j < nchunks; j++) { const int v = q[(size_t)j * NID_NCLS]; q[(size_t)j * NID_NCLS] = run; run += v; }
}

template <bool PTS>
__global__ void __launch_bounds__(256) k_scatter_sell(EvalParams p, int pair0, int L, const double* __restrict__ depth_all,
                                                      const int* __restrict__ task_pos_all, const int* __restrict__ chunk_off_all,
                                                      double* __restrict__ sd0, double* __restrict__ sd1,
                                                      double* __restrict__ sd2, unsigned* __restrict__ sid) {
  __shared__ int run[NID_NCLS];
  __shared__ int s_cts[NID_NCLS + 1];
  const int chunk = blockIdx.x, c = blockIdx.y, pair = pair0 + blockIdx.z;
  const double* depth = depth_all + (size_t)pair * p.N;
  const int* task_pos = task_pos_all + (size_t)pair * p.max_tasks;
  const int* chunk_off = chunk_off_all + (size_t)blockIdx.z * p.ncell * gridDim.x * NID_NCLS;
  if (p.n_c[pair * p.ncell + c] < NID_MIN_CELL_POINTS) return;  // inactive cells have no tasks
  const size_t base = (size_t)pair * p.N;
  const int* cts = p.cls_task_start + ((size_t)pair * p.ncell + c) * (NID_NCLS + 1);
  const int* off = chunk_off + ((size_t)c * gridDim.x + chunk) * NID_NCLS;
  for (int k = threadIdx.x; k < NID_NCLS; k += blockDim.x) run[k] = off[k];
  for (int k = threadIdx.x; k <= NID_NCLS; k += blockDim.x) s_cts[k] = cts[k];
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const size_t sbase = (size_t)pair * p.sell_cap;
  int row = 0, col = 0;
  const int key = sell_key(p, base, c, chunk * 256 + threadIdx.x, row, col);
  const unsigned mask = __match_any_sync(0xffffffffu, key);
  const int leader = __ffs(mask) - 1;
  const int rank = __popc(mask & ((1u << lane) - 1u));
  const int cnt = __popc(mask);
  int pos = 0;
  for (int w = 0; w < (int)(blockDim.x >> 5); w++) {  // warps in order: stable
    if (warp == w && lane == leader && key >= 0) {
      pos = run[key];
      run[key] = pos + cnt;
    }
    __syncthreads();
  }
  pos = __shfl_sync(0xffffffffu, pos, leader) + rank;
  if (key >= 0) {
    const size_t i = base + (size_t)row * p.cols + col;
    const int task = s_cts[key] + pos / L, o = pos % L;
    const size_t dst = sbase + (size_t)task_pos[task] + (size_t)(o >> 2) * 128 + (o & 3);
    if (PTS) { sd0[dst] = p.pwx[i]; sd1[dst] = p.pwy[i]; sd2[dst] = p.pwz[i]; }
    else sd0[dst] = depth[(size_t)row * p.cols + col];
    sid[dst] = ((unsigned)row << 16) | (unsigned)col;
  }
}


// ------------------------------------------------------------------------------------------------
// Device-side construction of the task / slice tables of the sliced layout from the (cell, class) counts of
// k_prepare: no D2H of the counts, no host loops, no H2D of tables, any number of pairs per launch.
// Per cell the tasks are numbered in class order (class v contributes ceil(cnt_v / L) tasks of L pixels, the last one
// possibly shorter); slices take the cell's tasks longest first, 32 at a time, ties in task order: every full task (in
// task order), then the partial tasks by decreasing length (ties by class). A slice is as long as its first task, so
// all slices that start with a full task hold 32 * L pixel slots and only the last <= 9 slices of a cell need a running sum.
#define NID_LAYOUT_THREADS 288  // >= NID_NCLS, whole warps
struct CellLayoutSm {
  int ts[NID_NCLS + 1];   // first task of every class, cell-local
  int fs[NID_NCLS + 1];   // full tasks in the classes before
  int nf[NID_NCLS];       // full tasks of the class
  int r[NID_NCLS];        // pixels of the class's partial task (0: none)
  int prank[NID_NCLS];    // rank of that partial task among the cell's partial tasks
  int sorted_r[NID_NCLS]; // partial-task lengths in rank order
  int tail_off[NID_NCLS / 32 + 4];  // pixel-slot offset of slice SF + j (the slices that start with a partial task)
  int wsum[2][NID_LAYOUT_THREADS / 32];
  int T, F, S, SF, slots;
};

__device__ __forceinline__ void cell_layout(const unsigned* __restrict__ cnt, int L, CellLayoutSm& s) {
  const int v = threadIdx.x, lane = v & 31, w = v >> 5;
  constexpr int NW = NID_LAYOUT_THREADS / 32;
  const int c = v < NID_NCLS ? (int)cnt[v] : 0;  // pixels of reference intensity v
  {  // n_c = pixels with a reference sample; cells under 300 get no tasks (computeH.cu:271)
    int n = v < 256 ? c : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
    if (lane == 0) s.wsum[0][w] = n;
  }
  __syncthreads();
  int n_c = 0;
#pragma unroll
  for (int i = 0; i < NW; i++) n_c += s.wsum[0][i];
  __syncthreads();
  const int cc = n_c >= NID_MIN_CELL_POINTS ? c : 0;
  const int nf = cc / L, r = cc - nf * L, nt = nf + (r > 0 ? 1 : 0);
  int a = nt, b = nf;  // inclusive scans over the classes
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int x = __shfl_up_sync(0xffffffffu, a, o), y = __shfl_up_sync(0xffffffffu, b, o);
    if (lane >= o) { a += x; b += y; }
  }
  if (lane == 31) { s.wsum[0][w] = a; s.wsum[1][w] = b; }
  __syncthreads();
  int oa = 0, ob = 0;
  for (int i = 0; i < w; i++) { oa += s.wsum[0][i]; ob += s.wsum[1][i]; }
  if (v < NID_NCLS) {
    s.ts[v] = oa + a - nt; s.fs[v] = ob + b - nf;
    s.nf[v] = nf; s.r[v] = r;
    if (v == NID_NCLS - 1) { s.ts[NID_NCLS] = oa + a; s.fs[NID_NCLS] = ob + b; }
  }
  __syncthreads();
  if (v < NID_NCLS && r > 0) {  // longest first, ties in class (= task) order
    int g = 0;
    for (int q = 0; q < NID_NCLS; q++) {
      const int rq = s.r[q];
      g += (rq > r || (rq == r && q < v)) ? 1 : 0;
    }
    s.prank[v] = g;
    s.sorted_r[g] = r;
  }
  __syncthreads();
  if (v == 0) {
    const int T = s.ts[NID_NCLS], F = s.fs[NID_NCLS];
    const int S = (T + 31) >> 5, SF = (F + 31) >> 5;
    int off = SF * 32 * L;
    s.tail_off[0] = off;
    for (int j = 0; SF + j < S; j++) {
      off += ((s.sorted_r[32 * (SF + j) - F] + 3) >> 2) * 128;
      s.tail_off[j + 1] = off;
    }
    s.T = T; s.F = F; s.S = S; s.SF = SF; s.slots = off;
  }
  __syncthreads();
}

// totals per (pair, cell): tasks, slices, pixel slots
__global__ void __launch_bounds__(NID_LAYOUT_THREADS) k_layout_totals(int pair0, int ncell, int L, const unsigned* __restrict__ cnt,
                                                                      int* __restrict__ tot) {
  __shared__ CellLayoutSm s;
  const int c = blockIdx.x, pair = pair0 + blockIdx.y;
  cell_layout(cnt + ((size_t)pair * ncell + c) * NID_NCLS, L, s);
  if (threadIdx.x == 0) {
    int* o = tot + ((size_t)blockIdx.y * ncell + c) * 3;
    o[0] = s.T; o[1] = s.S; o[2] = s.slots;
  }
}

// exclusive scan of the totals over the cells of a pair -> bases; one CTA per pair
__global__ void __launch_bounds__(256) k_layout_scan(EvalParams p, int pair0, const int* __restrict__ tot, int* __restrict__ base,
                                                     int* __restrict__ cell_task_start, int* __restrict__ cell_slice_start,
                                                     int* __restrict__ ntasks, int* __restrict__ nslices, int* __restrict__ sl_off,
                                                     int* __restrict__ overflow) {
  __shared__ int wsum[3][8];
  __shared__ int carry[3];
  const int pair = pair0 + blockIdx.x, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int* t = tot + (size_t)blockIdx.x * p.ncell * 3;
  int* bs = base + (size_t)blockIdx.x * p.ncell * 3;
  if (threadIdx.x < 3) carry[threadIdx.x] = 0;
  __syncthreads();
  for (int c0 = 0; c0 < p.ncell; c0 += 256) {
    const int c = c0 + threadIdx.x;
    int x[3], a[3];
#pragma unroll
    for (int k = 0; k < 3; k++) { x[k] = c < p.ncell ? t[3 * c + k] : 0; a[k] = x[k]; }
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
#pragma unroll
      for (int k = 0; k < 3; k++) {
        const int y = __shfl_up_sync(0xffffffffu, a[k], o);
        if (lane >= o) a[k] += y;
      }
    if (lane == 31)
#pragma unroll
      for (int k = 0; k < 3; k++) wsum[k][w] = a[k];
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 3; k++) {
      int o = carry[k];
      for (int i = 0; i < w; i++) o += wsum[k][i];
      a[k] += o - x[k];  // exclusive
    }
    if (c < p.ncell) {
      bs[3 * c] = a[0]; bs[3 * c + 1] = a[1]; bs[3 * c + 2] = a[2];
      cell_task_start[(size_t)pair * (p.ncell + 1) + c] = a[0];
      cell_slice_start[(size_t)pair * (p.ncell + 1) + c] = a[1];
    }
    __syncthreads();
    if (threadIdx.x == 255)
#pragma unroll
      for (int k = 0; k < 3; k++) carry[k] = a[k] + x[k];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const int nt = carry[0], ns = carry[1], slots = carry[2];
    cell_task_start[(size_t)pair * (p.ncell + 1) + p.ncell] = nt;
    cell_slice_start[(size_t)pair * (p.ncell + 1) + p.ncell] = ns;
    ntasks[pair] = nt;
    nslices[pair] = ns;
    sl_off[(size_t)pair * (p.max_slices + 1) + min(ns, p.max_slices)] = slots;
    if (nt > p.max_tasks || ns > p.max_slices || (size_t)slots > p.sell_cap) atomicExch(overflow, 1);  // (cannot happen by construction)
  }
}

// the tables of one (pair, cell)
__global__ void __launch_bounds__(NID_LAYOUT_THREADS) k_layout_write(EvalParams p, int pair0, int L, const unsigned* __restrict__ cnt,
                                                                     const int* __restrict__ base, int2* __restrict__ tasks,
                                                                     int* __restrict__ task_pos, int* __restrict__ sl_task,
                                                                     int* __restrict__ sl_off, int* __restrict__ sl_cell,
                                                                     int* __restrict__ cls_task_start) {
  __shared__ CellLayoutSm s;
  const int c = blockIdx.x, pair = pair0 + blockIdx.y;
  cell_layout(cnt + ((size_t)pair * p.ncell + c) * NID_NCLS, L, s);
  const int* bs = base + ((size_t)blockIdx.y * p.ncell + c) * 3;
  const int tb = bs[0], sb = bs[1], pb = bs[2];
  if (tb + s.T > p.max_tasks || sb + s.S > p.max_slices) return;  // flagged by k_layout_scan
  for (int v = threadIdx.x; v <= NID_NCLS; v += blockDim.x)
    cls_task_start[((size_t)pair * p.ncell + c) * (NID_NCLS + 1) + v] = tb + s.ts[v];
  int2* tk = tasks + (size_t)pair * p.max_tasks + tb;
  int* tp = task_pos + (size_t)pair * p.max_tasks + tb;
  int* st = sl_task + ((size_t)pair * p.max_slices + sb) * 32;
  int* sd = const_cast<int*>(p.sl_desc) + ((size_t)pair * p.max_slices + sb) * 32;
  unsigned short* tc = const_cast<unsigned short*>(p.task_cls) + (size_t)pair * p.max_tasks + tb;
  for (int t = threadIdx.x; t < s.T; t += blockDim.x) {
    int lo = 0, hi = NID_NCLS;  // class of task t: the last v with ts[v] <= t
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (s.ts[mid] <= t) lo = mid; else hi = mid;
    }
    const int v = lo, i = t - s.ts[v];
    const bool full = i < s.nf[v];
    const int len = full ? L : s.r[v];
    const int rank = full ? s.fs[v] + i : s.F + s.prank[v];
    const int slice = rank >> 5, ln = rank & 31;
    const int off = slice < s.SF ? slice * 32 * L : s.tail_off[slice - s.SF];
    tk[t] = make_int2(i * L, len | (v << 9) | (c << 18));
    tp[t] = pb + off + 4 * ln;
    st[rank] = tb + t;
    sd[rank] = len | (v << 9) | (c << 18);
    tc[t] = (unsigned short)v;
  }
  for (int q = s.T + threadIdx.x; q < s.S * 32; q += blockDim.x) { st[q] = -1; sd[q] = 0; }  // empty lanes of the cell's last slice
  for (int sl = threadIdx.x; sl < s.S; sl += blockDim.x) {
    sl_off[(size_t)pair * (p.max_slices + 1) + sb + sl] = pb + (sl < s.SF ? sl * 32 * L : s.tail_off[sl - s.SF]);
    sl_cell[(size_t)pair * p.max_slices + sb + sl] = c;
  }
}

// Packed target texture: texel = I | (Gx+256) << 8 | (Gy+256) << 17 with the central differences
// Gx = I(x+1,y) - I(x-1,y), Gy = I(x,y+1) - I(x,y-1) (types_six_dof_expmap.cpp:434-435 before the /2);
// one 2x2 gather then holds everything the bilinear samples of I, dI/du and dI/dv need. Border texels
// use clamped neighbours and are never consumed (the first row/column takes the literal formula).
__global__ void k_pack_tex(int rows, int cols, int pair0, const uint8_t* __restrict__ im_all, unsigned* __restrict__ out_all) {
  const int N = rows * cols;
  const uint8_t* im = im_all + (size_t)(pair0 + blockIdx.y) * N;
  unsigned* out = out_all + (size_t)blockIdx.y * N;  // scratch of the batch
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
    const int y = i / cols, x = i % cols;
    const int xm = max(x - 1, 0), xp = min(x + 1, cols - 1), ym = max(y - 1, 0), yp = min(y + 1, rows - 1);
    const int I = im[i];
    const int gx = (int)im[y * cols + xp] - (int)im[y * cols + xm];
    const int gy = (int)im[yp * cols + x] - (int)im[ym * cols + x];
    out[i] = (unsigned)I | ((unsigned)(gx + 256) << 8) | ((unsigned)(gy + 256) << 17);
  }
}

// Footprint-packed target image for pass 1: out[y*cols + x] = I(x,y) | I(x+1,y)<<8 | I(x,y+1)<<16 | I(x+1,y+1)<<24
// (neighbours clamped at the border; in-bounds samples never reach it): one aligned 32-bit load per sample.
__global__ void k_pack_fp(int rows, int cols, int pair0, const uint8_t* __restrict__ im_all, unsigned* __restrict__ out_all) {
  const int N = rows * cols;
  const uint8_t* im = im_all + (size_t)(pair0 + blockIdx.y) * N;
  unsigned* out = out_all + (size_t)(pair0 + blockIdx.y) * N;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
    const int y = i / cols, x = i % cols;
    const int xp = min(x + 1, cols - 1), yp = min(y + 1, rows - 1);
    out[i] = (unsigned)im[y * cols + x] | ((unsigned)im[y * cols + xp] << 8) | ((unsigned)im[yp * cols + x] << 16) |
             ((unsigned)im[yp * cols + xp] << 24);
  }
}

// ------------------------------------------------------------------------------------------------
// Per-job geometry of the fast path. Built on the host from the staged poses and handed to the pixel
// kernels BY VALUE: the kernel parameter space is a constant bank, so the entries are read with uniform
// constant loads instead of occupying ~40 registers of matrix entries per thread.
//   [0..11] M[3c + r]: T_cw1 * T_wc0 (depth form) or T_cw1 (point form), 3x4; pass 1 gets rows 0 and 1
//           pre-multiplied by fx and fy (it only needs u and v)
//   [12] 1/fx  [13] -cx/fx  [14] 1/fy  [15] -cy/fy  [16] fx  [17] fy  [18] cx  [19] cy
#define NID_GEO_STRIDE 20
template <int NG>
struct GeoTable {
  double g[NG][NID_GEO_STRIDE];
  // the launch's i-th job, its pair, the pair's slice count and packed target texture: the pixel kernels start without
  // a chain of dependent global loads (job list -> job_pair -> nslices / texture handle)
  unsigned long long tex[NG];
  int job[NG], pair[NG], nsl[NG];
};

// The reference's exact sequence for one pixel: CudaPoints3d.cu:20-28 then computeH.cu:152-158, from the
// job's T_cw1, the pair's T_wc0 and intrinsics in global memory (rare path).
template <bool PTS>
__device__ __noinline__ void exact_uv(const double* __restrict__ T1g, const double* __restrict__ T0g,
                                      const double* __restrict__ camg, double a0, double a1, double a2, unsigned id,
                                      double* out5) {
  const Cam cam{camg[0], camg[1], camg[2], camg[3]};
  double xw = a0, yw = a1, zw = a2;
  if (!PTS) backproject(T0g, cam, a0, (int)(id >> 16), (int)(id & 0xffffu), xw, yw, zw);
  const Pose P = load_pose(T1g);
  double x1, y1, z1, u, v;
  warp_project(P, cam, xw, yw, zw, x1, y1, z1, u, v);
  out5[0] = x1; out5[1] = y1; out5[2] = z1; out5[3] = u; out5[4] = v;
}

// Result of the shared front end of both passes.
struct Px {
  double xn, yn, rz;   // normalised camera-frame coordinates x/z, y/z and 1/z (pass 2)
  double dx, dy;       // fractional parts of (u, v)
  int ix, iy;
  bool ok;             // in bounds for the cost: u>=0 && u+3<=cols && v>=0 && v+3<=rows
  bool jac;            // ... and for the Jacobian (u+3<=cols-1)
  bool exact;          // (u, v) came from the reference's exact sequence
  bool fix;            // fast path could not decide: (u, v) within 2^-24 of an integer
};

// not near an integer: fraction in [2^-24, 1 - 2^-21)
__device__ __forceinline__ bool frac_is_safe(double d) {
  return (unsigned)(__double2hiint(d) - 0x3E700000) < (unsigned)(0x3FEFFFFF - 0x3E700000);
}

__device__ __forceinline__ void px_from_exact(const double* e, int rows, int cols, Px& r) {
  r.rz = 1.0 / e[2];  // types_six_dof_expmap.cpp:437
  r.xn = e[0] * r.rz; r.yn = e[1] * r.rz;
  const double u = e[3], v = e[4];
  r.ok = inb_cost(u, v, rows, cols);
  r.jac = inb_jac(u, v, rows, cols);
  r.ix = 0; r.iy = 0; r.dx = 0.0; r.dy = 0.0;
  if (r.ok) {
    r.ix = (int)u; r.iy = (int)v;
    r.dx = u - (double)r.ix; r.dy = v - (double)r.iy;
  }
  r.exact = true;
  r.fix = false;
}

// Branch-free fast path (so that the pixels of a batch interleave). g: the job's geometry entries.
// P1: pass 1 (rows 0/1 of M pre-scaled, only u, v wanted); else pass 2 (xn, yn, 1/z kept).
template <bool PTS, bool P1>
__device__ __forceinline__ void front(const double* __restrict__ g, int rows, int cols, double a0, double a1, double a2,
                                      unsigned id, Px& r) {
  double x1, y1, z1;
  if (PTS) {
    x1 = fma(g[0], a0, fma(g[3], a1, fma(g[6], a2, g[9])));
    y1 = fma(g[1], a0, fma(g[4], a1, fma(g[7], a2, g[10])));
    z1 = fma(g[2], a0, fma(g[5], a1, fma(g[8], a2, g[11])));
  } else {
    const double cxn = fma(u2d(id & 0xffffu), g[12], g[13]);
    const double cyn = fma(u2d(id >> 16), g[14], g[15]);
    const double d0 = fma(g[0], cxn, fma(g[3], cyn, g[6]));
    const double d1 = fma(g[1], cxn, fma(g[4], cyn, g[7]));
    const double d2 = fma(g[2], cxn, fma(g[5], cyn, g[8]));
    x1 = fma(a0, d0, g[9]);
    y1 = fma(a0, d1, g[10]);
    z1 = fma(a0, d2, g[11]);
  }
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(z1));
  double e = fma(-z1, y, 1.0);
  y = fma(y, e, y);
  e = fma(-z1, y, 1.0);
  y = fma(y, e, y);
  double u, v;
  if (P1) {
    u = fma(x1, y, g[18]);
    v = fma(y1, y, g[19]);
  } else {
    r.xn = x1 * y; r.yn = y1 * y; r.rz = y;
    u = fma(g[16], r.xn, g[18]);
    v = fma(g[17], r.yn, g[19]);
  }
  r.exact = false;
  const int ix = __double2int_rz(u), iy = __double2int_rz(v);  // NaN -> 0, saturating
  const double dx = u - u2d((unsigned)ix), dy = v - u2d((unsigned)iy);
  // u <= -1 or u >= cols-2 (same for v) is out of bounds whatever the last bits are; padding slots never count
  const bool inr = id != NID_PAD_ID && (unsigned)ix <= (unsigned)(cols - 3) && (unsigned)iy <= (unsigned)(rows - 3);
  const bool safe = frac_is_safe(dx) && frac_is_safe(dy);
  // with u, v not within 2^-24 of an integer the integer comparisons decide exactly like
  // `u>=0 && u+3<=cols && v>=0 && v+3<=rows` (types_six_dof_expmap.cpp:565; :433 with cols-1)
  r.ok = inr && safe && ix <= cols - 4 && iy <= rows - 4;
  r.jac = r.ok && ix <= cols - 5;
  r.fix = inr && !safe;
  const bool keep = P1 ? r.ok : r.jac;
  r.ix = keep ? ix : 0; r.iy = keep ? iy : 0;
  r.dx = dx; r.dy = dy;
}

// types_six_dof_expmap.h:321-326 in the reference's term order, without contraction (exact-path pixels:
// on a saturated plateau the `>= 255` clamp that follows sees the last bit of this sum)
__device__ __forceinline__ double bilinear_ref(double dx, double dy, unsigned p00, unsigned p01, unsigned p10, unsigned p11) {
  const double dxdy = __dmul_rn(dx, dy);
  const double w00 = __dadd_rn(__dsub_rn(__dsub_rn(1.0, dx), dy), dxdy);
  double a = __dmul_rn(dxdy, u2d(p11));
  a = __dadd_rn(a, __dmul_rn(__dsub_rn(dy, dxdy), u2d(p10)));
  a = __dadd_rn(a, __dmul_rn(__dsub_rn(dx, dxdy), u2d(p01)));
  return __dadd_rn(a, __dmul_rn(w00, u2d(p00)));
}

// Same interpolant for fast-path pixels, as p00 + dx d0 + dy ((p10 + dx d1) - (p00 + dx d0)): 4 fp64 operations.
// It differs from bilinear_ref by rounding only, which no decision of a fast-path pixel depends on: the spline
// weights are continuous across span boundaries, an all-zero footprint gives exactly 0 in both forms, and
// saturated footprints take the exact path.
__device__ __forceinline__ double bilinear_fast(double dx, double dy, double p00, double d0, double p10, double d1) {
  const double a = fma(dx, d0, p00), b = fma(dx, d1, p10);
  return fma(dy, b - a, a);
}

// pass-2 gather: component order for the footprint with top-left texel (ix, iy):
//   .w = (ix, iy)  .z = (ix+1, iy)  .x = (ix, iy+1)  .y = (ix+1, iy+1)
__device__ __forceinline__ uint4 gather_u32(cudaTextureObject_t tex, int ix, int iy) {
  return tex2Dgather<uint4>(tex, (float)(ix + 1), (float)(iy + 1), 0);
}

// Cubic B-spline weights without end-span cases. The reference's basis N_j lives on the clamped knot vector
// t_i = clamp(i-3, 0, B-3) (types_six_dof_expmap.cpp:738-764); on [0, B-3] it spans the same space as the B shifted
// copies U_j of the uniform cubic B-spline, and the change of basis is the identity except for a 3x3 block at
// either end (exact rationals, the same for every B >= 6):
//     N_0 = 6 U_0                N_{B-1} = 6 U_{B-1}
//     N_1 = -6 U_0 + 3/2 U_1     N_{B-2} = 3/2 U_{B-2} - 6 U_{B-1}
//     N_2 = U_0 - 1/2 U_1 + U_2  N_{B-3} = U_{B-3} - 1/2 U_{B-2} + U_{B-1}
// Histograms are sums of basis values, so pass 1 accumulates the *uniform* weights of every pixel (one branch-free
// formula, no coefficient table) and applies the block once per task row (fold_row); pass 2 uses the transposed
// block on its class table (fold_table) and the uniform derivative per pixel. The one place where this is not
// a rounding-level identity is a bin whose clamped sum is exactly zero in the reference while U-sums cancel only
// to rounding: that happens iff every contributing pixel sits at u == 0 exactly (N_1(0) = N_2(0) = 0), so pixels
// with u == 0 are counted apart and enter bin 0 with weight exactly 1.
__device__ __forceinline__ void bspline4_uniform(double f, double w[4]) {
  const double s6 = 1.0 / 6.0, h = 0.5;
  w[0] = fma(f, fma(f, fma(f, -s6, h), -h), s6);
  w[1] = fma(f * f, fma(f, h, -1.0), 2.0 / 3.0);
  w[2] = fma(f, fma(f, fma(f, -h, h), h), s6);
  w[3] = f * f * f * s6;
}
// h: one lane's row of uniform sums, element b at h[b * stride]; n0: its pixels with u == 0
__device__ __forceinline__ void fold_row(double* h, int stride, int B, double n0) {
  const double u0 = h[0], u1 = h[stride], u2 = h[2 * stride];
  h[0] = fma(6.0, u0, n0);
  h[stride] = fma(1.5, u1, -6.0 * u0);
  h[2 * stride] = (u0 - 0.5 * u1) + u2;
  const double t1 = h[(B - 1) * stride], t2 = h[(B - 2) * stride], t3 = h[(B - 3) * stride];
  h[(B - 1) * stride] = 6.0 * t1;
  h[(B - 2) * stride] = fma(1.5, t2, -6.0 * t1);
  h[(B - 3) * stride] = (t1 - 0.5 * t2) + t3;
}
// transposed block: sum_j N'_j W_j = sum_j U'_j W^_j
__device__ __forceinline__ void fold_table(double* w, int stride, int B) {
  const double w0 = w[0], w1 = w[stride], w2 = w[2 * stride];
  w[0] = fma(6.0, w0 - w1, w2);
  w[stride] = fma(1.5, w1, -0.5 * w2);
  const double v1 = w[(B - 1) * stride], v2 = w[(B - 2) * stride], v3 = w[(B - 3) * stride];
  w[(B - 1) * stride] = fma(6.0, v1 - v2, v3);
  w[(B - 2) * stride] = fma(1.5, v2, -0.5 * v3);
}

// ------------------------------------------------------------------------------------------------
// One group = four consecutive pixels of a lane's task (32 B of depths + 16 B of pixel ids per lane).
template <bool PTS>
struct Group {
  unsigned id[4];
  double a0[4], a1[4], a2[4];
  __device__ __forceinline__ void load(const double* q0, const double* q1, const double* q2, const unsigned* qi, size_t o) {
    // read-once stream: evict-first loads keep L1 for the target-image gathers
    const uint4 i4 = __ldcs(reinterpret_cast<const uint4*>(qi + o));
    id[0] = i4.x; id[1] = i4.y; id[2] = i4.z; id[3] = i4.w;
    const double2 xa = __ldcs(reinterpret_cast<const double2*>(q0 + o)), xb = __ldcs(reinterpret_cast<const double2*>(q0 + o + 2));
    a0[0] = xa.x; a0[1] = xa.y; a0[2] = xb.x; a0[3] = xb.y;
    if (PTS) {
      const double2 ya = __ldcs(reinterpret_cast<const double2*>(q1 + o)), yb = __ldcs(reinterpret_cast<const double2*>(q1 + o + 2));
      const double2 za = __ldcs(reinterpret_cast<const double2*>(q2 + o)), zb = __ldcs(reinterpret_cast<const double2*>(q2 + o + 2));
      a1[0] = ya.x; a1[1] = ya.y; a1[2] = yb.x; a1[3] = yb.y;
      a2[0] = za.x; a2[1] = za.y; a2[2] = zb.x; a2[3] = zb.y;
    } else {
#pragma unroll
      for (int j = 0; j < 4; j++) { a1[j] = 0.0; a2[j] = 0.0; }
    }
  }
};

// mbarrier and bulk-copy (cp.async.bulk) helpers: pass 2 of small cells stages the cell's log tables by one bulk copy
// (k_jac_sell, BULK)
__device__ __forceinline__ unsigned smem_u32(const void* ptr) { return (unsigned)__cvta_generic_to_shared(ptr); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

// what the rare exact paths need from global memory
struct ExactSrc {
  const double* T1;   // the job's T_cw1, column-major 4x4
  const double* T0;   // the pair's T_wc0
  const double* cam;  // fx fy cx cy
};

// where the current group of the lane lives in the pixel store: the rare paths re-read a pixel from there, so that
// the group's registers are free once the fast front end has consumed them
struct GroupAddr {
  const double *q0, *q1, *q2;
  const unsigned* qi;
};

template <bool PTS>
__device__ __forceinline__ void make_exact(const ExactSrc& xs, int rows, int cols, const GroupAddr& ga, int j, Px& r) {
  double ex[5];
  const double a0 = ga.q0[j], a1 = PTS ? ga.q1[j] : 0.0, a2 = PTS ? ga.q2[j] : 0.0;
  const unsigned id = ga.qi[j];
  exact_uv<PTS>(xs.T1, xs.T0, xs.cam, a0, a1, a2, id, ex);
  px_from_exact(ex, rows, cols, r);
}

// Pass 1 on W pixels of a group at once: projection (branch-free), W footprint loads in flight, uniform spline
// weights, then the accumulations in pixel order into the lane's private row h[b * T] (T = threads per CTA).
// fp: the pair's footprint-packed target image, fp[y*cols + x] = I(x,y) | I(x+1,y)<<8 | I(x,y+1)<<16 | I(x+1,y+1)<<24.
// n0 counts the lane's pixels with u == 0 exactly (see bspline4_uniform).
template <bool PTS, int W, int T>
__device__ __forceinline__ void hist_pixels(const double* __restrict__ g, const ExactSrc& xs, int rows, int cols,
                                            const Group<PTS>& G, int j0, const GroupAddr& ga,
                                            const unsigned* __restrict__ fp, double s, int NS, double* __restrict__ h,
                                            int& n0) {
  Px r[W];
  bool anyexact = false;
#pragma unroll
  for (int j = 0; j < W; j++) {
    front<PTS, true>(g, rows, cols, G.a0[j0 + j], G.a1[j0 + j], G.a2[j0 + j], G.id[j0 + j], r[j]);
    anyexact |= r[j].fix;
  }
  if (anyexact) {
#pragma unroll
    for (int j = 0; j < W; j++)
      if (r[j].fix) make_exact<PTS>(xs, rows, cols, ga, j0 + j, r[j]);
  }
  unsigned t[W];
#pragma unroll
  for (int j = 0; j < W; j++) t[j] = __ldg(fp + (unsigned)(r[j].iy * cols + r[j].ix));
  bool sat = false;
#pragma unroll
  for (int j = 0; j < W; j++) sat |= t[j] == 0xffffffffu;  // (qualified below: the common case is one compare per pixel)
  if (sat) {
    // saturated plateau: the clamp `>= 255 -> 254.999` (types_six_dof_expmap.cpp:572) depends on the last bit
    // of the bilinear weights, so the fractions must be the reference's own
#pragma unroll
    for (int j = 0; j < W; j++)
      if (r[j].ok && !r[j].exact && t[j] == 0xffffffffu) {
        anyexact = true;
        make_exact<PTS>(xs, rows, cols, ga, j0 + j, r[j]);
        t[j] = __ldg(fp + (unsigned)(r[j].iy * cols + r[j].ix));
      }
  }
  double ic[W];
#pragma unroll
  for (int j = 0; j < W; j++) {
    const int p00 = t[j] & 0xffu, p01 = (t[j] >> 8) & 0xffu, p10 = (t[j] >> 16) & 0xffu, p11 = t[j] >> 24;
    ic[j] = bilinear_fast(r[j].dx, r[j].dy, u2d(p00), i2d_small(p01 - p00), u2d(p10), i2d_small(p11 - p10));
  }
  if (anyexact) {
#pragma unroll
    for (int j = 0; j < W; j++)
      if (r[j].exact) {
        const unsigned p00 = t[j] & 0xffu, p01 = (t[j] >> 8) & 0xffu, p10 = (t[j] >> 16) & 0xffu, p11 = t[j] >> 24;
        ic[j] = clamp_intensity(bilinear_ref(r[j].dx, r[j].dy, p00, p01, p10, p11));
      }
  }
  double wt[W][4];
  int kt[W];
  bool acc[W];
#pragma unroll
  for (int j = 0; j < W; j++) {
    const double ub = ic[j] * s;
    kt[j] = min((int)ub, NS - 1);  // 0 <= ub <= NS (== NS only by rounding); only used where acc[j]
    bspline4_uniform(ub - u2d((unsigned)kt[j]), wt[j]);
    const bool zero = ub == 0.0;
    acc[j] = r[j].ok && !zero;
    n0 += (r[j].ok && zero) ? 1 : 0;
  }
#pragma unroll
  for (int j = 0; j < W; j++) {
    if (!acc[j]) continue;
    double* hk = h + kt[j] * T;
#pragma unroll
    for (int n = 0; n < 4; n++) hk[n * T] += wt[j][n];
  }
}

// Epilogue of pass 1: the warp's 32 rows go out as whole 8 B x B lines. Lane l first rotates its row inside the warp's
// own columns of the shared array -- value (l, b) to column (l + b) mod 32 of plane b -- so that the lanes which then
// write one task's row read B different banks; each store instruction covers 32/B' complete rows (B' = B rounded up
// to a power of two) instead of 32 partial sectors of 32 different rows.
// hw: plane b of this warp at hw[b * T + 0..31]; the row of task tk goes to Gj[tk * gstride + 0..B-1].
template <int T>
__device__ __forceinline__ void store_task_rows(double* hw, int B, int lane, int task, double* __restrict__ Gj, size_t gstride) {
  for (int b0 = 0; b0 < B; b0 += 8) {
    double v[8];
#pragma unroll
    for (int i = 0; i < 8; i++) v[i] = (b0 + i < B) ? hw[(b0 + i) * T + lane] : 0.0;
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 8; i++)
      if (b0 + i < B) hw[(b0 + i) * T + ((lane + b0 + i) & 31)] = v[i];
  }
  __syncwarp();
  const int BP2 = B <= 8 ? 8 : (B <= 16 ? 16 : 32);  // lanes per row
  const int rpi = 32 / BP2;                          // rows per store instruction
  const int b = lane & (BP2 - 1), sub = lane / BP2;
  {
    const double* src = hw + min(b, B - 1) * T;  // (lanes beyond the row length read a valid plane and store nothing)
    double* dst = Gj + b;
    const int nit = 32 / rpi;  // 8, 16 or 32 store instructions
    for (int i0 = 0; i0 < nit; i0 += 8) {
      double v[8];
      int tk[8];
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const int tl = (i0 + i) * rpi + sub;
        tk[i] = __shfl_sync(0xffffffffu, task, tl);
        v[i] = src[(tl + b) & 31];
      }
#pragma unroll
      for (int i = 0; i < 8; i++)
        if (b < B && tk[i] >= 0) dst[(size_t)tk[i] * gstride] = v[i];
    }
  }
  for (int b1 = BP2; b1 < B; b1 += BP2) {  // B > 32: remaining columns
    for (int t0 = 0; t0 < 32; t0 += rpi) {
      const int tl = t0 + sub, bb = b1 + b;
      const int tk = __shfl_sync(0xffffffffu, task, tl);
      if (bb < B && tk >= 0) Gj[(size_t)tk * gstride + bb] = hw[bb * T + ((tl + bb) & 31)];
    }
  }
  __syncwarp();
}

// Pass 1: per task the un-weighted target soft histogram h[B] of its pixels.
// grid (jobs of this launch, ceil(max_slices/(T/32))), T = 32..256 threads (fewer when few jobs are in flight, so
// that every SM gets work); shared: rows [B][T]. The job index is the fast grid dimension and slices are ordered
// longest first, so the long CTAs of every job start first and the short ones fill the tail. The next group's
// pixels are loaded before the current group is processed. NID_HIST_W pixels of a lane are in flight together.
#ifndef NID_HIST_W
#define NID_HIST_W 4
#endif
#ifndef NID_JAC_W
#define NID_JAC_W 2
#endif
#ifndef NID_HIST_TMAX
#define NID_HIST_TMAX 32  // largest CTA of pass 1 / pass 2 (pick_block shrinks it when few jobs are in flight); measured best:
                          // one-warp CTAs at 18 resident warps (113 registers) 2.28 us per C2 evaluation, 128-thread CTAs at 16 warps 2.49
#endif
#ifndef NID_JAC_TMAX
#define NID_JAC_TMAX 64
#endif
#ifndef NID_HIST_MINB
#define NID_HIST_MINB 2  // CTAs of 256 threads per SM (128 registers)
#endif
#ifndef NID_JAC_MINB
#define NID_JAC_MINB 4  // CTAs of 128 threads per SM (128 registers)
#endif
#ifndef NID_HIST_WARPS
#define NID_HIST_WARPS 18  // resident warps per SM the register budget is set for
#endif
#ifndef NID_JAC_WARPS
#define NID_JAC_WARPS (NID_JAC_MINB * 4)
#endif
// the small-cell instantiations (BULK: short slices, prologue-heavy) trade registers for resident warps (__maxnreg__): measured
// at 16x16 cells, us per evaluation by register budget (resident warps): 128 (16) 5.48, 120 (17) 5.28, 112 (18) 5.50,
// 104 (19) 5.52, 96 (21) 5.08, 88 (23) 5.56, 80 (25) 5.75; at 12x12 cells 4.70 with 112, 4.42 with 96. At 4x4 cells the
// full 128 registers are best (3.43 against 3.68 with 96).
#ifndef NID_JAC_REGS_SMALL
#define NID_JAC_REGS_SMALL 96
#endif
#define NID_JAC_WARPS_SMALL (2048 / NID_JAC_REGS_SMALL)  // resident warps the register file holds at that budget
template <bool PTS, int NG, int T>
__global__ void __launch_bounds__(T, NID_HIST_WARPS * 32 / T)
k_hist_sell(const __grid_constant__ EvalParams p, const __grid_constant__ GeoTable<NG> gt) {
  extern __shared__ __align__(16) double sm[];
  const int B = p.bins, NS = B - 3;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // (the job / pair / slice-count entries of the parameter table, which pass 2 uses, cost this kernel 24 bytes of spills:
  // measured slower at 4x4 and at 16x16 cells)
  const int job = job_at(p, NID_BLK_JOB);
  const int pair = p.job_pair[job];
  const double* g = gt.g[NID_BLK_JOB];
  const int slice = NID_BLK_CHUNK * (T >> 5) + warp;
  if (slice >= p.nslices[pair]) return;  // (no block-wide barrier below)
  const int* so = p.sl_off + (size_t)pair * (p.max_slices + 1) + slice;
  const int off0 = so[0], ngroups = (so[1] - off0) >> 7;
  const int task = p.sl_task[((size_t)pair * p.max_slices + slice) * 32 + lane];  // (for the epilogue; requested early)
  double* h = sm + threadIdx.x;  // h[b * T]
  for (int b = 0; b < B; b++) h[b * T] = 0.0;
  const size_t sbase = (size_t)pair * p.sell_cap + off0 + lane * 4;
  const double* q0 = p.sd0 + sbase;
  const double* q1 = PTS ? p.sd1 + sbase : nullptr;
  const double* q2 = PTS ? p.sd2 + sbase : nullptr;
  const unsigned* qi = p.sid + sbase;
  const unsigned* fp = p.fp1 + (size_t)pair * p.N;
  const ExactSrc xs{p.poses + 16 * job, p.Twc0 + 16 * pair, p.cam + 4 * pair};
  const double s = (double)NS / 255.0;
  int n0 = 0;
  Group<PTS> G;
  G.load(q0, q1, q2, qi, 0);
  for (int gi = 0; gi < ngroups; gi++) {
    Group<PTS> Gn = G;
    if (gi + 1 < ngroups) Gn.load(q0, q1, q2, qi, (size_t)(gi + 1) * 128);
#if NID_PREFETCH_L2 > 0
    if (gi + 1 + NID_PREFETCH_L2 < ngroups) {
      const size_t po = (size_t)(gi + 1 + NID_PREFETCH_L2) * 128;
      asm volatile("prefetch.global.L2 [%0];" ::"l"(q0 + po));
      asm volatile("prefetch.global.L2 [%0];" ::"l"(qi + po));
    }
#endif
    const size_t go = (size_t)gi * 128;
    const GroupAddr ga{q0 + go, PTS ? q1 + go : nullptr, PTS ? q2 + go : nullptr, qi + go};
#pragma unroll
    for (int j0 = 0; j0 < 4; j0 += NID_HIST_W) hist_pixels<PTS, NID_HIST_W, T>(g, xs, p.rows, p.cols, G, j0, ga, fp, s, NS, h, n0);
    G = Gn;
  }
  fold_row(h, T, B, (double)n0);  // uniform sums -> sums of the reference's clamped basis
  __syncwarp();
  store_task_rows<T>(sm + (threadIdx.x & ~31), B, lane, task, p.G + (size_t)job * p.g_stride * B, B);
}

// ------------------------------------------------------------------------------------------------
// Assembly (a7 + table half of a8): one CTA per (cell, job). From the per-class soft histograms h_v,
//     P_j[r][t] = sum_kk sum_{v: k_r(v) = r-kk} w_ref,v[kk] * h_v[t]     (kk = 0..3, classes in order)
//     P_t[t]    = sum_v h_v[t]
// normalises by n_c, computes H_t, H_j, err (computeH.cu:261-300; types_six_dof_expmap.cpp:609-635,
// .h:227) and, when want_jac, stores the scaled tables for pass 2:
//   W[r][t] = coefJ * (1 + log2 P_j[r][t]),  V[t] = coefT * (1 + log2 P_t[t])   (0 where P < 1e-30),
//   coefJ = -(s/(n_c Hj^2)) (Ht + Href), coefT = (s/(n_c Hj^2)) Hj  (types_six_dof_expmap.cpp:486-528).
// k_r(v) is monotone in v, so the classes of a span are a contiguous range (span_start).
#ifndef NID_ASM_THREADS
#define NID_ASM_THREADS 256
#endif
#define NID_ASM_SMALL 128
#ifndef NID_ASM_BATCH
#define NID_ASM_BATCH 12  // task rows a thread keeps in flight
#endif
#ifndef NID_ASM_CHUNK
#define NID_ASM_CHUNK 16  // task rows of a class that are summed in one go (see assemble_body)
#endif
#ifndef NID_ASM_MINB
#define NID_ASM_MINB 4
#endif
// NT threads per CTA: 256 in general, 128 for small cells (many cells per job, little work per cell: twice the CTAs
// resident per SM). Fixed per geometry, so results never depend on how a batch is launched.
template <int NT>
__device__ __forceinline__ void assemble_body(const EvalParams& p, int want_jac) {
  extern __shared__ __align__(16) double sm[];
  __shared__ double scratch[8];
  __shared__ int s_cts[NID_NCLS + 1];
  __shared__ int s_bnd[NT / 3 + 2];
  __shared__ int s_span[NID_SORTED_MAX_BINS];  // first class of every span (+ end)
  const int B = p.bins, BB = B * B, NS = B - 3;
  double* Pall = sm;                    // [BB + B]
  double* red = sm + BB + B;            // [NT] partial sums of P_t
  double* hvs = red + NT;  // [NID_NCLS][B] per-class soft histograms
  double* part = hvs + NID_NCLS * B;    // [4][BB] per-span partial sums of P_j
  double* wl = part + 4 * BB;           // [256][4] reference weights (up to 20 bins)
  const int c = blockIdx.x, job = job_at(p, blockIdx.y);
  const int pair = p.job_pair[job];
  const int nc = p.n_c[pair * p.ncell + c];
  const size_t o = (size_t)job * p.ncell + c;
  if (nc < NID_MIN_CELL_POINTS) {
    if (threadIdx.x == 0) { p.ht[o] = nan(""); p.hj[o] = nan(""); p.err[o] = nan(""); }
    return;
  }
  // ---- per-class soft histograms h_v[t] = sum over the tasks of class v of G[task][t], straight from pass 1's task
  // rows. The cell's tasks are one contiguous range ordered by class. A class of more than NID_ASM_CHUNK tasks is summed
  // in chunks of that many consecutive rows, the chunk sums then in chunk order (the summation order is part of the
  // result: it does not depend on the CTA size or on how the rows are dealt out). The rows are cut into runs of about
  // equal length at chunk boundaries, one run per group of threads that covers a row, and every thread streams through
  // its run with NID_ASM_BATCH independent row loads in flight, closing a segment (a whole class, or one chunk of a long
  // class) whenever the row index passes the segment's end. Chunk sums are parked in the chunk's first row of G (pass
  // 1's rows are dead once they are summed) and folded after a barrier. Without the chunks one dominant class (a
  // saturated or uniform region: thousands of pixels of one intensity) serialises on one thread group and the whole
  // cell waits for it: measured 17.6 us against 6.6 us for an ordinary cell of the same size.
  {
    const int* cts = p.cls_task_start + ((size_t)pair * p.ncell + c) * (NID_NCLS + 1);
    for (int i = threadIdx.x; i <= NID_NCLS; i += blockDim.x) s_cts[i] = cts[i];
    for (int i = threadIdx.x; i <= NS; i += blockDim.x) s_span[i] = p.span_start[i];
    if (NID_FEW_BINS(B)) for (int i = threadIdx.x; i < 1024; i += blockDim.x) wl[i] = p.lut_w[i];
    __syncthreads();
    // many bins: a thread owns two adjacent bins of a row (one 16-byte load; rows are 16-byte aligned when B is even),
    // which doubles the number of runs in flight; with few bins there are enough runs already
    const bool pairs = (B & 1) == 0;
    const int tpr = pairs ? B >> 1 : B;  // threads per row
    const int ng = NT / tpr;
    const int tfirst = s_cts[0], tlast = s_cts[NID_NCLS], ntask = tlast - tfirst;
    if ((int)threadIdx.x <= ng) {
      int bnd = tlast;
      if ((int)threadIdx.x < ng) {
        const int target = tfirst + (int)(((long long)threadIdx.x * ntask) / ng);
        int lo = 0, hi = NID_NCLS;  // the class that holds row `target`: the last v with s_cts[v] <= target
        while (hi - lo > 1) {
          const int mid = (lo + hi) >> 1;
          if (s_cts[mid] <= target) lo = mid; else hi = mid;
        }
        bnd = s_cts[lo] + ((target - s_cts[lo]) / NID_ASM_CHUNK) * NID_ASM_CHUNK;
      }
      s_bnd[threadIdx.x] = bnd;
    }
    for (int i = threadIdx.x; i < NID_NCLS * B; i += blockDim.x) {  // classes without tasks
      const int v = (int)(((unsigned)i * ((1048576u + (unsigned)B - 1u) / (unsigned)B)) >> 20);
      if (s_cts[v + 1] == s_cts[v]) hvs[i] = 0.0;
    }
    __syncthreads();
    const int g = threadIdx.x / tpr, tt = (threadIdx.x % tpr) * (pairs ? 2 : 1);
    double* Gjob = p.G + (size_t)job * p.g_stride * B;
    if (g < ng && s_bnd[g] < s_bnd[g + 1]) {
      int t = s_bnd[g];
      const int tend = s_bnd[g + 1];
      int v;
      {
        int lo = 0, hi = NID_NCLS;
        while (hi - lo > 1) {
          const int mid = (lo + hi) >> 1;
          if (s_cts[mid] <= t) lo = mid; else hi = mid;
        }
        v = lo;
      }
      int cend = s_cts[v + 1];
      bool multi = cend - s_cts[v] > NID_ASM_CHUNK;
      int seg0 = t, nxt = min(cend, seg0 + NID_ASM_CHUNK);
      const double* gp = Gjob + (size_t)t * B + tt;
      double a0 = 0.0, a1 = 0.0;
      auto close_segment = [&]() {
        double* dst = multi ? Gjob + (size_t)seg0 * B + tt : hvs + v * B + tt;
        if (pairs) *reinterpret_cast<double2*>(dst) = make_double2(a0, a1);
        else *dst = a0;
        a0 = 0.0; a1 = 0.0;
      };
      auto next_segment = [&]() {
        seg0 = nxt;
        if (nxt == cend) {
          do v++; while (s_cts[v + 1] == s_cts[v]);  // (a later class has rows: seg0 < tend)
          cend = s_cts[v + 1];
          multi = cend - s_cts[v] > NID_ASM_CHUNK;
        }
        nxt = min(cend, seg0 + NID_ASM_CHUNK);
      };
      if (pairs) {
        while (t < tend) {
          const int rem = tend - t;
          double2 x[8];
#pragma unroll
          for (int i = 0; i < 8; i++) x[i] = (i < rem) ? *reinterpret_cast<const double2*>(gp + i * B) : make_double2(0.0, 0.0);
#pragma unroll
          for (int i = 0; i < 8; i++) {
            if (i < rem) {
              if (t + i >= nxt) { close_segment(); next_segment(); }
              a0 += x[i].x; a1 += x[i].y;
            }
          }
          t += 8;
          gp += 8 * B;
        }
      } else {
        while (t < tend) {
          const int rem = tend - t;
          double x[NID_ASM_BATCH];
#pragma unroll
          for (int i = 0; i < NID_ASM_BATCH; i++) x[i] = (i < rem) ? __ldcs(gp + i * B) : 0.0;  // (read once: evict-first)
#pragma unroll
          for (int i = 0; i < NID_ASM_BATCH; i++) {
            if (i < rem) {
              if (t + i >= nxt) { close_segment(); next_segment(); }
              a0 += x[i];
            }
          }
          t += NID_ASM_BATCH;
          gp += NID_ASM_BATCH * B;
        }
      }
      close_segment();
    }
    __syncthreads();  // (the chunk sums this CTA parked in G are visible to all of its threads)
    if (g < ng) {
      for (int v = g; v < NID_NCLS; v += ng) {
        const int m = s_cts[v + 1] - s_cts[v];
        if (m <= NID_ASM_CHUNK) continue;
        const int nch = (m + NID_ASM_CHUNK - 1) / NID_ASM_CHUNK;
        const double* gp = Gjob + (size_t)s_cts[v] * B + tt;
        double a0 = 0.0, a1 = 0.0;
        for (int j0 = 0; j0 < nch; j0 += 8) {
          double2 x[8];
#pragma unroll
          for (int i = 0; i < 8; i++) {
            x[i] = make_double2(0.0, 0.0);
            if (j0 + i < nch) {
              const double* q = gp + (size_t)(j0 + i) * NID_ASM_CHUNK * B;
              if (pairs) x[i] = __ldcg(reinterpret_cast<const double2*>(q));
              else x[i].x = __ldcg(q);
            }
          }
#pragma unroll
          for (int i = 0; i < 8; i++)
            if (j0 + i < nch) { a0 += x[i].x; a1 += x[i].y; }
        }
        if (pairs) *reinterpret_cast<double2*>(hvs + v * B + tt) = make_double2(a0, a1);
        else hvs[v * B + tt] = a0;
      }
    }
  }
  __syncthreads();
  // ---- P_j: item (kk, r, t) sums the classes of span r-kk (in class order: the summation order is part of the result)
  {
    const unsigned mdiv = (1048576u + (unsigned)B - 1u) / (unsigned)B;  // idx / B == (idx * mdiv) >> 20 for idx < 2^20 / B
    for (int item = threadIdx.x; item < 4 * BB; item += blockDim.x) {
      const int kk = item / BB, idx = item - kk * BB;
      {
        const int r = (int)(((unsigned)idx * mdiv) >> 20), tt = idx - r * B;
        const int k = r - kk;
        double a = 0.0;
        if (k >= 0 && k < NS) {
          const int vlo = s_span[k], vhi = s_span[k + 1];
          const double* ph = hvs + vlo * B + tt;
          int n = vhi - vlo;
          if (NID_FEW_BINS(B)) {
            const double* pw = wl + 4 * vlo + kk;
            for (; n >= 4; n -= 4, pw += 16, ph += 4 * B) {
              a = fma(pw[0], ph[0], a); a = fma(pw[4], ph[B], a); a = fma(pw[8], ph[2 * B], a); a = fma(pw[12], ph[3 * B], a);
            }
            for (; n > 0; n--, pw += 4, ph += B) a = fma(pw[0], ph[0], a);
          } else {  // many bins: the 8 KB copy of the weight table would cost a resident CTA per SM
            const double* pw = p.lut_w + 4 * vlo + kk;
            for (; n > 0; n--, pw += 4, ph += B) a = fma(__ldg(pw), ph[0], a);
          }
        }
        part[kk * BB + idx] = a;
      }
    }
  }
  // Every sum below has ONE order whatever the CTA size (the 128-, 256- and 1024-thread variants of this kernel -- the
  // last one for a handful of evaluations in flight -- produce the same bits):
  // ---- P_t: ngt = max(1, 128 / B) groups; group g sums classes g, g + ngt, ... in order, the groups are then added in order
  const int ngt = max(1, 128 / B);
  if ((int)threadIdx.x < ngt * B) {
    const int g = threadIdx.x / B, tt = threadIdx.x % B;
    double a = 0.0;
    for (int v = g; v < NID_NCLS; v += ngt) a += hvs[v * B + tt];
    red[threadIdx.x] = a;
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < BB; idx += blockDim.x) {
    const double a = ((part[idx] + part[BB + idx]) + part[2 * BB + idx]) + part[3 * BB + idx];
    const double q = a / (double)nc;
    Pall[idx] = q;
    const double lg = (q < kSigma) ? 0.0 : log2(q);
    part[BB + idx] = -(q * lg);                 // entropy term of this entry (slots idx of the four planes are this thread's)
    part[idx] = (q < kSigma) ? 0.0 : 1.0 + lg;  // 1 + log2 P_j for the tables below
  }
  if ((int)threadIdx.x >= NT - B) {  // the last B threads (idle in the loop above for B <= 22)
    const int tt = threadIdx.x - (NT - B);
    double a = 0.0;
    for (int g = 0; g < ngt; g++) a += red[g * B + tt];
    const double q = a / (double)nc;
    Pall[BB + tt] = q;
    const double lg = (q < kSigma) ? 0.0 : log2(q);
    red[B + tt] = -(q * lg);                    // entropy term of bin tt (column tt of red belongs to this thread)
    red[tt] = (q < kSigma) ? 0.0 : 1.0 + lg;
  }
  __syncthreads();
  // ---- H_j: 128 partial sums (partial j takes the terms j, j + 128, ... in order), an xor tree inside each of the four
  // warps, the four warp sums in order. H_t: the same with one warp's worth of partials.
  {
    double ej = 0.0, et = 0.0;
    if (threadIdx.x < 128) {
      for (int idx = threadIdx.x; idx < BB; idx += 128) ej += part[BB + idx];
      if (threadIdx.x < 32)
        for (int tt = threadIdx.x; tt < B; tt += 32) et += red[B + tt];
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        ej += __shfl_xor_sync(0xffffffffu, ej, off);
        et += __shfl_xor_sync(0xffffffffu, et, off);
      }
      if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = ej;
      if (threadIdx.x == 0) scratch[4] = et;
    }
  }
  __syncthreads();
  const double Hj = ((scratch[0] + scratch[1]) + scratch[2]) + scratch[3];
  const double Ht = scratch[4];
  const double Href = p.href[pair * p.ncell + c];
  if (threadIdx.x == 0) {
    p.ht[o] = Ht; p.hj[o] = Hj;
    p.err[o] = (2 * Hj - Href - Ht) / Hj;
  }
  __syncthreads();
  if (p.hist) for (int i = threadIdx.x; i < BB + B; i += blockDim.x) p.hist[o * (BB + B) + i] = Pall[i];
  if (want_jac) {
    const double s_over = ((double)(B - 3) / 255.0) / ((double)nc * Hj * Hj);
    const double coefJ = -s_over * (Ht + Href);
    const double coefT = s_over * Hj;
    const int BP = wv_row(B);
    const unsigned mdiv = (1048576u + (unsigned)B - 1u) / (unsigned)B;
    double* wv = p.wv + o * (size_t)wv_stride(B);
    for (int i = threadIdx.x; i < BB; i += blockDim.x) {
      const int r = (int)(((unsigned)i * mdiv) >> 20);
      wv[r * BP + (i - r * B)] = part[i] * coefJ;
    }
    if ((int)threadIdx.x < B) wv[B * BP + threadIdx.x] = red[threadIdx.x] * coefT;
  }
}

__global__ void __launch_bounds__(NID_ASM_THREADS, NID_ASM_MINB) k_assemble(EvalParams p, int want_jac) {
  assemble_body<NID_ASM_THREADS>(p, want_jac);
}
__global__ void __launch_bounds__(NID_ASM_SMALL, 2 * NID_ASM_MINB) k_assemble_small(EvalParams p, int want_jac) {
  assemble_body<NID_ASM_SMALL>(p, want_jac);
}
// a handful of evaluations in flight (a lone LM solve): fewer CTAs than SMs, so every cell gets a whole SM's worth of threads
#define NID_ASM_WIDE 1024
__global__ void __launch_bounds__(NID_ASM_WIDE, 1) k_assemble_wide(EvalParams p, int want_jac) {
  assemble_body<NID_ASM_WIDE>(p, want_jac);
}

// Assembly for small cells (the reference's default 16x16 cells hold ~1200 pixels, i.e. ~130 task rows and at most a
// handful of pixels per class): one WARP per (cell, job) and no block barrier. Lane t owns bin t of P_t and column t of
// P_j; the warp streams the cell's task rows in task order, eight in flight, and a row of class v adds
// w_ref,v[m] * row[t] to P_j[k_r(v)+m][t] (types_six_dof_expmap.cpp:598-601 summed per task instead of per pixel).
// Same outputs as assemble_body (entropies, err, scaled log tables); the CTA-per-cell version spends its time on the
// 257-class bookkeeping and six barriers, which only pays off when a cell has thousands of task rows.
// Fixed per geometry (cells under NID_ASM_SMALL_PX pixels and at most 32 bins), so results never depend on the batch.
#define NID_ASMW_WARPS 8
#ifndef NID_ASMW_BATCH
#define NID_ASMW_BATCH 4  // task rows a lane keeps in flight (16x16 cells: 1.68 us per evaluation with 4, 1.70 with 6, 1.81 with 8, 2.08 with 12)
#endif
#ifndef NID_ASMW_MINB
#define NID_ASMW_MINB 4
#endif
#ifndef NID_ASMW_BATCH_LAT
#define NID_ASMW_BATCH_LAT 16
#endif
// Lanes are (g, t) = (lane / B, lane % B): NG = 32 / B sub-groups each stream every NG-th task row of the cell into
// their own copy of P_j / P_t (rows are B doubles, so one load instruction fetches NG whole rows); the copies are
// added in sub-group order at the end. Task order within a sub-group and sub-group order are fixed: deterministic.
// BATCH: task rows a lane keeps in flight -- NID_ASMW_BATCH when the device is full (more resident warps matter more),
// NID_ASMW_BATCH_LAT for a handful of evaluations (a lone solve: fewer dependent round trips per warp); same bits.
template <int BATCH>
__global__ void __launch_bounds__(NID_ASMW_WARPS * 32, BATCH > 8 ? 1 : NID_ASMW_MINB) k_assemble_warp(EvalParams p, int want_jac, int n_jobs) {
  extern __shared__ __align__(16) double sm[];  // per warp: NG copies of P_j as [B][B] (+ one row of P_t each)
  const int B = p.bins, BB = B * B;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int unit = blockIdx.x * NID_ASMW_WARPS + warp;
  if (unit >= n_jobs * p.ncell) return;
  const int c = unit % p.ncell, job = job_at(p, unit / p.ncell);
  const int pair = p.job_pair[job];
  const int nc = p.n_c[pair * p.ncell + c];
  const size_t o = (size_t)job * p.ncell + c;
  if (nc < NID_MIN_CELL_POINTS) {
    if (lane == 0) { p.ht[o] = nan(""); p.hj[o] = nan(""); p.err[o] = nan(""); }
    return;
  }
  const int NG = 32 / B;                 // sub-groups (1 for more than 16 bins)
  const int g = lane / B, t = lane - g * B;
  const bool mine = g < NG;              // lanes beyond NG * B idle
  const int stride = BB + B;             // one copy: P_j [B][B] | P_t [B]
  double* cp = sm + (size_t)warp * NG * stride;
  for (int i = lane; i < NG * stride; i += 32) cp[i] = 0.0;
  __syncwarp();
  double* Pj = cp + (mine ? g : 0) * stride + t;  // Pj[r * B]: column t of the sub-group's copy
  double pt = 0.0;
  // the rows a lane sees are ordered by class, hence by reference span: the four weighted sums of a span stay in registers
  // and go to the span's four rows of P_j when the span changes (13 times per cell at 16 bins instead of once per row)
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  int cur = -1;
  const int t0 = p.cell_task_start[pair * (p.ncell + 1) + c], t1 = p.cell_task_start[pair * (p.ncell + 1) + c + 1];
  // the lane's rows are t0 + g, t0 + g + NG, ...: one pointer per array, stepped by constant strides
  const unsigned short* tcp = p.task_cls + (size_t)pair * p.max_tasks + t0 + g;
  const double* gp = p.G + ((size_t)job * p.g_stride + t0 + g) * B + t;
  const int rstep = NG * B;
  for (int tb = t0; tb < t1; tb += BATCH * NG, tcp += BATCH * NG, gp += BATCH * rstep) {
    double x[BATCH];
    int cls[BATCH];
#pragma unroll
    for (int i = 0; i < BATCH; i++) {
      const bool in = mine && tb + i * NG + g < t1;
      x[i] = in ? __ldcs(gp + i * rstep) : 0.0;  // (read once: evict-first)
      cls[i] = in ? (int)__ldg(tcp + i * NG) : 256;
    }
#pragma unroll
    for (int i = 0; i < BATCH; i++) {
      pt += x[i];
      if (cls[i] < 256) {  // (class 256: valid points without a reference sample count in P_t only)
        const int k = __ldg(p.lut_k + cls[i]);
        if (k != cur) {
          if (cur >= 0) {
            double* q = Pj + cur * B;
#pragma unroll
            for (int m = 0; m < 4; m++) { q[m * B] += acc[m]; acc[m] = 0.0; }
          }
          cur = k;
        }
        const double2* w = reinterpret_cast<const double2*>(p.lut_w + 4 * cls[i]);  // (32-byte rows)
        const double2 w01 = __ldg(w), w23 = __ldg(w + 1);
        acc[0] = fma(w01.x, x[i], acc[0]); acc[1] = fma(w01.y, x[i], acc[1]);
        acc[2] = fma(w23.x, x[i], acc[2]); acc[3] = fma(w23.y, x[i], acc[3]);
      }
    }
  }
  if (cur >= 0) {
    double* q = Pj + cur * B;
#pragma unroll
    for (int m = 0; m < 4; m++) q[m * B] += acc[m];
  }
  if (mine) cp[g * stride + BB + t] = pt;
  __syncwarp();
  // add the copies in sub-group order: lane (r-chunk) ... every lane sums whole entries
  for (int i = lane; i < stride; i += 32) {
    double a = cp[i];
    for (int k = 1; k < NG; k++) a += cp[k * stride + i];
    cp[i] = a;
  }
  __syncwarp();
  // normalise, entropies (computeH.cu:261-300); the table 1 + log2 P replaces P in place
  double ej = 0.0, et = 0.0;
  const double dn = (double)nc;
  double* hist = p.hist ? p.hist + o * (size_t)(BB + B) : nullptr;
  for (int i = lane; i < stride; i += 32) {
    const double q = cp[i] / dn;
    const double lg = (q < kSigma) ? 0.0 : log2(q);
    if (i < BB) ej -= q * lg; else et -= q * lg;
    cp[i] = (q < kSigma) ? 0.0 : 1.0 + lg;
    if (hist) hist[i] = q;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    ej += __shfl_xor_sync(0xffffffffu, ej, off);
    et += __shfl_xor_sync(0xffffffffu, et, off);
  }
  const double Hj = ej, Ht = et;
  const double Href = p.href[pair * p.ncell + c];
  if (lane == 0) {
    p.ht[o] = Ht; p.hj[o] = Hj;
    p.err[o] = (2 * Hj - Href - Ht) / Hj;
  }
  __syncwarp();
  if (want_jac) {
    const double s_over = ((double)(B - 3) / 255.0) / ((double)nc * Hj * Hj);
    const double coefJ = -s_over * (Ht + Href);
    const double coefT = s_over * Hj;
    const int BP = wv_row(B);
    const unsigned mdiv = (1048576u + (unsigned)B - 1u) / (unsigned)B;
    double* wv = p.wv + o * (size_t)wv_stride(B);
    for (int i = lane; i < stride; i += 32) {
      const int r = (int)(((unsigned)i * mdiv) >> 20);  // (i >= BB: r = B, the row of V)
      wv[r * BP + (i - r * B)] = cp[i] * (i < BB ? coefJ : coefT);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Pass 2: per task the partial of  J[a] = sum_i g_i[a] * c_i,  c_i = q0 + f_i (q1 + f_i q2) with the
// quadratic of the pixel's (class, span); c_i = 0 at ub == 0 exactly (the reference's BsplineDer quirk).
// Pass-2 pixel by the reference's literal sequence: exact (u, v) for the cached intensity
// (types_six_dof_expmap.cpp:562-575), the second projection fx*(x/z)+cx for the Jacobian bounds test and the
// four gradient samples (:407-435). Taken when (u, v) is within 2^-24 of an integer, on saturated plateaus,
// and in the first image row / column, where (int)(u-1) truncates towards zero so that the five bilinear
// samples do not share their fractions. out: {x/z, y/z, 1/z, clamped ic, 2 gx, 2 gy}; returns the Jacobian validity.
template <bool PTS>
__device__ __noinline__ bool jac_pixel_literal(const double* __restrict__ T1g, const double* __restrict__ T0g,
                                               const double* __restrict__ camg, int rows, int cols,
                                               const uint8_t* __restrict__ im, double a0, double a1, double a2, unsigned id,
                                               double* out6) {
  double e[5];
  exact_uv<PTS>(T1g, T0g, camg, a0, a1, a2, id, e);
  const Cam cam{camg[0], camg[1], camg[2], camg[3]};
  const double u = e[3], v = e[4];
  double u2, v2;
  project_jac(cam, e[0], e[1], e[2], u2, v2);
  if (!inb_cost(u, v, rows, cols) || !inb_jac(u2, v2, rows, cols)) return false;
  const double iz = 1.0 / e[2];
  out6[0] = e[0] * iz; out6[1] = e[1] * iz; out6[2] = iz;
  out6[3] = clamp_intensity(interp_u8(im, cols, u, v));
  out6[4] = interp_u8(im, cols, u2 + 1.0, v2) - interp_u8(im, cols, u2 - 1.0, v2);
  out6[5] = interp_u8(im, cols, u2, v2 + 1.0) - interp_u8(im, cols, u2, v2 - 1.0);
  return true;
}

// 2^52 + v as a double (v < 2^32): differences of two such values are exact small integers
__device__ __forceinline__ double tapd(unsigned v) { return __hiloint2double(0x43300000, (int)v); }

// Pass 2 on W pixels of a group at once; acc[6] are the lane's Jacobian partial sums.
// wq: the lane's folded class table (fold_table), element t at wq[t * T].
template <bool PTS, int W, int T>
__device__ __forceinline__ void jac_pixels(const double* __restrict__ g, const ExactSrc& xs, int rows, int cols,
                                           const Group<PTS>& G, int j0, cudaTextureObject_t tex2,
                                           const uint8_t* __restrict__ im1, double s, int NS, double hfx, double hfy,
                                           const double* __restrict__ wq, double acc[6]) {
  Px r[W];
#pragma unroll
  for (int j = 0; j < W; j++) front<PTS, false>(g, rows, cols, G.a0[j0 + j], G.a1[j0 + j], G.a2[j0 + j], G.id[j0 + j], r[j]);
  uint4 t[W];
#pragma unroll
  for (int j = 0; j < W; j++) t[j] = gather_u32(tex2, r[j].ix, r[j].iy);
#pragma unroll
  for (int j = 0; j < W; j++) {
    // texel = I | (Gx+256) << 8 | (Gy+256) << 17; the biases cancel in the differences
    const double two52 = 4503599627370496.0;
    const double i00 = tapd(t[j].w & 0xffu), i01 = tapd(t[j].z & 0xffu), i10 = tapd(t[j].x & 0xffu), i11 = tapd(t[j].y & 0xffu);
    const double x00 = tapd((t[j].w >> 8) & 0x1ffu), x01 = tapd((t[j].z >> 8) & 0x1ffu);
    const double x10 = tapd((t[j].x >> 8) & 0x1ffu), x11 = tapd((t[j].y >> 8) & 0x1ffu);
    const double y00 = tapd(t[j].w >> 17), y01 = tapd(t[j].z >> 17), y10 = tapd(t[j].x >> 17), y11 = tapd(t[j].y >> 17);
    double ic = bilinear_fast(r[j].dx, r[j].dy, i00 - two52, i01 - i00, i10 - two52, i11 - i10);
    double gx2 = bilinear_fast(r[j].dx, r[j].dy, x00 - (two52 + 256.0), x01 - x00, x10 - (two52 + 256.0), x11 - x10);
    double gy2 = bilinear_fast(r[j].dx, r[j].dy, y00 - (two52 + 256.0), y01 - y00, y10 - (two52 + 256.0), y11 - y10);
    // rare: undecided by the fast path, saturated plateau, or first image row / column
    const bool sat = (t[j].w & t[j].z & t[j].x & t[j].y & 0xffu) == 0xffu;
    if (r[j].fix || (r[j].jac && (sat || r[j].ix < 1 || r[j].iy < 1))) {
      double o6[6];
      r[j].jac = jac_pixel_literal<PTS>(xs.T1, xs.T0, xs.cam, rows, cols, im1, G.a0[j0 + j], G.a1[j0 + j], G.a2[j0 + j], G.id[j0 + j], o6);
      if (r[j].jac) {
        r[j].xn = o6[0]; r[j].yn = o6[1]; r[j].rz = o6[2];
        ic = o6[3]; gx2 = o6[4]; gy2 = o6[5];
      }
    }
    const double ub = r[j].jac ? ic * s : 0.0;
    const int k = min((int)ub, NS - 1);  // 0 <= ub <= NS (== NS only by rounding)
    const double f = ub - u2d((unsigned)k);
    // c_i = sum_m N'_{k+m}(u_i) Wv[k+m] = sum_m U'_m(f) W^v[k+m]: uniform cubic derivative, folded class table
    const double dw0 = fma(f, fma(f, -0.5, 1.0), -0.5);
    const double dw1 = f * fma(f, 1.5, -2.0);
    const double dw2 = fma(f, fma(f, -1.5, 1.0), 0.5);
    const double dw3 = 0.5 * f * f;
    const double* q = wq + k * T;
    double ci = fma(dw3, q[3 * T], fma(dw2, q[2 * T], fma(dw1, q[T], dw0 * q[0])));
    if (ub == 0.0) ci = 0.0;  // the reference's BsplineDer quirk
    if (!r[j].jac) continue;  // (a padding slot may carry z = 0 and non-finite coordinates)
    // d(u,v)/d(xi), types_six_dof_expmap.cpp:438-450, in normalised coordinates xn = x/z, yn = y/z
    const double iz = r[j].rz, xn = r[j].xn, yn = r[j].yn;
    const double a = ci * gx2 * hfx, b = ci * gy2 * hfy;
    const double xy = xn * yn;
    acc[0] = fma(-b, fma(yn, yn, 1.0), fma(-a, xy, acc[0]));
    acc[1] = fma(b, xy, fma(a, fma(xn, xn, 1.0), acc[1]));
    acc[2] = fma(b, xn, fma(-a, yn, acc[2]));
    const double aiz = a * iz, biz = b * iz;
    acc[3] += aiz;
    acc[4] += biz;
    acc[5] = fma(-yn, biz, fma(-xn, aiz, acc[5]));
  }
}

// grid (jobs of this launch, ceil(max_slices/(T/32))), T = 32..128 threads.
template <bool PTS, int NG, int T, bool BULK>
__global__ void __launch_bounds__(T) __maxnreg__(BULK ? NID_JAC_REGS_SMALL : 65536 / (NID_JAC_WARPS * 32))
k_jac_sell(const __grid_constant__ EvalParams p, const __grid_constant__ GeoTable<NG> gt) {
  extern __shared__ __align__(16) double sm[];
  const int B = p.bins, NS = B - 3;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int job = gt.job[NID_BLK_JOB], pair = gt.pair[NID_BLK_JOB];
  const double* g = gt.g[NID_BLK_JOB];
  // shared: the lanes' class tables W^v [B][T] | per-warp log tables W|V (prologue only)
  const int slice = NID_BLK_CHUNK * (T >> 5) + warp;
  if (slice >= gt.nsl[NID_BLK_JOB]) return;  // (no block-wide barrier below)
  const int* so = p.sl_off + (size_t)pair * (p.max_slices + 1) + slice;
  const int off0 = so[0], ngroups = (so[1] - off0) >> 7;
  // (the lane's task descriptor from the slice's own table: no sl_task -> tasks chain of dependent loads in front of the
  // class table; 0 = no task)
  const int desc = p.sl_desc[((size_t)pair * p.max_slices + slice) * 32 + lane];
  const int task = desc != 0 ? 0 : -1;
  // the slice is as long as its first lane's task (tasks are dealt longest first): when that task ends in the first half
  // of its last group of four, no lane has a pixel in the second half and the last step of the slice is skipped
  // (small cells: slices are 2.6 groups long on average, half of them end that way)
  const bool half_last = (((__shfl_sync(0xffffffffu, desc, 0) & 0x1ff) - 1) & 3) < 2;
  double* wq = sm + threadIdx.x;  // wq[t * T]
  // the first group of pixels is requested before the prologue, so that it arrives while the class table is built
  const size_t sbase = (size_t)pair * p.sell_cap + off0 + lane * 4;
  const double* q0 = p.sd0 + sbase;
  const double* q1 = PTS ? p.sd1 + sbase : nullptr;
  const double* q2 = PTS ? p.sd2 + sbase : nullptr;
  const unsigned* qi = p.sid + sbase;
  Group<PTS> G;
  G.load(q0, q1, q2, qi, 0);
  // ---- class table of the lane's task (class v, cell of the slice):
  //   Wv[t] = V[t] + sum_kk w_ref,v[kk] W[k_r(v)+kk][t]     (class 256: V only)
  // from the cell's scaled log tables W|V (k_assemble), staged per warp with rows padded to B+1, then folded onto
  // the uniform basis (fold_table). Pass 2 then needs  c_i = sum_m U'_m(f_i) * W^v[k_i+m]  per pixel
  // (types_six_dof_expmap.cpp:467-528 re-associated).
  {
    // (the slice's cell comes from its own small table, so that the table loads below do not wait for the
    // sl_task -> tasks chain of dependent loads)
    const int cell = p.sl_cell[(size_t)pair * p.max_slices + slice];
    const double* wvg = p.wv + ((size_t)job * p.ncell + cell) * (size_t)wv_stride(B);
    // few bins: the cell's block W | V (rows of B + 1 doubles, see wv_row) is staged per warp. Short slices (small cells,
    // p.stage_bulk): as ONE bulk copy (cp.async.bulk, executed by the copy engine: no registers, no per-lane loads or
    // address arithmetic) that completes on the warp's mbarrier while the lanes fetch their task descriptors and
    // reference weights -- measured at 16x16 cells: 6.53 -> 6.13 us per evaluation
    double* Ww = sm + B * T + warp * wv_stride(B);
    unsigned long long* bar = reinterpret_cast<unsigned long long*>(sm + B * T + (T >> 5) * wv_stride(B)) + warp;
    constexpr bool bulk = BULK;  // (a launch-time choice, compiled in: the kernel has no register to spare for both paths)
    if (bulk) {
      if (lane == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        mbar_expect_tx(bar, (unsigned)(wv_stride(B) * sizeof(double)));
        bulk_g2s(Ww, wvg, (unsigned)(wv_stride(B) * sizeof(double)), bar);
      }
      __syncwarp();
    }
    const int cls = (desc >> 9) & 0x1ff;
    double wr[4] = {0.0, 0.0, 0.0, 0.0};
    int kr = 0;
    if (task >= 0 && cls < 256) {
      kr = p.lut_k[cls];
#pragma unroll
      for (int kk = 0; kk < 4; kk++) wr[kk] = p.lut_w[4 * cls + kk];
    }
    if (NID_FEW_BINS(B)) {
      // the cell's tables staged per warp (rows padded to B+1): the lanes then read their four rows bank-conflict free
      const int BP = B + 1;
      const double* Vw = Ww + B * BP;
      if (bulk) {
        mbar_wait(bar, 0u);  // the block has landed (every lane observes the barrier's phase itself)
      } else {
        // long slices (large cells): the prologue is a small part of the slice and the copy engine's latency exceeds
        // that of the lanes' own loads (measured at 4x4 cells: 3.81 us per evaluation with the bulk copy, 3.70 without)
        for (int i = lane; i < B * BP + B; i += 32) Ww[i] = wvg[i];
        __syncwarp();
      }
      if (task >= 0) {
        const double* Wr = Ww + kr * BP;
        for (int t = 0; t < B; t++) {
          double a = Vw[t];
#pragma unroll
          for (int kk = 0; kk < 4; kk++) a += wr[kk] * Wr[kk * BP + t];
          wq[t * T] = a;
        }
      }
    } else if (task >= 0) {
      // many bins: no staging area (it would cost a resident CTA per SM); the rows come through L1
      const double* Wr = wvg + kr * B;
      for (int t = 0; t < B; t++) {
        double a = __ldg(wvg + B * B + t);
#pragma unroll
        for (int kk = 0; kk < 4; kk++) a += wr[kk] * __ldg(Wr + kk * B + t);
        wq[t * T] = a;
      }
    }
    if (task >= 0) fold_table(wq, T, B);
  }
  const cudaTextureObject_t tex2 = (cudaTextureObject_t)gt.tex[NID_BLK_JOB];
  const uint8_t* im1 = p.im1 + (size_t)pair * p.N;
  const ExactSrc xs{p.poses + 16 * job, p.Twc0 + 16 * pair, p.cam + 4 * pair};
  const double s = (double)NS / 255.0;
  const double hfx = 0.5 * g[16], hfy = 0.5 * g[17];  // the /2 of the central differences folded in
  double acc[6] = {0, 0, 0, 0, 0, 0};
  for (int gi = 0; gi < ngroups; gi++) {
    Group<PTS> Gn = G;
    if (gi + 1 < ngroups) Gn.load(q0, q1, q2, qi, (size_t)(gi + 1) * 128);
#if NID_PREFETCH_L2 > 0
    if (gi + 1 + NID_PREFETCH_L2 < ngroups) {
      const size_t po = (size_t)(gi + 1 + NID_PREFETCH_L2) * 128;
      asm volatile("prefetch.global.L2 [%0];" ::"l"(q0 + po));
      asm volatile("prefetch.global.L2 [%0];" ::"l"(qi + po));
    }
#endif
#pragma unroll
    for (int j0 = 0; j0 < 4; j0 += NID_JAC_W) {
      if (BULK && j0 >= 2 && half_last && gi + 1 == ngroups) break;  // (small cells only: 5.07 -> 4.98 us; at 4x4 cells 3.43 -> 3.48)
      jac_pixels<PTS, NID_JAC_W, T>(g, xs, p.rows, p.cols, G, j0, tex2, im1, s, NS, hfx, hfy, wq, acc);
    }
    G = Gn;
  }
  // one partial per slice: fixed-order butterfly over the 32 lanes (lanes without a task hold zeros)
#pragma unroll
  for (int k = 0; k < 6; k++) {
    double vv = acc[k];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) vv += __shfl_xor_sync(0xffffffffu, vv, off);
    acc[k] = vv;
  }
  if (lane < 6) {
    double vv = acc[0];
#pragma unroll
    for (int k = 1; k < 6; k++) vv = lane == k ? acc[k] : vv;
    p.jpart[((size_t)job * p.max_slices + slice) * 6 + lane] = vv;
  }
}

// a8 tail of one (job, cell) by one warp: the slice partials of the cell summed in a fixed order -> der[6]
__device__ __forceinline__ void jac_tail_cell(const EvalParams& p, int job, int pair, int c, int lane) {
  double* der = p.der + ((size_t)job * p.ncell + c) * 6;
  if (p.n_c[pair * p.ncell + c] < NID_MIN_CELL_POINTS) {
    if (lane < 6) der[lane] = nan("");
    return;
  }
  const int s0 = p.cell_slice_start[pair * (p.ncell + 1) + c];
  const int s1 = p.cell_slice_start[pair * (p.ncell + 1) + c + 1];
  const double* jp = p.jpart + (size_t)job * p.max_slices * 6;
  double acc[6] = {0, 0, 0, 0, 0, 0};
  for (int t = s0 + lane; t < s1; t += 32) {
#pragma unroll
    for (int k = 0; k < 6; k++) acc[k] += jp[(size_t)t * 6 + k];
  }
#pragma unroll
  for (int k = 0; k < 6; k++) {
    double vv = acc[k];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) vv += __shfl_xor_sync(0xffffffffu, vv, off);
    if (lane == 0) der[k] = vv;
  }
}

// The same for geometries of many cells with few slices each (64 cells or more; chosen by geometry, so one context always
// sums the same way): component k of der[6] of one (job, cell) by one thread, in slice order. A cell has 5 slices at the
// reference's default geometry: a warp per cell with a butterfly per component is mostly idle lanes and shuffles there
// (0.19 -> 0.10 us per evaluation at 16x16 cells); with one cell of 300 slices it is the other way round (0.13 -> 0.34).
__device__ __forceinline__ void jac_tail_entry(const EvalParams& p, int job, int pair, int c, int k) {
  double* der = p.der + ((size_t)job * p.ncell + c) * 6;
  if (p.n_c[pair * p.ncell + c] < NID_MIN_CELL_POINTS) { der[k] = nan(""); return; }
  const int s0 = p.cell_slice_start[pair * (p.ncell + 1) + c];
  const int s1 = p.cell_slice_start[pair * (p.ncell + 1) + c + 1];
  const double* jp = p.jpart + ((size_t)job * p.max_slices + s0) * 6 + k;
  double acc = 0.0;
  int t = s0;
  for (; t + 8 <= s1; t += 8, jp += 48) {  // eight independent loads, then the ordered additions
    double v[8];
#pragma unroll
    for (int u = 0; u < 8; u++) v[u] = jp[6 * u];
#pragma unroll
    for (int u = 0; u < 8; u++) acc += v[u];
  }
  for (; t < s1; t++, jp += 6) acc += jp[0];
  der[k] = acc;
}

#define NID_TAIL_PER_THREAD(ncell) ((ncell) >= 64)
// one warp per (job, cell), or one thread per (job, cell, component)
__global__ void __launch_bounds__(256) k_jac_final_sorted(EvalParams p, int n_jobs) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (NID_TAIL_PER_THREAD(p.ncell)) {
    if (idx >= n_jobs * p.ncell * 6) return;
    const int k = idx % 6, c = (idx / 6) % p.ncell;
    const int job = job_at(p, idx / (6 * p.ncell));
    jac_tail_entry(p, job, p.job_pair[job], c, k);
  } else {
    const int wid = idx >> 5;
    if (wid >= n_jobs * p.ncell) return;
    const int job = job_at(p, wid / p.ncell), c = wid % p.ncell;
    jac_tail_cell(p, job, p.job_pair[job], c, threadIdx.x & 31);
  }
}
static int jac_final_blocks(const nid_ctx* c, int n) {
  const long long threads = NID_TAIL_PER_THREAD(c->ncell) ? (long long)n * c->ncell * 6 : (long long)n * c->ncell * 32;
  return (int)((threads + 255) / 256);
}

// the Gauss-Newton blocks of the launch's jobs written where the host reads them (see k_tail_gn)
__global__ void __launch_bounds__(128) k_gn_out(EvalParams p, double* __restrict__ gn_out) {
  gn_block(p, job_at(p, blockIdx.x), 1, gn_out);
}

// Latency mode of the LM driver: the Jacobian tail and the Gauss-Newton block of a job in ONE launch (one CTA per job:
// its warps finish the cells, then the block is summed exactly as k_gn does (gn_block)), written where the host reads it
// (gn_out may be pinned host memory: no copy is queued behind the kernel).
__global__ void __launch_bounds__(256) k_tail_gn(EvalParams p, double* __restrict__ gn_out) {
  const int job = job_at(p, blockIdx.x);
  const int pair = p.job_pair[job];
  for (int c = threadIdx.x >> 5; c < p.ncell; c += blockDim.x >> 5) jac_tail_cell(p, job, pair, c, threadIdx.x & 31);  // (at most 32 cells here)
  __syncthreads();  // (the der values this CTA wrote are visible to all of its threads)
  gn_block(p, job, 1, gn_out);
}

// Kernel-1 target texture: three stacked planes of 16-bit floats, rows [0,R) I, [R,2R) Gx/2, [2R,3R) Gy/2 with the
// central differences Gx = I(x+1,y) - I(x-1,y), Gy = I(x,y+1) - I(x,y-1) (types_six_dof_expmap.cpp:434-435); border
// texels use clamped neighbours and are never consumed (the first row / column takes the literal formula).
__global__ void k_pack_k1(int rows, int cols, const uint8_t* __restrict__ im, unsigned short* __restrict__ out) {
  const int N = rows * cols;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
    const int y = i / cols, x = i % cols;
    const int xm = max(x - 1, 0), xp = min(x + 1, cols - 1), ym = max(y - 1, 0), yp = min(y + 1, rows - 1);
    const int gx = (int)im[y * cols + xp] - (int)im[y * cols + xm];
    const int gy = (int)im[yp * cols + x] - (int)im[ym * cols + x];
    out[i] = __half_as_ushort(__float2half_rn((float)im[i]));
    out[N + i] = __half_as_ushort(__float2half_rn(0.5f * (float)gx));
    out[2 * N + i] = __half_as_ushort(__float2half_rn(0.5f * (float)gy));
  }
}

// ------------------------------------------------------------------------------------------------
// Kernel 1 on its own, batched over jobs (north_star kernel (1); parity + HBM roofline probe; the evaluation path
// fuses the same front end into both passes instead of storing its output). A streaming kernel:
//   in   the pair's depth plane, 2 B/px as the dataset's raw 16-bit values (metres = raw * factor, exact) or 8 B/px fp64
//   out  {I_c, g_x, g_y, valid} as one float4 per pixel (16 B/px), valid: 0 invalid, 1 cost only, 3 cost + Jacobian
// A CTA of 128 threads owns 512 consecutive pixels; thread t takes pixels t, t+128, t+256, t+384 of them, so every
// warp load is 32 consecutive depths and every warp store 512 contiguous bytes (evict-first: written once, never read
// here). The first version of this kernel was issue-bound at 217 instructions per pixel (profiles/r02_k1_*): two
// thirds of them unpacking and converting the twelve integer taps and re-deriving the viewing ray. Now:
//  * the target lives in a 16-bit-float gather texture of three stacked planes {I, Gx/2, Gy/2} (small integers and
//    half-integers: exact in fp16), so one gather per channel delivers four ready-made floats: no unpacking, no
//    integer-to-float conversion, and the /2 of the central differences is already in the texels;
//  * the ray d = M (cxn, cyn, 1) is affine in (col, row): it is evaluated once per thread and stepped by 128 columns
//    (three DADDs per pixel instead of ten fp64 operations and two conversions);
//  * the validity logic is branch-free bit arithmetic and full chunks skip the per-pixel range checks.
// fp64 is kept for what decides something -- SE3 warp, projection, the (int) truncation and the in-bounds tests,
// with the same exact fall-backs as pass 2 for (u, v) within 2^-24 of an integer, saturated footprints and the first
// image row / column -- and the three bilinear samples, whose results are stored as floats anyway, are evaluated in
// fp32 from the fp64 fractions. One Newton step on the reciprocal leaves (u, v) within 2^-36 of their exact values:
// far inside the 2^-24 guard band.
#ifndef NID_WS_MINB
#define NID_WS_MINB 8
#endif
// Kernel-1 pixel i by the reference's literal sequence (rare path; re-reads its depth): cost validity and intensity
// from (u, v), Jacobian validity and gradient from the second projection (types_six_dof_expmap.cpp:562-575, :407-435).
// out3 = {I_c, 2 g_x, 2 g_y}; returns valid bits (1 cost, 2 Jacobian).
template <bool U16>
__device__ __noinline__ unsigned warp_sample_literal(const EvalParams& p, int job, int pair, int i, const double* __restrict__ depth64,
                                                     const uint16_t* __restrict__ depth16, const double* __restrict__ factor_all,
                                                     float* out3) {
  const size_t pbase = (size_t)pair * p.N;
  const double z = U16 ? __dmul_rn((double)depth16[pbase + i], factor_all[pair]) : depth64[pbase + i];
  const int row = i / p.cols, col = i - row * p.cols;
  const unsigned id = ((unsigned)row << 16) | (unsigned)col;
  const double* T1 = p.poses + 16 * job;
  const double* T0 = p.Twc0 + 16 * pair;
  const double* camg = p.cam + 4 * pair;
  double e[5];
  exact_uv<false>(T1, T0, camg, z, 0.0, 0.0, id, e);
  out3[0] = 0.f; out3[1] = 0.f; out3[2] = 0.f;
  if (!inb_cost(e[3], e[4], p.rows, p.cols)) return 0u;
  const uint8_t* im1 = p.im1 + pbase;
  out3[0] = (float)clamp_intensity(interp_u8(im1, p.cols, e[3], e[4]));
  double o6[6];
  if (!jac_pixel_literal<false>(T1, T0, camg, p.rows, p.cols, im1, z, 0.0, 0.0, id, o6)) return 1u;
  out3[1] = (float)o6[4]; out3[2] = (float)o6[5];
  return 3u;
}
#ifndef NID_WS_W
#define NID_WS_W 4
#endif
// Geometry entries of this kernel (fill_geo_k1): [0..2] A, [3..5] B, [6..8] C with the ray d = A col + B row + C
// (rows 0 and 1 pre-multiplied by fx, fy), [9..11] translation (same scaling), [12..14] 128 A, [15..17] B - cols A
// (the step into the next image row), [18] cx, [19] cy.
template <int NG, bool U16>
__global__ void __launch_bounds__(128, NID_WS_MINB)
k_warp_sample_jobs(const __grid_constant__ EvalParams p, const __grid_constant__ GeoTable<NG> gt,
                   const double* __restrict__ depth64, const uint16_t* __restrict__ depth16,
                   const double* __restrict__ factor_all, float4* __restrict__ out) {
  constexpr int W = NID_WS_W;
  const int jb = blockIdx.x, cb_ = blockIdx.y;  // job index fast
  const int job = job_at(p, jb);
  const int pair = p.job_pair[job];
  const double* g = gt.g[jb];
  const int i0 = cb_ * (128 * W) + threadIdx.x;
  const bool full = (cb_ + 1) * (128 * W) <= p.N;  // (uniform per CTA)
  const size_t pbase = (size_t)pair * p.N;
  // depths first: W independent loads in flight
  double z[W];
  if (U16) {
    const double factor = factor_all[pair];
    unsigned raw[W];
#pragma unroll
    for (int j = 0; j < W; j++) raw[j] = (full || i0 + j * 128 < p.N) ? (unsigned)__ldcs(depth16 + pbase + i0 + j * 128) : 0u;
#pragma unroll
    for (int j = 0; j < W; j++) z[j] = __dmul_rn(u2d(raw[j]), factor);  // NID_pose_estimation.cpp:105-106, one rounding
  } else {
#pragma unroll
    for (int j = 0; j < W; j++) z[j] = (full || i0 + j * 128 < p.N) ? __ldcs(depth64 + pbase + i0 + j * 128) : 0.0;
  }
  int row = i0 / p.cols, col = i0 - row * p.cols;
  double d0, d1, d2;
  {
    const double fc = u2d((unsigned)col), fr = u2d((unsigned)row);
    d0 = fma(g[0], fc, fma(g[3], fr, g[6]));
    d1 = fma(g[1], fc, fma(g[4], fr, g[7]));
    d2 = fma(g[2], fc, fma(g[5], fr, g[8]));
  }
  // what survives the front end, per pixel: the footprint corner, the two fractions as floats, three flag bits
  // (1 cost-valid, 2 Jacobian-valid, 4 take the literal path); the rare paths re-read everything else
  int jxs[W], jys[W];
  unsigned flags = 0;
  float dxf[W], dyf[W];
  const int c3 = p.cols - 3, r3 = p.rows - 3;
#pragma unroll
  for (int j = 0; j < W; j++) {
    // depth outside [0.01, 100] is a NaN point in the reference (CudaPoints3d.cu:16-19)
    const unsigned valid = (z[j] >= 0.01) & (z[j] <= 100.0);
    const double x1 = fma(z[j], d0, g[9]), y1 = fma(z[j], d1, g[10]), z1 = fma(z[j], d2, g[11]);
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(z1));
    y = fma(y, fma(-z1, y, 1.0), y);
    const double u = fma(x1, y, g[18]), v = fma(y1, y, g[19]);
    const int jx = __double2int_rz(u), jy = __double2int_rz(v);  // NaN -> 0, saturating
    const double dx = u - u2d((unsigned)jx), dy = v - u2d((unsigned)jy);
    // with u, v not within 2^-24 of an integer the integer comparisons decide exactly like
    // `u>=0 && u+3<=cols && v>=0 && v+3<=rows` (types_six_dof_expmap.cpp:565; :433 with cols-1)
    const unsigned band = valid & ((unsigned)jx <= (unsigned)c3) & ((unsigned)jy <= (unsigned)r3);
    const unsigned safe = (unsigned)frac_is_safe(dx) & (unsigned)frac_is_safe(dy);
    const unsigned ok = band & safe & (jx < c3) & (jy < r3);
    const unsigned jac = ok & (jx < c3 - 1);
    const unsigned lit = (band & (safe ^ 1u)) | (ok & ((jx < 1) | (jy < 1)));  // undecided, or first row / column
    flags |= (ok | (jac << 1) | (lit << 2)) << (4 * j);
    jxs[j] = ok ? jx : 0; jys[j] = ok ? jy : 0;
    dxf[j] = (float)dx; dyf[j] = (float)dy;
    if (j + 1 < W) {
      col += 128;
      d0 += g[12]; d1 += g[13]; d2 += g[14];
      while (col >= p.cols) { col -= p.cols; d0 += g[15]; d1 += g[16]; d2 += g[17]; }
    }
  }
  const cudaTextureObject_t tex = p.k1tex[pair];
  float4* o = out + (size_t)job * p.N + i0;
#pragma unroll
  for (int j = 0; j < W; j++) {
    // one gather per plane: .w (ix,iy) .z (ix+1,iy) .x (ix,iy+1) .y (ix+1,iy+1)
    const float gxc = (float)(jxs[j] + 1), gyc = (float)(jys[j] + 1);
    const float4 I = tex2Dgather<float4>(tex, gxc, gyc, 0);
    const float4 X = tex2Dgather<float4>(tex, gxc, gyc + (float)p.rows, 0);
    const float4 Y = tex2Dgather<float4>(tex, gxc, gyc + (float)(2 * p.rows), 0);
    const float fx_ = dxf[j], fy_ = dyf[j];
    const float w11 = fx_ * fy_, w01 = fx_ - w11, w10 = fy_ - w11, w00 = (1.0f - fx_) - w10;
    float ic = fmaf(w11, I.y, fmaf(w10, I.x, fmaf(w01, I.z, w00 * I.w)));
    float gx = fmaf(w11, X.y, fmaf(w10, X.x, fmaf(w01, X.z, w00 * X.w)));
    float gy = fmaf(w11, Y.y, fmaf(w10, Y.x, fmaf(w01, Y.z, w00 * Y.w)));
    const unsigned f = flags >> (4 * j);
    unsigned vc = f & 1u, vj = (f >> 1) & 1u;
    const unsigned sat = fminf(fminf(I.x, I.y), fminf(I.z, I.w)) == 255.0f;
    if (((f >> 2) | (vc & sat)) & 1u) {
      if (full || i0 + j * 128 < p.N) {
        float r3_[3];
        const unsigned vv = warp_sample_literal<U16>(p, job, pair, i0 + j * 128, depth64, depth16, factor_all, r3_);
        vc = vv & 1u; vj = (vv >> 1) & 1u;
        ic = r3_[0]; gx = 0.5f * r3_[1]; gy = 0.5f * r3_[2];
      }
    }
    ic = vc ? ic : 0.f;
    gx = vj ? gx : 0.f; gy = vj ? gy : 0.f;
    const float fl = vc ? (vj ? 3.f : 1.f) : 0.f;
    if (full || i0 + j * 128 < p.N) __stcs(o + j * 128, make_float4(ic, gx, gy, fl));
  }
}

// ================================================================================================ launchers
int launch_count_classes(nid_ctx* c, int pair) {
  EvalParams p = make_params(c, 1);
  int g = (c->N + 255) / 256;
  if (g > c->sm_count * 8) g = c->sm_count * 8;
  k_count_classes<<<g, 256, 0, c->stream>>>(p, pair, c->cnt);
  NID_LAUNCH_CHECK(c, "k_count_classes");
  return NID_OK;
}

// pairs [pair0, pair0 + n), n <= c->setup_batch: tables on the device, then the regrouping scatter
int launch_layout_and_scatter(nid_ctx* c, int pair0, int n) {
  EvalParams p = make_params(c, 1);
  const int L = c->task_px;
  const dim3 gcell(c->ncell, n);
  k_layout_totals<<<gcell, NID_LAYOUT_THREADS, 0, c->stream>>>(pair0, c->ncell, L, c->cnt, c->lay_tot);
  NID_LAUNCH_CHECK(c, "k_layout_totals");
  k_layout_scan<<<n, 256, 0, c->stream>>>(p, pair0, c->lay_tot, c->lay_base, c->cell_task_start, c->cell_slice_start, c->ntasks,
                                         c->nslices, c->sl_off, c->d_flag + 1);
  NID_LAUNCH_CHECK(c, "k_layout_scan");
  k_layout_write<<<gcell, NID_LAYOUT_THREADS, 0, c->stream>>>(p, pair0, L, c->cnt, c->lay_base, c->tasks, c->task_pos, c->sl_task,
                                                             c->sl_off, c->sl_cell, c->cls_task_start);
  NID_LAUNCH_CHECK(c, "k_layout_write");
  const size_t sb = (size_t)pair0 * c->sell_cap;
  cudaError_t e = cudaMemsetAsync(c->sid + sb, 0xFF, sizeof(unsigned) * c->sell_cap * n, c->stream);
  if (e != cudaSuccess) return check_cuda(e, "memset sid");
  e = cudaMemsetAsync(c->sd0 + sb, 0, sizeof(double) * c->sell_cap * n, c->stream);
  if (e != cudaSuccess) return check_cuda(e, "memset sd0");
  const int nchunks = (c->rb * c->cb + 255) / 256;
  const dim3 grid(nchunks, c->ncell, n);
  k_chunk_count<<<grid, 256, 0, c->stream>>>(p, pair0, c->chunk_cnt);
  NID_LAUNCH_CHECK(c, "k_chunk_count");
  k_chunk_scan<<<dim3((c->ncell * NID_NCLS + 255) / 256, n), 256, 0, c->stream>>>(c->ncell, nchunks, c->chunk_cnt);
  NID_LAUNCH_CHECK(c, "k_chunk_scan");
  if (c->sell_points) {
    cudaMemsetAsync(c->sd1 + sb, 0, sizeof(double) * c->sell_cap * n, c->stream);
    cudaMemsetAsync(c->sd2 + sb, 0, sizeof(double) * c->sell_cap * n, c->stream);
    k_scatter_sell<true><<<grid, 256, 0, c->stream>>>(p, pair0, L, c->depth, c->task_pos, c->chunk_cnt, c->sd0, c->sd1, c->sd2, c->sid);
  } else {
    k_scatter_sell<false><<<grid, 256, 0, c->stream>>>(p, pair0, L, c->depth, c->task_pos, c->chunk_cnt, c->sd0, nullptr, nullptr, c->sid);
  }
  NID_LAUNCH_CHECK(c, "k_scatter_sell");
  return NID_OK;
}

// footprint-packed planes and packed gather texels of the targets of pairs [pair0, pair0 + n), n <= c->setup_batch
int launch_pack(nid_ctx* c, int pair0, int n) {
  int g = (c->N + 255) / 256;
  g = std::min(g, std::max(8, c->sm_count * 8 / n));
  k_pack_fp<<<dim3(g, n), 256, 0, c->stream>>>(c->rows, c->cols, pair0, c->im1, c->fp1);
  NID_LAUNCH_CHECK(c, "k_pack_fp");
  k_pack_tex<<<dim3(g, n), 256, 0, c->stream>>>(c->rows, c->cols, pair0, c->im1, c->d_pack);
  NID_LAUNCH_CHECK(c, "k_pack_tex");
  return NID_OK;
}

size_t hist_sell_smem(const nid_ctx* c, int T = 256) { return sizeof(double) * ((size_t)c->bins * T); }
size_t jac_sell_smem(const nid_ctx* c, int T = 128) {
  const size_t B = c->bins;
  // class tables [B][T] | per warp: the staged block W | V | per warp: its mbarrier (few bins)
  return sizeof(double) * (B * T + (NID_FEW_BINS(c->bins) ? (size_t)(T / 32) * (wv_stride(c->bins) + 1) : 0));
}

// Threads per CTA of the pixel kernels: the largest of 32..tmax that still gives every SM about two CTAs; a
// handful of jobs (a single LM solve) then spreads its slices over the whole GPU instead of a few dozen SMs.
static int pick_block(const nid_ctx* c, int ns, int n_jobs, int tmax) {
  for (int T = tmax; T > 32; T >>= 1)
    if ((long long)n_jobs * ((ns + T / 32 - 1) / (T / 32)) >= 2LL * c->sm_count) return T;
  return 32;
}
// cells of fewer than NID_ASM_SMALL_PX pixels take the warp assembly (at most 32 bins) or the 128-thread one
#ifndef NID_ASM_SMALL_PX
#define NID_ASM_SMALL_PX 8192
#endif
static bool assemble_small(const nid_ctx* c) { return (long long)c->rb * c->cb < NID_ASM_SMALL_PX; }
static bool assemble_warp(const nid_ctx* c) { return assemble_small(c) && c->bins <= 32; }
static size_t assemble_warp_smem(const nid_ctx* c) {
  return sizeof(double) * (size_t)NID_ASMW_WARPS * (32 / c->bins) * ((size_t)c->bins * c->bins + c->bins);
}
size_t assemble_smem(const nid_ctx* c, int threads) {
  return sizeof(double) * ((size_t)5 * c->bins * c->bins + c->bins + threads + (size_t)NID_NCLS * c->bins + (NID_FEW_BINS(c->bins) ? 1024 : 0));
}

// Host side of the geometry table: job s0 + i of js -> gt.g[i] from the host mirrors of its pose and pair, the pair's
// T_wc0 and intrinsics. pass1: rows 0 and 1 of M pre-multiplied by fx, fy.
template <int NG>
static void fill_geo(const nid_ctx* c, GeoTable<NG>& gt, const JobSet& js, int s0, int n, bool pass1) {
  for (int i = 0; i < n; i++) {
    const int job = js.h_list ? js.h_list[js.first + s0 + i] : js.first + s0 + i;
    const double* T1 = js.h_poses + 16 * (size_t)job;
    const int pair = js.h_pair[job];
    const double* T0 = c->h_Twc0.data() + 16 * (size_t)pair;
    const double* cam = c->h_cam.data() + 4 * (size_t)pair;
    double* g = gt.g[i];
    gt.job[i] = job; gt.pair[i] = pair;
    gt.nsl[i] = c->h_nslices[pair];
    gt.tex[i] = c->tex2.empty() ? 0ull : (unsigned long long)c->tex2[pair].tex;
    for (int col = 0; col < 4; col++)
      for (int r = 0; r < 3; r++) {
        double m;
        if (c->sell_points) m = T1[4 * col + r];
        else {
          m = T1[r] * T0[4 * col] + T1[4 + r] * T0[4 * col + 1] + T1[8 + r] * T0[4 * col + 2];
          if (col == 3) m += T1[12 + r];
        }
        if (pass1 && r < 2) m *= cam[r];
        g[3 * col + r] = m;
      }
    g[12] = 1.0 / cam[0]; g[13] = -cam[2] / cam[0]; g[14] = 1.0 / cam[1]; g[15] = -cam[3] / cam[1];
    g[16] = cam[0]; g[17] = cam[1]; g[18] = cam[2]; g[19] = cam[3];
  }
}

template <bool PTS, int NG>
static int launch_hist_chunks(nid_ctx* c, const EvalParams& p, int ns, const JobSet& js) {
  // (many bins: the rows take the shared memory that one-warp CTAs would need for 18 resident warps: 128-thread CTAs)
  const int T = pick_block(c, ns, js.n, c->bins > 20 ? 128 : NID_HIST_TMAX);
  const size_t sm = hist_sell_smem(c, T);
  for (int s0 = 0; s0 < js.n; s0 += NG) {
    const int n = std::min(NG, js.n - s0);
    GeoTable<NG> gt;
    fill_geo(c, gt, js, s0, n, true);
    EvalParams q = p;
    q.job0 = js.first + s0;
    const dim3 grid = NID_GRID(n, (ns + T / 32 - 1) / (T / 32));
    switch (T) {
      case 256: k_hist_sell<PTS, NG, 256><<<grid, 256, sm, js.stream>>>(q, gt); c->last_hist_func = (const void*)k_hist_sell<PTS, NG, 256>; break;
      case 128: k_hist_sell<PTS, NG, 128><<<grid, 128, sm, js.stream>>>(q, gt); c->last_hist_func = (const void*)k_hist_sell<PTS, NG, 128>; break;
      case 64: k_hist_sell<PTS, NG, 64><<<grid, 64, sm, js.stream>>>(q, gt); c->last_hist_func = (const void*)k_hist_sell<PTS, NG, 64>; break;
      default: k_hist_sell<PTS, NG, 32><<<grid, 32, sm, js.stream>>>(q, gt); c->last_hist_func = (const void*)k_hist_sell<PTS, NG, 32>; break;
    }
    NID_LAUNCH_CHECK(c, "k_hist_sell");
  }
  return NID_OK;
}
template <bool PTS, int NG>
static int launch_jac_chunks(nid_ctx* c, const EvalParams& p, int ns, const JobSet& js) {
  // CTA size by geometry (it does not change any result): small cells have short slices, and one-warp CTAs let the SM
  // replace every finished slice at once -- measured at 16x16 cells 5.93 -> 5.47 us per evaluation with 32 threads, at
  // 4x4 cells 3.41 -> 3.66 (there two slices per CTA share the L1 lines of the target gathers)
  const int T = pick_block(c, ns, js.n, (long long)c->rb * c->cb < NID_SMALL_CELL_PX ? 32 : NID_JAC_TMAX);
  const size_t sm = jac_sell_smem(c, T);
  for (int s0 = 0; s0 < js.n; s0 += NG) {
    const int n = std::min(NG, js.n - s0);
    GeoTable<NG> gt;
    fill_geo(c, gt, js, s0, n, false);
    EvalParams q = p;
    q.job0 = js.first + s0;
    const dim3 grid = NID_GRID(n, (ns + T / 32 - 1) / (T / 32));
#define NID_JAC_LAUNCH(TT, BK)                                                 \
  do {                                                                         \
    k_jac_sell<PTS, NG, TT, BK><<<grid, TT, sm, js.stream>>>(q, gt);          \
    c->last_jac_func = (const void*)k_jac_sell<PTS, NG, TT, BK>;               \
  } while (0)
    const bool bulk = q.stage_bulk && NID_FEW_BINS(c->bins);
    switch (T) {
      case 128: if (bulk) NID_JAC_LAUNCH(128, true); else NID_JAC_LAUNCH(128, false); break;
      case 64: if (bulk) NID_JAC_LAUNCH(64, true); else NID_JAC_LAUNCH(64, false); break;
      default: if (bulk) NID_JAC_LAUNCH(32, true); else NID_JAC_LAUNCH(32, false); break;
    }
#undef NID_JAC_LAUNCH
    NID_LAUNCH_CHECK(c, "k_jac_sell");
  }
  return NID_OK;
}
#define NID_GEO_SMALL 8
#define NID_GEO_LARGE 96
static int launch_hist_w(nid_ctx* c, const EvalParams& p, int ns, const JobSet& js) {
  if (c->sell_points)
    return js.n <= NID_GEO_SMALL ? launch_hist_chunks<true, NID_GEO_SMALL>(c, p, ns, js) : launch_hist_chunks<true, NID_GEO_LARGE>(c, p, ns, js);
  return js.n <= NID_GEO_SMALL ? launch_hist_chunks<false, NID_GEO_SMALL>(c, p, ns, js) : launch_hist_chunks<false, NID_GEO_LARGE>(c, p, ns, js);
}
static int launch_jac_w(nid_ctx* c, const EvalParams& p, int ns, const JobSet& js) {
  if (c->sell_points)
    return js.n <= NID_GEO_SMALL ? launch_jac_chunks<true, NID_GEO_SMALL>(c, p, ns, js) : launch_jac_chunks<true, NID_GEO_LARGE>(c, p, ns, js);
  return js.n <= NID_GEO_SMALL ? launch_jac_chunks<false, NID_GEO_SMALL>(c, p, ns, js) : launch_jac_chunks<false, NID_GEO_LARGE>(c, p, ns, js);
}

// the natural-order kernels (nid_kernels.cu)
__global__ void k_hist(EvalParams p);
__global__ void k_entropy(EvalParams p);
__global__ void k_jac(EvalParams p);
__global__ void k_jac_final(EvalParams p, int n_jobs);

// Pass 1 of the jobs of js. Sorted: pixel kernel + assembly (histograms, entropies, err; unless p2 == none also the
// scaled log tables pass 2 needs). Natural: strip histograms, then the cost tail k_entropy unless k_jac will write it.
int launch_pass1(nid_ctx* c, const JobSet& js, Pass2 p2) {
  const EvalParams p = make_params(c, js);
  const int n = js.n;
  if (!use_sorted(c)) {
    const size_t smem = sizeof(double) * p.hist_stride;
    ktime_mark(c, js.stream, 0);
    k_hist<<<dim3(p.S, p.ncell, n), 256, smem, js.stream>>>(p);
    NID_LAUNCH_CHECK(c, "k_hist");
    ktime_mark(c, js.stream, 1);
    if (p2 != Pass2::all) {
      k_entropy<<<dim3(p.ncell, n), 256, smem, js.stream>>>(p);
      NID_LAUNCH_CHECK(c, "k_entropy");
    }
    ktime_mark(c, js.stream, 2);
    return NID_OK;
  }
  const int tables = p2 != Pass2::none;
  const int ns = c->max_nslices_prepared;
  ktime_mark(c, js.stream, 0);
  // (no slices at all: every cell of every prepared pair is inactive; the assembly reports NaN)
  const int r = ns > 0 ? launch_hist_w(c, p, ns, js) : NID_OK;
  if (r != NID_OK) return r;
  ktime_mark(c, js.stream, 1);
  if (assemble_warp(c)) {
    const int units = c->ncell * n;
    if (units <= 2 * c->sm_count * NID_ASMW_WARPS)
      k_assemble_warp<NID_ASMW_BATCH_LAT><<<(units + NID_ASMW_WARPS - 1) / NID_ASMW_WARPS, NID_ASMW_WARPS * 32, assemble_warp_smem(c), js.stream>>>(p, tables, n);
    else
      k_assemble_warp<NID_ASMW_BATCH><<<(units + NID_ASMW_WARPS - 1) / NID_ASMW_WARPS, NID_ASMW_WARPS * 32, assemble_warp_smem(c), js.stream>>>(p, tables, n);
  } else if (c->opt_asm_wide && (c->ncell * n <= c->sm_count || c->opt_asm_wide == 2 ||
                                 (!assemble_small(c) && assemble_smem(c, NID_ASM_THREADS) > (size_t)100 * 1024))) {
    // the 1024-thread variant (same bits): for a handful of evaluations in flight (fewer units than SMs), and whenever the
    // shared memory of a CTA leaves room for one or two CTAs per SM only (more than ~30 bins) -- 1024 threads then fill the
    // SM where 256 leave it mostly empty (C3, 32 bins: 5.57 -> 4.00 us per evaluation; 40 bins at 640x480: 4.59 -> 2.55;
    // but 28 bins: 1.97 -> 2.09, 24 bins: 1.44 -> 1.88, 16 bins: 0.87 -> 1.51, so not there)
    k_assemble_wide<<<dim3(c->ncell, n), NID_ASM_WIDE, assemble_smem(c, NID_ASM_WIDE), js.stream>>>(p, tables);
  } else if (assemble_small(c)) k_assemble_small<<<dim3(c->ncell, n), NID_ASM_SMALL, assemble_smem(c, NID_ASM_THREADS), js.stream>>>(p, tables);
  else k_assemble<<<dim3(c->ncell, n), NID_ASM_THREADS, assemble_smem(c, NID_ASM_THREADS), js.stream>>>(p, tables);
  NID_LAUNCH_CHECK(c, "k_assemble");
  ktime_mark(c, js.stream, 2);
  return NID_OK;
}

// Pass 2 + Jacobian tail of the jobs of js; their pass 1 must have run at their current poses (sorted: with the tables).
int launch_pass2(nid_ctx* c, const JobSet& js) {
  const EvalParams p = make_params(c, js);
  const int n = js.n;
  if (!use_sorted(c)) {
    k_jac<<<dim3(p.S, p.ncell, n), 256, sizeof(double) * p.hist_stride, js.stream>>>(p);
    NID_LAUNCH_CHECK(c, "k_jac");
    ktime_mark(c, js.stream, 3);
    k_jac_final<<<(n * p.ncell * 6 + 255) / 256, 256, 0, js.stream>>>(p, n);
    NID_LAUNCH_CHECK(c, "k_jac_final");
    ktime_mark(c, js.stream, 4);
    return NID_OK;
  }
  const int ns = c->max_nslices_prepared;
  const int r = ns > 0 ? launch_jac_w(c, p, ns, js) : NID_OK;
  if (r != NID_OK) return r;
  ktime_mark(c, js.stream, 3);
  k_jac_final_sorted<<<jac_final_blocks(c, n), 256, 0, js.stream>>>(p, n);
  NID_LAUNCH_CHECK(c, "k_jac_final_sorted");
  ktime_mark(c, js.stream, 4);
  return NID_OK;
}

int launch_sorted_tail_gn(nid_ctx* c, const JobSet& js, double delta, double* gn_out) {
  EvalParams p = make_params(c, js);
  p.huber_delta = delta;
  p.huber_dsqr = huber_dsqr(delta);
  const int n = js.n;
  const int ns = c->max_nslices_prepared;
  const int r = ns > 0 ? launch_jac_w(c, p, ns, js) : NID_OK;
  if (r != NID_OK) return r;
  if (c->ncell <= 32) {
    k_tail_gn<<<n, 256, 0, js.stream>>>(p, gn_out);
    NID_LAUNCH_CHECK(c, "k_tail_gn");
  } else {
    // many cells (the reference's default geometry has 256): one CTA per job would walk them eight at a time (measured
    // ~120 us of a 240 us round); a warp per (job, cell) for the tails, then the block sums
    k_jac_final_sorted<<<jac_final_blocks(c, n), 256, 0, js.stream>>>(p, n);
    NID_LAUNCH_CHECK(c, "k_jac_final_sorted");
    k_gn_out<<<n, 128, 0, js.stream>>>(p, gn_out);
    NID_LAUNCH_CHECK(c, "k_gn_out");
  }
  return NID_OK;
}

// ------------------------------------------------------------------------------------------------
// Latency mode of the LM driver as ONE graph launch per round. A round is always the same chain -- the staged poses
// and slot list to the device, pass 1, assembly, pass 2, Jacobian tail + Gauss-Newton block -- over the same nslots job
// slots; only the geometry tables, which the pixel kernels take as launch parameters (constant bank: they cost the
// kernels no registers), change from round to round. The chain is captured once and kept with the context; per round
// the two pixel-kernel nodes get their new parameter block (cudaGraphExecKernelNodeSetParams) and the graph is
// launched: one driver call instead of a copy and five launches, and no launch gaps between the kernels.
// Measured (B200, one 640x480 pair, 4x4 cells, 16 bins, 4 slots): 148 -> 115 us per round.
// The graph is rebuilt whenever anything its nodes captured by value has changed (buffers, layout sizes, options):
// the signature below is compared at every round.
struct LatencyGraph {
  Graph graph;
  GraphExec exec;  // (declared after its graph: destroyed first)
  cudaGraphNode_t hist_node = nullptr, jac_node = nullptr;
  cudaKernelNodeParams hist_np{}, jac_np{};
  EvalParams hist_q, jac_q;  // first argument of the two pixel kernels as captured
  // signature
  EvalParams sig;  // (holds the slot list and the device pose table)
  int nslots = 0, ns = 0, task_px = 0;
  size_t h2d_bytes = 0;
  double delta = 0.0;
  const double* gn_out = nullptr;
  const void* h_src = nullptr;
  cudaStream_t stream = nullptr;
};

void LatencyGraphDelete::operator()(LatencyGraph* g) const { delete g; }

static int capture_latency_graph(nid_ctx* c, LatencyGraph* g, const JobSet& js, size_t h2d_bytes, double delta, double* gn_out) {
  g->exec.reset();
  g->graph.reset();
  cudaError_t e = cudaStreamBeginCapture(js.stream, cudaStreamCaptureModeThreadLocal);
  if (e != cudaSuccess) return check_cuda(e, "cudaStreamBeginCapture");
  int r = NID_OK;
  e = cudaMemcpyAsync(js.d_poses, js.h_poses, h2d_bytes, cudaMemcpyHostToDevice, js.stream);
  if (e != cudaSuccess) r = check_cuda(e, "H2D poses + list (capture)");
  if (r == NID_OK) r = launch_pass1(c, js, Pass2::some);
  if (r == NID_OK) r = launch_sorted_tail_gn(c, js, delta, gn_out);
  cudaGraph_t graph = nullptr;
  e = cudaStreamEndCapture(js.stream, &graph);
  g->graph.reset(graph);
  if (r != NID_OK) return r;
  if (e != cudaSuccess) return check_cuda(e, "cudaStreamEndCapture");
  size_t nn = 0;
  e = cudaGraphGetNodes(g->graph, nullptr, &nn);
  if (e != cudaSuccess) return check_cuda(e, "cudaGraphGetNodes");
  std::vector<cudaGraphNode_t> nodes(nn);
  e = cudaGraphGetNodes(g->graph, nodes.data(), &nn);
  if (e != cudaSuccess) return check_cuda(e, "cudaGraphGetNodes");
  g->hist_node = g->jac_node = nullptr;
  for (cudaGraphNode_t nd : nodes) {
    cudaGraphNodeType ty;
    if (cudaGraphNodeGetType(nd, &ty) != cudaSuccess || ty != cudaGraphNodeTypeKernel) continue;
    cudaKernelNodeParams np{};
    if (cudaGraphKernelNodeGetParams(nd, &np) != cudaSuccess) continue;
    if (np.func == c->last_hist_func && !g->hist_node) {
      g->hist_node = nd; g->hist_np = np;
      memcpy(&g->hist_q, np.kernelParams[0], sizeof(EvalParams));
    } else if (np.func == c->last_jac_func && !g->jac_node) {
      g->jac_node = nd; g->jac_np = np;
      memcpy(&g->jac_q, np.kernelParams[0], sizeof(EvalParams));
    }
  }
  if (!g->hist_node || !g->jac_node) { set_error("latency graph: pixel-kernel nodes not found"); return NID_ERR_STATE; }
  cudaGraphExec_t exec = nullptr;
  e = cudaGraphInstantiate(&exec, g->graph, 0);
  if (e != cudaSuccess) return check_cuda(e, "cudaGraphInstantiate");
  g->exec.reset(exec);
  return NID_OK;
}

// One round of the latency mode over the slots js.h_list[0 .. js.n) (every slot of the solve, each exactly once): the
// staging block of h2d_bytes at js.h_poses (poses, then the slot list js.d_list points into) is copied to js.d_poses first.
int launch_latency_round(nid_ctx* c, const JobSet& js, size_t h2d_bytes, double delta, double* gn_out) {
  const int nslots = js.n;
  const int ns = c->max_nslices_prepared;
  const bool graph_ok = c->opt_lm_graph && !c->opt_time_kernels && ns > 0 && nslots <= NID_GEO_SMALL;
  if (!graph_ok) {
    cudaError_t e = cudaMemcpyAsync(js.d_poses, js.h_poses, h2d_bytes, cudaMemcpyHostToDevice, js.stream);
    if (e != cudaSuccess) return check_cuda(e, "H2D poses + list");
    int r = launch_pass1(c, js, Pass2::some);
    if (r != NID_OK) return r;
    return launch_sorted_tail_gn(c, js, delta, gn_out);
  }
  if (!c->lm_graph) c->lm_graph.reset(new LatencyGraph());
  LatencyGraph* g = c->lm_graph.get();
  const EvalParams sig = make_params(c, js);
  const bool same = g->exec && memcmp(&sig, &g->sig, sizeof(sig)) == 0 && g->nslots == nslots && g->ns == ns && g->task_px == c->task_px &&
                    g->h2d_bytes == h2d_bytes && g->delta == delta && g->gn_out == gn_out && g->h_src == (const void*)js.h_poses &&
                    g->stream == js.stream;
  if (!same) {
    const int r = capture_latency_graph(c, g, js, h2d_bytes, delta, gn_out);
    if (r != NID_OK) { c->lm_graph.reset(); return r; }
    g->sig = sig; g->nslots = nslots; g->ns = ns; g->task_px = c->task_px; g->h2d_bytes = h2d_bytes; g->delta = delta;
    g->gn_out = gn_out; g->h_src = js.h_poses; g->stream = js.stream;
    // (the graph just captured holds this round's geometry already)
  } else {
    GeoTable<NID_GEO_SMALL> gt;
    for (int pass = 0; pass < 2; pass++) {
      fill_geo(c, gt, js, 0, nslots, pass == 0);
      cudaKernelNodeParams np = pass == 0 ? g->hist_np : g->jac_np;
      void* args[2] = {pass == 0 ? (void*)&g->hist_q : (void*)&g->jac_q, (void*)&gt};
      np.kernelParams = args;
      np.extra = nullptr;
      const cudaError_t e = cudaGraphExecKernelNodeSetParams(g->exec, pass == 0 ? g->hist_node : g->jac_node, &np);
      if (e != cudaSuccess) return check_cuda(e, "cudaGraphExecKernelNodeSetParams");
    }
  }
  const cudaError_t e = cudaGraphLaunch(g->exec, js.stream);
  if (e != cudaSuccess) return check_cuda(e, "cudaGraphLaunch");
  c->launches += 4;
  return NID_OK;
}

// Geometry table of kernel 1 (see k_warp_sample_jobs): the ray of pixel (col, row) is affine in (col, row)
template <int NG>
static void fill_geo_k1(const nid_ctx* c, GeoTable<NG>& gt, const JobSet& js, int s0, int n) {
  fill_geo(c, gt, js, s0, n, true);  // [0..11] M with rows 0/1 scaled by fx, fy; [12] 1/fx [13] -cx/fx [14] 1/fy [15] -cy/fy
  for (int i = 0; i < n; i++) {
    double* g = gt.g[i];
    const double ifx = g[12], cxo = g[13], ify = g[14], cyo = g[15], cx = g[18], cy = g[19];
    double A[3], B[3], C[3];
    for (int r = 0; r < 3; r++) {
      A[r] = g[r] * ifx;
      B[r] = g[3 + r] * ify;
      C[r] = g[r] * cxo + g[3 + r] * cyo + g[6 + r];
    }
    for (int r = 0; r < 3; r++) {
      g[r] = A[r]; g[3 + r] = B[r]; g[6 + r] = C[r];
      g[12 + r] = 128.0 * A[r];
      g[15 + r] = B[r] - (double)c->cols * A[r];
    }
    g[18] = cx; g[19] = cy;
  }
}

// target planes of kernel 1 for one pair (built on first use; the evaluation path does not need them)
int launch_pack_k1(nid_ctx* c, int pair, unsigned short* d_out) {
  int g = (c->N + 255) / 256;
  if (g > c->sm_count * 8) g = c->sm_count * 8;
  k_pack_k1<<<g, 256, 0, c->stream>>>(c->rows, c->cols, c->im1 + (size_t)pair * c->N, d_out);
  NID_LAUNCH_CHECK(c, "k_pack_k1");
  return NID_OK;
}

// all jobs of a launch must take their depth from the same kind of plane (raw 16-bit or fp64): u16 says which
int launch_warp_sample_jobs(nid_ctx* c, const JobSet& js, float4* d_out, bool u16) {
  const EvalParams p = make_params(c, js);
  const int chunks = (c->N + 128 * NID_WS_W - 1) / (128 * NID_WS_W);
  for (int s0 = 0; s0 < js.n; s0 += NID_GEO_LARGE) {
    const int n = std::min(NID_GEO_LARGE, js.n - s0);
    GeoTable<NID_GEO_LARGE> gt;
    fill_geo_k1(c, gt, js, s0, n);
    EvalParams q = p;
    q.job0 = js.first + s0;
    const dim3 grid(n, chunks);
    if (u16) k_warp_sample_jobs<NID_GEO_LARGE, true><<<grid, 128, 0, js.stream>>>(q, gt, nullptr, c->depth16, c->depth_factor, d_out);
    else k_warp_sample_jobs<NID_GEO_LARGE, false><<<grid, 128, 0, js.stream>>>(q, gt, c->depth, nullptr, nullptr, d_out);
    NID_LAUNCH_CHECK(c, "k_warp_sample_jobs");
  }
  return NID_OK;
}

int sorted_init(nid_ctx* c) {
  cudaError_t e;
  if (c->bins > NID_SORTED_MAX_BINS || c->bins < NID_SORTED_MIN_BINS) return NID_OK;  // natural-order kernels only
#define NID_SMEM_ATTR(k, bytes)                                                                     \
  e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes));            \
  if (e != cudaSuccess) return check_cuda(e, "smem attr " #k);
  // shared-memory carve-out of the pixel kernels: what their resident CTAs need and no more, the rest of the 256 KB
  // stays L1 for the target-image gathers. (hint only; per kernel: threads T, CTAs per SM = warps per SM * 32 / T)
#define NID_CARVE(k, bytes, ctas)                                                                                  \
  {                                                                                                                 \
    const int pct = (int)std::min<size_t>(100, (((bytes) + 1024) * (size_t)(ctas) * 100 + 228 * 1024 - 1) / (228 * 1024)); \
    cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, pct);                                   \
  }
#define NID_SMEM_ATTR_PX(PTS, NG)                                           \
  NID_SMEM_ATTR((k_hist_sell<PTS, NG, 256>), hist_sell_smem(c, 256));       \
  NID_SMEM_ATTR((k_hist_sell<PTS, NG, 128>), hist_sell_smem(c, 128));       \
  NID_SMEM_ATTR((k_hist_sell<PTS, NG, 64>), hist_sell_smem(c, 64));         \
  NID_SMEM_ATTR((k_hist_sell<PTS, NG, 32>), hist_sell_smem(c, 32));         \
  NID_SMEM_ATTR((k_jac_sell<PTS, NG, 128, false>), jac_sell_smem(c, 128));  \
  NID_SMEM_ATTR((k_jac_sell<PTS, NG, 64, false>), jac_sell_smem(c, 64));    \
  NID_SMEM_ATTR((k_jac_sell<PTS, NG, 32, false>), jac_sell_smem(c, 32));    \
  NID_SMEM_ATTR((k_jac_sell<PTS, NG, 128, true>), jac_sell_smem(c, 128));   \
  NID_SMEM_ATTR((k_jac_sell<PTS, NG, 64, true>), jac_sell_smem(c, 64));     \
  NID_SMEM_ATTR((k_jac_sell<PTS, NG, 32, true>), jac_sell_smem(c, 32));     \
  NID_CARVE((k_hist_sell<PTS, NG, 128>), hist_sell_smem(c, 128), NID_HIST_WARPS / 4);  \
  NID_CARVE((k_hist_sell<PTS, NG, 64>), hist_sell_smem(c, 64), NID_HIST_WARPS / 2);    \
  NID_CARVE((k_hist_sell<PTS, NG, 32>), hist_sell_smem(c, 32), NID_HIST_WARPS);        \
  NID_CARVE((k_jac_sell<PTS, NG, 64, false>), jac_sell_smem(c, 64), NID_JAC_WARPS / 2);  \
  NID_CARVE((k_jac_sell<PTS, NG, 32, false>), jac_sell_smem(c, 32), NID_JAC_WARPS);      \
  NID_CARVE((k_jac_sell<PTS, NG, 64, true>), jac_sell_smem(c, 64), NID_JAC_WARPS_SMALL / 2);   \
  NID_CARVE((k_jac_sell<PTS, NG, 32, true>), jac_sell_smem(c, 32), NID_JAC_WARPS_SMALL);
  NID_SMEM_ATTR_PX(true, NID_GEO_SMALL)
  NID_SMEM_ATTR_PX(false, NID_GEO_SMALL)
  NID_SMEM_ATTR_PX(true, NID_GEO_LARGE)
  NID_SMEM_ATTR_PX(false, NID_GEO_LARGE)
#undef NID_SMEM_ATTR_PX
  NID_SMEM_ATTR(k_assemble, assemble_smem(c, NID_ASM_THREADS));
  NID_SMEM_ATTR(k_assemble_small, assemble_smem(c, NID_ASM_THREADS));
  NID_SMEM_ATTR(k_assemble_wide, assemble_smem(c, NID_ASM_WIDE));
  if (c->bins <= 32) {
    NID_SMEM_ATTR(k_assemble_warp<NID_ASMW_BATCH>, assemble_warp_smem(c));
    NID_SMEM_ATTR(k_assemble_warp<NID_ASMW_BATCH_LAT>, assemble_warp_smem(c));
  }
#undef NID_SMEM_ATTR
  return NID_OK;
}

}  // namespace nid
