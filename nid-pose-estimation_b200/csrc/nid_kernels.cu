// sm_100a kernels of the NID cost + Jacobian path and their launchers.
// Citations: file:line in arpg/NID-Pose-Estimation. See DESIGN.md for the data layout and the
// roofline of each kernel.
#include <math.h>

#include <algorithm>

#include "nid_ctx.h"
#include "nid_device.cuh"

namespace nid {

#define NID_LAUNCH_CHECK(c, what)                         \
  do {                                                    \
    (c)->launches++;                                      \
    cudaError_t e__ = cudaGetLastError();                 \
    if (e__ != cudaSuccess) return check_cuda(e__, what); \
  } while (0)

// ------------------------------------------------------------------------------------------------
// reference-intensity lookup: for v in 0..255 the span index k_r and the 4 spline weights
// (CudaComputeHref.cu:102-116; types_six_dof_expmap.cpp:683-699)
__global__ void k_build_lut(int bins, double* __restrict__ lut_w, int* __restrict__ lut_k) {
  int v = threadIdx.x;
  if (v >= 256) return;
  double obs = (double)v;
  if (obs >= 255.0) obs = 254.999;
  double ub = __ddiv_rn(__dmul_rn(obs, (double)(bins - 3)), 255.0);
  int k = (int)floor(ub);
  double w[4], dw[4];
  bspline4<false>(ub, k, bins, w, dw);
  lut_k[v] = k;
#pragma unroll
  for (int m = 0; m < 4; m++) lut_w[4 * v + m] = w[m];
}

// ------------------------------------------------------------------------------------------------
// a1: depth -> world points (CudaPoints3d.cu:5-32), SoA planes, NaN for invalid depth. Pair pair0 + blockIdx.y.
// U16: the depth arrives as the raw 16-bit plane of the dataset and is converted like the reference's driver does,
// `depth.convertTo(CV_64F, depth_factor)` (NID_pose_estimation.cpp:105-106): one rounding of raw * factor; the fp64
// plane is kept for the regrouping scatter and kernel 1.
template <bool U16>
__global__ void k_points(int rows, int cols, int pair0, double* __restrict__ depth_all, const uint16_t* __restrict__ d16_all,
                         const double* __restrict__ factor_all, const double* __restrict__ Twc0_all,
                         const double* __restrict__ cam_all, double* __restrict__ pwx_all, double* __restrict__ pwy_all,
                         double* __restrict__ pwz_all) {
  const int N = rows * cols;
  const int pair = pair0 + blockIdx.y;
  const size_t b = (size_t)pair * N;
  const double* camp = cam_all + 4 * pair;
  Cam cam{camp[0], camp[1], camp[2], camp[3]};
  double T[16];
#pragma unroll
  for (int i = 0; i < 16; i++) T[i] = Twc0_all[16 * pair + i];
  const double factor = U16 ? factor_all[pair] : 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
    double z;
    if (U16) { z = __dmul_rn((double)d16_all[b + i], factor); depth_all[b + i] = z; }
    else z = depth_all[b + i];
    double x = nan(""), y = nan(""), zz = nan("");
    if (!(z < 0.01 || z > 100)) {
      backproject(T, cam, z, i / cols, i % cols, x, y, zz);
    }
    pwx_all[b + i] = x; pwy_all[b + i] = y; pwz_all[b + i] = zz;
  }
}

// 2x2 downsampling of a pair (nid_set_pairs_downsampled): destination pixel (i, j) of pair blockIdx.y covers source
// pixels (2i..2i+1, 2j..2j+1); an odd last source row or column is dropped. Images: (a + b + c + d + 2) >> 2, exact in
// integers. Depth: the mean of the valid samples (the test of k_points, with NaN and Inf invalid too), summed in the fixed
// order (2i,2j), (2i,2j+1), (2i+1,2j), (2i+1,2j+1) without contraction; 0 (invalid) when no sample is valid.
// The pointers are those of the first source / destination pair of the batch.
__global__ void k_downsample2(int src_cols, int rows, int cols, const double* __restrict__ src_depth,
                              const uint8_t* __restrict__ src_im0, const uint8_t* __restrict__ src_im1, size_t src_N,
                              double* __restrict__ dst_depth, uint8_t* __restrict__ dst_im0, uint8_t* __restrict__ dst_im1,
                              size_t dst_N) {
  const int N = rows * cols;
  const size_t sb = (size_t)blockIdx.y * src_N, db = (size_t)blockIdx.y * dst_N;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
    const int r = i / cols, c = i % cols;
    const size_t s[4] = {sb + (size_t)(2 * r) * src_cols + 2 * c, sb + (size_t)(2 * r) * src_cols + 2 * c + 1,
                         sb + (size_t)(2 * r + 1) * src_cols + 2 * c, sb + (size_t)(2 * r + 1) * src_cols + 2 * c + 1};
    dst_im0[db + i] = (uint8_t)(((unsigned)src_im0[s[0]] + src_im0[s[1]] + src_im0[s[2]] + src_im0[s[3]] + 2) >> 2);
    dst_im1[db + i] = (uint8_t)(((unsigned)src_im1[s[0]] + src_im1[s[1]] + src_im1[s[2]] + src_im1[s[3]] + 2) >> 2);
    double sum = 0.0;
    int n = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const double z = src_depth[s[k]];
      if (z >= 0.01 && z <= 100) { sum = __dadd_rn(sum, z); n++; }
    }
    dst_depth[db + i] = n ? __ddiv_rn(sum, (double)n) : 0.0;
  }
}

__global__ void k_points_aos(int N, const double* __restrict__ pwx, const double* __restrict__ pwy,
                             const double* __restrict__ pwz, double* __restrict__ out) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
    out[3 * i] = pwx[i]; out[3 * i + 1] = pwy[i]; out[3 * i + 2] = pwz[i];
  }
}

__global__ void k_points_soa(int N, const double* __restrict__ in, double* __restrict__ pwx, double* __restrict__ pwy,
                             double* __restrict__ pwz) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
    double x = in[3 * i], y = in[3 * i + 1], z = in[3 * i + 2];
    if (isnan(x) || isnan(y) || isnan(z)) { x = nan(""); y = nan(""); z = nan(""); }  // computeH.cu:147
    pwx[i] = x; pwy[i] = y; pwz[i] = z;
  }
}

__global__ void k_import_flags(int N, const double* __restrict__ bs_value, uint8_t* __restrict__ inb0) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x)
    inb0[i] = isnan(bs_value[4 * (size_t)i]) ? 0 : 1;
}

// doubles -> uint8 with the reference's clamp (>=255 -> 254.999 is handled by the LUT, so 255 stays
// 255 here); flags non-integral values
__global__ void k_check_integral(int N, const double* __restrict__ src, uint8_t* __restrict__ dst, int* flag,
                                 int is_ref) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
    double v = src[i];
    if (is_ref) {
      // the reference clamps im0 before use (CudaComputeHref.cu:102-105)
      if (v < 0.0) v = 0.0;
      if (v >= 255.0) v = 255.0;
    } else if (v < 0.0 || v > 255.0) {
      atomicOr(flag, 1);
      v = 0.0;
    }
    double r = rint(v);
    if (r != v) atomicOr(flag, 1);
    dst[i] = (uint8_t)r;
  }
}

// ------------------------------------------------------------------------------------------------
// a2 part 1: in-bounds flag at the prepare pose and per-cell counts of reference intensities
// (CudaComputeHref.cu:76-131; computeHref types_six_dof_expmap.cpp:655-702)
// Pair pair0 + blockIdx.y at the initial pose poses16[16 * blockIdx.y].
__global__ void k_prepare(EvalParams p, int pair0, const double* __restrict__ poses16, uint8_t* __restrict__ inb0,
                          unsigned int* __restrict__ cnt) {
  const int pair = pair0 + blockIdx.y;
  const size_t base = (size_t)pair * p.N;
  const double* cp = p.cam + 4 * pair;
  Cam cam{cp[0], cp[1], cp[2], cp[3]};
  Pose P = load_pose(poses16 + 16 * blockIdx.y);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < p.N; i += gridDim.x * blockDim.x) {
    int row = i / p.cols, col = i % p.cols;
    uint8_t flag = 0;
    double x0 = p.pwx[base + i];
    if (!isnan(x0) && row < p.rb * p.cell && col < p.cb * p.cell) {
      double x1, y1, z1, u, v;
      warp_project(P, cam, x0, p.pwy[base + i], p.pwz[base + i], x1, y1, z1, u, v);
      int key = 256;  // valid point, no reference sample
      if (inb_cost(u, v, p.rows, p.cols)) {
        flag = 1;
        key = p.im0[base + i];
      }
      int c = (row / p.rb) * p.cell + (col / p.cb);
      atomicAdd(&cnt[((size_t)pair * p.ncell + c) * NID_NCLS + key], 1u);
    }
    inb0[base + i] = flag;
  }
}

// a2 part 2: n_c, reference marginal and H_ref per cell (CudaComputeHref.cu:204-221;
// types_six_dof_expmap.cpp:710-723). One block per (cell, pair pair0 + blockIdx.y), one thread per intensity value.
__global__ void __launch_bounds__(256) k_href(EvalParams p, int pair0, const unsigned int* __restrict__ cnt,
                                              int* __restrict__ n_c, double* __restrict__ href) {
  const int pair = pair0 + blockIdx.y;
  extern __shared__ double sm[];
  double* pro = sm;  // [bins]
  __shared__ double s_con[256][4];  // class v's contribution to bins k_r(v) .. k_r(v)+3
  __shared__ int s_k[256];
  __shared__ unsigned int s_cnt[256];
  __shared__ int s_part[8];
  __shared__ int s_n;
  const int c = blockIdx.x;
  const unsigned int* cc = cnt + ((size_t)pair * p.ncell + c) * NID_NCLS;
  const int t = threadIdx.x;
  const unsigned int mine = cc[t];
  s_cnt[t] = mine;
  s_k[t] = p.lut_k[t];
#pragma unroll
  for (int m = 0; m < 4; m++) s_con[t][m] = mine ? (double)mine * p.lut_w[4 * t + m] : 0.0;
  __syncthreads();
  {  // n_c: integer sum, any order
    int n = (int)mine;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
    if ((t & 31) == 0) s_part[t >> 5] = n;
  }
  if (t < p.bins) {
    // fixed order over intensity values -> deterministic; only the classes of spans t-3 .. t reach bin t
    // (k_r(v) is monotone in v: span_start)
    const int NS = p.bins - 3;
    const int vlo = p.span_start[max(t - 3, 0)], vhi = p.span_start[min(t, NS - 1) + 1];
    double acc = 0.0;
    for (int v = vlo; v < vhi; v++) {
      const int m = t - s_k[v];
      if (m >= 0 && m < 4 && s_cnt[v]) acc += s_con[v][m];
    }
    pro[t] = acc;
  }
  __syncthreads();
  if (t == 0) {
    int n = 0;
    for (int w = 0; w < 8; w++) n += s_part[w];
    s_n = n;
  }
  __syncthreads();
  if (t == 0) {
    int n = s_n;
    n_c[pair * p.ncell + c] = n;
    double H = nan("");
    if (n >= NID_MIN_CELL_POINTS) {
      H = 0.0;
      for (int b = 0; b < p.bins; b++) {
        double q = pro[b] / (double)n;
        if (q < kSigma) continue;
        H -= q * log2(q);
      }
    }
    href[pair * p.ncell + c] = H;
  }
}

// reference-layout per-pixel spline data for the CudaComputeHref shim (CudaComputeHref.cu:107-131)
__global__ void k_ref_weights(EvalParams p, int pair, double* __restrict__ bs_value, int* __restrict__ bs_index) {
  const size_t base = (size_t)pair * p.N;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < p.N; i += gridDim.x * blockDim.x) {
    if (p.inb0[base + i]) {
      int v = p.im0[base + i];
      bs_index[i] = p.lut_k[v];
#pragma unroll
      for (int m = 0; m < 4; m++) bs_value[4 * i + m] = p.lut_w[4 * v + m];
    } else {
      bs_index[i] = 0;
#pragma unroll
      for (int m = 0; m < 4; m++) bs_value[4 * i + m] = nan("");
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Pass 1 (a6, cost half): warp + sample + target/joint B-spline histograms of one strip of one cell.
// grid (S, ncell, jobs). The CTA accumulates into a private shared-memory histogram and stores its
// partial; partials are merged in a fixed order by the consumers.
__global__ void __launch_bounds__(256) k_hist(EvalParams p) {
  extern __shared__ double sm[];
  const int B = p.bins;
  double* Pj = sm;           // [B*B]
  double* Pt = sm + B * B;   // [B]
  const int strip = blockIdx.x, c = blockIdx.y, job = job_at(p, blockIdx.z);
  const int pair = p.job_pair[job];
  double* out = p.part + (((size_t)job * p.ncell + c) * p.S + strip) * p.hist_stride;
  if (p.n_c[pair * p.ncell + c] < NID_MIN_CELL_POINTS) return;
  for (int i = threadIdx.x; i < p.hist_stride; i += blockDim.x) sm[i] = 0.0;
  __syncthreads();

  const size_t base = (size_t)pair * p.N;
  const double* cp = p.cam + 4 * pair;
  const Cam cam{cp[0], cp[1], cp[2], cp[3]};
  const Pose P = load_pose(p.poses + 16 * job);
  const int ci = c / p.cell, cj = c % p.cell;
  const int r0 = ci * p.rb + strip * p.strip_rows;
  const int r1 = min(ci * p.rb + p.rb, r0 + p.strip_rows);
  const int c0 = cj * p.cb;
  const int npx = max(r1 - r0, 0) * p.cb;
  const uint8_t* im1 = p.im1 + base;
  const double scale = (double)(B - 3);

  for (int t = threadIdx.x; t < npx; t += blockDim.x) {
    const int row = r0 + t / p.cb, col = c0 + t % p.cb;
    const size_t i = base + (size_t)row * p.cols + col;
    const double x0 = p.pwx[i];
    if (isnan(x0)) continue;
    double x1, y1, z1, u, v;
    warp_project(P, cam, x0, p.pwy[i], p.pwz[i], x1, y1, z1, u, v);
    if (!inb_cost(u, v, p.rows, p.cols)) continue;
    double ic = clamp_intensity(interp_u8(im1, p.cols, u, v));
    double ub = __ddiv_rn(__dmul_rn(ic, scale), 255.0);
    int kt = (int)floor(ub);
    double wt[4], dw[4];
    bspline4<false>(ub, kt, B, wt, dw);
#pragma unroll
    for (int n = 0; n < 4; n++) atomicAdd(&Pt[kt + n], wt[n]);
    if (p.inb0[i]) {
      const int v0 = p.im0[i];
      const int kr = p.lut_k[v0];
#pragma unroll
      for (int m = 0; m < 4; m++) {
        const double wr = p.lut_w[4 * v0 + m];
#pragma unroll
        for (int n = 0; n < 4; n++) atomicAdd(&Pj[(kr + m) * B + kt + n], wr * wt[n]);
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < p.hist_stride; i += blockDim.x) out[i] = sm[i];
}

// Merge the S strip partials of (job, cell) in strip order, normalise by n_c and compute the two
// entropies (a7: computeH.cu:261-300; types_six_dof_expmap.cpp:609-635). Leaves P_j|P_t in `sm`.
// Returns through Ht/Hj on every thread.
__device__ __forceinline__ void merge_entropy(const EvalParams& p, int job, int c, int nc, double* sm,
                                              double* scratch, double& Ht, double& Hj) {
  const int B = p.bins;
  const double* in = p.part + ((size_t)job * p.ncell + c) * p.S * p.hist_stride;
  double ej = 0.0, et = 0.0;
  for (int i = threadIdx.x; i < p.hist_stride; i += blockDim.x) {
    double acc = 0.0;
    for (int s = 0; s < p.S; s++) acc += in[(size_t)s * p.hist_stride + i];
    acc = acc / (double)nc;
    sm[i] = acc;
    double h = (acc < kSigma) ? 0.0 : acc * log2(acc);
    if (i < B * B) ej -= h; else et -= h;
  }
  Hj = block_sum(ej, scratch);
  Ht = block_sum(et, scratch);
}

// cost-only tail: one CTA per (cell, job)
__global__ void __launch_bounds__(256) k_entropy(EvalParams p) {
  extern __shared__ double sm[];
  __shared__ double scratch[8];
  const int c = blockIdx.x, job = job_at(p, blockIdx.y);
  const int pair = p.job_pair[job];
  const int nc = p.n_c[pair * p.ncell + c];
  const size_t o = (size_t)job * p.ncell + c;
  if (nc < NID_MIN_CELL_POINTS) {
    if (threadIdx.x == 0) { p.ht[o] = nan(""); p.hj[o] = nan(""); p.err[o] = nan(""); }
    return;
  }
  double Ht, Hj;
  merge_entropy(p, job, c, nc, sm, scratch, Ht, Hj);
  if (p.hist) for (int i = threadIdx.x; i < p.hist_stride; i += blockDim.x) p.hist[o * p.hist_stride + i] = sm[i];
  if (threadIdx.x == 0) {
    p.ht[o] = Ht; p.hj[o] = Hj;
    p.err[o] = (2 * Hj - p.href[pair * p.ncell + c] - Ht) / Hj;  // types_six_dof_expmap.h:227
  }
}

// Pass 2 (a6 Jacobian half + a8): every CTA rebuilds the merged histograms of its cell, turns them
// into the table W[r][t] = coefJ*(1+log2 P_j) and V[t] = coefT*(1+log2 P_t), and reduces
//   J[a] = sum_i g_i[a] * sum_m dw_i[m] * ( V[kt+m] + sum_k wr_i[k] W[kr+k][kt+m] )
// which is the reference's sum (types_six_dof_expmap.cpp:395-528; computeH.cu:179-258,303-368)
// re-associated so that the 6 x bins^2 derivative tensor never has to be materialised.
__global__ void __launch_bounds__(256) k_jac(EvalParams p) {
  extern __shared__ double sm[];
  __shared__ double scratch[8];
  __shared__ double red[8][6];
  const int B = p.bins;
  const int strip = blockIdx.x, c = blockIdx.y, job = job_at(p, blockIdx.z);
  const int pair = p.job_pair[job];
  const int nc = p.n_c[pair * p.ncell + c];
  const size_t o = (size_t)job * p.ncell + c;
  if (nc < NID_MIN_CELL_POINTS) {
    if (strip == 0 && threadIdx.x == 0) { p.ht[o] = nan(""); p.hj[o] = nan(""); p.err[o] = nan(""); }
    return;
  }
  double Ht, Hj;
  merge_entropy(p, job, c, nc, sm, scratch, Ht, Hj);
  const double Href = p.href[pair * p.ncell + c];
  if (strip == 0) {
    if (p.hist) for (int i = threadIdx.x; i < p.hist_stride; i += blockDim.x) p.hist[o * p.hist_stride + i] = sm[i];
    if (threadIdx.x == 0) {
      p.ht[o] = Ht; p.hj[o] = Hj;
      p.err[o] = (2 * Hj - Href - Ht) / Hj;
    }
  }
  __syncthreads();
  {
    const double s_over = ((double)(B - 3) / 255.0) / ((double)nc * Hj * Hj);
    const double coefJ = -s_over * (Ht + Href);
    const double coefT = s_over * Hj;
    for (int i = threadIdx.x; i < p.hist_stride; i += blockDim.x) {
      double q = sm[i];
      double L = (q < kSigma) ? 0.0 : (1.0 + log2(q));
      sm[i] = L * (i < B * B ? coefJ : coefT);
    }
  }
  __syncthreads();
  const double* W = sm;
  const double* V = sm + B * B;

  const size_t base = (size_t)pair * p.N;
  const double* cp = p.cam + 4 * pair;
  const Cam cam{cp[0], cp[1], cp[2], cp[3]};
  const Pose P = load_pose(p.poses + 16 * job);
  const int ci = c / p.cell, cj = c % p.cell;
  const int r0 = ci * p.rb + strip * p.strip_rows;
  const int r1 = min(ci * p.rb + p.rb, r0 + p.strip_rows);
  const int c0 = cj * p.cb;
  const int npx = max(r1 - r0, 0) * p.cb;
  const uint8_t* im1 = p.im1 + base;
  const double scale = (double)(B - 3);
  double acc[6] = {0, 0, 0, 0, 0, 0};

  for (int t = threadIdx.x; t < npx; t += blockDim.x) {
    const int row = r0 + t / p.cb, col = c0 + t % p.cb;
    const size_t i = base + (size_t)row * p.cols + col;
    const double x0 = p.pwx[i];
    if (isnan(x0)) continue;
    double x, y, z, u, v;
    warp_project(P, cam, x0, p.pwy[i], p.pwz[i], x, y, z, u, v);
    double u2, v2;
    project_jac(cam, x, y, z, u2, v2);
    if (!inb_cost(u, v, p.rows, p.cols) || !inb_jac(u2, v2, p.rows, p.cols)) continue;
    const double ic = clamp_intensity(interp_u8(im1, p.cols, u, v));
    const double gx = (interp_u8(im1, p.cols, u2 + 1.0, v2) - interp_u8(im1, p.cols, u2 - 1.0, v2)) / 2;
    const double gy = (interp_u8(im1, p.cols, u2, v2 + 1.0) - interp_u8(im1, p.cols, u2, v2 - 1.0)) / 2;
    const double ub = __ddiv_rn(__dmul_rn(ic, scale), 255.0);
    const int kt = (int)floor(ub);
    double wt[4], dw[4];
    bspline4<true>(ub, kt, B, wt, dw);
    double ci_ = 0.0;
    if (p.inb0[i]) {
      const int v0 = p.im0[i];
      const int kr = p.lut_k[v0];
      double wr[4];
#pragma unroll
      for (int k = 0; k < 4; k++) wr[k] = p.lut_w[4 * v0 + k];
#pragma unroll
      for (int m = 0; m < 4; m++) {
        double a = V[kt + m];
#pragma unroll
        for (int k = 0; k < 4; k++) a += wr[k] * W[(kr + k) * B + kt + m];
        ci_ += dw[m] * a;
      }
    } else {
#pragma unroll
      for (int m = 0; m < 4; m++) ci_ += dw[m] * V[kt + m];
    }
    // d(u,v)/d(xi), types_six_dof_expmap.cpp:438-450
    const double iz = 1.0 / z, iz2 = iz * iz;
    const double a = ci_ * gx * cam.fx, b = ci_ * gy * cam.fy;
    acc[0] += a * (-x * y * iz2) + b * (-(1.0 + y * y * iz2));
    acc[1] += a * (1.0 + x * x * iz2) + b * (x * y * iz2);
    acc[2] += a * (-y * iz) + b * (x * iz);
    acc[3] += a * iz;
    acc[4] += b * iz;
    acc[5] += a * (-x * iz2) + b * (-y * iz2);
  }
  // deterministic block reduction of the 6-vector
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 6; k++) {
    double vv = acc[k];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) vv += __shfl_xor_sync(0xffffffffu, vv, off);
    if (lane == 0) red[wid][k] = vv;
  }
  __syncthreads();
  if (threadIdx.x < 6) {
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) t += red[w][threadIdx.x];
    p.jpart[(o * p.S + strip) * 6 + threadIdx.x] = t;
  }
}

// a8 tail: fixed-order sum of the strip partials -> der[6] per cell (NaN for inactive cells)
__global__ void k_jac_final(EvalParams p, int n_jobs) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  int total = n_jobs * p.ncell * 6;
  if (idx >= total) return;
  int k = idx % 6;
  const int job = job_at(p, (idx / 6) / p.ncell), c = (idx / 6) % p.ncell;
  size_t o = (size_t)job * p.ncell + c;
  idx = (int)(o * 6 + k);
  int pair = p.job_pair[job];
  if (p.n_c[pair * p.ncell + c] < NID_MIN_CELL_POINTS) { p.der[idx] = nan(""); return; }
  double t = 0.0;
  for (int s = 0; s < p.S; s++) t += p.jpart[(o * p.S + s) * 6 + k];
  p.der[idx] = t;
}

// a11: Huber-weighted Gauss-Newton block over the active cells of a job, in cell order
// (base_unary_edge.hpp:43-72, robust_kernel_impl.cpp:78-90, sparse_optimizer.cpp:102-116).
// One thread per (job, entry): entry 0 chi2, 1..36 H, 37..42 b, 43 active count.
__global__ void __launch_bounds__(128) k_gn(EvalParams p, int want_jac) {
  gn_block(p, job_at(p, blockIdx.x), want_jac, p.gn);
}

// ------------------------------------------------------------------------------------------------
// a12: hard-binned NID (NID_standard_property.cpp:342-485). One CTA per (cell, job); integer counts.
__global__ void __launch_bounds__(256) k_hard(EvalParams p, double* __restrict__ out) {
  extern __shared__ unsigned int cnts[];  // [B*B joint][B ref][B cur][1 n]
  __shared__ double scratch[8];
  const int B = p.bins;
  const int c = blockIdx.x, job = blockIdx.y;
  const int pair = p.job_pair[job];
  const int nslots = B * B + 2 * B + 1;
  for (int i = threadIdx.x; i < nslots; i += blockDim.x) cnts[i] = 0;
  __syncthreads();
  unsigned int* cj = cnts;
  unsigned int* cr = cnts + B * B;
  unsigned int* cc = cr + B;
  unsigned int* cn = cc + B;
  const size_t base = (size_t)pair * p.N;
  const double* cp = p.cam + 4 * pair;
  const Cam cam{cp[0], cp[1], cp[2], cp[3]};
  const Pose P = load_pose(p.poses + 16 * job);
  const int r0 = (c / p.cell) * p.rb, c0 = (c % p.cell) * p.cb;
  const int npx = p.rb * p.cb;
  const uint8_t* im1 = p.im1 + base;
  for (int t = threadIdx.x; t < npx; t += blockDim.x) {
    const int row = r0 + t / p.cb, col = c0 + t % p.cb;
    const size_t i = base + (size_t)row * p.cols + col;
    const double x0 = p.pwx[i];
    if (isnan(x0)) continue;
    double x1, y1, z1, u, v;
    warp_project(P, cam, x0, p.pwy[i], p.pwz[i], x1, y1, z1, u, v);
    if (!inb_cost(u, v, p.rows, p.cols)) continue;
    double i0 = (double)p.im0[i];
    if (i0 >= 255.0) i0 = 254.999;
    int kr = (int)floor(__ddiv_rn(__dmul_rn(i0, (double)B), 255.0));
    double ic = clamp_intensity(interp_u8(im1, p.cols, u, v));
    int kt = (int)floor(__ddiv_rn(__dmul_rn(ic, (double)B), 255.0));
    atomicAdd(&cj[kr * B + kt], 1u);  // the only per-pixel atomic: marginals and n are sums of the joint counts
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * B; i += blockDim.x) {
    unsigned int a = 0;
    if (i < B) for (int k = 0; k < B; k++) a += cj[i * B + k];          // reference marginal: row sums
    else for (int k = 0; k < B; k++) a += cj[k * B + (i - B)];          // target marginal: column sums
    cr[i] = a;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int a = 0;
    for (int k = 0; k < B; k++) a += cr[k];
    *cn = a;
  }
  __syncthreads();
  const unsigned int n = *cn;
  double hj = 0, hr = 0, hc = 0;
  for (int i = threadIdx.x; i < B * B + 2 * B; i += blockDim.x) {
    unsigned int k = cnts[i];
    if (!k) continue;
    double q = (double)k / (double)n;
    double h = (q < kSigma) ? 0.0 : q * log2(q);
    if (i < B * B) hj -= h; else if (i < B * B + B) hr -= h; else hc -= h;
  }
  hj = block_sum(hj, scratch);
  hr = block_sum(hr, scratch);
  hc = block_sum(hc, scratch);
  if (threadIdx.x == 0) {
    double nid = 0.0;
    if (n >= NID_MIN_CELL_POINTS) {
      nid = (2 * hj - hr - hc) / hj;
      if (hr == 0.0 && hc == 0.0 && hj == 0.0) nid = 0.0;
    }
    out[(size_t)job * (p.ncell + 1) + c] = nid;
  }
}

__global__ void k_hard_total(int n_jobs, int ncell, double* __restrict__ out) {
  int job = blockIdx.x * blockDim.x + threadIdx.x;
  if (job >= n_jobs) return;
  double t = 0.0;
  for (int c = 0; c < ncell; c++) { double v = out[(size_t)job * (ncell + 1) + c]; t += v * v; }
  out[(size_t)job * (ncell + 1) + ncell] = sqrt(t);
}

// ------------------------------------------------------------------------------------------------
// Kernel 1 standalone: warp + bilinear sample + image gradient per pixel (parity and HBM roofline).
template <bool F64>
__global__ void __launch_bounds__(256) k_warp_sample(EvalParams p, int pair, const double* __restrict__ pose16,
                                                     float4* __restrict__ out4, double* __restrict__ out8) {
  const size_t base = (size_t)pair * p.N;
  const double* cp = p.cam + 4 * pair;
  const Cam cam{cp[0], cp[1], cp[2], cp[3]};
  const Pose P = load_pose(pose16);
  const uint8_t* im1 = p.im1 + base;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < p.N; i += gridDim.x * blockDim.x) {
    const double x0 = p.pwx[base + i];
    double u = nan(""), v = nan(""), ic = nan(""), gx = nan(""), gy = nan(""), z1 = nan("");
    int vc = 0, vj = 0;
    if (!isnan(x0)) {
      double x1, y1;
      warp_project(P, cam, x0, p.pwy[base + i], p.pwz[base + i], x1, y1, z1, u, v);
      double u2, v2;
      project_jac(cam, x1, y1, z1, u2, v2);
      vc = inb_cost(u, v, p.rows, p.cols);
      vj = vc && inb_jac(u2, v2, p.rows, p.cols);
      ic = 0; gx = 0; gy = 0;
      if (vc) ic = clamp_intensity(interp_u8(im1, p.cols, u, v));
      if (vj) {
        gx = (interp_u8(im1, p.cols, u2 + 1.0, v2) - interp_u8(im1, p.cols, u2 - 1.0, v2)) / 2;
        gy = (interp_u8(im1, p.cols, u2, v2 + 1.0) - interp_u8(im1, p.cols, u2, v2 - 1.0)) / 2;
      }
    }
    if (F64) {
      double* o = out8 + 8 * (size_t)i;
      if (isnan(x0)) {
#pragma unroll
        for (int k = 0; k < 8; k++) o[k] = nan("");
      } else {
        o[0] = u; o[1] = v; o[2] = ic; o[3] = gx; o[4] = gy; o[5] = vc; o[6] = vj; o[7] = z1;
      }
    } else {
      float4 r;
      r.x = (float)ic; r.y = (float)gx; r.z = (float)gy; r.w = (float)(vc + 2 * vj);
      if (isnan(x0)) { r.x = 0.f; r.y = 0.f; r.z = 0.f; r.w = 0.f; }
      out4[i] = r;
    }
  }
}

// ================================================================================================ launchers
static inline int grid_for(int n, int threads, int cap) {
  int g = (n + threads - 1) / threads;
  return g < cap ? (g < 1 ? 1 : g) : cap;
}

int launch_build_lut(nid_ctx* c) {
  k_build_lut<<<1, 256, 0, c->stream>>>(c->bins, c->lut_w, c->lut_k);
  NID_LAUNCH_CHECK(c, "k_build_lut");
  return NID_OK;
}

int launch_points(nid_ctx* c, int pair0, int n, bool u16) {
  const dim3 grid(grid_for(c->N, 256, std::max(8, c->sm_count * 8 / n)), n);
  if (u16) k_points<true><<<grid, 256, 0, c->stream>>>(c->rows, c->cols, pair0, c->depth, c->depth16, c->depth_factor, c->Twc0, c->cam, c->pwx, c->pwy, c->pwz);
  else k_points<false><<<grid, 256, 0, c->stream>>>(c->rows, c->cols, pair0, c->depth, nullptr, nullptr, c->Twc0, c->cam, c->pwx, c->pwy, c->pwz);
  NID_LAUNCH_CHECK(c, "k_points");
  return NID_OK;
}

int launch_downsample2(nid_ctx* dst, int dst_pair0, const nid_ctx* src, int src_pair0, int n) {
  const dim3 grid(grid_for(dst->N, 256, std::max(8, dst->sm_count * 8 / n)), n);
  const size_t sb = (size_t)src_pair0 * src->N, db = (size_t)dst_pair0 * dst->N;
  k_downsample2<<<grid, 256, 0, dst->stream>>>(src->cols, dst->rows, dst->cols, src->depth + sb, src->im0 + sb, src->im1 + sb,
                                               (size_t)src->N, dst->depth + db, dst->im0 + db, dst->im1 + db, (size_t)dst->N);
  NID_LAUNCH_CHECK(dst, "k_downsample2");
  return NID_OK;
}

int launch_points_aos(nid_ctx* c, int pair, double* d_out) {
  size_t b = (size_t)pair * c->N;
  k_points_aos<<<grid_for(c->N, 256, c->sm_count * 8), 256, 0, c->stream>>>(c->N, c->pwx + b, c->pwy + b, c->pwz + b, d_out);
  NID_LAUNCH_CHECK(c, "k_points_aos");
  return NID_OK;
}

int launch_points_soa(nid_ctx* c, int pair, const double* d_in) {
  size_t b = (size_t)pair * c->N;
  k_points_soa<<<grid_for(c->N, 256, c->sm_count * 8), 256, 0, c->stream>>>(c->N, d_in, c->pwx + b, c->pwy + b, c->pwz + b);
  NID_LAUNCH_CHECK(c, "k_points_soa");
  return NID_OK;
}

int launch_import_flags(nid_ctx* c, int pair, const double* d_bsv) {
  k_import_flags<<<grid_for(c->N, 256, c->sm_count * 8), 256, 0, c->stream>>>(c->N, d_bsv, c->inb0 + (size_t)pair * c->N);
  NID_LAUNCH_CHECK(c, "k_import_flags");
  return NID_OK;
}

int launch_check_integral(nid_ctx* c, const double* d_src, uint8_t* d_dst, int is_ref) {
  k_check_integral<<<grid_for(c->N, 256, c->sm_count * 8), 256, 0, c->stream>>>(c->N, d_src, d_dst, c->d_flag, is_ref);
  NID_LAUNCH_CHECK(c, "k_check_integral");
  return NID_OK;
}

int launch_prepare(nid_ctx* c, int pair0, int n, const double* d_poses16) {
  EvalParams p = make_params(c, 1);
  cudaError_t e = cudaMemsetAsync(c->cnt + (size_t)pair0 * c->ncell * NID_NCLS, 0, sizeof(unsigned int) * c->ncell * NID_NCLS * n, c->stream);
  if (e != cudaSuccess) return check_cuda(e, "memset cnt");
  const dim3 grid(grid_for(c->N, 256, std::max(8, c->sm_count * 8 / n)), n);
  k_prepare<<<grid, 256, 0, c->stream>>>(p, pair0, d_poses16, c->inb0, c->cnt);
  NID_LAUNCH_CHECK(c, "k_prepare");
  return NID_OK;
}

int launch_href(nid_ctx* c, int pair0, int n) {
  EvalParams p = make_params(c, 1);
  k_href<<<dim3(c->ncell, n), 256, sizeof(double) * c->bins, c->stream>>>(p, pair0, c->cnt, c->n_c, c->href);
  NID_LAUNCH_CHECK(c, "k_href");
  return NID_OK;
}

int launch_ref_weights(nid_ctx* c, int pair) {
  EvalParams p = make_params(c, 1);
  k_ref_weights<<<grid_for(c->N, 256, c->sm_count * 8), 256, 0, c->stream>>>(p, pair, c->d_bsv, c->d_bsi);
  NID_LAUNCH_CHECK(c, "k_ref_weights");
  return NID_OK;
}

int launch_gn(nid_ctx* c, const JobSet& js, double delta, int want_jac) {
  EvalParams p = make_params(c, js.slots);
  p.huber_delta = delta;
  p.huber_dsqr = (double)(float)(delta * delta);  // `float dsqr`, robust_kernel_impl.h:84
  p.job0 = js.first;
  p.job_list = js.d_list;
  k_gn<<<js.n, 128, 0, c->stream>>>(p, want_jac);
  NID_LAUNCH_CHECK(c, want_jac ? "k_gn" : "k_gn(chi2)");
  return NID_OK;
}

int launch_hard(nid_ctx* c, int n_jobs) {
  EvalParams p = make_params(c, n_jobs);
  size_t smem = sizeof(unsigned int) * (p.bins * p.bins + 2 * p.bins + 1);
  dim3 g(p.ncell, n_jobs);
  k_hard<<<g, 256, smem, c->stream>>>(p, c->hard);
  NID_LAUNCH_CHECK(c, "k_hard");
  k_hard_total<<<(n_jobs + 127) / 128, 128, 0, c->stream>>>(n_jobs, p.ncell, c->hard);
  NID_LAUNCH_CHECK(c, "k_hard_total");
  return NID_OK;
}

int launch_warp_sample(nid_ctx* c, int pair, const double* d_pose16, int f64) {
  EvalParams p = make_params(c, 1);
  int g = grid_for(c->N, 256, c->sm_count * 8);
  if (f64) k_warp_sample<true><<<g, 256, 0, c->stream>>>(p, pair, d_pose16, nullptr, c->d_pix);
  else k_warp_sample<false><<<g, 256, 0, c->stream>>>(p, pair, d_pose16, (float4*)c->d_pix4.get(), nullptr);
  NID_LAUNCH_CHECK(c, "k_warp_sample");
  return NID_OK;
}

}  // namespace nid
