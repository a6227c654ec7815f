// Device-side building blocks of the NID path (sm_100a). All arithmetic fp64.
// Citations: file:line in arpg/NID-Pose-Estimation.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace nid {

constexpr double kSigma = 1e-30;  // types_six_dof_expmap.h:281

struct Cam {
  double fx, fy, cx, cy;
};

// 3x4 part of a column-major 4x4
struct Pose {
  double m[12];  // m[4*c + r] -> stored as r0c0,r1c0,r2c0, r0c1,... (3 per column)
};

__device__ __forceinline__ Pose load_pose(const double* __restrict__ p16) {
  Pose P;
#pragma unroll
  for (int c = 0; c < 4; c++)
#pragma unroll
    for (int r = 0; r < 3; r++) P.m[3 * c + r] = p16[4 * c + r];
  return P;
}

// computeH.cu:152-158 evaluated in the reference's operation order without fused
// multiply-adds, so that (u, v) and the in-bounds decisions taken from them are bit-identical to a
// contraction-free CPU evaluation of the same expressions.
__device__ __forceinline__ void warp_project(const Pose& P, const Cam& cam, double x0, double y0, double z0,
                                             double& x1, double& y1, double& z1, double& u, double& v) {
  x1 = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(P.m[0], x0), __dmul_rn(P.m[3], y0)), __dmul_rn(P.m[6], z0)), P.m[9]);
  y1 = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(P.m[1], x0), __dmul_rn(P.m[4], y0)), __dmul_rn(P.m[7], z0)), P.m[10]);
  z1 = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(P.m[2], x0), __dmul_rn(P.m[5], y0)), __dmul_rn(P.m[8], z0)), P.m[11]);
  u = __dadd_rn(__ddiv_rn(__dmul_rn(cam.fx, x1), z1), cam.cx);
  v = __dadd_rn(__ddiv_rn(__dmul_rn(cam.fy, y1), z1), cam.cy);
}

// The CPU edge projects a second time in linearizeOplus, as fx*(x/z)+cx (types_six_dof_expmap.cpp:407-421);
// its Jacobian bounds test (:433) and gradient samples (:434-435) use this value, which can differ from
// warp_project's (fx*x)/z+cx in the last bit -- visible only when (u, v) sits on an integer.
__device__ __forceinline__ void project_jac(const Cam& cam, double x1, double y1, double z1, double& u2, double& v2) {
  u2 = __dadd_rn(__dmul_rn(cam.fx, __ddiv_rn(x1, z1)), cam.cx);
  v2 = __dadd_rn(__dmul_rn(cam.fy, __ddiv_rn(y1, z1)), cam.cy);
}

// CudaPoints3d.cu:20-28 (same order, no contraction)
__device__ __forceinline__ void backproject(const double* __restrict__ T, const Cam& cam, double z, int row, int col,
                                            double& xw, double& yw, double& zw) {
  double x0 = __ddiv_rn(__dmul_rn(z, __dsub_rn((double)col, cam.cx)), cam.fx);
  double y0 = __ddiv_rn(__dmul_rn(z, __dsub_rn((double)row, cam.cy)), cam.fy);
  xw = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(T[0], x0), __dmul_rn(T[4], y0)), __dmul_rn(T[8], z)), T[12]);
  yw = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(T[1], x0), __dmul_rn(T[5], y0)), __dmul_rn(T[9], z)), T[13]);
  zw = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(T[2], x0), __dmul_rn(T[6], y0)), __dmul_rn(T[10], z)), T[14]);
}

// in-bounds tests: cost `u+3<=cols` (types_six_dof_expmap.cpp:565), Jacobian `u+3<=cols-1` (:433)
__device__ __forceinline__ bool inb_cost(double u, double v, int rows, int cols) {
  return u >= 0 && __dadd_rn(u, 3.0) <= (double)cols && v >= 0 && __dadd_rn(v, 3.0) <= (double)rows;
}
__device__ __forceinline__ bool inb_jac(double u, double v, int rows, int cols) {
  return u >= 0 && __dadd_rn(u, 3.0) <= (double)(cols - 1) && v >= 0 && __dadd_rn(v, 3.0) <= (double)rows;
}

// types_six_dof_expmap.h:310-328: bilinear with (int) truncation (so u in (-1,0) extrapolates from
// columns 0/1, which the gradient taps u-1 / v-1 rely on). The Jacobian bounds test admits u == 0 and v == 0
// exactly (types_six_dof_expmap.cpp:433), whose taps u-1 / v-1 == -1.0 truncate to column / row -1: upstream
// that is an out-of-bounds cv::Mat access (undefined). Defined here, and in the oracle, as the continuous
// extension of the (-1, 0) case: the index is clamped to 0 and the fraction becomes -1 (extrapolation from
// columns / rows 0 and 1), so no byte outside the image is ever read.
__device__ __forceinline__ double interp_u8(const uint8_t* __restrict__ im, int cols, double x, double y) {
  int ix = max((int)x, 0);
  int iy = max((int)y, 0);
  double dx = x - (double)ix;
  double dy = y - (double)iy;
  double dxdy = __dmul_rn(dx, dy);
  const uint8_t* r0 = im + (size_t)iy * cols + ix;
  const uint8_t* r1 = r0 + cols;
  double p00 = (double)__ldg(r0), p01 = (double)__ldg(r0 + 1);
  double p10 = (double)__ldg(r1), p11 = (double)__ldg(r1 + 1);
  // the reference's term order without fused multiply-adds: on a saturated plateau the `>= 255` clamp that
  // follows sees the last bit of this sum
  double a = __dmul_rn(dxdy, p11);
  a = __dadd_rn(a, __dmul_rn(__dsub_rn(dy, dxdy), p10));
  a = __dadd_rn(a, __dmul_rn(__dsub_rn(dx, dxdy), p01));
  return __dadd_rn(a, __dmul_rn(__dadd_rn(__dsub_rn(__dsub_rn(1.0, dx), dy), dxdy), p00));
}

__device__ __forceinline__ double clamp_intensity(double ic) {
  // types_six_dof_expmap.cpp:572-575
  if (ic >= 255.0) ic = 254.999;
  if (ic < 0.0) ic = 0.0;
  return ic;
}

// Clamped uniform knots t_k = clamp(k-3, 0, B-3) (computeH.cu:99-112 tables in closed form)
__device__ __forceinline__ int knot_i(int k, int bins) { return min(max(k - 3, 0), bins - 3); }

__device__ __forceinline__ double rcp_small(int d) {
  // knot differences on this knot vector are 1, 2 or 3
  return d == 1 ? 1.0 : (d == 2 ? 0.5 : (1.0 / 3.0));
}

// The four non-zero cubic basis functions N_{k..k+3}(ub), k = floor(ub), and optionally their
// derivatives. Non-recursive de Boor triangle (Piegl & Tiller A2.2/A2.3); equal to the reference's
// Cox-de Boor recursion (types_six_dof_expmap.cpp:738-800) everywhere, including its one quirk:
// the derivative is returned as 0 at ub == 0 exactly (SURVEY A-3).
template <bool WANT_DER>
__device__ __forceinline__ void bspline4(double ub, int k, int bins, double w[4], double dw[4]) {
  const int mu = k + 3;  // t_mu <= ub < t_{mu+1}
  double left[4], right[4];
#pragma unroll
  for (int j = 1; j <= 3; j++) {
    left[j] = ub - (double)knot_i(mu + 1 - j, bins);
    right[j] = (double)knot_i(mu + j, bins) - ub;
  }
  double N[4];
  double Q[3] = {0, 0, 0};
  N[0] = 1.0;
#pragma unroll
  for (int j = 1; j <= 3; j++) {
    double saved = 0.0;
#pragma unroll
    for (int r = 0; r < j; r++) {
      // right[r+1] + left[j-r] == t_{mu+r+1} - t_{mu+1-j+r}
      int den = knot_i(mu + r + 1, bins) - knot_i(mu + 1 - j + r, bins);
      double temp = N[r] * rcp_small(den);
      N[r] = saved + right[r + 1] * temp;
      saved = left[j - r] * temp;
    }
    N[j] = saved;
    if (WANT_DER && j == 2) {
      Q[0] = N[0]; Q[1] = N[1]; Q[2] = N[2];
    }
  }
#pragma unroll
  for (int r = 0; r < 4; r++) w[r] = N[r];
  if (WANT_DER) {
#pragma unroll
    for (int r = 0; r < 4; r++) {
      const int i = mu - 3 + r;
      double d = 0.0;
      if (r >= 1) d += 3.0 * Q[r - 1] * rcp_small(knot_i(i + 3, bins) - knot_i(i, bins));
      if (r <= 2) d -= 3.0 * Q[r] * rcp_small(knot_i(i + 4, bins) - knot_i(i + 1, bins));
      dw[r] = (ub == 0.0) ? 0.0 : d;
    }
  }
}

// ---- fast variants used by the sorted kernels -----------------------------------------------------
// exact small-integer -> double without the I2F.F64 path: bits(2^52 + v) - 2^52 (one move + one DADD)
__device__ __forceinline__ double u2d(unsigned v) { return __hiloint2double(0x43300000, (int)v) - 4503599627370496.0; }
__device__ __forceinline__ double i2d_small(int v) {  // |v| < 2^20
  return __hiloint2double(0x43300000, v + 1048576) - (4503599627370496.0 + 1048576.0);
}

// Centre sample and central-difference gradient (types_six_dof_expmap.cpp:434-435 via .h:310-328) from
// 12 taps instead of 5 x 4: for u,v >= 1 the five bilinear samples share their fractional weights.
// The first image row/column (where (int)(u-1) truncates towards zero) takes the literal formula.
__device__ __forceinline__ void sample_grad_u8(const uint8_t* __restrict__ im, int cols, double u, double v,
                                               double& ic, double& gx, double& gy) {
  const int ix = (int)u, iy = (int)v;
  if (ix >= 1 && iy >= 1) {
    const double dx = u - u2d((unsigned)ix), dy = v - u2d((unsigned)iy);
    const double w11 = dx * dy, w10 = dy - w11, w01 = dx - w11, w00 = 1.0 - dx - dy + w11;
    const uint8_t* r0 = im + (size_t)(iy - 1) * cols + (ix - 1);
    const uint8_t* r1 = r0 + cols;
    const uint8_t* r2 = r1 + cols;
    const uint8_t* r3 = r2 + cols;
    const int a01 = __ldg(r0 + 1), a02 = __ldg(r0 + 2);
    const int a10 = __ldg(r1), a11 = __ldg(r1 + 1), a12 = __ldg(r1 + 2), a13 = __ldg(r1 + 3);
    const int a20 = __ldg(r2), a21 = __ldg(r2 + 1), a22 = __ldg(r2 + 2), a23 = __ldg(r2 + 3);
    const int a31 = __ldg(r3 + 1), a32 = __ldg(r3 + 2);
    ic = w11 * u2d(a22) + w10 * u2d(a21) + w01 * u2d(a12) + w00 * u2d(a11);
    gx = (w11 * i2d_small(a23 - a21) + w10 * i2d_small(a22 - a20) + w01 * i2d_small(a13 - a11) + w00 * i2d_small(a12 - a10)) * 0.5;
    gy = (w11 * i2d_small(a32 - a12) + w10 * i2d_small(a31 - a11) + w01 * i2d_small(a22 - a02) + w00 * i2d_small(a21 - a01)) * 0.5;
  } else {
    ic = interp_u8(im, cols, u, v);
    gx = (interp_u8(im, cols, u + 1.0, v) - interp_u8(im, cols, u - 1.0, v)) / 2;
    gy = (interp_u8(im, cols, u, v + 1.0) - interp_u8(im, cols, u, v - 1.0)) / 2;
  }
}

__device__ __forceinline__ double interp_u8_fast(const uint8_t* __restrict__ im, int cols, double x, double y) {
  const int ix = (int)x, iy = (int)y;  // x, y >= 0 here
  const double dx = x - u2d((unsigned)ix), dy = y - u2d((unsigned)iy);
  const double dxdy = dx * dy;
  const uint8_t* r0 = im + (size_t)iy * cols + ix;
  const uint8_t* r1 = r0 + cols;
  return dxdy * u2d(__ldg(r1 + 1)) + (dy - dxdy) * u2d(__ldg(r1)) + (dx - dxdy) * u2d(__ldg(r0 + 1)) +
         (1.0 - dx - dy + dxdy) * u2d(__ldg(r0));
}

// deterministic block-wide sum (fixed tree): every thread gets the total. `scratch` >= blockDim/32 doubles.
__device__ __forceinline__ double block_sum(double v, double* scratch) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int nw = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if (lane == 0) scratch[wid] = v;
  __syncthreads();
  double t = 0.0;
  for (int i = 0; i < nw; i++) t += scratch[i];
  return t;
}

}  // namespace nid
