// Host-side pose algebra and 6x6 solve used by the LM driver and the apps (fp64, header-only).
// The reference takes these from Eigen and g2o's SE3Quat; neither is available to (or wanted by) this
// build, so the few operations the path needs are written out with the same conventions:
//   pose7 = {tx,ty,tz,qx,qy,qz,qw}  (g2o SE3Quat::toVector, se3quat.h:144-154)
//   mat16 = column-major 4x4        (Eigen .data(), se3quat.h:270-278)
//   update T <- exp(xi) * T, xi = (omega, upsilon)   (types_six_dof_expmap.h:74-77, se3quat.h:223-257)
#pragma once
#include <cmath>
#include <cstring>
#include <limits>
#include <utility>

namespace nidhost {

struct Pose7 {
  double t[3];
  double q[4];  // x y z w
};

inline void q_normalize_pos_w(double q[4]) {  // se3quat.h:280-285
  if (q[3] < 0) for (int i = 0; i < 4; i++) q[i] = -q[i];
  double n = std::sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  for (int i = 0; i < 4; i++) q[i] /= n;
}

// rotation matrix -> quaternion, branch structure of Eigen's Quaternion(Matrix3)
inline void q_from_R(const double R[3][3], double q[4]) {
  double tr = R[0][0] + R[1][1] + R[2][2];
  if (tr > 0.0) {
    double s = std::sqrt(tr + 1.0);
    q[3] = 0.5 * s;
    s = 0.5 / s;
    q[0] = (R[2][1] - R[1][2]) * s;
    q[1] = (R[0][2] - R[2][0]) * s;
    q[2] = (R[1][0] - R[0][1]) * s;
  } else {
    int i = 0;
    if (R[1][1] > R[0][0]) i = 1;
    if (R[2][2] > R[i][i]) i = 2;
    int j = (i + 1) % 3, k = (j + 1) % 3;
    double s = std::sqrt(R[i][i] - R[j][j] - R[k][k] + 1.0);
    q[i] = 0.5 * s;
    s = 0.5 / s;
    q[3] = (R[k][j] - R[j][k]) * s;
    q[j] = (R[j][i] + R[i][j]) * s;
    q[k] = (R[k][i] + R[i][k]) * s;
  }
}

inline void q_to_R(const double q[4], double R[3][3]) {
  const double x2 = 2 * q[0], y2 = 2 * q[1], z2 = 2 * q[2];
  const double wx = x2 * q[3], wy = y2 * q[3], wz = z2 * q[3];
  const double xx = x2 * q[0], xy = y2 * q[0], xz = z2 * q[0];
  const double yy = y2 * q[1], yz = z2 * q[1], zz = z2 * q[2];
  R[0][0] = 1 - (yy + zz); R[0][1] = xy - wz; R[0][2] = xz + wy;
  R[1][0] = xy + wz; R[1][1] = 1 - (xx + zz); R[1][2] = yz - wx;
  R[2][0] = xz - wy; R[2][1] = yz + wx; R[2][2] = 1 - (xx + yy);
}

inline void q_mul(const double a[4], const double b[4], double o[4]) {
  double r[4];
  r[3] = a[3] * b[3] - a[0] * b[0] - a[1] * b[1] - a[2] * b[2];
  r[0] = a[3] * b[0] + a[0] * b[3] + a[1] * b[2] - a[2] * b[1];
  r[1] = a[3] * b[1] + a[1] * b[3] + a[2] * b[0] - a[0] * b[2];
  r[2] = a[3] * b[2] + a[2] * b[3] + a[0] * b[1] - a[1] * b[0];
  std::memcpy(o, r, sizeof(r));
}

inline void q_rot(const double q[4], const double v[3], double o[3]) {
  double c[3] = {2 * (q[1] * v[2] - q[2] * v[1]), 2 * (q[2] * v[0] - q[0] * v[2]), 2 * (q[0] * v[1] - q[1] * v[0])};
  double r[3] = {v[0] + q[3] * c[0] + (q[1] * c[2] - q[2] * c[1]), v[1] + q[3] * c[1] + (q[2] * c[0] - q[0] * c[2]),
                 v[2] + q[3] * c[2] + (q[0] * c[1] - q[1] * c[0])};
  o[0] = r[0]; o[1] = r[1]; o[2] = r[2];
}

inline Pose7 pose_from_Rt(const double R[3][3], const double t[3]) {
  Pose7 P;
  q_from_R(R, P.q);
  q_normalize_pos_w(P.q);
  P.t[0] = t[0]; P.t[1] = t[1]; P.t[2] = t[2];
  return P;
}

inline Pose7 pose_from_mat16(const double m[16]) {
  double R[3][3], t[3];
  for (int r = 0; r < 3; r++) {
    for (int c = 0; c < 3; c++) R[r][c] = m[4 * c + r];
    t[r] = m[12 + r];
  }
  return pose_from_Rt(R, t);
}

inline void pose_to_mat16(const Pose7& P, double m[16]) {
  double R[3][3];
  q_to_R(P.q, R);
  for (int c = 0; c < 3; c++) {
    for (int r = 0; r < 3; r++) m[4 * c + r] = R[r][c];
    m[4 * c + 3] = 0.0;
  }
  m[12] = P.t[0]; m[13] = P.t[1]; m[14] = P.t[2]; m[15] = 1.0;
}

inline Pose7 pose_mul(const Pose7& a, const Pose7& b) {  // se3quat.h:102-108
  Pose7 r;
  double rt[3];
  q_rot(a.q, b.t, rt);
  for (int i = 0; i < 3; i++) r.t[i] = a.t[i] + rt[i];
  q_mul(a.q, b.q, r.q);
  q_normalize_pos_w(r.q);
  return r;
}

inline Pose7 pose_inverse(const Pose7& a) {  // se3quat.h:124-129
  Pose7 r;
  r.q[0] = -a.q[0]; r.q[1] = -a.q[1]; r.q[2] = -a.q[2]; r.q[3] = a.q[3];
  double nt[3] = {-a.t[0], -a.t[1], -a.t[2]};
  q_rot(r.q, nt, r.t);
  return r;
}

inline Pose7 pose_exp(const double xi[6]) {  // se3quat.h:223-257
  const double* w = xi;
  const double* up = xi + 3;
  const double th = std::sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]);
  double O[3][3] = {{0, -w[2], w[1]}, {w[2], 0, -w[0]}, {-w[1], w[0], 0}};
  double O2[3][3];
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) {
      double s = 0;
      for (int k = 0; k < 3; k++) s += O[i][k] * O[k][j];
      O2[i][j] = s;
    }
  double R[3][3], V[3][3];
  if (th < 0.00001) {
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) V[i][j] = R[i][j] = (i == j) + O[i][j] + O2[i][j];
  } else {
    const double a = std::sin(th) / th, b = (1 - std::cos(th)) / (th * th), c = (th - std::sin(th)) / std::pow(th, 3);
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) {
        R[i][j] = (i == j) + a * O[i][j] + b * O2[i][j];
        V[i][j] = (i == j) + b * O[i][j] + c * O2[i][j];
      }
  }
  double t[3];
  for (int i = 0; i < 3; i++) t[i] = V[i][0] * up[0] + V[i][1] * up[1] + V[i][2] * up[2];
  return pose_from_Rt(R, t);
}

// 6x6 adjoint (row-major) of a rigid column-major 4x4 E = [R t; 0 1] for xi = (omega, upsilon):
// E * exp(xi) * E^-1 = exp(Ad * xi), Ad = [[R, 0], [t^ R, R]].
inline void adjoint6(const double E[16], double Ad[36]) {
  double R[3][3], tx[3][3];
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) R[r][c] = E[4 * c + r];
  const double* t = E + 12;
  tx[0][0] = 0; tx[0][1] = -t[2]; tx[0][2] = t[1];
  tx[1][0] = t[2]; tx[1][1] = 0; tx[1][2] = -t[0];
  tx[2][0] = -t[1]; tx[2][1] = t[0]; tx[2][2] = 0;
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) {
      double s = 0;
      for (int k = 0; k < 3; k++) s += tx[r][k] * R[k][c];
      Ad[6 * r + c] = R[r][c];
      Ad[6 * r + c + 3] = 0.0;
      Ad[6 * (r + 3) + c] = s;
      Ad[6 * (r + 3) + c + 3] = R[r][c];
    }
}

// A Gauss-Newton block {chi2, H[36] row-major, b[6], n_active} of a camera whose pose is E * T, re-expressed for the update
// T <- exp(xi) * T of the body pose T: J_body = J_cam * Ad(E), so H -> Ad^T H Ad and b -> Ad^T b; chi2 and n_active stay.
inline void gn_block_to_body(const double Ad[36], const double in[44], double out[44]) {
  const double* H = in + 1;
  double HA[36];
  for (int i = 0; i < 6; i++)
    for (int j = 0; j < 6; j++) {
      double s = 0;
      for (int k = 0; k < 6; k++) s += H[6 * i + k] * Ad[6 * k + j];
      HA[6 * i + j] = s;
    }
  for (int i = 0; i < 6; i++) {
    for (int j = 0; j < 6; j++) {
      double s = 0;
      for (int k = 0; k < 6; k++) s += Ad[6 * k + i] * HA[6 * k + j];
      out[1 + 6 * i + j] = s;
    }
    double s = 0;
    for (int k = 0; k < 6; k++) s += Ad[6 * k + i] * in[37 + k];
    out[37 + i] = s;
  }
  out[0] = in[0];
  out[43] = in[43];
}

// The block of a group of n jobs sharing one pose: the sum of the jobs' blocks in job order (blocks[44 * i ..]), each first
// taken to the body frame when Ad is given (Ad[36 * i ..] per job). The first block is copied, not added to zero, so that a
// group of one without Ad returns its job's block bit for bit.
inline void gn_combine(int n, const double* blocks, const double* Ad, double out[44]) {
  double tmp[44];
  for (int i = 0; i < n; i++) {
    const double* g = blocks + 44 * (size_t)i;
    if (Ad) {
      gn_block_to_body(Ad + 36 * (size_t)i, g, tmp);
      g = tmp;
    }
    if (i == 0) std::memcpy(out, g, sizeof(double) * 44);
    else for (int k = 0; k < 44; k++) out[k] += g[k];
  }
}

// Is m a rigid column-major 4x4: bottom row exactly (0, 0, 0, 1), R^T R = I to tol per entry, det R > 0?
inline bool is_rigid(const double m[16], double tol = 1e-9) {
  if (!(m[3] == 0.0 && m[7] == 0.0 && m[11] == 0.0 && m[15] == 1.0)) return false;
  for (int i = 0; i < 16; i++) if (!std::isfinite(m[i])) return false;
  for (int a = 0; a < 3; a++)
    for (int b = 0; b < 3; b++) {
      double s = 0;
      for (int r = 0; r < 3; r++) s += m[4 * a + r] * m[4 * b + r];
      if (std::fabs(s - (a == b ? 1.0 : 0.0)) > tol) return false;
    }
  const double det = m[0] * (m[5] * m[10] - m[9] * m[6]) - m[4] * (m[1] * m[10] - m[9] * m[2]) + m[8] * (m[1] * m[6] - m[5] * m[2]);
  return det > 0;
}

// out = A * B for column-major 4x4 (out may not alias A or B)
inline void mat16_mul(const double A[16], const double B[16], double out[16]) {
  for (int c = 0; c < 4; c++)
    for (int r = 0; r < 4; r++) {
      double s = 0;
      for (int k = 0; k < 4; k++) s += A[4 * k + r] * B[4 * c + k];
      out[4 * c + r] = s;
    }
}

// Huber, robust_kernel_impl.cpp:78-90 with the `float dsqr` of robust_kernel_impl.h:84
inline void huber(double e2, double delta, double rho[3]) {
  const double dsqr = (double)(float)(delta * delta);
  if (e2 <= dsqr) {
    rho[0] = e2; rho[1] = 1; rho[2] = 0;
  } else {
    const double s = std::sqrt(e2);
    rho[0] = 2 * s * delta - dsqr;
    rho[1] = delta / s;
    rho[2] = -0.5 * rho[1] / e2;
  }
}

// 6x6 symmetric solve as linear_solver_dense.h:104-110 does it: LDL^T with symmetric pivoting on the
// largest |diagonal|, accepted only if no negative pivot shows up. Returns false otherwise (x untouched).
inline bool ldlt6_solve(const double H[36], const double b[6], double x[6]) {
  const int n = 6;
  double A[6][6];
  for (int i = 0; i < n; i++) for (int j = 0; j < n; j++) A[i][j] = H[6 * i + j];
  int perm[6];
  int sign = 0;
  bool zero_seen = false;
  for (int k = 0; k < n; k++) {
    int piv = k;
    double best = std::fabs(A[k][k]);
    for (int i = k + 1; i < n; i++)
      if (std::fabs(A[i][i]) > best) { best = std::fabs(A[i][i]); piv = i; }
    perm[k] = piv;
    if (piv != k) {
      for (int j = 0; j < k; j++) std::swap(A[k][j], A[piv][j]);
      for (int i = piv + 1; i < n; i++) std::swap(A[i][k], A[i][piv]);
      std::swap(A[k][k], A[piv][piv]);
      for (int i = k + 1; i < piv; i++) std::swap(A[i][k], A[piv][i]);
    }
    if (k > 0) {
      double tmp[6];
      for (int j = 0; j < k; j++) tmp[j] = A[j][j] * A[k][j];
      double s = 0;
      for (int j = 0; j < k; j++) s += A[k][j] * tmp[j];
      A[k][k] -= s;
      for (int i = k + 1; i < n; i++) {
        double s2 = 0;
        for (int j = 0; j < k; j++) s2 += A[i][j] * tmp[j];
        A[i][k] -= s2;
      }
    }
    const double d = A[k][k];
    const bool valid = std::fabs(d) > 0.0;
    if (k == 0 && !valid) {
      for (int j = 0; j < n; j++) perm[j] = j;
      break;
    }
    if (valid) for (int i = k + 1; i < n; i++) A[i][k] /= d;
    if (zero_seen && valid) sign = 2;
    else if (!valid) zero_seen = true;
    if (sign == 1) { if (d < 0) sign = 2; }
    else if (sign == -1) { if (d > 0) sign = 2; }
    else if (sign == 0) { if (d > 0) sign = 1; else if (d < 0) sign = -1; }
  }
  if (!(sign == 1 || sign == 0)) return false;
  double y[6];
  for (int i = 0; i < n; i++) y[i] = b[i];
  for (int k = 0; k < n; k++) std::swap(y[k], y[perm[k]]);
  for (int i = 0; i < n; i++) for (int j = 0; j < i; j++) y[i] -= A[i][j] * y[j];
  const double tiny = std::numeric_limits<double>::min();
  for (int i = 0; i < n; i++) y[i] = (std::fabs(A[i][i]) > tiny) ? y[i] / A[i][i] : 0.0;
  for (int i = n - 1; i >= 0; i--) for (int j = i + 1; j < n; j++) y[i] -= A[j][i] * y[j];
  for (int k = n - 1; k >= 0; k--) std::swap(y[k], y[perm[k]]);
  for (int i = 0; i < n; i++) x[i] = y[i];
  return true;
}

// The reference's initial-guess perturbation (NID_pose_estimation.cpp:186-208): T_wc1 -> perturbed T_cw1
inline Pose7 reference_perturbation(const double Twc1[16]) {
  const double t_off = 0.02, r_off = 0.005;
  const double td[3] = {0.5 * t_off, -t_off, -t_off};
  const double a = r_off * M_PI, c = std::cos(a), s = std::sin(a);
  const double Rx[3][3] = {{1, 0, 0}, {0, c, -s}, {0, s, c}};
  const double Ry[3][3] = {{c, 0, s}, {0, 1, 0}, {-s, 0, c}};
  const double Rz[3][3] = {{c, -s, 0}, {s, c, 0}, {0, 0, 1}};
  auto mm = [](const double A[3][3], const double B[3][3], double C[3][3]) {
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) {
        double v = 0;
        for (int k = 0; k < 3; k++) v += A[i][k] * B[k][j];
        C[i][j] = v;
      }
  };
  double Rxy[3][3], Rd[3][3], Rcw[3][3], R2[3][3], tcw[3];
  mm(Rx, Ry, Rxy);
  mm(Rxy, Rz, Rd);
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) Rcw[i][j] = Twc1[4 * i + j];
  for (int i = 0; i < 3; i++) {
    double v = 0;
    for (int j = 0; j < 3; j++) v += (-Rcw[i][j]) * Twc1[12 + j];
    tcw[i] = v + td[i];
  }
  mm(Rd, Rcw, R2);
  return pose_from_Rt(R2, tcw);
}

}  // namespace nidhost
