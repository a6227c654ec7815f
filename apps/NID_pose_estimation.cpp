// NID_pose_estimation <config.yaml> -- the reference's first binary (NID_pose_estimation.cpp:55-399) on the
// B200-native path: same YAML keys (config_eth_cvg.yaml), same ETH-CVG layout, same perturbation of the ground-truth
// pose, same LM schedule (optimize(10)), same printed lines and the same nid_error.csv row. The g2o graph is
// replaced by the C-ABI of include/nid_b200.h: nid_set_pair (Calculate3Dpoint), nid_prepare (CudaComputeHref),
// nid_solve (optimizer.optimize). Optional extra keys: cell (16), bin_num (10), iterations (10), use_gpu is
// accepted and must be 1: there is no CPU path in this build.
// pyramid_levels (1): with L > 1 the solve is coarse-to-fine, for starting poses farther from the answer than the
// reference's perturbation. Level l (1..L-1) halves the resolution l times (nid_set_pairs_downsampled) with cell
// max(1, cell >> l), so that a cell keeps its pixel count; nid_solve_pyramid_jobs solves levels L-1 .. 1 with `iterations`
// each, then level 0 is prepared and solved at the pose they hand down, exactly as with L == 1. One extra line per
// coarse level reports its outer iterations; every other printed line and the CSV row keep their formats.
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <fstream>
#include <iostream>

#include "../include/nid_b200.h"
#include "../nid-pose-estimation_b200/host/nid_host_math.hpp"
#include "nid_io.hpp"

static void die(const char* what) {
  std::fprintf(stderr, "%s: %s\n", what, nid_last_error());
  std::exit(1);
}

int main(int argc, char** argv) {
  if (argc != 2) {
    std::cout << "usage './program path_to_config.yaml', image1's timestamp should be smaller than image2" << std::endl;
    return 0;
  }
  try {
    const nidio::Config cfg = nidio::read_config(argv[1]);
    const int cell = cfg.integer("cell", 16), bins = cfg.integer("bin_num", 10), iters = cfg.integer("iterations", 10);
    const int levels = cfg.integer("pyramid_levels", 1);
    if (levels < 1 || levels > 8) {
      std::fprintf(stderr, "pyramid_levels must be in [1, 8]\n");
      return 2;
    }
    if (cfg.has("use_gpu") && cfg.integer("use_gpu") == 0) {
      std::fprintf(stderr, "use_gpu: 0 requested, but this build has no CPU evaluation path\n");
      return 2;
    }
    const int pose_id0 = atoi(cfg.str("image0_id").c_str()), pose_id1 = atoi(cfg.str("image1_id").c_str());
    std::cout << "optimize relative pose between " << pose_id0 << " and " << pose_id1 << ", in string " << cfg.str("image0_id") << ","
              << cfg.str("image1_id") << std::endl;
    nidio::Pair P = nidio::load_pair(cfg);
    std::cout << "id of two image is " << pose_id0 << "," << pose_id1 << std::endl;
    const auto t_start = std::chrono::steady_clock::now();

    double T_cw1[16];
    nidio::invert_rigid(P.T_wc1.data(), T_cw1);
    std::cout << "before add disturbance the T_wc1 inverse is \n";
    nidio::print_mat4(T_cw1);
    const nidhost::Pose7 gt = nidhost::pose_from_mat16(T_cw1);

    // perturbation of NID_pose_estimation.cpp:186-208: t += (0.01, -0.02, -0.02), R <- Rx Ry Rz (0.005 pi each) * R
    const double t_offset = 0.02, r_offset = 0.005;
    const double ang = r_offset * M_PI, c = std::cos(ang), s = std::sin(ang);
    const double Rx[3][3] = {{1, 0, 0}, {0, c, -s}, {0, s, c}}, Ry[3][3] = {{c, 0, s}, {0, 1, 0}, {-s, 0, c}}, Rz[3][3] = {{c, -s, 0}, {s, c, 0}, {0, 0, 1}};
    double Rxy[3][3], Rd[3][3], Rn[3][3];
    for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) { Rxy[i][j] = 0; for (int k = 0; k < 3; k++) Rxy[i][j] += Rx[i][k] * Ry[k][j]; }
    for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) { Rd[i][j] = 0; for (int k = 0; k < 3; k++) Rd[i][j] += Rxy[i][k] * Rz[k][j]; }
    for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) { Rn[i][j] = 0; for (int k = 0; k < 3; k++) Rn[i][j] += Rd[i][k] * T_cw1[4 * j + k]; }
    const double tn[3] = {T_cw1[12] + 0.5 * t_offset, T_cw1[13] - t_offset, T_cw1[14] - t_offset};
    nidhost::Pose7 est = nidhost::pose_from_Rt(Rn, tn);
    double M0[16];
    nidhost::pose_to_mat16(est, M0);
    std::cout << "original matrix to be optimized \n";
    nidio::print_mat4(M0);
    std::cout << "the error to be minimized is (6d minimal form) \n";
    for (int i = 0; i < 3; i++) std::cout << gt.t[i] - est.t[i] << " ";
    for (int i = 0; i < 3; i++) std::cout << gt.q[i] - est.q[i] << (i < 2 ? " " : "\n");

    nid_ctx* ctx = nullptr;
    if (nid_create(&ctx, 0, P.rows, P.cols, cell, bins, 3, 1, 1) != NID_OK) die("nid_create");
    if (nid_set_option(ctx, "task_px", 16) != NID_OK) die("nid_set_option");  // one pair, one solve: latency-bound (nid_b200.h)
    if (nid_set_pair(ctx, 0, P.depth0.data(), P.im0.data(), P.im1.data(), P.T_wc0.data(), P.intr) != NID_OK) die("nid_set_pair");
    double pose7[7] = {est.t[0], est.t[1], est.t[2], est.q[0], est.q[1], est.q[2], est.q[3]};
    if (levels > 1) {
      // coarse levels 1 .. L-1, each derived on the device from the one above it
      std::vector<nid_ctx*> lv(levels, nullptr);
      lv[0] = ctx;
      for (int l = 1; l < levels; l++) {
        if (nid_create(&lv[l], 0, P.rows >> l, P.cols >> l, std::max(1, cell >> l), bins, 3, 1, 1) != NID_OK) die("nid_create (pyramid level)");
        if (nid_set_option(lv[l], "task_px", 16) != NID_OK) die("nid_set_option");
        if (nid_set_pairs_downsampled(lv[l], 0, lv[l - 1], 0, 1) != NID_OK) die("nid_set_pairs_downsampled");
      }
      std::vector<int> its(levels - 1, iters), lstats(3 * (levels - 1));
      if (nid_solve_pyramid_jobs(lv.data() + 1, levels - 1, 1, nullptr, pose7, its.data(), std::sqrt(0.95), lstats.data()) != NID_OK)
        die("nid_solve_pyramid_jobs");
      for (int l = levels - 1; l >= 1; l--)
        std::cout << "pyramid level " << l << " (" << (P.rows >> l) << "x" << (P.cols >> l) << "): outer iterations " << lstats[3 * (l - 1)]
                  << std::endl;
      for (int l = 1; l < levels; l++) nid_destroy(lv[l]);
      nidhost::Pose7 pc;
      for (int i = 0; i < 3; i++) pc.t[i] = pose7[i];
      for (int i = 0; i < 4; i++) pc.q[i] = pose7[3 + i];
      nidhost::pose_to_mat16(pc, M0);  // level 0 is prepared at the pose the coarse levels handed down
    }
    std::vector<int> counter(cell * cell);
    std::vector<double> Href(cell * cell);
    if (nid_prepare(ctx, 0, M0, counter.data(), Href.data()) != NID_OK) die("nid_prepare");
    int edges = 0;
    for (double h : Href) edges += !std::isnan(h);  // edges whose Href is NaN are put on level 1 (:323-325)

    std::cout << "enter optimization ............. 0" << std::endl;
    std::vector<double> trace(10 * (size_t)std::max(iters, 1));
    int stats[3] = {0, 0, 0};
    const auto t_opt = std::chrono::steady_clock::now();
    if (nid_solve(ctx, 0, pose7, iters, std::sqrt(0.95), trace.data(), stats) != NID_OK) die("nid_solve");
    const double opt_s = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_opt).count();
    // the verbose line of SparseOptimizer::optimize (sparse_optimizer.cpp:434-440); per-iteration times are not
    // recorded by nid_solve, the total is spread evenly
    for (int i = 0; i < stats[0]; i++) {
      const double* t = &trace[10 * (size_t)i];
      std::cerr << "iteration= " << i << "\t chi2= " << std::fixed << t[0] << std::defaultfloat << "\t time= " << opt_s / stats[0]
                << "\t cumTime= " << opt_s * (i + 1) / stats[0] << "\t edges= " << edges << "\t schur= 0\t lambda= " << std::fixed
                << t[1] << std::defaultfloat << "\t levenbergIter= " << (int)t[2] << std::endl;
    }
    std::cout << "the final error is \n";
    const double err[6] = {gt.t[0] - pose7[0], gt.t[1] - pose7[1], gt.t[2] - pose7[2], gt.q[0] - pose7[3], gt.q[1] - pose7[4], gt.q[2] - pose7[5]};
    for (int i = 0; i < 6; i++) std::cout << err[i] << (i < 5 ? " " : "\n");
    std::ofstream of("nid_error.csv", std::ofstream::out | std::ofstream::app);
    of << err[0] << "," << err[1] << "," << err[2] << "," << err[3] << "," << err[4] << "," << err[5] << "," << pose_id0 << "," << pose_id1 << std::endl;
    nidhost::Pose7 fin;
    for (int i = 0; i < 3; i++) fin.t[i] = pose7[i];
    for (int i = 0; i < 4; i++) fin.q[i] = pose7[3 + i];
    double Mf[16];
    nidhost::pose_to_mat16(fin, Mf);
    std::cout << "pose optimized \n";
    nidio::print_mat4(Mf);
    std::cout << "use " << std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count() << " in release mode" << std::endl;
    std::cout << "outer iterations " << stats[0] << ", cost+Jacobian evaluations " << stats[1] << ", cost evaluations " << stats[2]
              << ", kernels launched " << nid_launch_count(ctx) << std::endl;
    nid_destroy(ctx);
  } catch (const std::exception& e) {
    std::fprintf(stderr, "error: %s\n", e.what());
    return 1;
  }
  return 0;
}
