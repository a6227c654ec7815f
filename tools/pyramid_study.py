#!/usr/bin/env python
"""Does a coarse-to-fine solve (nid_solve_pyramid_jobs over levels from nid_set_pairs_downsampled) widen the convergence
basin or shorten a solve on this library's synthetic pairs?

640x480, 16 synthetic pairs (seeds 1000+p), at C2 (4x4 cells, 16 bins) and at the reference's default (16x16 cells, 10
bins); level l has cell max(1, cell >> l) (constant pixels per cell) and 10 iterations. Starting poses: the reference's
perturbation (NID_pose_estimation.cpp:186-208) scaled by s (translation offsets x s, the three 0.005 pi angles x s).
For every (config, s, n_levels): the fraction of solves that end within 1e-3 rad and 1e-3 m of the ground truth, the median
final errors, the batched rate (16 problems in one call, level prepares included), the single-solve latency (one problem
per call, host clock around blocking calls, warmed up) and the time of the downsampling calls and of the level prepares.
The card's name and power limit are read in the same run.

    python tools/pyramid_study.py [--out FILE] [--pairs 16] [--reps 5]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def rot(ax, ay, az):
    cx, sx, cy, sy, cz, sz = np.cos(ax), np.sin(ax), np.cos(ay), np.sin(ay), np.cos(az), np.sin(az)
    Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
    Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
    Rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]])
    return Rx @ Ry @ Rz


def scaled_perturbation(orc, synth, T_wc1, s):
    """T_cw1 of the ground truth with t += s (0.01, -0.02, -0.02) and R <- Rx Ry Rz (s 0.005 pi each) R."""
    M = synth.mat16_inverse(T_wc1).reshape(4, 4).T
    a = s * 0.005 * np.pi
    R = rot(a, a, a) @ M[:3, :3]
    t = M[:3, 3] + s * np.array([0.01, -0.02, -0.02])
    return orc.se3_from_Rt(R.reshape(9), t)


def pose_errors(orc, pose, gt):
    """rotation angle (rad) and translation distance (m) between two T_cw1 poses {t, q}"""
    q, qg = pose[3:] / np.linalg.norm(pose[3:]), gt[3:] / np.linalg.norm(gt[3:])
    ang = 2 * np.arccos(min(1.0, abs(float(np.dot(q, qg)))))
    return ang, float(np.linalg.norm(pose[:3] - gt[:3]))


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                       text=True).strip().splitlines()[0]
    except Exception as e:  # (the numbers below are then without their card: say so)
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--pairs", type=int, default=16)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--rows", type=int, default=480)
    ap.add_argument("--cols", type=int, default=640)
    args = ap.parse_args()
    nid = importlib.import_module("nid-pose-estimation_b200")
    synth = importlib.import_module("nid-pose-estimation_b200.synth")
    from oracle import binding as orc
    n, R, Cn = args.pairs, args.rows, args.cols
    pairs = [synth.make_pair(1000 + p, R, Cn) for p in range(n)]
    gts = [orc.se3_from_mat16(synth.mat16_inverse(p.T_wc1)) for p in pairs]
    scales = (1, 2, 4, 8)
    out = {"card": card(), "rows": R, "cols": Cn, "pairs": n, "seeds": f"1000..{1000 + n - 1}", "iterations_per_level": 10,
           "success": "rotation < 1e-3 rad and translation < 1e-3 m from the ground truth (within_1e-2: 1e-2 rad, 1e-2 m)",
           "configs": []}
    for cell, bins in ((4, 16), (16, 10)):
        # level contexts: level 0 set from the host, every coarser level derived from the one above it
        ctxs = [nid.Context(R, Cn, cell, bins, n_pairs=n, max_jobs=n)]
        for i, p in enumerate(pairs):
            ctxs[0].set_pair(i, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
        ds_ms = []
        for l in (1, 2):
            ctxs.append(nid.Context(R >> l, Cn >> l, max(1, cell >> l), bins, n_pairs=n, max_jobs=n))
        for rep in range(args.reps + 1):
            t = []
            for l in (1, 2):
                t0 = time.perf_counter()
                ctxs[l].set_pairs_downsampled(0, ctxs[l - 1], 0, n)
                ctxs[l].sync()
                t.append((time.perf_counter() - t0) * 1e3)
            if rep:
                ds_ms.append(t)
        cfg = {"cell": cell, "bins": bins, "level_geometry": [[R >> l, Cn >> l, max(1, cell >> l)] for l in range(3)],
               "downsample_ms_16_pairs": {f"level{l}": float(np.median([t[l - 1] for t in ds_ms])) for l in (1, 2)},
               "rows": []}
        # level prepares of 16 pairs at the reference perturbation
        M = np.stack([orc.se3_to_mat16(orc.reference_perturbation(p.T_wc1)) for p in pairs])
        prep = {}
        for l in range(3):
            ctxs[l].prepare_pairs(0, M)
            ts = []
            for _ in range(args.reps):
                t0 = time.perf_counter()
                ctxs[l].prepare_pairs(0, M)
                ts.append((time.perf_counter() - t0) * 1e3)
            prep[f"level{l}"] = float(np.median(ts))
        cfg["prepare_ms_16_pairs"] = prep
        for s in scales:
            pose0 = np.stack([scaled_perturbation(orc, synth, p.T_wc1, s) for p in pairs])
            for L in (1, 2, 3):
                lv = ctxs[:L]
                poses, st = nid.solve_pyramid_jobs(lv, pose0)  # (also the warm-up of this shape)
                errs = np.array([pose_errors(orc, poses[j], gts[j]) for j in range(n)])
                err0 = np.array([pose_errors(orc, pose0[j], gts[j]) for j in range(n)])
                ok = (errs[:, 0] < 1e-3) & (errs[:, 1] < 1e-3)
                ok2 = (errs[:, 0] < 1e-2) & (errs[:, 1] < 1e-2)
                tb = []
                for _ in range(args.reps):
                    t0 = time.perf_counter()
                    nid.solve_pyramid_jobs(lv, pose0)
                    tb.append(time.perf_counter() - t0)
                tl = []
                for j in range(n):
                    nid.solve_pyramid_jobs(lv, pose0[j:j + 1], job_pair=[j])
                    t0 = time.perf_counter()
                    nid.solve_pyramid_jobs(lv, pose0[j:j + 1], job_pair=[j])
                    tl.append((time.perf_counter() - t0) * 1e3)
                row = {"scale": s, "n_levels": L, "start_rot_rad": float(np.median(err0[:, 0])),
                       "start_trans_m": float(np.median(err0[:, 1])), "converged_fraction": float(ok.mean()),
                       "within_1e-2_fraction": float(ok2.mean()),
                       "median_rot_err_rad": float(np.median(errs[:, 0])), "median_trans_err_m": float(np.median(errs[:, 1])),
                       "batched_solves_per_s": float(n / np.median(tb)), "single_solve_ms_median": float(np.median(tl)),
                       "outer_iters_mean_per_level": [float(v) for v in st[:, :, 0].mean(axis=0)]}
                cfg["rows"].append(row)
                print(json.dumps({"cell": cell, "bins": bins, **row}), flush=True)
        out["configs"].append(cfg)
        for c in ctxs:
            c.close()
    txt = json.dumps(out, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        open(args.out, "w").write(txt + "\n")
    print(txt)


if __name__ == "__main__":
    main()
