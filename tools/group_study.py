#!/usr/bin/env python
"""Does a joint solve over several pairs that share one pose (nid_solve_groups) end closer to the truth than a single-pair
solve, and what does it cost?

640x480, 16 synthetic scenes, at C2 (4x4 cells, 16 bins) and at the reference's default (16x16 cells, 10 bins), 10
iterations. Variants: one camera (a plain single-pair solve), 2- and 4-camera rigs (synth.make_rig: camera 0 is the body,
the others tilted 15-25 degrees; the 1- and 2-camera variants are the first cameras of the 4-camera rig of the same seed),
and 3 reference keyframes of one target frame (synth.make_keyframes). Starting poses: the reference's perturbation
(NID_pose_estimation.cpp:186-208) of the body (rig) or target (keyframes) pose scaled by s = 1, 2, 4; every pair is
prepared at its camera's starting pose. For every (config, variant, s): the fraction of solves that end within 1e-3 rad and
1e-3 m of the ground truth, the median final errors, the batched rate (16 groups in one call, lock-step) and the latency of
one group per call (latency mode; host clock around the blocking call, warmed up). The card's name and power limit are read
in the same run.

    python tools/group_study.py [--out FILE] [--scenes 16] [--reps 5]
"""
import argparse
import importlib
import json
import multiprocessing as mp
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from pyramid_study import card, pose_errors, scaled_perturbation  # noqa: E402

VARIANTS = (("cam1", 1), ("rig2", 2), ("rig4", 4), ("kf3", 3))


def _scene(args):
    seed, rows, cols = args
    synth = importlib.import_module("nid-pose-estimation_b200.synth")
    return synth.make_rig(2000 + seed, 4, rows, cols), synth.make_keyframes(3000 + seed, 3, rows, cols)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--scenes", type=int, default=16)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--rows", type=int, default=480)
    ap.add_argument("--cols", type=int, default=640)
    args = ap.parse_args()
    n, R, Cn = args.scenes, args.rows, args.cols
    t0 = time.perf_counter()
    with mp.get_context("fork").Pool(min(n, os.cpu_count() or 1)) as pool:
        scenes = pool.map(_scene, [(s, R, Cn) for s in range(n)])
    gen_s = time.perf_counter() - t0
    nid = importlib.import_module("nid-pose-estimation_b200")
    synth = importlib.import_module("nid-pose-estimation_b200.synth")
    from oracle import binding as orc
    # per variant: the pairs of every group, their T_cb (None: identity), the frame whose pose is solved (ground truth)
    var = {}
    for name, G in VARIANTS:
        groups = []
        for rig, kf in scenes:
            if name == "kf3":
                groups.append((kf, None, kf[0].T_wc1))
            else:
                groups.append((rig.pairs[:G], rig.T_cb[:G] if G > 1 else None, rig.T_wb1))
        var[name] = groups
    out = {"card": card(), "rows": R, "cols": Cn, "scenes": n, "seeds": f"rig 2000..{2000 + n - 1}, keyframes 3000..{3000 + n - 1}",
           "iterations": 10, "scene_generation_s": gen_s,
           "success": "rotation < 1e-3 rad and translation < 1e-3 m from the ground truth (within_1e-2: 1e-2 rad, 1e-2 m)",
           "configs": []}
    n_pairs = sum(len(g[0]) for v in var.values() for g in v)
    for cell, bins in ((4, 16), (16, 10)):
        ctx = nid.Context(R, Cn, cell, bins, n_pairs=n_pairs, max_jobs=4 * n)
        base, first = {}, 0
        for name, _ in VARIANTS:
            base[name] = first
            for pairs, _, _ in var[name]:
                for p in pairs:
                    ctx.set_pair(first, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
                    first += 1
        cfg = {"cell": cell, "bins": bins, "rows": []}
        for s in (1, 2, 4):
            for name, G in VARIANTS:
                groups = var[name]
                gts = [orc.se3_from_mat16(synth.mat16_inverse(T)) for _, _, T in groups]
                pose0 = np.stack([scaled_perturbation(orc, synth, T, s) for _, _, T in groups])
                eye = np.eye(4).reshape(16)
                T_cb = np.concatenate([np.tile(eye, (G, 1)) if E is None else E for _, E, _ in groups])
                use_T = name.startswith("rig")
                M = np.stack([orc.se3_to_mat16(pose0[j]) for j in range(n) for _ in range(G)])
                M = np.stack([(T_cb[i].reshape(4, 4).T @ M[i].reshape(4, 4).T).T.reshape(16) for i in range(n * G)])
                ctx.prepare_pairs(base[name], M)
                jp = np.arange(base[name], base[name] + n * G, dtype=np.int32)
                kw = dict(job_pair=jp, T_cb=T_cb if use_T else None)
                poses, st, _ = ctx.solve_groups(pose0, [G] * n, **kw)  # (also the warm-up of this shape)
                errs = np.array([pose_errors(orc, poses[j], gts[j]) for j in range(n)])
                err0 = np.array([pose_errors(orc, pose0[j], gts[j]) for j in range(n)])
                ok = (errs[:, 0] < 1e-3) & (errs[:, 1] < 1e-3)
                ok2 = (errs[:, 0] < 1e-2) & (errs[:, 1] < 1e-2)
                tb = []
                for _ in range(args.reps):
                    t1 = time.perf_counter()
                    ctx.solve_groups(pose0, [G] * n, **kw)
                    tb.append(time.perf_counter() - t1)
                tl = []
                for j in range(n):
                    sl = slice(j * G, (j + 1) * G)
                    kj = dict(job_pair=jp[sl], T_cb=T_cb[sl] if use_T else None)
                    ctx.solve_groups(pose0[j:j + 1], [G], **kj)
                    t1 = time.perf_counter()
                    ctx.solve_groups(pose0[j:j + 1], [G], **kj)
                    tl.append((time.perf_counter() - t1) * 1e3)
                row = {"scale": s, "variant": name, "pairs_per_group": G, "start_rot_rad": float(np.median(err0[:, 0])),
                       "start_trans_m": float(np.median(err0[:, 1])), "converged_fraction": float(ok.mean()),
                       "within_1e-2_fraction": float(ok2.mean()),
                       "median_rot_err_rad": float(np.median(errs[:, 0])), "median_trans_err_m": float(np.median(errs[:, 1])),
                       "batched_groups_per_s": float(n / np.median(tb)), "single_group_ms_median": float(np.median(tl)),
                       "outer_iters_mean": float(st[:, 0].mean()), "trial_evals_mean": float(st[:, 2].mean())}
                cfg["rows"].append(row)
                print(json.dumps({"cell": cell, "bins": bins, **row}), flush=True)
        out["configs"].append(cfg)
        ctx.close()
    txt = json.dumps(out, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        open(args.out, "w").write(txt + "\n")
    print(txt)


if __name__ == "__main__":
    main()
