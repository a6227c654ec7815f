"""Small evaluations of every kernel family for compute-sanitizer (memcheck / racecheck / initcheck)."""
import importlib, os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
nid = importlib.import_module("nid-pose-estimation_b200")
synth = importlib.import_module("nid-pose-estimation_b200.synth")
from oracle import binding as orc
for (rows, cols, cell, bins) in ((120, 160, 2, 16), (120, 160, 4, 10), (96, 128, 1, 9), (120, 160, 2, 40), (100, 130, 3, 6),
                                 (120, 160, 8, 32)):
    p = synth.make_pair(1000, rows, cols, invalid_depth_frac=0.03)
    pose0 = orc.reference_perturbation(p.T_wc1)
    M0 = orc.se3_to_mat16(pose0)
    ctx = nid.Context(rows, cols, cell, bins, n_pairs=3, max_jobs=12)
    for s in range(2):
        ctx.set_pair(s, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
        ctx.prepare(s, M0)
    # batched set-up from raw 16-bit depth, tables built on the device (pairs 1 and 2)
    keep = ctx.set_pairs_u16(1, np.stack([p.depth0_u16] * 2), np.stack([p.im0] * 2), np.stack([p.im1] * 2), np.stack([p.T_wc0] * 2),
                             np.stack([p.intr] * 2))
    ctx.prepare_pairs(1, np.stack([M0] * 2))
    jp = np.arange(12, dtype=np.int32) % 3
    poses = np.stack([M0] * 12)
    ctx.eval_jobs(poses, jp, True)
    ctx.eval(0, M0, False)
    ctx.solve_jobs(np.stack([pose0] * 12), jp, 3)   # lock-step, two half-batches, job lists
    ctx.solve(0, pose0, 2)                          # latency mode (speculative trial poses, one graph launch per round)
    ctx.solve(0, pose0, 2)                          # replay of the cached graph (parameter update of the pixel-kernel nodes)
    ctx.set_option("lm_graph", 0)
    ctx.solve(0, pose0, 2)                          # the same round as plain launches (k_tail_gn writes to pinned memory)
    ctx.set_option("asm_wide", 0)
    ctx.eval_jobs(poses, jp, True)                  # 128/256-thread assembly instead of the 1024-thread one
    ctx.set_option("asm_wide", 1)
    ctx.set_option("lm_graph", 1)
    ctx.warp_sample_jobs(poses, jp)                 # mixed fp64 / u16 depth planes -> fp64 variant
    ctx.warp_sample_jobs(poses[:4], np.array([1, 2, 1, 2], dtype=np.int32))  # u16 variant
    ctx.hard_eval_jobs(poses, jp)
    ctx.set_target(1, p.im0)
    ctx.prepare(1, M0)
    ctx.eval(1, M0, True)
    ctx.close()
    print("ok", rows, cols, cell, bins)
