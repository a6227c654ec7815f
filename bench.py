#!/usr/bin/env python
"""bench.py — NID cost+Jacobian evals/s @640x480 (BASELINE.json metric), one rank per GPU.

A "step" evaluates the cost + 6-DoF Jacobian (the a9-equivalent, want_jac=1) of every frame pair this rank
owns once, at a pose that changes every step. Workload = BASELINE config[1] (C2): 640x480, 4x4 cells, 16-bin
B-spline NID. The rank owns `--pairs` pair slots (default 384) whose device footprint (several GB) exceeds the 126 MB L2,
so every step streams its inputs from HBM ("inputs larger than L2").

  value : evals/s with inputs resident in HBM (poses staged, results left on the device), CUDA events on
          the library's stream, max over ranks.
  e2e   : the same evaluations through the reference-facing C-ABI call with HOST buffers
          (nid_eval_jobs: H2D poses from pinned memory, kernels, D2H Htarget/Hjoint/der, sync).
  --impl reference : the reference's CPU implementation of the path (the fp64 restatement in oracle/,
          OpenMP over cells on all host cores) on the same workload, bounded sample per step.

Further legs on the same line (each with its own CPU figure at N=1):
  pair_setup : nid_set_pairs_u16 + nid_prepare_pairs from pinned host buffers (the step before the path).
  pose_solves: complete optimize(10) LM runs of every slot (nid_solve_jobs).
  c4   : BASELINE config 4 as stated: 1024 DISTINCT pairs (16 seeded scenes x 64 seeded exposure / illumination
         variants), set-up + solve + gather of {pose7, iterations} through shard.py (NCCL all-gather), sharded in
         blocks over the ranks; strong scaling (the 1024 pairs are the whole job).
  c5   : BASELINE config 5 as stated: the 6 x 64^2 = 24 576-pose hard-binned cost-surface sweep of one pair
         (NID_standard_property semantics, 16x16 cells, 8 bins), pose q on rank q mod G, totals gathered through shard.py.
  old_gpu_path : the reference's own CUDA code (oracle/_ref, compiled unmodified) timed on the one geometry it is
         memory-safe for on a 148-SM part (592x512), next to this library at that geometry.

Multi-GPU: whole problems are sharded across ranks (no data-path collective); NCCL is only used for the barrier, the
max-over-ranks of the device time and the result gathers of c4 / c5.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ROWS, COLS, CELL, BINS = 480, 640, 4, 16
ALGO_BYTES_PER_EVAL = ROWS * COLS * 12 + CELL * CELL * 8 * 8  # SURVEY 8(d): fp32 depth + I_ref + I_tgt planes, outputs
DISTINCT_PAIRS = 6
C4_PAIRS, C4_SCENES = 1024, 16
C5_GRID, C5_AXES, C5_SPAN = 64, 6, 0.05
FP64_PEAK_WARP_INST_PER_CLK_SMSP = 0.49  # measured: profiles/r01_pipe_bench.txt (DFMA, 16 warps/SM, 4 chains each)


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md), through NVML when the
    binding is importable (sub-millisecond polls), else through nvidia-smi."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.sm, self.mx, self.reasons, self.n = [], [], set(), 0
        self._stop = threading.Event()
        self._t = None
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[gpu_index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else gpu_index
            self._h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self._nvml = pynvml
        except Exception:
            self._nvml = None

    def _poll_nvml(self):
        nv = self._nvml
        if not self.mx:
            self.mx.append(float(nv.nvmlDeviceGetMaxClockInfo(self._h, nv.NVML_CLOCK_SM)))
        self.sm.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
        self.n += 1
        if self.n % 4 == 1:  # the reasons query is the slow one: every fourth poll
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
            for name, bit in (("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                              ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap)):
                if r & bit:
                    self.reasons.add(name)

    def _poll_smi(self):
        out = subprocess.check_output(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-i", str(self.gpu)], timeout=5).decode().strip()
        r = [x.strip() for x in out.split(",")]
        if r[1].replace(".", "").isdigit():
            self.sm.append(float(r[1]))
        if r[2].replace(".", "").isdigit():
            self.mx.append(float(r[2]))
        for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
            if v.lower().startswith("active"):
                self.reasons.add(name)
        self.n += 1

    def _run(self):
        while not self._stop.is_set():
            try:
                if self._nvml is not None:
                    self._poll_nvml()
                else:
                    self._poll_smi()
            except Exception:
                if self._nvml is not None:
                    self._nvml = None  # fall back to nvidia-smi
                    continue
            self._stop.wait(0.0005 if self._nvml is not None else 0.02)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.n:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"], "samples": 0}
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                "reasons": sorted(self.reasons), "samples": self.n, "source": "nvml" if self._nvml is not None else "nvidia-smi"}


def make_poses(orc, pose0_list, step, n_slots):
    """pose of slot s at step k: small seeded se(3) offset on the left of that pair's initial guess."""
    rng = np.random.default_rng(77 + step)
    xi = rng.uniform(-1, 1, size=(n_slots, 6)) * np.array([2e-3, 2e-3, 2e-3, 5e-3, 5e-3, 5e-3])
    return np.stack([orc.se3_to_mat16(orc.se3_mul(orc.se3_exp(xi[s]), pose0_list[s % len(pose0_list)])) for s in range(n_slots)])


def peaks():
    """HBM copy peak in GB/s: the driver-written MEASURED_PEAKS.json when present, else the fallback
    B200_PROFILING.md states."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            d = json.load(open(path))
            flat = {}

            def walk(prefix, o):
                if isinstance(o, dict):
                    for k, v in o.items():
                        walk(f"{prefix}.{k}" if prefix else str(k), v)
                elif isinstance(o, (int, float)):
                    flat[prefix.lower()] = float(o)
            walk("", d)
            cands = [(k, v) for k, v in flat.items() if "hbm" in k and v > 100]
            for pref in ("sustain", "burst", ""):
                for k, v in cands:
                    if pref in k:
                        return v, f"measured (MEASURED_PEAKS.json {k})"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def _traffic_json():
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return None


def measured_traffic(kernel, n_evals):
    """DRAM bytes per launch of `kernel` from the committed ncu --set full capture (profiles/traffic.json), or None."""
    d = _traffic_json()
    try:
        return d["dram_bytes_per_eval"][kernel] * n_evals, d["source"]
    except Exception:
        return None, None


def measured_pipes(kernel):
    """fp64-pipe / issue utilisation of `kernel` from the committed ncu --set full capture (profiles/traffic.json), or None."""
    d = _traffic_json()
    try:
        return dict(d["pipes"][kernel], source=d["source"].split(" ")[0])
    except Exception:
        return None


def fp64_roofline(kernel, n_evals, kernel_ms, sm_mhz, n_sm=148):
    """fp64-pipe roofline of `kernel`: fp64 warp instructions per launch (counted by ncu in the committed capture,
    per evaluation) / the kernel's live device time, against the measured DFMA issue peak of the part
    (0.49 warp instructions per clock per SM sub-partition, profiles/r01_pipe_bench.txt) at the SM clock sampled during
    the run."""
    d = _traffic_json()
    try:
        per_eval = d["fp64_warp_inst_per_eval"][kernel]
    except Exception:
        return None
    mhz = sm_mhz or 1965.0
    peak = FP64_PEAK_WARP_INST_PER_CLK_SMSP * 4 * n_sm * mhz * 1e6 / 1e9
    achieved = per_eval * n_evals / (kernel_ms * 1e-3) / 1e9
    return {"kernel": kernel, "achieved": achieved, "peak": peak, "unit": "G fp64 warp-instructions/s", "frac": achieved / peak,
            "fp64_warp_inst_per_launch": per_eval * n_evals, "peak_source": "tools/pipe_bench.cu: 0.49 DFMA warp-instr/clk/SMSP x 4 x 148 SMs "
            f"x {mhz:.0f} MHz", "count_source": d.get("source")}


def cpu_layout(cores):
    """Use every host core: `workers` independent evaluations in flight, each an OpenMP team of `team` threads over
    the 16 cells (team divides 16 so that cells split evenly)."""
    best = (1, 1)
    for team in (1, 2, 4, 8, 16):
        workers = max(1, cores // team)
        if team <= cores and workers * team >= best[0] * best[1]:
            best = (workers, team)
    return best


class CpuArm:
    """The reference's CPU implementation of the path (oracle/ restatement: the reference's own CPU code needs
    Eigen/OpenCV, absent here) on the bench workload; `workers` problems evaluated concurrently (ctypes releases
    the GIL), `team` OpenMP threads each."""

    def __init__(self, orc, synth, workers, team):
        self.orc, self.workers, self.team = orc, workers, team
        p = synth.make_pair(1000, ROWS, COLS)
        self.pose0 = orc.reference_perturbation(p.T_wc1)
        self.P = [orc.Problem(p.im0, p.depth0, p.im1, p.T_wc0, p.intr, CELL, BINS, threads=team) for _ in range(workers)]
        for P in self.P:
            P.prepare(self.pose0)
            P.eval(self.pose0, True)  # warm

    def _par(self, work):
        ts = [threading.Thread(target=work, args=(w,)) for w in range(self.workers)]
        t0 = time.perf_counter()
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        return time.perf_counter() - t0

    def run(self, evals_per_worker, seed):
        """evals_per_worker cost+Jacobian evaluations on every worker; returns (evals, seconds)."""
        orc = self.orc

        def work(w):
            rng = np.random.default_rng(seed * 131 + w)
            for _ in range(evals_per_worker):
                xi = rng.uniform(-1, 1, size=6) * 2e-3
                self.P[w].eval(orc.se3_mul(orc.se3_exp(xi), self.pose0), True)
        return evals_per_worker * self.workers, self._par(work)

    def solves(self):
        """one complete optimize(10) per worker (LM of optimization_algorithm_levenberg.cpp:61-225); (solves, seconds)"""
        def work(w):
            self.P[w].prepare(self.pose0)
            self.P[w].optimize(self.pose0, 10)
        return self.workers, self._par(work)


def cpu_eval_rate(orc, synth, workers, team, budget_s):
    """evals/s of the CPU arm, bounded sample of about budget_s seconds."""
    arm = CpuArm(orc, synth, workers, team)
    n, el = arm.run(1, 0)
    per = max(1, min(200, int(budget_s / max(el, 1e-3))))
    n, el = arm.run(per, 1)
    return n / el, n, el, arm


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on the host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import binding as orc
    synth = importlib.import_module("nid-pose-estimation_b200.synth")
    cores = os.cpu_count() or 1
    workers, team = cpu_layout(cores)
    arm = CpuArm(orc, synth, workers, team)
    evals_per_worker = 2  # bounded sample of the workload per step
    for k in range(args.warmup):
        arm.run(evals_per_worker, k)
    n, el = 0, 0.0
    for k in range(args.steps):
        a, b = arm.run(evals_per_worker, 100 + k)
        n += a
        el += b
    v = n / el
    line = {
        "impl": "reference", "metric": "NID cost+Jacobian evals/s @640x480", "value": v, "unit": "evals/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "C2: 640x480 pair, 4x4 cells, 16-bin cubic B-spline NID, cost+Jacobian", "rows": ROWS,
                   "cols": COLS, "cell": CELL, "bins": BINS},
        "cpu_baseline": {"value": v, "unit": "evals/s", "cores": workers * team, "kind": "port",
                         "sample": f"{evals_per_worker * workers} evals/step of one seeded 640x480 pair: {workers} evaluations in "
                                   f"flight x {team} OpenMP threads over the 16 cells (the reference CPU path cannot be "
                                   "compiled here: Eigen/OpenCV absent)"},
        "e2e": {"value": v, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------- legs
def pinned_pairs(torch, pairs):
    """depth16 / im0 / im1 of a list of pairs stacked into pinned host buffers (+ T_wc0, intr)"""
    n, N = len(pairs), pairs[0].rows * pairs[0].cols
    d16 = torch.empty((n, N), dtype=torch.uint16).pin_memory()
    im0 = torch.empty((n, N), dtype=torch.uint8).pin_memory()
    im1 = torch.empty((n, N), dtype=torch.uint8).pin_memory()
    dn, an, bn = d16.numpy(), im0.numpy(), im1.numpy()
    for i, p in enumerate(pairs):
        dn[i] = p.depth0_u16.reshape(-1)
        an[i] = p.im0.reshape(-1)
        bn[i] = p.im1.reshape(-1)
    T = np.stack([p.T_wc0 for p in pairs])
    K = np.stack([p.intr for p in pairs])
    return (d16, im0, im1), dn, an, bn, T, K


def leg_c4(args, nid, synth, orc, shard, torch, dist, rank, world, local_rank, barrier):
    """BASELINE config 4: 1024 distinct pairs, set-up + optimize(10) + gather, block-sharded over the ranks."""
    n_total = args.c4_pairs
    per_scene = max(1, n_total // C4_SCENES)
    mine = shard.owned(n_total, world, rank, "block")
    scenes = sorted(set(int(p) // per_scene for p in mine))
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=min(len(scenes), max(1, (os.cpu_count() or 2) // max(1, min(world, 8))))) as ex:
        seqs = dict(zip(scenes, ex.map(lambda s: synth.make_sequence(2000 + s, per_scene, ROWS, COLS), scenes)))
    pairs = [seqs[int(p) // per_scene][int(p) % per_scene] for p in mine]
    gen_s = time.perf_counter() - t0
    keep, dn, an, bn, T, K = pinned_pairs(torch, pairs)
    pose0 = []
    for gp, p in zip(mine, pairs):  # the reference perturbation plus a small offset seeded by the GLOBAL pair index
        xi = np.random.default_rng(4000 + int(gp)).uniform(-1, 1, size=6) * np.array([1e-3, 1e-3, 1e-3, 2e-3, 2e-3, 2e-3])
        pose0.append(orc.se3_mul(orc.se3_exp(xi), orc.reference_perturbation(p.T_wc1)))
    pose0 = np.stack(pose0)
    init = np.stack([orc.se3_to_mat16(q) for q in pose0])
    n = len(pairs)
    # pairs per set-up submission. Smaller blocks for many ranks (128 pairs per rank at N=8) were measured and do not pay:
    # one block of 128 31.6 ms, two of 64 32.8 ms, four of 32 38.3 ms -- solves of fewer problems per call fill the device
    # less, and the concurrent upload competes with them
    block = min(n, 256)
    chunk = min(block, 128)      # problems per nid_solve_jobs call
    # two contexts ping-pong: while one solves its block of pairs, the other one's block is uploaded and prepared
    # (set-up runs on its own host thread and its own stream; the ctypes calls release the GIL)
    ctxs = [nid.Context(ROWS, COLS, CELL, BINS, n_pairs=block, max_jobs=chunk, device=local_rank) for _ in range(2 if n > block else 1)]
    blocks = [(b0, min(n, b0 + block)) for b0 in range(0, n, block)]

    def setup(k):
        b0, b1 = blocks[k]
        cx = ctxs[k % len(ctxs)]
        cx.set_pairs_u16(0, dn[b0:b1], an[b0:b1], bn[b0:b1], T[b0:b1], K[b0:b1])
        cx.prepare_pairs(0, init[b0:b1])

    def run_once():
        rows = np.zeros((n, 10))
        t_first = None
        with ThreadPoolExecutor(max_workers=1) as ex:
            fut = ex.submit(setup, 0)
            for k, (b0, b1) in enumerate(blocks):
                fut.result()
                if t_first is None:
                    t_first = time.perf_counter()
                if k + 1 < len(blocks):
                    fut = ex.submit(setup, k + 1)
                cx = ctxs[k % len(ctxs)]
                for c0 in range(b0, b1, chunk):
                    c1 = min(b1, c0 + chunk)
                    out, st = cx.solve_jobs(pose0[c0:c1], np.arange(c0 - b0, c1 - b0, dtype=np.int32))
                    rows[c0:c1, :7] = out
                    rows[c0:c1, 7:] = st
        return rows, t_first

    run_once()  # warm (allocations, first-touch)
    barrier()
    t0 = time.perf_counter()
    rows, t_setup = run_once()
    table = shard.gather_results(rows, n_total, world, rank, "block", device=torch.device("cuda", local_rank) if world > 1 else None)
    torch.cuda.synchronize()
    el = time.perf_counter() - t0
    setup_s = t_setup - t0
    if world > 1:
        t = torch.tensor([el, setup_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        el, setup_s = t.tolist()
    for cx in ctxs:
        cx.close()
    assert np.all(np.isfinite(table)), "c4: non-finite rows in the gathered table"
    res = {"value": n_total / el, "unit": "pairs/s", "pairs": n_total, "pairs_per_rank": int(n), "seconds": el,
           "first_block_setup_seconds": setup_s, "scaling": "strong", "sharding": "block (shard.py)",
           "overlap": f"two contexts ping-pong: the set-up of the next block of {block} pairs overlaps the solves of the current one",
           "gather": "NCCL all_gather of {pose7, outer_iters, jac_evals, cost_evals} per pair" if world > 1 else "single rank",
           "mean_outer_iters": float(table[:, 7].mean()), "mean_jac_evals": float(table[:, 8].mean()),
           "mean_cost_evals": float(table[:, 9].mean()), "host_generation_seconds_untimed": gen_s,
           "workload": f"{n_total} distinct pairs = {C4_SCENES} seeded scenes x {per_scene} seeded exposure / illumination variants "
                       "(synth.make_sequence), each with its own initial pose; timed: nid_set_pairs_u16 from pinned host buffers + "
                       "nid_prepare_pairs + nid_solve_jobs (optimize(10)) + result gather, wall clock, max over ranks",
           "table_checksum": float(np.sum(table[:, :7] * np.arange(1, 8)))}
    return res


def c5_poses(orc, synth, p):
    """the 6 x 64 x 64 lattice of SURVEY 8(d): for axis a, offsets (d_a, d_(a+1) mod 6) on a uniform grid over +-0.05"""
    gt = orc.se3_from_mat16(synth.mat16_inverse(p.T_wc1))
    lat = -C5_SPAN + 2 * C5_SPAN * np.arange(C5_GRID) / (C5_GRID - 1)
    out = np.zeros((C5_AXES * C5_GRID * C5_GRID, 16))
    q = 0
    for a in range(C5_AXES):
        for i in range(C5_GRID):
            for j in range(C5_GRID):
                d = np.zeros(6)
                d[a] = lat[i]
                d[(a + 1) % 6] += lat[j]
                out[q] = orc.se3_to_mat16(orc.se3_mul(orc.se3_exp(d), gt))
                q += 1
    return out


def leg_c5(args, nid, synth, orc, shard, torch, dist, rank, world, local_rank, barrier):
    """BASELINE config 5: 24 576 hard-binned cost evaluations of one pair, pose q on rank q mod G."""
    p = synth.make_pair(1000, ROWS, COLS)
    poses = c5_poses(orc, synth, p)
    n_total = poses.shape[0]
    mine = shard.owned(n_total, world, rank, "cyclic")
    chunk = 2048
    ctx = nid.Context(ROWS, COLS, 16, 8, n_pairs=1, max_jobs=chunk, device=local_rank)
    ctx.set_pair(0, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
    my_poses = np.ascontiguousarray(poses[mine])

    def run_once():
        tot = np.zeros(len(mine))
        for c0 in range(0, len(mine), chunk):
            c1 = min(len(mine), c0 + chunk)
            tot[c0:c1], _ = ctx.hard_eval_jobs(my_poses[c0:c1])
        return tot

    run_once()
    barrier()
    t0 = time.perf_counter()
    tot = run_once()
    table = shard.gather_results(tot, n_total, world, rank, "cyclic", device=torch.device("cuda", local_rank) if world > 1 else None)
    torch.cuda.synchronize()
    el = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([el], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        el = t.item()
    # the gathered table against this rank's own GPU on rows other ranks computed: bit-equal
    rng = np.random.default_rng(5)
    probe = rng.choice(n_total, size=64, replace=False)
    again, _ = ctx.hard_eval_jobs(np.ascontiguousarray(poses[probe]))
    verified = bool(np.array_equal(again, table[probe, 0]))
    ctx.close()
    gt_row = int(np.argmin(np.abs(table[:, 0] - table[:, 0].min())))
    return {"value": n_total / el, "unit": "hard-binned cost evals/s", "poses": n_total, "poses_per_rank": int(len(mine)), "seconds": el,
            "scaling": "strong", "sharding": "cyclic q mod G (shard.py)",
            "gather": "NCCL all_gather of sqrt(sum nid_c^2) per pose" if world > 1 else "single rank",
            "rows_rechecked_bit_equal_on_rank0": 64 if verified else 0, "surface_min": float(table[:, 0].min()),
            "surface_min_at_row": gt_row, "surface_max": float(table[:, 0].max()),
            "workload": "NID_standard_property semantics (NID_standard_property.cpp:342-485), 640x480, 16x16 cells, 8 hard bins, "
                        "6 axes x 64 x 64 lattice over +-0.05 m / rad around the true pose; timed: nid_hard_eval_jobs with host poses "
                        "in and host totals out + gather, wall clock, max over ranks",
            "table_checksum": float(np.sum(table[:, 0]))}, p, poses


def leg_old_gpu(nid, synth, orc, torch):
    """The reference's own CUDA path (oracle/_ref, unmodified computeH.cu) next to this library at 592x512 (the one
    geometry the unguarded reference kernels are memory-safe for on 148 SMs), 16x16 cells / 10 bins (the reference's
    defaults, NID_pose_estimation.cpp:26-28) and 4x4 cells / 10 bins."""
    from oracle import ref_gpu
    if not ref_gpu.available():
        return {"unavailable": "oracle/_ref not built (upstream tree absent at build time)"}
    out = {"geometry": f"{ref_gpu.SAFE_ROWS}x{ref_gpu.SAFE_COLS}", "unit": "cost+Jacobian evals/s",
           "note": "reference: g2o::CudaComputeH as shipped (per-call cudaMalloc/H2D/memset/3 kernels/D2H/cudaFree, global fp64 atomics), "
                   "one call at a time as its LM loop issues them; ours: nid_eval_jobs, 32 jobs per call, same pair and poses"}
    p = synth.make_pair(1000, ref_gpu.SAFE_ROWS, ref_gpu.SAFE_COLS)
    pose0 = orc.reference_perturbation(p.T_wc1)
    rng = np.random.default_rng(3)
    poses = [orc.se3_to_mat16(orc.se3_mul(orc.se3_exp(rng.uniform(-1, 1, 6) * 2e-3), pose0)) for _ in range(32)]
    for cell, bins in ((16, 10), (4, 10)):
        P = orc.Problem(p.im0, p.depth0, p.im1, p.T_wc0, p.intr, cell, bins)
        nc, href = P.prepare(pose0)
        bv, bi = P.ref_weights()
        R = ref_gpu.RefGpu(p, cell, bins)
        R.set_prepare(nc, bv, bi, np.where(np.isnan(href), 0.0, href))
        R.compute_h(poses[0], True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        n_ref = 8
        for k in range(n_ref):
            R.compute_h(poses[k], True)
        torch.cuda.synchronize()
        ref_rate = n_ref / (time.perf_counter() - t0)
        R.close()
        ctx = nid.Context(p.rows, p.cols, cell, bins, n_pairs=1, max_jobs=32)
        ctx.set_pair(0, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
        ctx.prepare(0, orc.se3_to_mat16(pose0))
        M = np.stack(poses)
        ctx.eval_jobs(M, np.zeros(32, dtype=np.int32), True)
        t0 = time.perf_counter()
        for _ in range(10):
            ctx.eval_jobs(M, np.zeros(32, dtype=np.int32), True)
        ours = 320 / (time.perf_counter() - t0)
        t0 = time.perf_counter()
        for k in range(32):
            ctx.eval(0, poses[k], True)
        ours1 = 32 / (time.perf_counter() - t0)
        ctx.close()
        out[f"cell{cell}_bins{bins}"] = {"reference_cuda": ref_rate, "ours_batched": ours, "ours_one_call_at_a_time": ours1,
                                         "ratio_batched": ours / ref_rate, "ratio_one_at_a_time": ours1 / ref_rate}
    return out


def leg_single_pair(nid, synth, orc):
    """Latency of the flow the reference's NID_pose_estimation runs per frame pair (one pair per process,
    NID_pose_estimation.cpp:253-350): set-up, one evaluation, one optimize(10), each a blocking call, wall clock. Twice:
    with the library's defaults, and with the 16-pixel tasks its header recommends to latency-bound callers
    (nid_set_option "task_px"; throughput-bound callers keep 32: 144k against 126k evaluations/s at this geometry)."""
    p = synth.make_pair(1000, ROWS, COLS)
    pose0 = orc.reference_perturbation(p.T_wc1)
    M0 = orc.se3_to_mat16(pose0)
    out = {"workload": "one 640x480 pair, 4x4 cells, 16 bins, one context (n_pairs=1, max_jobs=1), blocking calls, wall clock per call",
           "lm": "latency mode: 4 speculative trial poses per round, one CUDA-graph launch per round"}
    for name, opts in (("default", {}), ("task_px_16", {"task_px": 16})):
        ctx = nid.Context(ROWS, COLS, 4, 16, n_pairs=1, max_jobs=1)
        for k, v in opts.items():
            ctx.set_option(k, v)

        def t(f, n):
            f()
            ctx.sync()
            t0 = time.perf_counter()
            for _ in range(n):
                f()
            ctx.sync()
            return (time.perf_counter() - t0) / n * 1e3
        r = {"set_pair_ms": t(lambda: ctx.set_pair(0, p.depth0, p.im0, p.im1, p.T_wc0, p.intr), 10),
             "prepare_ms": t(lambda: ctx.prepare(0, M0), 10),
             "eval_cost_ms": t(lambda: ctx.eval(0, M0, False), 50),
             "eval_cost_jac_ms": t(lambda: ctx.eval(0, M0, True), 50),
             "solve_ms": t(lambda: ctx.solve(0, pose0), 10)}
        _, _, st = ctx.solve(0, pose0)
        r["outer_iters"], r["jac_evals"], r["cost_evals"] = (int(v) for v in st)
        out[name] = r
        ctx.close()
    return out


def leg_shim(nid, synth, orc, torch):
    """The reference-API drop-in path: the exact-signature entry points (Calculate3Dpoint, CudaComputeHref,
    g2o::CudaComputeH; csrc/ref_shims.cu) driven like NID_pose_estimation.cpp:253-276 and the LM loop drive them,
    one blocking call at a time with the reference's fp64 host buffers, at the reference's default geometry."""
    import ctypes as C
    _dp, _ip = C.POINTER(C.c_double), C.POINTER(C.c_int)
    L = nid.lib()
    p = synth.make_pair(1000, ROWS, COLS)
    cell, bins, N = 16, 10, ROWS * COLS
    d = lambda a: a.ctypes.data_as(_dp)
    depth = p.depth0.reshape(-1).copy()
    Twc0, intr = p.T_wc0.copy(), p.intr.copy()
    points = np.zeros(3 * N)
    im0 = p.im0.astype(np.float64).reshape(-1).copy()
    im1 = p.im1.astype(np.float64).reshape(-1).copy()
    pose0 = orc.reference_perturbation(p.T_wc1)
    M0 = orc.se3_to_mat16(pose0)
    t0 = time.perf_counter()
    L.nid_shim_Calculate3Dpoint(d(depth), d(Twc0), d(points), d(intr), ROWS, COLS)
    bs_value = np.zeros(4 * N)
    bs_index = np.zeros(N, dtype=np.int32)
    bs_counter = np.zeros(cell * cell, dtype=np.int32)
    Href = np.zeros(cell * cell)
    L.nid_shim_CudaComputeHref(d(im0), d(points), d(M0), d(intr), bins, 3, cell, ROWS, COLS, d(bs_value),
                               bs_index.ctypes.data_as(_ip), bs_counter.ctypes.data_as(_ip), d(Href))
    setup_s = time.perf_counter() - t0
    rng = np.random.default_rng(9)
    poses = [orc.se3_to_mat16(orc.se3_mul(orc.se3_exp(rng.uniform(-1, 1, 6) * 2e-3), pose0)) for _ in range(40)]
    Ht, Hj, der = np.zeros(cell * cell), np.zeros(cell * cell), np.zeros(6 * cell * cell)

    def call(M, jac):
        Ht[:] = 0
        Hj[:] = 0
        L.nid_shim_CudaComputeH(jac, d(im0), d(im1), d(points), bs_counter.ctypes.data_as(_ip), d(bs_value),
                                bs_index.ctypes.data_as(_ip), d(M), d(intr), bins, 3, cell, ROWS, COLS, d(Href), None, None,
                                d(Ht), d(Hj), d(der))
    call(poses[0], 1)
    t0 = time.perf_counter()
    for M in poses:
        call(M, 1)
    rate_j = len(poses) / (time.perf_counter() - t0)
    t0 = time.perf_counter()
    for M in poses:
        call(M, 0)
    rate_c = len(poses) / (time.perf_counter() - t0)
    L.nid_shim_reset()
    return {"geometry": f"{ROWS}x{COLS}, 16x16 cells, 10 bins (NID_pose_estimation.cpp:26-28)", "cost_jacobian_calls_per_s": rate_j,
            "cost_only_calls_per_s": rate_c, "setup_ms": 1e3 * setup_s,
            "call": "g2o::CudaComputeH(calculate_der, ...) with the reference's signature and fp64 host / managed buffers, blocking, one "
                    "evaluation per call (each call compares the two images with the uploaded copies: 4.9 MB of memcmp)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--pairs", type=int, default=384, help="pair slots per rank (384 x ~18 MB of device data >> L2)")
    ap.add_argument("--solves", type=int, default=1, help="also time complete LM pose solves of every slot (0: skip)")
    ap.add_argument("--cpu-budget", type=float, default=12.0)
    ap.add_argument("--c4-pairs", type=int, default=C4_PAIRS, help="BASELINE config 4: distinct pairs of the whole job (0: skip the leg)")
    ap.add_argument("--c5", type=int, default=1, help="BASELINE config 5: the 24 576-pose hard-binned sweep (0: skip)")
    ap.add_argument("--old-gpu", type=int, default=1, help="time the reference's own CUDA code beside ours (0: skip)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step (Htarget, Hjoint, der of every pair slot) as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the NID path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    nid = importlib.import_module("nid-pose-estimation_b200")
    synth = importlib.import_module("nid-pose-estimation_b200.synth")
    shard = importlib.import_module("nid-pose-estimation_b200.shard")
    from oracle import binding as orc  # pose algebra for the synthetic workload + the cpu_baseline legs only

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    n_slots = args.pairs
    ctx = nid.Context(ROWS, COLS, CELL, BINS, n_pairs=n_slots, max_jobs=n_slots, device=local_rank)
    for kv in filter(None, os.environ.get("NID_OPTS", "").split(",")):  # developer knob, e.g. NID_OPTS=task_px=64
        k, v = kv.split("=")
        ctx.set_option(k, int(v))
    distinct = [synth.make_pair(1000 + rank * DISTINCT_PAIRS + i, ROWS, COLS) for i in range(DISTINCT_PAIRS)]
    pose0 = [orc.reference_perturbation(p.T_wc1) for p in distinct]
    # ---------------- pair set-up (the step before the path): batched, raw 16-bit depth, pinned host buffers
    keep, dn, an, bn, T, K = pinned_pairs(torch, [distinct[s % DISTINCT_PAIRS] for s in range(n_slots)])
    init = np.stack([orc.se3_to_mat16(pose0[s % DISTINCT_PAIRS]) for s in range(n_slots)])
    ctx.set_pairs_u16(0, dn, an, bn, T, K)   # first pass pays the one-time allocations: not timed
    ctx.prepare_pairs(0, init)
    barrier()
    t0 = time.perf_counter()
    ctx.set_pairs_u16(0, dn, an, bn, T, K)
    ctx.prepare_pairs(0, init)
    t_prep = time.perf_counter() - t0
    job_pair = np.arange(n_slots, dtype=np.int32)
    total_steps = args.warmup + args.steps
    n_pose_sets = min(total_steps, 8)
    poses = [make_poses(orc, pose0, k, n_slots) for k in range(n_pose_sets)]

    # ---------------- device-resident throughput (`value`)
    for k in range(args.warmup):
        ctx.stage_jobs(poses[k % n_pose_sets], job_pair)
        ctx.eval_staged(n_slots, True)
    ctx.sync()
    launches0 = ctx.launch_count()
    barrier()
    with ClockSampler(local_rank) as clk:
        ctx.event_record(0)
        for k in range(args.warmup, total_steps):
            ctx.stage_jobs(poses[k % n_pose_sets], job_pair)
            ctx.eval_staged(n_slots, True)
        ctx.event_record(1)
        ms = ctx.event_elapsed_ms()
        barrier()
    launches = ctx.launch_count() - launches0
    Ht, Hj, der = ctx.fetch_results(n_slots, True)
    assert np.all(np.isfinite(Hj)) and np.all(np.isfinite(der)), "non-finite results in the timed region"
    if args.dump_outputs:  # fp64, 1 KB per pair slot
        os.makedirs(args.dump_outputs, exist_ok=True)
        suffix = f"_rank{rank}" if world > 1 else ""
        for name, a in (("Htarget", Ht), ("Hjoint", Hj), ("der", der)):
            np.save(os.path.join(args.dump_outputs, f"{name}{suffix}.npy"), a)

    # ---------------- end to end through the host-buffer C-ABI call (`e2e`)
    for k in range(args.warmup):
        ctx.eval_jobs(poses[k % n_pose_sets], job_pair, True)
    barrier()
    t0 = time.perf_counter()
    for k in range(args.warmup, total_steps):
        ctx.eval_jobs(poses[k % n_pose_sets], job_pair, True)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0

    # ---------------- per-kernel device time, live (roofline of the dominant kernel)
    ctx.set_option("time_kernels", 1)
    for k in range(min(args.steps, 20)):
        ctx.stage_jobs(poses[k % n_pose_sets], job_pair)
        ctx.eval_staged(n_slots, True)
    ctx.sync()
    kt = ctx.kernel_times()
    ctx.set_option("time_kernels", 0)

    # ---------------- kernel 1 on its own (warp + sample, north_star kernel (1)): HBM roofline probe
    probe = None
    try:
        n_probe = min(n_slots, 96)
        pp = [np.ascontiguousarray(q[:n_probe]) for q in poses]
        for k in range(3):
            ctx.warp_sample_jobs(pp[k % n_pose_sets], job_pair[:n_probe], fetch=False)
        reps = max(10, min(args.steps, 50))
        ctx.event_record(0)
        for k in range(reps):
            ctx.warp_sample_jobs(pp[k % n_pose_sets], job_pair[:n_probe], fetch=False)
        ctx.event_record(1)
        probe_ms = ctx.event_elapsed_ms() / reps
        probe = {"kernel": "k_warp_sample_jobs", "ms_per_launch": probe_ms, "jobs_per_launch": n_probe,
                 "algorithmic_bytes_per_launch": ROWS * COLS * 24 * n_probe,
                 "moved_bytes_per_launch": ROWS * COLS * (2 + 6 + 16) * n_probe,
                 "note": "one launch = kernel 1 for 96 pair slots: raw 16-bit depth in (2 B/px), fp16 target planes gathered "
                         "(6 B/px), float4 {I_c, g_x, g_y, valid} out (16 B/px); algorithmic bytes = SURVEY 8(d) 24 B/px; the "
                         "evaluation path fuses this front end into both passes instead of storing its output"}
    except Exception as e:  # noqa: BLE001 - the probe must not take the bench line down
        probe = {"kernel": "k_warp_sample_jobs", "error": str(e)}

    # ---------------- complete LM pose solves (optimize(10), reference perturbation), all slots in lockstep
    solve_s, solve_stats = 0.0, None
    if args.solves:
        n_solve = min(n_slots, 128)
        p7 = np.stack([pose0[s % DISTINCT_PAIRS] for s in range(n_solve)])
        ctx.solve_jobs(p7, job_pair[:n_solve])  # warm
        barrier()
        t0 = time.perf_counter()
        reps_solve = 3
        for _ in range(reps_solve):
            _, solve_stats = ctx.solve_jobs(p7, job_pair[:n_solve])
        torch.cuda.synchronize()
        solve_s = (time.perf_counter() - t0) / reps_solve
    ctx.close()
    del ctx

    if world > 1:
        t = torch.tensor([ms, e2e_s * 1e3, solve_s * 1e3, t_prep * 1e3], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms, solve_ms, prep_ms = t.tolist()
    else:
        e2e_ms, solve_ms, prep_ms = e2e_s * 1e3, solve_s * 1e3, t_prep * 1e3

    # ---------------- BASELINE configs 4 and 5 as stated, old-GPU path
    c4 = c5 = old = None
    c5_pair = c5_all = None
    try:
        if args.c4_pairs > 0:
            c4 = leg_c4(args, nid, synth, orc, shard, torch, dist, rank, world, local_rank, barrier)
    except Exception as e:  # noqa: BLE001
        c4 = {"error": repr(e)}
    try:
        if args.c5:
            c5, c5_pair, c5_all = leg_c5(args, nid, synth, orc, shard, torch, dist, rank, world, local_rank, barrier)
    except Exception as e:  # noqa: BLE001
        c5 = {"error": repr(e)}
    shim = single = None
    if rank == 0 and world == 1 and args.old_gpu:
        try:
            old = leg_old_gpu(nid, synth, orc, torch)
        except Exception as e:  # noqa: BLE001
            old = {"error": repr(e)}
        try:
            shim = leg_shim(nid, synth, orc, torch)
        except Exception as e:  # noqa: BLE001
            shim = {"error": repr(e)}
        try:
            single = leg_single_pair(nid, synth, orc)
        except Exception as e:  # noqa: BLE001
            single = {"error": repr(e)}

    if rank == 0:
        evals = args.steps * n_slots * world
        value = evals / (ms * 1e-3)
        e2e_value = evals / (e2e_ms * 1e-3)
        peak, peak_src = peaks()
        clocks = clk.summary()
        dom = max(("k_hist_sell", "k_jac_sell"), key=lambda n: kt[n][0])
        per_launch_jobs = min(n_slots, 96)  # the pixel kernels take 96 jobs per launch (one geometry table)
        launches_per_step = -(-n_slots // 96)
        dom_ms = kt[dom][0] / max(kt[dom][1], 1) / launches_per_step  # kernel_times brackets all launches of one evaluation step
        share = {n: kt[n][0] for n in kt}
        tot = sum(share.values()) or 1.0
        achieved = ALGO_BYTES_PER_EVAL * (n_slots / launches_per_step) / (dom_ms * 1e-3) / 1e9
        traffic, traffic_src = measured_traffic(dom, n_slots / launches_per_step)
        line = {
            "metric": "NID cost+Jacobian evals/s @640x480", "value": value, "unit": "evals/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "C2: 640x480 pair, 4x4 cells, 16-bin cubic B-spline NID, cost+Jacobian",
                       "rows": ROWS, "cols": COLS, "cell": CELL, "bins": BINS, "pairs_per_gpu": n_slots,
                       "evals_per_step": n_slots * world,
                       "l2": f"inputs larger than L2: {n_slots} pair slots x ~18 MB of device data per GPU streamed every step"},
            "e2e": {"value": e2e_value, "unit": "evals/s", "h2d_bytes_per_step": n_slots * (16 * 8 + 4),
                    "d2h_bytes_per_step": n_slots * CELL * CELL * 8 * 8,
                    "call": "nid_eval_jobs (host poses in, host Htarget/Hjoint/der out, blocking)"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "binding_roof": "fp64 issue (see fp64 below): all arithmetic of this path is fp64 (SURVEY 7: fp32 breaks "
                                         "the 1e-5 Jacobian bar), so the kernel is bounded by the fp64 pipe and instruction issue, "
                                         "not by HBM; the HBM figure is SURVEY 8(d)'s algorithmic bytes over the kernel time",
                         "algorithmic_bytes_per_launch": ALGO_BYTES_PER_EVAL * (n_slots / launches_per_step),
                         "evals_per_launch": n_slots / launches_per_step,
                         "kernel_ms_per_launch": dom_ms,
                         "ncu_pipes": measured_pipes(dom),
                         "fp64": fp64_roofline(dom, n_slots / launches_per_step, dom_ms, clocks.get("sm_mhz")),
                         "kernel_share_of_step": {n: share[n] / tot for n in share}},
            "clocks": clocks,
        }
        if probe and "ms_per_launch" in probe:
            probe["achieved"] = probe["algorithmic_bytes_per_launch"] / (probe["ms_per_launch"] * 1e-3) / 1e9
            probe["moved"] = probe["moved_bytes_per_launch"] / (probe["ms_per_launch"] * 1e-3) / 1e9
            probe["unit"] = "GB/s"
            probe["peak"] = peak
            probe["frac"] = probe["achieved"] / peak
            probe["frac_moved"] = probe["moved"] / peak
        line["roofline"]["warp_sample_probe"] = probe
        line["pair_setup"] = {"value": n_slots * world / (prep_ms * 1e-3), "unit": "pairs/s", "pairs": n_slots * world,
                              "call": "nid_set_pairs_u16 (raw 16-bit depth + two 8-bit images per pair from pinned host buffers, "
                                      "1.2 MB per pair) + nid_prepare_pairs (in-bounds set, n_c, H_ref, task tables built on the "
                                      "device, regrouped pixel store), wall clock, max over ranks"}
        if args.solves and solve_ms > 0:
            n_solve = min(n_slots, 128)
            line["pose_solves"] = {"value": n_solve * world / (solve_ms * 1e-3), "unit": "solves/s",
                                   "solves": n_solve * world, "ms": solve_ms,
                                   "mean_outer_iters": float(solve_stats[:, 0].mean()),
                                   "mean_jac_evals": float(solve_stats[:, 1].mean()),
                                   "mean_cost_evals": float(solve_stats[:, 2].mean()),
                                   "call": "nid_solve_jobs: optimize(10) LM schedule, 6x6 solves on the host overlapped with the other half-batch's kernels, wall clock"}
        # ---------------- CPU figures (rank 0, N=1 only; bounded samples)
        if world == 1:
            cpu_v, cpu_n, cpu_el, _ = cpu_eval_rate(orc, synth, 1, 1, args.cpu_budget / 3)
            workers, team = cpu_layout(os.cpu_count() or 1)
            cores = workers * team
            cpu_vm, cpu_nm, cpu_elm, arm = cpu_eval_rate(orc, synth, workers, team, args.cpu_budget / 3)
            line["cpu_baseline"] = {"value": cpu_vm, "unit": "evals/s", "cores": cores, "kind": "port",
                                    "single_thread_value": cpu_v,
                                    "sample": f"{cpu_nm} evals in {cpu_elm:.1f}s on {cores} threads ({workers} evaluations in flight x "
                                              f"{team} OpenMP threads over the cells) and {cpu_n} evals in {cpu_el:.1f}s on 1 thread, one "
                                              "seeded 640x480 pair (oracle/ restatement; the reference CPU path needs Eigen/OpenCV, "
                                              "absent here)"}
            if args.cpu_budget >= 3:
                ns, els = arm.solves()
                line["cpu_baseline"]["pose_solves"] = {"value": ns / els, "unit": "solves/s", "cores": cores,
                                                       "sample": f"{ns} optimize(10) runs in {els:.1f}s, {workers} in flight x {team} threads"}
                if c5_pair is not None:
                    p = c5_pair
                    idx = np.random.default_rng(6).choice(c5_all.shape[0], size=32, replace=False)
                    t0 = time.perf_counter()
                    for q in idx:
                        orc.hard_nid(p.im0, p.depth0, p.im1, p.T_wc0, c5_all[q], p.intr, 16, 8, threads=cores)
                    elh = time.perf_counter() - t0
                    line["cpu_baseline"]["hard_binned"] = {"value": len(idx) / elh, "unit": "hard-binned cost evals/s", "cores": cores,
                                                           "sample": f"{len(idx)} poses of the c5 sweep in {elh:.1f}s, OpenMP over the 256 cells"}
        else:
            line["cpu_baseline"] = None
        if c4 is not None:
            line["c4"] = c4
        if c5 is not None:
            line["c5"] = c5
        if old is not None:
            line["old_gpu_path"] = old
        if shim is not None:
            line["reference_api_shim"] = shim
        if single is not None:
            line["single_pair_latency"] = single
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
