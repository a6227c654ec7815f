"""bench.py's reference arm runs without a GPU (it times the CPU restatement of the path) and prints the contract's line."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "3"],
                                  timeout=600).decode().strip().splitlines()
    assert len(out) == 1
    d = json.loads(out[0])
    assert d["impl"] == "reference" and d["unit"] == "evals/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["metric"] == "NID cost+Jacobian evals/s @640x480" and d["config"]["workload"].startswith("C2")
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and d["vs_baseline"] is None


def test_non_zero_ranks_of_the_reference_arm_do_no_work():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], env=env, timeout=120)
    assert out.decode().strip() == ""


def test_roofline_helpers_read_the_committed_ncu_capture():
    """bench.py takes roofline.traffic and roofline.ncu_pipes from profiles/traffic.json (written by
    tools/profile_summary.py from the committed ncu --set full capture): the file must name the two pixel kernels."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    for k in ("k_hist_sell", "k_jac_sell"):
        t, src = bench.measured_traffic(k, 96)
        assert t is not None and t > 96 * 3.6e6 and src.startswith("profiles/")  # at least the algorithmic bytes
        p = bench.measured_pipes(k)
        assert p is not None and 0 < p["fp64_pipe_pct"] < 100 and 0 < p["issue_active_pct"] <= 100
    peak, src = bench.peaks()
    assert 1000 < peak < 10000 and src


def test_fp64_roofline_and_sweep_helpers():
    """roofline.fp64 comes from the executed fp64 warp instructions per evaluation in profiles/traffic.json; the C5 lattice is
    the 6 x 64 x 64 grid of SURVEY 8(d) around the true pose; the CPU layout uses every core in teams that divide 16 cells."""
    import importlib
    import importlib.util
    import numpy as np
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    r = bench.fp64_roofline("k_jac_sell", 96, 0.36, 1965.0)
    assert r is not None and 0.2 < r["frac"] < 0.9 and r["unit"].startswith("G fp64")
    assert abs(r["peak"] - 0.49 * 4 * 148 * 1.965) < 1.0
    assert bench.fp64_roofline("no_such_kernel", 96, 0.36, 1965.0) is None
    assert bench.cpu_layout(16) == (1, 16) and bench.cpu_layout(32) == (2, 16) and bench.cpu_layout(8) == (1, 8) and bench.cpu_layout(1) == (1, 1)
    sys.path.insert(0, ROOT)
    synth = importlib.import_module("nid-pose-estimation_b200.synth")
    from oracle import binding as orc
    p = synth.make_pair(1000, 48, 64)
    poses = bench.c5_poses(orc, synth, p)
    assert poses.shape == (6 * 64 * 64, 16)
    gt = synth.mat16_inverse(p.T_wc1)
    # the lattice has no point exactly at the true pose (64 is even), and is symmetric: first and last offsets are +-0.05
    first = orc.se3_from_mat16(poses[0])
    d = orc.se3_mul(first, orc.se3_inverse(orc.se3_from_mat16(gt)))
    assert abs(2 * np.arcsin(min(1.0, np.linalg.norm(d[3:6]))) - np.hypot(0.05, 0.05)) < 1e-3  # rotation axes 0 and 1 at -0.05 rad each
    assert len({tuple(np.round(q, 12)) for q in poses[:4096]}) == 4096


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(tmp_path, orc, synth):
    """--dump-outputs writes what the timed path returned in its last step: slot s of a step k is pair s mod 6 at
    make_poses(step k)[s]; checked against the oracle for two slots that share a pair."""
    import importlib.util
    import numpy as np
    warmup, steps, slots = 3, 2, 7
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(warmup),
                                   "--pairs", str(slots), "--solves", "0", "--c4-pairs", "0", "--c5", "0", "--old-gpu", "0",
                                   "--cpu-budget", "0", "--dump-outputs", str(tmp_path)], timeout=900).decode().strip().splitlines()
    d = json.loads(out[-1])
    assert d["steps"] == steps and d["warmup"] == warmup
    Ht, Hj, der = (np.load(tmp_path / f"{n}.npy") for n in ("Htarget", "Hjoint", "der"))
    assert Ht.shape == Hj.shape == (slots, 16) and der.shape == (slots, 16, 6)
    assert Ht.dtype == Hj.dtype == der.dtype == np.float64
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    pairs = [synth.make_pair(1000 + i, bench.ROWS, bench.COLS) for i in range(bench.DISTINCT_PAIRS)]
    pose0 = [orc.reference_perturbation(p.T_wc1) for p in pairs]
    last = warmup + steps - 1
    M = bench.make_poses(orc, pose0, last % min(warmup + steps, 8), slots)
    p = pairs[0]
    P = orc.Problem(p.im0, p.depth0, p.im1, p.T_wc0, p.intr, bench.CELL, bench.BINS, threads=4)
    P.set_quirks(0, 1)
    P.prepare(pose0[0])
    for s in (0, bench.DISTINCT_PAIRS):
        Hto, Hjo, _, Jo = P.eval(orc.se3_from_mat16(M[s]), True)
        np.testing.assert_allclose(Ht[s], Hto, rtol=1e-10)
        np.testing.assert_allclose(Hj[s], Hjo, rtol=1e-10)
        assert np.max(np.abs(der[s] - Jo) / np.abs(Jo).max(axis=1, keepdims=True)) < 1e-5


def test_make_sequence_variants():
    import importlib
    import numpy as np
    sys.path.insert(0, ROOT)
    synth = importlib.import_module("nid-pose-estimation_b200.synth")
    seq = synth.make_sequence(1000, 5, 60, 80)
    p = synth.make_pair(1000, 60, 80)
    assert np.array_equal(seq[0].im0, p.im0) and np.array_equal(seq[0].im1, p.im1) and np.array_equal(seq[0].depth0_u16, p.depth0_u16)
    assert np.array_equal(seq[0].T_wc1, p.T_wc1)
    for k in range(1, 5):
        assert not np.array_equal(seq[k].im0, p.im0) and not np.array_equal(seq[k].im1, p.im1)
        assert np.array_equal(seq[k].depth0_u16, p.depth0_u16) and np.array_equal(seq[k].T_wc0, p.T_wc0)
    again = synth.make_sequence(1000, 5, 60, 80)
    assert all(np.array_equal(a.im1, b.im1) and np.array_equal(a.im0, b.im0) for a, b in zip(seq, again))
