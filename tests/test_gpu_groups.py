"""Joint pose solves over groups of pairs (nid_solve_groups): a multi-camera rig whose cameras share one body pose, and
several reference keyframes of one target frame. Groups of one are nid_solve_jobs bit for bit, in lock-step and in latency
mode; joint groups follow the oracle's LM over the edges of all their pairs (tests/group_oracle.py) to the bars of
test_gpu_parity.py::test_lm_solve_matches_oracle."""
import ctypes as C

import numpy as np
import pytest

import group_oracle

pytestmark = pytest.mark.gpu

DELTA = np.sqrt(0.95)
NID_ERR_ARG, NID_ERR_STATE = -2, -3


def _oracle_problem(orc, p, cell, bins):
    P = orc.Problem(p.im0, p.depth0, p.im1, p.T_wc0, p.intr, cell, bins, threads=4)
    P.set_quirks(0, 1)  # warp with the 4x4 like the CUDA code does
    return P


def _oracle_stats(its, counts):
    """iterations, linearisations, trial poses: the oracle's cost count also holds the re-evaluation at the end of
    every iteration, which the device solver does not repeat"""
    return [its, counts[0], counts[1] - its]


def _group(synth, orc, kind, seed, rows, cols):
    """(pairs, T_cb [n,16] or None, initial body pose7, ground-truth depth scale) of one group"""
    if kind == "single":
        p = synth.make_pair(seed, rows, cols)
        return [p], None, orc.reference_perturbation(p.T_wc1)
    if kind.startswith("rig"):
        rig = synth.make_rig(seed, int(kind[3:]), rows, cols)
        return rig.pairs, rig.T_cb, orc.reference_perturbation(rig.T_wb1)
    kf = synth.make_keyframes(seed, int(kind[2:]), rows, cols)
    return kf, None, orc.reference_perturbation(kf[0].T_wc1)


def _job_pose7(orc, T_cb, g, pose7):
    return pose7 if T_cb is None else orc.se3_mul(orc.se3_from_mat16(T_cb[g]), pose7)


def _load(ctx, orc, pairs, T_cb, pose0, pair0=0):
    for g, p in enumerate(pairs):
        ctx.set_pair(pair0 + g, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
        ctx.prepare(pair0 + g, orc.se3_to_mat16(_job_pose7(orc, T_cb, g, pose0)))


def _assert_matches_oracle(orc, pairs, T_cb, pose0, cell, bins, pose, stats, trace):
    probs = []
    for g, p in enumerate(pairs):
        P = _oracle_problem(orc, p, cell, bins)
        P.prepare(_job_pose7(orc, T_cb, g, pose0))
        probs.append(P)
    poseo, its, traceo, counts = group_oracle.optimize_group(probs, T_cb, pose0, 10, DELTA)
    assert np.array_equal(stats, _oracle_stats(its, counts))
    assert np.array_equal(trace[:its, 2], traceo[:, 2])  # same number of LM trials per iteration
    np.testing.assert_allclose(trace[:its, 0], traceo[:, 0], rtol=1e-7)
    depth = float(np.median(pairs[0].depth0))
    assert np.max(np.abs(pose[:3] - poseo[:3])) < 1e-4 * depth
    assert 2 * np.max(np.abs(pose[3:6] - poseo[3:6])) < 1e-4


@pytest.mark.parametrize("n", [9, 3])  # lock-step with both halves / latency mode
@pytest.mark.parametrize("reuse", [1, 0])
def test_groups_of_one_equal_solve_jobs(nid, orc, make_pair, n, reuse):
    pairs = [make_pair(1000 + i, 120, 160) for i in range(n)]
    ctx = nid.Context(120, 160, 4, 16, n_pairs=n, max_jobs=9)
    ctx.set_option("lm_reuse", reuse)
    pose0 = []
    for i, p in enumerate(pairs):
        ctx.set_pair(i, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
        pose0.append(orc.reference_perturbation(p.T_wc1))
        ctx.prepare(i, orc.se3_to_mat16(pose0[i]))
    pose0 = np.stack(pose0)
    jp = np.arange(n, dtype=np.int32)[::-1].copy()
    want, want_st = ctx.solve_jobs(pose0, jp)
    got, st, trace = ctx.solve_groups(pose0, [1] * n, jp)
    assert got.tobytes() == want.tobytes() and np.array_equal(st, want_st)
    eye = np.tile(np.eye(4).reshape(16), (n, 1))
    got_e, st_e, trace_e = ctx.solve_groups(pose0, [1] * n, jp, T_cb=eye)
    assert got_e.tobytes() == want.tobytes() and np.array_equal(st_e, want_st) and trace_e.tobytes() == trace.tobytes()
    # nid_solve's trace is the trace of a group of one
    for j in (0, n - 1):
        pose, tr, s = ctx.solve(int(jp[j]), pose0[j])
        assert pose.tobytes() == want[j].tobytes() and np.array_equal(s, want_st[j])
        assert tr.tobytes() == trace[j, :s[0]].tobytes()
        assert not trace[j, s[0]:].any()


@pytest.mark.parametrize("kind", ["kf3", "rig2", "rig4"])
@pytest.mark.parametrize("cell,bins,rows,cols", [(4, 16, 120, 160), (16, 10, 240, 320)])
def test_group_matches_oracle(nid, orc, synth, kind, cell, bins, rows, cols):
    pairs, T_cb, pose0 = _group(synth, orc, kind, 11, rows, cols)
    G = len(pairs)
    ctx = nid.Context(rows, cols, cell, bins, n_pairs=G, max_jobs=G)
    _load(ctx, orc, pairs, T_cb, pose0)
    pose, st, trace = ctx.solve_groups(pose0[None], [G], None, T_cb)
    assert st[0, 0] >= 2
    _assert_matches_oracle(orc, pairs, T_cb, pose0, cell, bins, pose[0], st[0], trace[0])


def test_lockstep_equals_latency_mode_for_rig_groups(nid, orc, synth):
    a, Ta, pa = _group(synth, orc, "rig4", 21, 120, 160)
    b, Tb, pb = _group(synth, orc, "rig2", 22, 120, 160)
    ctx = nid.Context(120, 160, 4, 16, n_pairs=6, max_jobs=12)  # room for two trials of every job: latency mode
    _load(ctx, orc, a, Ta, pa)
    _load(ctx, orc, b, Tb, pb, pair0=4)
    poses0, T_cb = np.stack([pa, pb]), np.concatenate([Ta, Tb])
    lat = ctx.solve_groups(poses0, [4, 2], None, T_cb)
    ctx.set_option("lm_speculate", 0)
    lock = ctx.solve_groups(poses0, [4, 2], None, T_cb)
    for x, y in zip(lat, lock):
        assert x.tobytes() == y.tobytes()
    assert lat[1][:, 2].sum() > lat[1][:, 1].sum()  # some trials were rejected


def test_mixed_group_sizes_equal_groups_solved_alone(nid, orc, synth):
    kinds = [("single", 31), ("kf3", 32), ("rig2", 33), ("rig4", 34)]
    groups = [_group(synth, orc, k, s, 120, 160) for k, s in kinds]
    sizes = [len(g[0]) for g in groups]
    ctx = nid.Context(120, 160, 4, 16, n_pairs=sum(sizes), max_jobs=sum(sizes))
    T_cb, first = [], 0
    for pairs, E, pose0 in groups:
        _load(ctx, orc, pairs, E, pose0, pair0=first)
        T_cb.append(np.tile(np.eye(4).reshape(16), (len(pairs), 1)) if E is None else E)
        first += len(pairs)
    T_cb = np.concatenate(T_cb)
    poses0 = np.stack([g[2] for g in groups])
    jp = np.arange(sum(sizes), dtype=np.int32)
    poses, st, trace = ctx.solve_groups(poses0, sizes, jp, T_cb)  # 10 jobs in 10 slots: lock-step
    first = 0
    for j, (pairs, E, pose0) in enumerate(groups):
        sl = slice(first, first + sizes[j])
        alone = ctx.solve_groups(pose0[None], [sizes[j]], jp[sl], T_cb[sl])  # latency mode
        assert alone[0][0].tobytes() == poses[j].tobytes()
        assert np.array_equal(alone[1][0], st[j]) and alone[2][0].tobytes() == trace[j].tobytes()
        first += sizes[j]


def test_natural_path_rig_group_matches_oracle(nid, orc, synth):
    cell, bins = 4, 16
    pairs, T_cb, pose0 = _group(synth, orc, "rig2", 41, 120, 160)
    ctx = nid.Context(120, 160, cell, bins, n_pairs=2, max_jobs=2)
    ctx.set_option("path", 1)
    _load(ctx, orc, pairs, T_cb, pose0)
    pose, st, trace = ctx.solve_groups(pose0[None], [2], None, T_cb)
    _assert_matches_oracle(orc, pairs, T_cb, pose0, cell, bins, pose[0], st[0], trace[0])


def _raw(nid, ctx, n_groups, sizes, jp, T_cb, poses, stats, trace, max_iters=10):
    ip = C.POINTER(C.c_int)
    dp = C.POINTER(C.c_double)
    arr = lambda a, t: None if a is None else a.ctypes.data_as(t)
    return nid.lib().nid_solve_groups(ctx._h, n_groups, arr(sizes, ip), arr(jp, ip), arr(T_cb, dp), arr(poses, dp), max_iters,
                                      float(DELTA), arr(stats, ip), arr(trace, dp))


def test_errors_leave_outputs_untouched(nid, orc, make_pair):
    ctx = nid.Context(120, 160, 4, 16, n_pairs=3, max_jobs=4)
    p = make_pair(1000, 120, 160)
    pose0 = orc.reference_perturbation(p.T_wc1)
    for i in range(2):  # pair 2 is never prepared
        ctx.set_pair(i, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
        ctx.prepare(i, orc.se3_to_mat16(pose0))
    eye = np.tile(np.eye(4).reshape(16), (4, 1))
    not_orth = eye.copy(); not_orth[1, 0] = 1 + 1e-7
    bottom = eye.copy(); bottom[0, 3] = 1e-3
    mirror = eye.copy(); mirror[1, 0] = -1.0
    I32 = lambda *v: np.array(v, dtype=np.int32)
    cases = [
        (NID_ERR_ARG, 0, I32(1), I32(0), None),           # n_groups < 1
        (NID_ERR_ARG, 2, I32(1, 0), I32(0, 1), None),     # a group size < 1
        (NID_ERR_ARG, 2, I32(3, 2), None, None),          # more jobs than max_jobs
        (NID_ERR_ARG, 1, None, None, None),               # NULL group_size
        (NID_ERR_ARG, 2, I32(1, 1), I32(0, 3), None),     # job_pair out of range
        (NID_ERR_ARG, 2, I32(1, 1), I32(0, -1), None),
        (NID_ERR_ARG, 2, I32(2, 2), I32(0, 1, 0, 1), not_orth),
        (NID_ERR_ARG, 2, I32(2, 2), I32(0, 1, 0, 1), bottom),
        (NID_ERR_ARG, 2, I32(2, 2), I32(0, 1, 0, 1), mirror),
        (NID_ERR_STATE, 2, I32(1, 2), I32(0, 1, 2), None),  # pair 2 not prepared
    ]
    for rc, ng, sizes, jp, T_cb in cases:
        poses = np.full((2, 7), 7.5)
        stats = np.full((2, 3), -7, dtype=np.int32)
        trace = np.full((2, 10, 10), 3.25)
        assert _raw(nid, ctx, ng, sizes, jp, T_cb, poses, stats, trace) == rc
        assert np.all(poses == 7.5) and np.all(stats == -7) and np.all(trace == 3.25)
    stats = np.full((1, 3), -7, dtype=np.int32)
    assert _raw(nid, ctx, 1, I32(1), I32(0), None, None, stats, None) == NID_ERR_ARG  # NULL poses7
    assert np.all(stats == -7)
    # the same pair in several jobs of one group is allowed
    poses, st, _ = ctx.solve_groups(pose0[None], [2], [0, 0])
    assert st[0, 0] >= 1


def test_group_without_active_cells_keeps_its_pose(nid, orc, make_pair):
    """16x16 cells of 60x80 pixels hold 15 pixels each, under NID_MIN_CELL_POINTS: no cell is active."""
    p = make_pair(1000, 60, 80)
    pose0 = orc.reference_perturbation(p.T_wc1)
    ctx = nid.Context(60, 80, 16, 16, n_pairs=1, max_jobs=3)
    ctx.set_pair(0, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
    nc, _ = ctx.prepare(0, orc.se3_to_mat16(pose0))
    assert nc.max() < 300
    poses, st, trace = ctx.solve_groups(pose0[None], [3], [0, 0, 0])
    assert np.array_equal(st[0], [1, 1, 1])
    assert poses[0].tobytes() == pose0.tobytes()
