"""State and memory-safety properties of the C-ABI that the round-1 review asked for: the asynchronous staged API
never reuses a pinned staging slot while a copy from it is pending, staged jobs survive a nid_prepare of another
pair, nid_eval_staged refuses more jobs than were staged, forced strip counts cannot overflow the partial buffers,
and the gradient taps of points with u == 0 / v == 0 exactly never read outside the image."""
import dataclasses

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

NATURAL, SORTED = 1, 2


def _two_pairs(nid, orc, make_pair, path, max_jobs=8, rows=120, cols=160):
    pa, pb = make_pair(1000, rows, cols), make_pair(1001, rows, cols)
    ctx = nid.Context(rows, cols, 4, 16, n_pairs=2, max_jobs=max_jobs)
    ctx.set_option("path", path)
    pose0 = []
    for i, p in enumerate((pa, pb)):
        ctx.set_pair(i, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
        pose0.append(orc.reference_perturbation(p.T_wc1))
        ctx.prepare(i, orc.se3_to_mat16(pose0[i]))
    return ctx, pose0


@pytest.mark.parametrize("path", [NATURAL, SORTED])
def test_pipelined_stage_eval_without_sync(nid, orc, make_pair, path):
    """stage A, eval, stage B (no synchronisation in between): the evaluation of A must see A's poses on the device
    (the natural-order kernels read them for every pixel, the sorted ones on their exact paths)."""
    ctx, pose0 = _two_pairs(nid, orc, make_pair, path)
    rng = np.random.default_rng(11)
    jp = np.array([0, 1, 1, 0, 0, 1, 0, 1], dtype=np.int32)

    def batch():
        return np.stack([orc.se3_to_mat16(orc.se3_mul(orc.se3_exp(rng.normal(size=6) * 3e-3), pose0[j])) for j in jp])
    for _ in range(12):
        A, B = batch(), batch()
        ref = ctx.eval_jobs(A, jp, True)
        ctx.stage_jobs(A, jp)
        ctx.eval_staged(len(jp), True)
        ctx.stage_jobs(B, jp)          # must not disturb the evaluation of A that is still in flight
        got = ctx.fetch_results(len(jp), True)
        for x, y in zip(got, ref):
            if path == SORTED:
                assert np.array_equal(x, y)
            else:
                np.testing.assert_allclose(x, y, rtol=1e-9, atol=1e-12)
    # many steps in flight (more than the staging ring holds): the last one is still right
    steps = [batch() for _ in range(9)]
    for S in steps:
        ctx.stage_jobs(S, jp)
        ctx.eval_staged(len(jp), True)
    got = ctx.fetch_results(len(jp), True)
    ref = ctx.eval_jobs(steps[-1], jp, True)
    for x, y in zip(got, ref):
        np.testing.assert_allclose(x, y, rtol=1e-9, atol=1e-12)


def test_staged_jobs_survive_prepare_and_kernel1_calls(nid, orc, make_pair):
    ctx, pose0 = _two_pairs(nid, orc, make_pair, SORTED)
    M0, M1 = orc.se3_to_mat16(pose0[0]), orc.se3_to_mat16(pose0[1])
    ref = ctx.eval_jobs(np.stack([M0]), np.array([0], dtype=np.int32), True)
    ctx.stage_jobs(np.stack([M0]), np.array([0], dtype=np.int32))
    ctx.prepare(1, M1)                # another pair, another pose: takes its own pose scratch
    ctx.warp_sample_f64(1, M1)
    ctx.eval_staged(1, True)
    got = ctx.fetch_results(1, True)
    for x, y in zip(got, ref):
        assert np.array_equal(x, y)
    with pytest.raises(nid.NidError, match="staged"):
        ctx.eval_staged(2, True)      # only one job was staged
    ctx.hard_eval_jobs(np.stack([M0, M1]), np.array([0, 1], dtype=np.int32))
    with pytest.raises(nid.NidError, match="staged"):
        ctx.eval_staged(1, True)      # hard-binned jobs are not evaluation jobs


def test_forced_strips_cannot_overflow_partials(nid, orc, make_pair):
    p = make_pair(1000, 120, 160)
    n_jobs = 96
    ctx = nid.Context(p.rows, p.cols, 2, 16, n_pairs=1, max_jobs=n_jobs)
    ctx.set_option("path", NATURAL)
    ctx.set_pair(0, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
    pose0 = orc.reference_perturbation(p.T_wc1)
    ctx.prepare(0, orc.se3_to_mat16(pose0))
    rng = np.random.default_rng(2)
    poses = np.stack([orc.se3_to_mat16(orc.se3_mul(orc.se3_exp(rng.normal(size=6) * 2e-3), pose0)) for _ in range(n_jobs)])
    jp = np.zeros(n_jobs, dtype=np.int32)
    ref = ctx.eval_jobs(poses, jp, True)
    ctx.set_option("force_strips", 32)  # 96 x 32 (job, strip) slots would not fit: clamped by the library
    got = ctx.eval_jobs(poses, jp, True)
    for x, y in zip(got, ref):
        np.testing.assert_allclose(x, y, rtol=1e-9, atol=1e-12)
    with pytest.raises(nid.NidError):
        ctx.set_option("force_strips", -1)


@pytest.mark.parametrize("path", [NATURAL, SORTED])
def test_first_row_and_column_points_at_identity(nid, orc, make_pair, synth, path):
    """T_cw1 = T_wc0^-1 with valid depth in the first image row and column: those points have u == 0 or v == 0, the
    Jacobian bounds test admits them (types_six_dof_expmap.cpp:433) and their gradient taps sit at -1.0 exactly.
    Upstream that indexes the image at -1 (undefined); here and in the oracle it is the continuous extension
    (nid_device.cuh interp_u8). Two pair slots hold different images: slot 1 must not see slot 0's bytes."""
    pa = make_pair(1000, 120, 160)
    pb = make_pair(1001, 120, 160)
    pa = dataclasses.replace(pa, im1=pa.im0.copy())
    pb = dataclasses.replace(pb, im1=pb.im0.copy())
    ctx = nid.Context(pa.rows, pa.cols, 2, 16, n_pairs=2, max_jobs=2)
    ctx.set_option("path", path)
    for slot, p in enumerate((pa, pb)):
        pose_id = orc.se3_from_mat16(synth.mat16_inverse(p.T_wc0))
        P = orc.Problem(p.im0, p.depth0, p.im1, p.T_wc0, p.intr, 2, 16, threads=4)
        P.set_quirks(0, 1)
        ctx.set_pair(slot, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
        M = orc.se3_to_mat16(pose_id)
        nc, href = ctx.prepare(slot, M)
        nco, hrefo = P.prepare(pose_id)
        assert np.array_equal(nc, nco)
        px = P.pixels(pose_id)
        assert np.sum((px[:, 0] == 0.0) & (px[:, 6] == 1)) > 20 and np.sum((px[:, 1] == 0.0) & (px[:, 6] == 1)) > 20
        Ht, Hj, J = ctx.eval(slot, M, True)
        Hto, Hjo, erro, Jo = P.eval(pose_id, True)
        np.testing.assert_allclose(Ht, Hto, rtol=1e-11)
        np.testing.assert_allclose(Hj, Hjo, rtol=1e-11)
        scale = np.abs(Jo).max(axis=1, keepdims=True)
        assert np.max(np.abs(J - Jo) / scale) < 1e-8
        got = ctx.warp_sample_f64(slot, M)
        m = ~np.isnan(px[:, 0])
        np.testing.assert_allclose(got[m, 2:5], px[m, 2:5], rtol=1e-12, atol=1e-10)


@pytest.mark.parametrize("cell,bins", [(4, 16), (8, 10)])
def test_batched_u16_setup_equals_single_pair_setup(nid, orc, make_pair, cell, bins):
    """nid_set_pairs_u16 + nid_prepare_pairs (raw 16-bit depth, task tables built on the device, several pairs per
    launch, more pairs than one set-up batch) against nid_set_pair + nid_prepare pair by pair: same n_c and H_ref, and
    bit-identical evaluations."""
    n = 37  # > one set-up batch of 32
    pairs = [make_pair(1000 + (i % 5), 120, 160, invalid_depth_frac=0.02 * (i % 3)) for i in range(n)]
    pose0 = [orc.reference_perturbation(p.T_wc1) for p in pairs]
    rng = np.random.default_rng(4)
    init = np.stack([orc.se3_to_mat16(orc.se3_mul(orc.se3_exp(rng.normal(size=6) * 2e-3), pose0[i])) for i in range(n)])
    A = nid.Context(120, 160, cell, bins, n_pairs=n, max_jobs=n)
    keep = A.set_pairs_u16(0, np.stack([p.depth0_u16 for p in pairs]), np.stack([p.im0 for p in pairs]),
                           np.stack([p.im1 for p in pairs]), np.stack([p.T_wc0 for p in pairs]),
                           np.stack([p.intr for p in pairs]))
    ncA, hrefA = A.prepare_pairs(0, init)
    del keep
    Bc = nid.Context(120, 160, cell, bins, n_pairs=n, max_jobs=n)
    for i, p in enumerate(pairs):
        Bc.set_pair(i, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
        nc, href = Bc.prepare(i, init[i])
        assert np.array_equal(nc, ncA[i]) and np.array_equal(href, hrefA[i], equal_nan=True)
    assert np.array_equal(A.points3d(3), Bc.points3d(3), equal_nan=True)
    jp = np.arange(n, dtype=np.int32)
    ra = A.eval_jobs(init, jp, True)
    rb = Bc.eval_jobs(init, jp, True)
    for x, y in zip(ra, rb):
        assert np.array_equal(x, y, equal_nan=True)
    # against the oracle for one pair of the second batch
    i = 34
    P = orc.Problem(pairs[i].im0, pairs[i].depth0, pairs[i].im1, pairs[i].T_wc0, pairs[i].intr, cell, bins, threads=4)
    P.set_quirks(0, 1)
    pose_i = orc.se3_from_mat16(init[i])
    nco, hrefo = P.prepare(pose_i)
    assert np.array_equal(ncA[i], nco)
    Hto, Hjo, _, Jo = P.eval(pose_i, True)
    act = ~np.isnan(hrefo)
    np.testing.assert_allclose(ra[0][i][act], Hto[act], rtol=1e-11)
    np.testing.assert_allclose(ra[1][i][act], Hjo[act], rtol=1e-11)
    # a re-prepare of a sub-range at other poses only touches that range
    A.prepare_pairs(5, init[5:9] )
    rc = A.eval_jobs(init, jp, True)
    for x, y in zip(ra, rc):
        assert np.array_equal(x, y, equal_nan=True)


def test_kernel1_from_raw_u16_depth(nid, orc, make_pair):
    """nid_warp_sample_jobs on pairs uploaded as raw 16-bit depth (2 B/px in) against the oracle's per-pixel record and
    against the same pairs uploaded as fp64 depth: flags identical, values to float precision."""
    pairs = [make_pair(1003, 120, 160, invalid_depth_frac=0.03), make_pair(1004, 120, 160)]
    A = nid.Context(120, 160, 4, 16, n_pairs=2, max_jobs=4)
    keep = A.set_pairs_u16(0, np.stack([p.depth0_u16 for p in pairs]), np.stack([p.im0 for p in pairs]),
                           np.stack([p.im1 for p in pairs]), np.stack([p.T_wc0 for p in pairs]), np.stack([p.intr for p in pairs]))
    A.sync()
    B = nid.Context(120, 160, 4, 16, n_pairs=2, max_jobs=4)
    for i, p in enumerate(pairs):
        B.set_pair(i, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
    base = [orc.reference_perturbation(p.T_wc1) for p in pairs]
    xi = np.array([0.002, -0.001, 0.0015, 0.004, -0.003, 0.002])
    jp = [0, 1, 1, 0]
    poses = [base[0], base[1], orc.se3_mul(orc.se3_exp(xi), base[1]), orc.se3_mul(orc.se3_exp(-xi), base[0])]
    M = np.stack([orc.se3_to_mat16(q) for q in poses])
    ga, gb = A.warp_sample_jobs(M, jp), B.warp_sample_jobs(M, jp)
    assert np.array_equal(ga, gb)  # same arithmetic once the depth is in a register
    for j, (pr, pose) in enumerate(zip(jp, poses)):
        P = orc.Problem(pairs[pr].im0, pairs[pr].depth0, pairs[pr].im1, pairs[pr].T_wc0, pairs[pr].intr, 4, 16, threads=4)
        P.set_quirks(0, 1)
        exp = P.pixels(pose)
        m = ~np.isnan(exp[:, 0])
        assert np.array_equal(ga[j, m, 3], exp[m, 5] + 2 * exp[m, 6])
        np.testing.assert_allclose(ga[j, m, 0], exp[m, 2], rtol=1e-6, atol=1e-5)
        np.testing.assert_allclose(ga[j, m, 1:3], exp[m, 3:5], rtol=1e-6, atol=1e-5)
        assert np.all(ga[j, ~m] == 0)


@pytest.mark.parametrize("cell,bins", [(4, 16), (8, 10)])
def test_lm_reuse_of_the_accepted_trial_is_bit_identical(nid, orc, make_pair, cell, bins):
    """nid_solve_jobs linearises at the pose of the accepted trial without recomputing that pose's histograms (option
    lm_reuse, default on): poses, iteration counts and the LM trace must equal a solve that recomputes everything,
    bit for bit; solo and batched, and against the oracle's LM run."""
    pairs = [make_pair(1000 + i, 120, 160) for i in range(9)]
    n = len(pairs)
    ctx = nid.Context(120, 160, cell, bins, n_pairs=n, max_jobs=n)
    pose0 = []
    for i, p in enumerate(pairs):
        ctx.set_pair(i, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
        pose0.append(orc.reference_perturbation(p.T_wc1))
        ctx.prepare(i, orc.se3_to_mat16(pose0[i]))
    pose0 = np.stack(pose0)
    jp = np.arange(n, dtype=np.int32)
    out1, st1 = ctx.solve_jobs(pose0, jp)
    solo1 = [ctx.solve(i, pose0[i]) for i in range(n)]
    ctx.set_option("lm_reuse", 0)
    out0, st0 = ctx.solve_jobs(pose0, jp)
    solo0 = [ctx.solve(i, pose0[i]) for i in range(n)]
    assert np.array_equal(out1, out0) and np.array_equal(st1, st0)
    for i in range(n):
        assert np.array_equal(solo1[i][0], solo0[i][0]) and np.array_equal(solo1[i][1], solo0[i][1])
        assert np.array_equal(solo1[i][0], out1[i]) and np.array_equal(solo1[i][2], st1[i])
    assert st1[:, 2].sum() > st1[:, 1].sum()  # some rejected trials happened (cost evaluations exceed Jacobian ones)
    # latency mode (speculative trial poses, default for up to four problems) against the plain state machine
    ctx.set_option("lm_reuse", 1)
    ctx.set_option("lm_speculate", 0)
    for i in (0, 3, 8):
        pose, trace, st = ctx.solve(i, pose0[i])
        assert np.array_equal(pose, solo1[i][0]) and np.array_equal(trace, solo1[i][1]) and np.array_equal(st, solo1[i][2])
    ctx.set_option("lm_speculate", 4)
    out2, st2 = ctx.solve_jobs(pose0[:2], jp[:2])
    assert np.array_equal(out2, out1[:2]) and np.array_equal(st2, st1[:2])
    P = orc.Problem(pairs[2].im0, pairs[2].depth0, pairs[2].im1, pairs[2].T_wc0, pairs[2].intr, cell, bins, threads=4)
    P.set_quirks(0, 1)
    P.prepare(pose0[2])
    poseo, its, traceo, counts = P.optimize(pose0[2], 10)
    assert st1[2, 0] == its
    np.testing.assert_allclose(solo1[2][1][:, 0], traceo[:, 0], rtol=1e-7)
    assert np.max(np.abs(out1[2] - poseo)) < 1e-7


@pytest.mark.parametrize("cell,bins,rows,cols", [(8, 10, 240, 320), (2, 16, 120, 160), (2, 40, 120, 160), (1, 9, 96, 128)])
def test_launch_shape_options_do_not_change_any_bit(nid, orc, make_pair, cell, bins, rows, cols):
    """How the work is launched is chosen by geometry and by the number of evaluations in flight -- bulk-copy or linear
    staging of the log tables in pass 2, the 1024-thread assembly for a handful of jobs, one job or twelve per launch --
    and none of it may change a result: every combination must reproduce the default bit for bit."""
    p = make_pair(1003, rows, cols, invalid_depth_frac=0.04)
    pose0 = orc.reference_perturbation(p.T_wc1)
    poses = np.stack([orc.se3_to_mat16(orc.se3_mul(orc.se3_exp(1e-3 * (k + 1) * np.array([1, -1, 0.5, 2, -2, 1.0])), pose0)) for k in range(12)])
    ctx = nid.Context(rows, cols, cell, bins, n_pairs=1, max_jobs=12)
    ctx.set_pair(0, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
    ctx.prepare(0, orc.se3_to_mat16(pose0))
    ref = ctx.eval_jobs(poses, np.zeros(12, np.int32), True)
    assert np.isfinite(ref[2][~np.isnan(ref[0])]).all()
    for bulk in (0, 1):
        for wide in (0, 1):
            ctx.set_option("stage_bulk", bulk)
            ctx.set_option("asm_wide", wide)
            got = ctx.eval_jobs(poses, np.zeros(12, np.int32), True)
            for a, b in zip(ref, got):
                assert np.array_equal(a, b, equal_nan=True), (bulk, wide)
            one = ctx.eval(0, poses[5], True)  # one job in flight: other CTA sizes, the wide assembly when allowed
            for a, b in zip(ref, one):
                assert np.array_equal(a[5], b, equal_nan=True), (bulk, wide)
    ctx.close()


def test_latency_mode_graph_survives_changes_of_the_context(nid, orc, make_pair):
    """The latency mode replays one captured CUDA graph per round (nid_sorted.cu, launch_latency_round). Everything the
    graph captured by value may change between solves -- another pair in the slot, another prepare pose (other slice
    counts), another task length, another Huber delta, another number of problems -- and every solve must equal the
    same solve without the graph, bit for bit."""
    pairs = [make_pair(1000 + i, 120, 160) for i in range(3)]
    ctx = nid.Context(120, 160, 2, 12, n_pairs=3, max_jobs=3)
    pose0 = []
    for i, p in enumerate(pairs):
        ctx.set_pair(i, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
        pose0.append(orc.reference_perturbation(p.T_wc1))
        ctx.prepare(i, orc.se3_to_mat16(pose0[i]))
    pose0 = np.stack(pose0)

    def both(f):
        ctx.set_option("lm_graph", 1)
        a = f()
        a2 = f()  # replay of the cached graph
        ctx.set_option("lm_graph", 0)
        b = f()
        for x, y, z in zip(a, a2, b):
            assert np.array_equal(x, y) and np.array_equal(x, z)
        return a

    both(lambda: ctx.solve(0, pose0[0]))
    both(lambda: ctx.solve(1, pose0[1], 10, 0.5))                      # another pair, another delta
    both(lambda: ctx.solve_jobs(pose0, np.arange(3, dtype=np.int32)))  # three problems: other slot count
    q = make_pair(1010, 120, 160, invalid_depth_frac=0.3)              # fewer valid pixels: other slice counts
    ctx.set_pair(0, q.depth0, q.im0, q.im1, q.T_wc0, q.intr)
    q0 = orc.reference_perturbation(q.T_wc1)
    ctx.prepare(0, orc.se3_to_mat16(q0))
    pose, trace, st = both(lambda: ctx.solve(0, q0))
    ctx.set_option("task_px", 32)
    for i in range(3):
        ctx.prepare(i, orc.se3_to_mat16(pose0[i] if i else q0))
    pose32, trace32, st32 = both(lambda: ctx.solve(0, q0))
    assert np.array_equal(st, st32) and np.max(np.abs(pose - pose32)) < 1e-9  # (another task length: another summation order)
    P = orc.Problem(q.im0, q.depth0, q.im1, q.T_wc0, q.intr, 2, 12, threads=4)
    P.set_quirks(0, 1)
    P.prepare(q0)
    poseo, its, traceo, counts = P.optimize(q0, 10)
    assert st[0] == its and np.max(np.abs(pose - poseo)) < 1e-7


@pytest.mark.parametrize("cell,bins,rows,cols", [(8, 10, 240, 320), (16, 10, 480, 640), (4, 16, 120, 160), (5, 20, 200, 250)])
def test_small_and_odd_cells_against_the_oracle_with_pixels_out_of_bounds_at_prepare(nid, orc, make_pair, cell, bins, rows,
                                                                                    cols):
    """Small cells (1200 to 2000 pixels: a handful of pixels per reference intensity, short tasks) at odd cell and bin
    counts, prepared at a pose that puts part of the frame out of bounds, so that many valid pixels have no reference
    sample: against the oracle at the prepare pose and away from it, histograms included, and the cost-only evaluation
    equal to the cost of the cost+Jacobian one, bit for bit."""
    p = make_pair(1004, rows, cols, invalid_depth_frac=0.05)
    pose0 = orc.reference_perturbation(p.T_wc1)
    shift = orc.se3_mul(orc.se3_exp(np.array([0, 0.05, 0, 0, 0, 0])), pose0)  # part of the frame starts out of bounds
    P = orc.Problem(p.im0, p.depth0, p.im1, p.T_wc0, p.intr, cell, bins, threads=8)
    P.set_quirks(0, 1)
    nco, hrefo = P.prepare(shift)
    act = ~np.isnan(hrefo)
    ctx = nid.Context(rows, cols, cell, bins, max_jobs=2)
    ctx.set_option("keep_hist", 1)
    ctx.set_pair(0, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
    nc, href = ctx.prepare(0, orc.se3_to_mat16(shift))
    assert np.array_equal(nc, nco)
    out = []
    for pose in (shift, orc.se3_mul(orc.se3_exp(np.array([0.002, -0.03, 0.0015, 0.004, -0.003, 0.002])), shift)):
        Ht, Hj, J = ctx.eval(0, orc.se3_to_mat16(pose), True)
        Hto, Hjo, erro, Jo = P.eval(pose, True)
        np.testing.assert_allclose(Ht[act], Hto[act], rtol=1e-11)
        np.testing.assert_allclose(Hj[act], Hjo[act], rtol=1e-11)
        scale = np.abs(Jo[act]).max(axis=1, keepdims=True)
        assert np.max(np.abs(J[act] - Jo[act]) / scale) < 1e-8
        assert np.all(np.isnan(Ht[~act])) and np.all(np.isnan(J[~act]))
        c0 = int(np.where(act)[0][0])
        pt, pj = ctx.debug_hist(0, c0)
        pto, pjo = P.last_hist(c0)
        np.testing.assert_allclose(pj, pjo, rtol=1e-10, atol=1e-16)
        np.testing.assert_allclose(pt, pto, rtol=1e-10, atol=1e-16)
        out.append((Ht, Hj, J))
    Ht2, Hj2, _ = ctx.eval(0, orc.se3_to_mat16(shift), False)
    assert np.array_equal(Ht2[act], out[0][0][act]) and np.array_equal(Hj2[act], out[0][1][act])
    ctx.close()


def test_every_cell_inactive(nid, orc, make_pair):
    """Cells of fewer than 300 pixels can never reach the reference's 300-point threshold (computeH.cu:271): everything is
    NaN, nothing is launched on an empty pixel store, and a solve leaves the pose where it was."""
    p = make_pair(1000, 120, 160)
    ctx = nid.Context(120, 160, 8, 10, max_jobs=2)   # 15 x 20 = 300 pixels per cell, minus the ones that leave the image
    ctx.set_pair(0, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
    pose0 = orc.reference_perturbation(p.T_wc1)
    M0 = orc.se3_to_mat16(pose0)
    nc, href = ctx.prepare(0, M0)
    P = orc.Problem(p.im0, p.depth0, p.im1, p.T_wc0, p.intr, 8, 10)
    P.set_quirks(0, 1)
    nco, hrefo = P.prepare(pose0)
    assert np.array_equal(nc, nco) and np.all(np.isnan(hrefo[nc < 300])) and np.array_equal(np.isnan(href), np.isnan(hrefo))
    inactive = nc < 300
    assert 8 <= inactive.sum() < nc.size
    Ht, Hj, J = ctx.eval(0, M0, True)
    assert np.all(np.isnan(Ht[inactive])) and np.all(np.isnan(Hj[inactive])) and np.all(np.isnan(J[inactive]))
    # a geometry in which every single cell is inactive
    ctx2 = nid.Context(120, 160, 10, 10, max_jobs=2)  # 12 x 16 = 192 pixels per cell
    ctx2.set_pair(0, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
    nc2, href2 = ctx2.prepare(0, M0)
    assert np.all(nc2 < 300) and np.all(np.isnan(href2))
    Ht, Hj, J = ctx2.eval(0, M0, True)
    assert np.all(np.isnan(Ht)) and np.all(np.isnan(Hj)) and np.all(np.isnan(J))
    Ht, Hj, _ = ctx2.eval(0, M0, False)
    assert np.all(np.isnan(Ht))
    pose, trace, st = ctx2.solve(0, pose0, 3)
    assert np.array_equal(pose, pose0)
