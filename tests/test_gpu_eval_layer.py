"""The evaluation layer drives both kernel families through the same job lists: the natural-order kernels (the only
path above 40 bins) run the lock-step LM's rounds like the sorted ones, and a contiguous evaluation launches the same
kernels on either path. The LM bars are those of test_gpu_parity.py::test_lm_solve_matches_oracle."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

DELTA = np.sqrt(0.95)
NATURAL, SORTED = 1, 2  # nid_set_option("path", ...)


def _problem(orc, p, cell, bins):
    P = orc.Problem(p.im0, p.depth0, p.im1, p.T_wc0, p.intr, cell, bins, threads=4)
    P.set_quirks(0, 1)  # warp with the 4x4 like the CUDA code does
    return P


def _assert_pose_close(pose, poseo, depth):
    assert np.max(np.abs(pose[:3] - poseo[:3])) < 1e-4 * depth
    assert 2 * np.max(np.abs(pose[3:6] - poseo[3:6])) < 1e-4


def _oracle_stats(its, counts):
    """iterations, linearisations, trial poses: the oracle's cost count also holds the re-evaluation at the end of
    every iteration (sparse_optimizer.cpp:404-433), which the device solver does not repeat"""
    return [its, counts[0], counts[1] - its]


def _solo_solve_matches_oracle(ctx, P, p, pose0):
    pose, trace, stats = ctx.solve(0, pose0, 10, DELTA)
    poseo, its, traceo, counts = P.optimize(pose0, 10, DELTA)
    assert np.array_equal(stats, _oracle_stats(its, counts))
    assert np.array_equal(trace[:, 2], traceo[:, 2])           # same number of LM trials per iteration
    np.testing.assert_allclose(trace[:, 0], traceo[:, 0], rtol=1e-7)
    _assert_pose_close(pose, poseo, float(np.median(p.depth0)))


@pytest.mark.parametrize("cell,bins,rows,cols", [(4, 16, 240, 320), (16, 10, 480, 640)])
def test_natural_path_solve_matches_oracle(nid, orc, make_pair, cell, bins, rows, cols):
    p = make_pair(1000, rows, cols)
    pose0 = orc.reference_perturbation(p.T_wc1)
    ctx = nid.Context(rows, cols, cell, bins)
    ctx.set_option("path", NATURAL)
    ctx.set_pair(0, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
    ctx.prepare(0, orc.se3_to_mat16(pose0))
    P = _problem(orc, p, cell, bins)
    P.prepare(pose0)
    _solo_solve_matches_oracle(ctx, P, p, pose0)


def test_48_bins_evaluation_and_solve_match_oracle(nid, orc, make_pair):
    """Above 40 bins the automatic path is the natural-order one (three kernels for a cost+Jacobian evaluation)."""
    cell, bins = 4, 48
    p = make_pair(1000, 240, 320)
    pose0 = orc.reference_perturbation(p.T_wc1)
    M0 = orc.se3_to_mat16(pose0)
    ctx = nid.Context(p.rows, p.cols, cell, bins)
    ctx.set_pair(0, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
    nc, href = ctx.prepare(0, M0)
    P = _problem(orc, p, cell, bins)
    nco, hrefo = P.prepare(pose0)
    assert np.array_equal(nc, nco)
    act = ~np.isnan(hrefo)
    assert act.any()
    np.testing.assert_allclose(href[act], hrefo[act], rtol=1e-12)
    pose = orc.se3_mul(orc.se3_exp(np.array([0.002, -0.001, 0.0015, 0.004, -0.003, 0.002])), pose0)
    n0 = ctx.launch_count()
    Ht, Hj, J = ctx.eval(0, orc.se3_to_mat16(pose), True)
    assert ctx.launch_count() - n0 == 3  # k_hist, k_jac, k_jac_final
    Hto, Hjo, erro, Jo = P.eval(pose, True)
    np.testing.assert_allclose(Ht[act], Hto[act], rtol=1e-11)
    np.testing.assert_allclose(Hj[act], Hjo[act], rtol=1e-11)
    assert np.all(np.isnan(Ht[~act])) and np.all(np.isnan(J[~act]))
    scale = np.max(np.abs(Jo[act]), axis=1, keepdims=True)
    assert np.max(np.abs(J[act] - Jo[act]) / scale) < 1e-8
    _solo_solve_matches_oracle(ctx, P, p, pose0)


def test_natural_path_solve_jobs_matches_oracle(nid, orc, make_pair):
    """Nine problems in one lock-step solve on the natural-order path: the job lists have holes where problems wait
    for a trial pose or have finished, and every problem must follow its own oracle run."""
    cell, bins = 4, 16
    pairs = [make_pair(1000 + i, 120, 160) for i in range(9)]
    n = len(pairs)
    ctx = nid.Context(120, 160, cell, bins, n_pairs=n, max_jobs=n)
    ctx.set_option("path", NATURAL)
    pose0 = []
    for i, p in enumerate(pairs):
        ctx.set_pair(i, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
        pose0.append(orc.reference_perturbation(p.T_wc1))
        ctx.prepare(i, orc.se3_to_mat16(pose0[i]))
    pose0 = np.stack(pose0)
    out, stats = ctx.solve_jobs(pose0, np.arange(n, dtype=np.int32), 10, DELTA)
    rounds = stats[:, 1] + stats[:, 2]  # one evaluation per problem and round
    assert len(set(rounds.tolist())) > 1  # the problems finish at different rounds
    for i, p in enumerate(pairs):
        P = _problem(orc, p, cell, bins)
        P.prepare(pose0[i])
        poseo, its, traceo, counts = P.optimize(pose0[i], 10, DELTA)
        assert np.array_equal(stats[i], _oracle_stats(its, counts)), i
        _assert_pose_close(out[i], poseo, float(np.median(p.depth0)))


@pytest.mark.parametrize("path,counts,timed", [(NATURAL, (3, 2, 4), (3, 2, 2, 1)), (SORTED, (4, 2, 5), (3, 2, 2, 3))],
                         ids=["natural", "sorted"])
@pytest.mark.parametrize("n_jobs", [1, 12])
def test_launch_counts_of_an_evaluation(nid, orc, make_pair, path, counts, timed, n_jobs):
    """Kernels launched by a cost+Jacobian evaluation, a cost-only one and a Gauss-Newton evaluation. Natural: k_hist,
    k_jac, k_jac_final / k_hist, k_entropy; sorted: pixel kernel, assembly, pixel kernel, Jacobian tail / pixel kernel,
    assembly; both then k_gn. The kernel timer's four buckets count each kernel it brackets once per evaluation: the
    natural path's cost tail (k_entropy, in the assembly's bucket) runs in the cost-only evaluation only."""
    p = make_pair(1000, 120, 160)
    pose0 = orc.reference_perturbation(p.T_wc1)
    M0 = orc.se3_to_mat16(pose0)
    ctx = nid.Context(120, 160, 4, 16, max_jobs=n_jobs)
    ctx.set_option("path", path)
    ctx.set_pair(0, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
    ctx.prepare(0, M0)
    poses = np.stack([orc.se3_to_mat16(orc.se3_mul(orc.se3_exp(1e-3 * k * np.array([1, -1, 0.5, 2, -2, 1.0])), pose0))
                      for k in range(n_jobs)])
    ctx.set_option("time_kernels", 1)
    got = []
    for call in (lambda: ctx.eval_jobs(poses, np.zeros(n_jobs, np.int32), True),
                 lambda: ctx.eval_jobs(poses, np.zeros(n_jobs, np.int32), False),
                 lambda: ctx.eval_gn(0, M0, DELTA)):
        n0 = ctx.launch_count()
        call()
        got.append(ctx.launch_count() - n0)
    assert tuple(got) == counts
    kt = ctx.kernel_times()
    assert tuple(calls for ms, calls in kt.values()) == timed
    assert all(ms > 0 for ms, calls in kt.values() if calls)
