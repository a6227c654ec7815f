"""Parity past 256 cells, at the 300-point activity threshold, and of the Gauss-Newton blocks against their own inputs.

Every other GPU test uses grids of at most 16 x 16 = 256 cells. Three pieces of device code have limits or branches
above that size:
- gn_block (csrc/nid_ctx.h) stages cells NID_GN_CHUNK = 256 at a time; its second chunk and a partial last chunk only
  run on larger grids. It builds every chi2, H and b: k_gn (nid_eval_gn, the lock-step LM), k_tail_gn and k_gn_out
  (latency mode).
- the sorted path's task descriptor keeps the cell index in bits 18-30 (count | cls << 9 | cell << 18); bits 26-30 hold
  a value only from cell index 256 on, bit 30 from 4096 on.
- every kernel that decides activity compares a cell's point count with 300 (NID_MIN_CELL_POINTS; k_hard: n >= 300).

The grids below are the seeded synthetic pair at the reference-perturbed start; the tests assert that each grid still
reaches the edge it is here for. The bars are those of test_gpu_parity.py, with an absolute floor where a saturated
plateau makes H_ref or a Jacobian row zero up to rounding (_assert_href_close, _jrel). The Gauss-Newton blocks are also
recomputed in fp64 numpy from the error and Jacobian the device returned with them: that isolates gn_block from the
evaluation, and a lost or doubled chunk, or a cell misplaced across a chunk boundary, changes a sum by a whole term."""
import types

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

DELTA = np.sqrt(0.95)
NATURAL, SORTED = 1, 2  # nid_set_option("path", ...)
GN_CHUNK = 256          # NID_GN_CHUNK, csrc/nid_ctx.h
MIN_POINTS = 300        # NID_MIN_CELL_POINTS
XI = np.array([0.002, -0.001, 0.0015, 0.004, -0.003, 0.002])

# cell: rows, cols, bins, make_pair keywords, Gauss-Newton chunks (the last one's size)
GRIDS = {
    4: (240, 320, 16, {}, 1, 16),
    17: (480, 640, 10, {}, 2, 33),                                # 28 x 37 pixels per cell
    32: (960, 1280, 10, {}, 4, 256),                              # 30 x 40: one cell at exactly 300 points
    64: (960, 1280, 10, {"invalid_depth_frac": 0.001}, 16, 256),  # 15 x 20 = 300: cells at 300 and at 299 points
    90: (1800, 1350, 10, {}, 32, 164),                            # 20 x 15 = 300: active cells with index >= 4096
}


@pytest.fixture(scope="module")
def grid(orc, make_pair):
    """The oracle side of one geometry, prepared at the reference-perturbed start; oracle results are cached by key."""
    made = {}

    def get(cell):
        if cell not in made:
            rows, cols, bins, kw, _, _ = GRIDS[cell]
            p = make_pair(1000, rows, cols, **kw)
            P = orc.Problem(p.im0, p.depth0, p.im1, p.T_wc0, p.intr, cell, bins, threads=8)
            P.set_quirks(0, 1)  # warp with the 4x4 like the CUDA code does
            pose0 = orc.reference_perturbation(p.T_wc1)
            nc, href = P.prepare(pose0)
            g = types.SimpleNamespace(p=p, P=P, cell=cell, bins=bins, pose0=pose0, nc=nc, href=href,
                                      act=~np.isnan(href), cache={})
            g.poses = (pose0, orc.se3_mul(orc.se3_exp(XI), pose0))
            made[cell] = g
        return made[cell]
    return get


def _oracle(g, key, fn):
    if key not in g.cache:
        g.cache[key] = fn()
    return g.cache[key]


def _oracle_eval(g, k):
    """the oracle's (Ht, Hj, err, J) at g.poses[k]"""
    return _oracle(g, ("eval", k), lambda: g.P.eval(g.poses[k], True))


def _context(nid, orc, g, path, max_jobs=1):
    ctx = nid.Context(g.p.rows, g.p.cols, g.cell, g.bins, max_jobs=max_jobs)
    ctx.set_option("path", path)
    ctx.set_option("keep_hist", 1)
    ctx.set_pair(0, g.p.depth0, g.p.im0, g.p.im1, g.p.T_wc0, g.p.intr)
    nc, href = ctx.prepare(0, orc.se3_to_mat16(g.pose0))
    return ctx, nc, href


def _jrel(J, Jo):
    """max over active cells of |dJ| / max|J_cell|; the NaN patterns must agree. The larger grids hold saturated
    plateaus: a cell whose reference patch is constant has a joint histogram that is the product of its marginals, so its
    err is 1 at every pose and its Jacobian is zero up to rounding (|J| ~ 1e-13, on either side). A row's scale is
    therefore taken as at least 1e-3 of the median row's: rounding noise is not held to a relative bar."""
    act = ~np.isnan(Jo[:, 0])
    assert np.array_equal(np.isnan(J[:, 0]), ~act)
    scale = np.max(np.abs(Jo[act]), axis=1, keepdims=True)
    scale = np.maximum(scale, 1e-3 * np.median(scale))
    return np.max(np.abs(J[act] - Jo[act]) / scale)


def _assert_href_close(href, hrefo):
    """H_ref at rtol 1e-12, or within 1e-12 bits where it is near zero. A saturated plateau has H_ref ~ 1.2e-3 (all weight
    of intensity 255 in one spline span); the entropy's rounding error is absolute, set by that of the bin masses. The
    reference sums the bin masses pixel by pixel: on the 30 x 40 cell of 1200 pixels at 255 in the 32 x 32 grid that
    rounds the dominant mass by 2.5e-11 and H_ref by 3.0e-14 (2.4e-11 relative); the device sums count x weight per
    intensity and lands on the exact value (checked in rational arithmetic)."""
    np.testing.assert_allclose(href, hrefo, rtol=1e-12, atol=1e-12)


def _assert_grid_reaches_its_edges(g):
    ncell = g.cell * g.cell
    chunks, last = GRIDS[g.cell][4:]
    assert -(-ncell // GN_CHUNK) == chunks and ncell - (chunks - 1) * GN_CHUNK == last
    idx = np.nonzero(g.act)[0]
    assert np.array_equal(g.act, g.nc >= MIN_POINTS)
    # every chunk of gn_block sums active cells, except (90 x 90) the partial last one
    used = np.unique(idx // GN_CHUNK)
    assert np.array_equal(used, np.arange(chunks if g.cell != 90 else chunks - 1))
    if g.cell == 17:
        assert g.act.all()  # the partial second chunk is all active cells
    if g.cell == 32:
        assert np.any(g.nc == MIN_POINTS)
    if g.cell == 64:
        assert np.sum(g.nc == MIN_POINTS) > 100 and np.sum(g.nc == MIN_POINTS - 1) > 100
    if g.cell == 90:
        assert np.sum(idx >= 4096) > 1000  # cell << 18 sets bit 30 of the task descriptor
        assert np.all(g.nc[g.act] == MIN_POINTS)  # 300-pixel cells: every active cell sits at the threshold


@pytest.mark.parametrize("path,cell", [(SORTED, 17), (SORTED, 32), (SORTED, 64), (SORTED, 90), (NATURAL, 17), (NATURAL, 32)])
def test_prepare_and_eval_past_256_cells(nid, orc, grid, path, cell):
    g = grid(cell)
    _assert_grid_reaches_its_edges(g)
    ctx, nc, href = _context(nid, orc, g, path, max_jobs=12 if path == SORTED else 1)
    act = g.act
    assert np.array_equal(nc, g.nc)
    assert np.array_equal(np.isnan(href), ~act)
    _assert_href_close(href[act], g.href[act])
    idx = np.nonzero(act)[0]
    show = sorted({idx[0], idx[len(idx) // 2], idx[-1], idx[np.searchsorted(idx, min(GN_CHUNK, idx[-1]))]} |
                  ({idx[np.searchsorted(idx, 4096)]} if cell == 90 else set()))
    for k, pose in enumerate(g.poses):
        M = orc.se3_to_mat16(pose)
        Ht, Hj, J = ctx.eval(0, M, True)
        Hto, Hjo, erro, Jo = _oracle_eval(g, k)
        np.testing.assert_allclose(Ht[act], Hto[act], rtol=1e-11)
        np.testing.assert_allclose(Hj[act], Hjo[act], rtol=1e-11)
        assert np.all(np.isnan(Ht[~act])) and np.all(np.isnan(Hj[~act]))
        assert _jrel(J, Jo) < 1e-8
        err = (2 * Hj - href - Ht) / Hj
        np.testing.assert_allclose(err[act], erro[act], rtol=1e-10)
        if k == 0:
            g.P.eval(pose, True)  # (the oracle's histograms are those of its last evaluation)
            for c in show:
                pt, pj = ctx.debug_hist(0, int(c))
                pto, pjo = g.P.last_hist(int(c))
                np.testing.assert_allclose(pt, pto, rtol=1e-11, atol=1e-16)
                np.testing.assert_allclose(pj, pjo, rtol=1e-11, atol=1e-16)
        # the cost-only call gives the entropies of the cost+Jacobian call and leaves der alone
        Ht2, Hj2, J2 = ctx.eval(0, M, False)
        if path == SORTED:
            assert np.array_equal(Ht2, Ht, equal_nan=True) and np.array_equal(Hj2, Hj, equal_nan=True)
        np.testing.assert_allclose(Ht2[act], Ht[act], rtol=1e-13)
        np.testing.assert_allclose(Hj2[act], Hj[act], rtol=1e-13)
        assert np.all(np.isnan(J2))
    if path == SORTED:
        # twelve jobs in one submission: each equals the same evaluation submitted alone, bit for bit
        rng = np.random.default_rng(cell)
        poses = np.stack([orc.se3_to_mat16(orc.se3_mul(orc.se3_exp(rng.uniform(-1, 1, 6) * 3e-3), g.pose0))
                          for _ in range(12)])
        Ht, Hj, J = ctx.eval_jobs(poses, np.zeros(12, np.int32), True)
        for j in range(12):
            a, b, c = ctx.eval(0, poses[j], True)
            assert np.array_equal(a, Ht[j], equal_nan=True) and np.array_equal(b, Hj[j], equal_nan=True)
            assert np.array_equal(c, J[j], equal_nan=True), j


@pytest.mark.parametrize("cell", [64, 90])
def test_hard_binned_at_the_threshold(nid, orc, grid, synth, cell):
    """k_hard's `n >= 300` against the oracle at poses where cells of exactly 300 and of 299 in-bounds points occur: a
    cell of 300 points contributes its NID, a cell of 299 contributes 0."""
    g = grid(cell)
    p = g.p
    gt = orc.se3_from_mat16(synth.mat16_inverse(p.T_wc1))
    poses = [gt, g.pose0, g.poses[1]]
    # the in-bounds counts of the hard-binned cells are the prepare counts at the same pose (same warp, same bounds test)
    Pc = orc.Problem(p.im0, p.depth0, p.im1, p.T_wc0, p.intr, cell, g.bins, threads=8)
    Pc.set_quirks(0, 1)
    counts = [Pc.prepare(q)[0] for q in poses]
    Ms = np.stack([orc.se3_to_mat16(q) for q in poses])
    ctx = nid.Context(p.rows, p.cols, cell, g.bins, max_jobs=len(poses))
    ctx.set_pair(0, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
    total, cells = ctx.hard_eval_jobs(Ms, np.zeros(len(poses), np.int32))
    both = 0
    for k, M in enumerate(Ms):
        to, co = orc.hard_nid(p.im0, p.depth0, p.im1, p.T_wc0, M, p.intr, cell, g.bins, threads=8)
        np.testing.assert_allclose(cells[k], co, rtol=1e-12, atol=1e-15)
        assert total[k] == pytest.approx(to, rel=1e-12)
        at, below = counts[k] == MIN_POINTS, counts[k] == MIN_POINTS - 1
        assert np.all(co[counts[k] < MIN_POINTS] == 0)
        if np.any(co[at] != 0) and np.any(below):
            both += 1
    assert both >= 1


# ---------------------------------------------------------------------------------------------- Gauss-Newton blocks
def _huber(e, delta, dsqr):
    """rho(e^2), rho'(e^2) of robust_kernel_impl.cpp:78-90 with the threshold dsqr"""
    chi = e * e
    inl = chi <= dsqr
    sq = np.sqrt(chi)
    return np.where(inl, chi, 2 * sq * delta - dsqr), np.where(inl, 1.0, delta / sq)


def _float_dsqr(delta):
    return float(np.float32(delta * delta))  # robust_kernel_impl.h:84 keeps delta^2 as a float


def _gn_terms(err, J, delta, dsqr):
    """per active cell, in cell order, the terms of chi2, H (row-major) and b: [n_active, 43]"""
    act = ~np.isnan(err)
    e, Jc = err[act], J[act]
    r0, r1 = _huber(e, delta, dsqr)
    tH = ((Jc[:, :, None] * r1[:, None, None]) * Jc[:, None, :]).reshape(-1, 36)
    tb = -(r1[:, None] * Jc) * e[:, None]
    return np.concatenate([r0[:, None], tH, tb], axis=1)


def _gn_block(err, J, delta, dsqr):
    """(the block summed in cell order, the sum of the absolute values of each entry's terms)"""
    T = _gn_terms(err, J, delta, dsqr)
    return np.cumsum(T, axis=0)[-1], np.abs(T).sum(axis=0)


def _flat(chi2, H, b):
    return np.concatenate([[chi2], np.reshape(H, 36), b])


def _half_outlier_delta(err):
    e2 = np.sort(err[~np.isnan(err)] ** 2)
    return float(np.sqrt(0.5 * (e2[len(e2) // 2 - 1] + e2[len(e2) // 2])))


@pytest.mark.parametrize("path", [SORTED, NATURAL])
@pytest.mark.parametrize("cell", [4, 17, 32, 90])
def test_eval_gn_against_oracle_and_its_own_outputs(nid, orc, grid, path, cell):
    g = grid(cell)
    ctx, _, _ = _context(nid, orc, g, path)
    M0 = orc.se3_to_mat16(g.pose0)
    _, _, erro, Jo = _oracle_eval(g, 0)
    act = g.act
    half = _half_outlier_delta(erro)
    frac = np.mean(erro[act] ** 2 > _float_dsqr(half))
    assert 0.4 < frac < 0.6
    for delta in (DELTA, half):
        chi2, H, b, err, J = ctx.eval_gn(0, M0, delta)
        assert np.array_equal(np.isnan(err), ~act)
        np.testing.assert_allclose(err[act], erro[act], rtol=1e-10)
        assert _jrel(J, Jo) < 1e-8
        chi2o, Ho, bo = _oracle(g, ("gn", delta), lambda: g.P.gn_system(g.pose0, delta))
        assert chi2 == pytest.approx(chi2o, rel=1e-10)
        np.testing.assert_allclose(H, Ho, rtol=1e-7, atol=1e-9 * np.abs(Ho).max())
        np.testing.assert_allclose(b, bo, rtol=1e-7, atol=1e-9 * np.abs(bo).max())
        # the block from the device's own err and J: equal up to the rounding of one term in each (FMA contraction)
        s, a = _gn_block(err, J, delta, _float_dsqr(delta))
        d = np.abs(_flat(chi2, H, b) - s)
        assert np.all(d <= 1e-13 * a), (np.argmax(d / a), np.max(d / a))
    # the numpy block reproduces the oracle's from the oracle's own inputs, which ties its Huber rule to the reference
    for delta in (DELTA, half):
        s, a = _gn_block(erro, Jo, delta, _float_dsqr(delta))
        chi2o, Ho, bo = g.cache[("gn", delta)]
        assert np.all(np.abs(_flat(chi2o, Ho, bo) - s) <= 1e-13 * a)
        for c in np.nonzero(act)[0][:4]:
            r0, r1 = _huber(erro[c:c + 1], delta, _float_dsqr(delta))
            assert np.array_equal(orc.huber(erro[c] ** 2, delta)[:2], [r0[0], r1[0]])


def _boundary_deltas(err):
    """Per active cell whose f = float32(e^2) differs from e^2 by more than 1e-9 relative: a delta whose double delta^2
    lies on the other side of e^2 (by at least 1e-10 relative) and rounds to f. The reference classifies the cell by f;
    a comparison with the double delta^2 classifies it the other way. -> [(cell, delta, f > e^2)]"""
    out = []
    for c in np.nonzero(~np.isnan(err))[0]:
        e2 = err[c] ** 2
        f32 = np.float32(e2)
        f = float(f32)
        if abs(f - e2) <= 1e-9 * e2:
            continue
        if f > e2:  # halfway between e^2 and the lower end of f's rounding interval
            d2 = 0.5 * (e2 + 0.5 * (f + float(np.nextafter(f32, np.float32(0)))))
        else:
            d2 = 0.5 * (e2 + 0.5 * (f + float(np.nextafter(f32, np.float32(np.inf)))))
        delta = float(np.sqrt(d2))
        d2 = delta * delta
        if _float_dsqr(delta) == f and abs(d2 - e2) >= 1e-10 * e2 and (d2 - e2) * (f - e2) < 0:
            out.append((int(c), delta, f > e2))
    return out


@pytest.mark.parametrize("path", [SORTED, NATURAL])
def test_float_dsqr_on_the_device(nid, orc, grid, path):
    """The Huber threshold is the float delta^2 (robust_kernel_impl.h:84). For cells whose e^2 lies between delta^2 and
    float(delta^2), the two rules classify differently; the device must follow the reference's."""
    g = grid(4)
    ctx, _, _ = _context(nid, orc, g, path)
    M0 = orc.se3_to_mat16(g.pose0)
    _, _, erro, Jo = _oracle_eval(g, 0)
    tol = 1e-10  # chi2 against the oracle
    picked = {True: [], False: []}
    cands = []
    for c, delta, above in _boundary_deltas(erro):
        chi2o, Ho, bo = g.P.gn_system(g.pose0, delta)
        right, _ = _gn_block(erro, Jo, delta, _float_dsqr(delta))
        wrong, _ = _gn_block(erro, Jo, delta, delta * delta)
        assert right[0] == pytest.approx(chi2o, rel=1e-13)  # the oracle classifies by f
        cands.append((abs(wrong[0] - chi2o) / chi2o, c, delta, above, (chi2o, Ho, bo)))
    for sep, c, delta, above, o in sorted(cands, reverse=True):
        if len(picked[above]) < 2:
            picked[above].append((sep, c, delta, o))
    assert len(picked[True]) == 2 and len(picked[False]) == 2  # cells above and below their float threshold
    for sep, c, delta, (chi2o, Ho, bo) in picked[True] + picked[False]:
        assert sep >= 100 * tol  # the wrong rule would fail this test by a wide margin
        chi2, H, b, err, J = ctx.eval_gn(0, M0, delta)
        assert chi2 == pytest.approx(chi2o, rel=tol), c
        np.testing.assert_allclose(H, Ho, rtol=1e-7, atol=1e-9 * np.abs(Ho).max())
        np.testing.assert_allclose(b, bo, rtol=1e-7, atol=1e-9 * np.abs(bo).max())
        got = _flat(chi2, H, b)
        s, a = _gn_block(err, J, delta, _float_dsqr(delta))
        assert np.all(np.abs(got - s) <= 1e-13 * a), c
        sw, _ = _gn_block(err, J, delta, delta * delta)
        assert np.max(np.abs(got - sw) / a) > 100 * 1e-13  # and the device's own inputs tell the rules apart too


# ---------------------------------------------------------------------------------------------- LM solves
def _oracle_stats(its, counts):
    """iterations, linearisations, trial poses: the oracle's cost count also holds the re-evaluation at the end of
    every iteration, which the device solver does not repeat"""
    return [its, counts[0], counts[1] - its]


def _assert_pose_close(pose, poseo, depth, tol=1e-7):
    assert np.max(np.abs(pose[:3] - poseo[:3])) < tol * depth
    assert 2 * np.max(np.abs(pose[3:6] - poseo[3:6])) < tol


def _starts(orc, g, n):
    rng = np.random.default_rng(17)
    return [g.pose0] + [orc.se3_mul(orc.se3_exp(rng.uniform(-1, 1, 6) * 2e-3), g.pose0) for _ in range(n - 1)]


@pytest.mark.parametrize("delta_kind", ["0.95", "half"])
@pytest.mark.parametrize("way", ["latency", "lockstep", "solve_jobs", "natural"])
def test_solves_past_256_cells(nid, orc, grid, way, delta_kind):
    """Every way of reaching a Gauss-Newton kernel on two chunks of cells: nid_solve in latency mode (k_jac_final_sorted
    + k_gn_out), with lm_speculate 0 (lock-step, k_gn), a 5-problem solve_jobs (lock-step) and the natural path."""
    g = grid(17)
    delta = DELTA if delta_kind == "0.95" else _half_outlier_delta(_oracle_eval(g, 0)[2])
    depth = float(np.median(g.p.depth0))
    n = 5 if way == "solve_jobs" else 1
    ctx, _, _ = _context(nid, orc, g, NATURAL if way == "natural" else SORTED, max_jobs=n)
    if way == "lockstep":
        ctx.set_option("lm_speculate", 0)
    starts = _starts(orc, g, n)
    oracle = [_oracle(g, ("optimize", delta, k), lambda: g.P.optimize(starts[k], 10, delta)) for k in range(n)]
    if way == "solve_jobs":
        out, stats = ctx.solve_jobs(np.stack(starts), np.zeros(n, np.int32), 10, delta)
        for k, (poseo, its, traceo, counts) in enumerate(oracle):
            assert np.array_equal(stats[k], _oracle_stats(its, counts)), k
            _assert_pose_close(out[k], poseo, depth)
        return
    pose, trace, stats = ctx.solve(0, g.pose0, 10, delta)
    poseo, its, traceo, counts = oracle[0]
    assert np.array_equal(stats, _oracle_stats(its, counts))
    assert np.array_equal(trace[:, 2], traceo[:, 2])  # LM trials per iteration
    np.testing.assert_allclose(trace[:, 0], traceo[:, 0], rtol=1e-7)
    _assert_pose_close(pose, poseo, depth)


def test_latency_solve_on_8100_cells(nid, orc, grid):
    g = grid(90)
    ctx, _, _ = _context(nid, orc, g, SORTED)
    pose, trace, stats = ctx.solve(0, g.pose0, 10, DELTA)
    poseo, its, traceo, counts = g.P.optimize(g.pose0, 10, DELTA)
    assert np.array_equal(stats, _oracle_stats(its, counts))
    assert np.array_equal(trace[:, 2], traceo[:, 2])
    np.testing.assert_allclose(trace[:, 0], traceo[:, 0], rtol=1e-7)
    _assert_pose_close(pose, poseo, float(np.median(g.p.depth0)))
