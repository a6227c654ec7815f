"""Coarse-to-fine pose solves: half-resolution pair levels built on the device (nid_set_pairs_downsampled) and the LM solve
chained across them (nid_solve_pyramid_jobs). A derived slot is held bit for bit to a slot set from the host with the
numpy restatement of the downsampling below; every level of a pyramid solve is held to the CPU oracle prepared at the pose
the library handed to that level."""
import ctypes as C
import importlib
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DELTA = np.sqrt(0.95)
NS_ROT = 1e-4      # rad
NS_TRANS = 1e-4    # x scene depth
ERR_ARG, ERR_STATE = -2, -3


# ---------------------------------------------------------------------------------------------- numpy restatement
def down2(depth, im0, im1, intr):
    """One 2x2 level: images (a+b+c+d+2)>>2; depth = mean of the valid samples (0.01 <= z <= 100) summed in the order
    (2i,2j), (2i,2j+1), (2i+1,2j), (2i+1,2j+1), 0 when none is valid; intrinsics fx/2, fy/2, (cx-0.5)/2, (cy-0.5)/2.
    An odd last row or column is dropped."""
    R, Cn = depth.shape[0] // 2, depth.shape[1] // 2

    def blocks(a):
        a = a[:2 * R, :2 * Cn]
        return [a[0::2, 0::2], a[0::2, 1::2], a[1::2, 0::2], a[1::2, 1::2]]

    def img(a):
        b = [x.astype(np.int32) for x in blocks(a)]
        return ((b[0] + b[1] + b[2] + b[3] + 2) >> 2).astype(np.uint8)

    s = np.zeros((R, Cn))
    n = np.zeros((R, Cn), dtype=np.int32)
    with np.errstate(invalid="ignore"):
        for z in blocks(depth):
            ok = (z >= 0.01) & (z <= 100)
            s = np.where(ok, s + np.where(ok, z, 0.0), s)
            n += ok
    d = np.where(n > 0, s / np.maximum(n, 1), 0.0)
    k = np.array([intr[0] * 0.5, intr[1] * 0.5, (intr[2] - 0.5) * 0.5, (intr[3] - 0.5) * 0.5, 1.0])
    return d, img(im0), img(im1), k


def levels_np(depth, im0, im1, intr, n):
    out = [(depth, im0, im1, np.asarray(intr, dtype=np.float64))]
    for _ in range(n - 1):
        out.append(down2(*out[-1]))
    return out


# ---------------------------------------------------------------------------------------------- fixtures / helpers
def _dirty_depth(p, seed):
    """p.depth0 (already with invalid_depth_frac zeros) plus injected NaN, 0 and > 100 m samples."""
    d = p.depth0.copy().reshape(-1)
    rng = np.random.default_rng(seed)
    idx = rng.choice(d.size, size=3 * max(4, d.size // 300), replace=False)
    k = idx.size // 3
    d[idx[:k]] = np.nan
    d[idx[k:2 * k]] = 0.0
    d[idx[2 * k:]] = 150.0
    return d.reshape(p.depth0.shape)


def _fill_source(ctx, pair, p, kind, seed):
    """Set `pair` of ctx from p; returns the fp64 depth the device holds (what the downsampling reads)."""
    if kind == "f64":
        depth = _dirty_depth(p, seed)
        ctx.set_pair(pair, depth, p.im0, p.im1, p.T_wc0, p.intr)
        return depth
    keep = ctx.set_pairs_u16(pair, p.depth0_u16[None], p.im0[None], p.im1[None], p.T_wc0[None], p.intr[None])
    ctx.sync()
    del keep
    return p.depth0_u16.astype(np.float64) * p.intr[4]


def _inbounds(nid, ctx, pair):
    out = np.zeros(ctx.n, dtype=np.uint8)
    assert nid.lib().nid_get_inbounds(ctx._h, pair, out.ctypes.data_as(C.POINTER(C.c_uint8))) == 0
    return out


def _poses16(orc, p, scale=1.0):
    pose = orc.reference_perturbation(p.T_wc1)
    M0 = orc.se3_to_mat16(pose)
    M1 = orc.se3_to_mat16(orc.se3_mul(orc.se3_exp(np.array([0.002, -0.001, 0.0015, 0.004, -0.003, 0.002]) * scale), pose))
    return M0, M1


def assert_same_slots(nid, ctx, a, b, M0, M1, paths=(1, 2)):
    """Slots a and b of ctx hold the same pair: world points, prepare, in-bounds set, evaluations, hard-binned NID and
    kernel 1 agree bit for bit. The natural-order path (1) accumulates its histograms with shared-memory atomics, whose
    order varies from run to run, so there its evaluations are held to rounding (the sorted path 2 is deterministic)."""
    pa, pb = ctx.points3d(a), ctx.points3d(b)
    assert np.array_equal(pa, pb, equal_nan=True)
    assert np.isfinite(pa).any()
    for path in paths:
        ctx.set_option("path", path)
        nca, ha = ctx.prepare(a, M0)
        ncb, hb = ctx.prepare(b, M0)
        assert np.array_equal(nca, ncb) and np.array_equal(ha, hb, equal_nan=True)
        assert np.array_equal(_inbounds(nid, ctx, a), _inbounds(nid, ctx, b))
        Ht, Hj, der = ctx.eval_jobs(np.stack([M0, M1, M0, M1]), job_pair=[a, a, b, b])
        for x in (Ht, Hj, der):
            if path == 2:
                assert np.array_equal(x[:2], x[2:], equal_nan=True)
            else:
                np.testing.assert_allclose(x[:2], x[2:], rtol=1e-10, atol=1e-10 * np.nanmax(np.abs(x)))
    ctx.set_option("path", 0)
    tot, cells = ctx.hard_eval_jobs(np.stack([M0, M1, M0, M1]), job_pair=[a, a, b, b])
    assert np.array_equal(tot[:2], tot[2:]) and np.array_equal(cells[:2], cells[2:], equal_nan=True)
    ws = ctx.warp_sample_jobs(np.stack([M0, M1, M0, M1]), [a, a, b, b])
    assert np.array_equal(ws[:2], ws[2:], equal_nan=True)


# ---------------------------------------------------------------------------------------------- 1, 2: the derived slot
@pytest.mark.parametrize("kind", ["f64", "u16"])
@pytest.mark.parametrize("rows,cols", [(480, 640), (121, 163), (240, 320)])
def test_derived_slot_equals_host_set_slot(nid, orc, make_pair, rows, cols, kind):
    p = make_pair(1000, rows, cols, invalid_depth_frac=0.1)
    src = nid.Context(rows, cols, 4, 16)
    depth = _fill_source(src, 0, p, kind, 7)
    dst = nid.Context(rows // 2, cols // 2, 4, 16, n_pairs=2, max_jobs=4)
    dst.set_pairs_downsampled(0, src, 0)
    d, a, b, k = down2(depth, p.im0, p.im1, p.intr)
    dst.set_pair(1, d, a, b, p.T_wc0, k)
    assert_same_slots(nid, dst, 0, 1, *_poses16(orc, p))


def test_chained_levels_and_batched_call(nid, orc, make_pair):
    rows, cols = 240, 320
    p = make_pair(1001, rows, cols, invalid_depth_frac=0.1)
    l0 = nid.Context(rows, cols, 4, 16)
    depth = _fill_source(l0, 0, p, "f64", 11)
    l1 = nid.Context(rows // 2, cols // 2, 4, 16)
    l2 = nid.Context(rows // 4, cols // 4, 2, 16, n_pairs=2, max_jobs=4)
    l1.set_pairs_downsampled(0, l0, 0)
    l2.set_pairs_downsampled(0, l1, 0)
    d, a, b, k = levels_np(depth, p.im0, p.im1, p.intr, 3)[2]
    l2.set_pair(1, d, a, b, p.T_wc0, k)
    assert_same_slots(nid, l2, 0, 1, *_poses16(orc, p))
    # one call over five pairs (dst_pair0 != src_pair0) == five single calls
    src = nid.Context(120, 160, 2, 16, n_pairs=6)
    ps = [make_pair(1000 + i, 120, 160, invalid_depth_frac=0.1) for i in range(6)]
    for i, q in enumerate(ps):
        _fill_source(src, i, q, "f64", 20 + i)
    batched = nid.Context(60, 80, 2, 16, n_pairs=8, max_jobs=2)
    single = nid.Context(60, 80, 2, 16, n_pairs=8, max_jobs=2)
    batched.set_pairs_downsampled(2, src, 1, 5)
    for i in range(5):
        single.set_pairs_downsampled(2 + i, src, 1 + i, 1)
    for i in range(5):
        s = 2 + i
        assert np.array_equal(batched.points3d(s), single.points3d(s), equal_nan=True)
        M0, M1 = _poses16(orc, ps[1 + i])
        assert all(np.array_equal(x, y, equal_nan=True) for x, y in zip(batched.prepare(s, M0), single.prepare(s, M0)))
        for x, y in zip(batched.eval_jobs(np.stack([M0, M1]), job_pair=[s, s]), single.eval_jobs(np.stack([M0, M1]), job_pair=[s, s])):
            assert np.array_equal(x, y, equal_nan=True)


# ---------------------------------------------------------------------------------------------- 3: stream ordering
def test_stream_ordering_against_asynchronous_refills(nid, orc, make_pair):
    rows, cols = 480, 640
    pa, pb = make_pair(1002, rows, cols), make_pair(1003, rows, cols)
    src = nid.Context(rows, cols, 4, 16)
    dst = nid.Context(rows // 2, cols // 2, 4, 16, n_pairs=2, max_jobs=4)

    def u16(p):
        return src.set_pairs_u16(0, p.depth0_u16[None], p.im0[None], p.im1[None], p.T_wc0[None], p.intr[None])

    def np_level(p):
        return down2(p.depth0_u16.astype(np.float64) * p.intr[4], p.im0, p.im1, p.intr)

    # derive, then refill the source slot at once: the destination holds the OLD pair
    keep = u16(pa)
    src.sync()
    dst.set_pairs_downsampled(0, src, 0)
    keep = u16(pb)
    src.sync()
    dst.sync()
    d, a, b, k = np_level(pa)
    dst.set_pair(1, d, a, b, pa.T_wc0, k)
    assert_same_slots(nid, dst, 0, 1, *_poses16(orc, pa), paths=(2,))
    # refill asynchronously, then derive at once: the destination holds the NEW pair
    keep = u16(pa)
    dst.set_pairs_downsampled(0, src, 0)
    dst.sync()
    src.sync()
    del keep
    d, a, b, k = np_level(pa)
    dst.set_pair(1, d, a, b, pa.T_wc0, k)
    assert_same_slots(nid, dst, 0, 1, *_poses16(orc, pa), paths=(2,))


# ---------------------------------------------------------------------------------------------- 4: errors
def _pyr_raw(nid, levels, poses, n, job_pair=None, its=None):
    """nid_solve_pyramid_jobs straight through ctypes, on the caller's array (to see that it is left untouched)."""
    L = len(levels)
    hs = (C.c_void_p * L)(*[None if c is None else c._h.value for c in levels])
    it = np.full(L, 10, dtype=np.int32) if its is None else np.ascontiguousarray(its, dtype=np.int32)
    jp = None if job_pair is None else np.ascontiguousarray(job_pair, dtype=np.int32)
    ip = C.POINTER(C.c_int)
    stats = np.full((n, L, 3), -7, dtype=np.int32)
    rc = nid.lib().nid_solve_pyramid_jobs(hs, L, n, None if jp is None else jp.ctypes.data_as(ip),
                                          poses.ctypes.data_as(C.POINTER(C.c_double)), it.ctypes.data_as(ip), float(DELTA),
                                          stats.ctypes.data_as(ip))
    return rc, stats


def test_errors_leave_everything_untouched(nid, orc, make_pair):
    L = nid.lib()
    p = make_pair(1000, 120, 160)
    src = nid.Context(120, 160, 2, 16, n_pairs=2, max_jobs=2)
    src.set_pair(0, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
    dst = nid.Context(60, 80, 2, 16, n_pairs=2, max_jobs=2)
    bad = nid.Context(61, 80, 2, 16, n_pairs=2)
    ds = L.nid_set_pairs_downsampled
    assert ds(bad._h, 0, src._h, 0, 1) == ERR_ARG                  # geometry
    assert ds(dst._h, -1, src._h, 0, 1) == ERR_ARG                 # ranges
    assert ds(dst._h, 0, src._h, 0, 0) == ERR_ARG
    assert ds(dst._h, 1, src._h, 0, 2) == ERR_ARG
    assert ds(dst._h, 0, src._h, 1, 2) == ERR_ARG
    assert ds(None, 0, src._h, 0, 1) == ERR_ARG                    # NULLs
    assert ds(dst._h, 0, None, 0, 1) == ERR_ARG
    assert ds(dst._h, 0, src._h, 1, 1) == ERR_STATE                # source pair 1 is not set
    assert ds(dst._h, 0, src._h, 0, 1) == 0
    # point-form source, point-form destination
    dp = C.POINTER(C.c_double)
    pts = np.ascontiguousarray(src.points3d(0))
    f0, f1 = p.im0.astype(np.float64), p.im1.astype(np.float64)
    ptsrc = nid.Context(120, 160, 2, 16)
    assert L.nid_set_pair_points(ptsrc._h, 0, pts.ctypes.data_as(dp), f0.ctypes.data_as(dp), f1.ctypes.data_as(dp),
                                 p.intr.ctypes.data_as(dp)) == 0
    assert ds(dst._h, 0, ptsrc._h, 0, 1) == ERR_STATE
    ptdst = nid.Context(60, 80, 2, 16)
    d, a, b, k = down2(p.depth0, p.im0, p.im1, p.intr)
    ptdst.set_pair(0, d, a, b, p.T_wc0, k)
    pts2 = np.ascontiguousarray(ptdst.points3d(0))
    a64, b64 = a.astype(np.float64), b.astype(np.float64)
    assert L.nid_set_pair_points(ptdst._h, 0, pts2.ctypes.data_as(dp), a64.ctypes.data_as(dp), b64.ctypes.data_as(dp),
                                 k.ctypes.data_as(dp)) == 0
    assert ds(ptdst._h, 0, src._h, 0, 1) == ERR_STATE
    # the pyramid solve: nothing is written on failure
    pose0 = orc.reference_perturbation(p.T_wc1)
    poses = np.ascontiguousarray(np.stack([pose0, pose0]))
    before = poses.copy()
    src.set_pair(1, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
    dst.set_pairs_downsampled(1, src, 1)
    rc, st = _pyr_raw(nid, [src, dst], poses, 2, job_pair=[1, 1])    # repeated job pairs
    assert rc == ERR_ARG
    one = nid.Context(60, 80, 2, 16, n_pairs=2, max_jobs=1)
    one.set_pairs_downsampled(0, src, 0, 2)
    rc, st = _pyr_raw(nid, [src, one], poses, 2)                     # n > max_jobs at a level
    assert rc == ERR_ARG
    part = nid.Context(60, 80, 2, 16, n_pairs=2, max_jobs=2)
    part.set_pairs_downsampled(0, src, 0, 1)
    rc, st = _pyr_raw(nid, [src, part], poses, 2)                    # pair 1 not set at level 1
    assert rc == ERR_STATE
    rc, st = _pyr_raw(nid, [src, None], poses, 2)                    # a NULL level
    assert rc == ERR_ARG
    rc, st = _pyr_raw(nid, [src, dst], poses, 2, its=[10, -1])
    assert rc == ERR_ARG
    assert np.array_equal(poses, before) and np.all(st == -7)
    # different devices, where there are two
    try:
        other = nid.Context(60, 80, 2, 16, device=1)
    except nid.NidError:
        return
    assert ds(other._h, 0, src._h, 0, 1) == ERR_ARG


# ---------------------------------------------------------------------------------------------- 5: policy and modes
def _pyramid(nid, ps, levels_n, cell_of, bins):
    """Contexts of a pyramid over pairs ps (level 0 set from the host, the rest derived)."""
    p0 = ps[0]
    ctxs = [nid.Context(p0.rows, p0.cols, cell_of(0), bins, n_pairs=len(ps), max_jobs=len(ps))]
    for i, p in enumerate(ps):
        ctxs[0].set_pair(i, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
    for l in range(1, levels_n):
        ctxs.append(nid.Context(p0.rows >> l, p0.cols >> l, cell_of(l), bins, n_pairs=len(ps), max_jobs=len(ps)))
        ctxs[l].set_pairs_downsampled(0, ctxs[l - 1], 0, len(ps))
    return ctxs


def test_one_level_is_prepare_and_solve_and_jobs_are_independent(nid, orc, make_pair):
    ps = [make_pair(1000 + i, 240, 320) for i in range(6)]
    pose0 = np.stack([orc.reference_perturbation(p.T_wc1) for p in ps])
    ctxs = _pyramid(nid, ps, 2, lambda l: max(1, 4 >> l), 16)
    got, st = nid.solve_pyramid_jobs(ctxs[:1], pose0)
    ctxs[0].prepare_pairs(0, np.stack([orc.se3_to_mat16(q) for q in pose0]))
    ref, st_ref = ctxs[0].solve_jobs(pose0)
    assert np.array_equal(got, ref) and np.array_equal(st[:, 0], st_ref)
    # two levels: six jobs in lock-step == one job at a time (latency mode), bit for bit
    many, st6 = nid.solve_pyramid_jobs(ctxs, pose0)
    for j in range(6):
        one, st1 = nid.solve_pyramid_jobs(ctxs, pose0[j:j + 1], job_pair=[j])
        assert np.array_equal(many[j], one[0]) and np.array_equal(st6[j], st1[0])
    assert np.all(st6[:, 1, 0] >= 1) and np.all(st6[:, 0, 0] >= 1)


# ---------------------------------------------------------------------------------------------- 6: oracle per level
@pytest.mark.parametrize("levels_n", [2, 3])
@pytest.mark.parametrize("cell,bins,rows,cols", [(4, 16, 240, 320), (16, 10, 480, 640)])
def test_every_level_matches_the_oracle(nid, orc, make_pair, cell, bins, rows, cols, levels_n):
    p = make_pair(1000, rows, cols)
    ctxs = _pyramid(nid, [p], levels_n, lambda l: max(1, cell >> l), bins)
    pose0 = orc.reference_perturbation(p.T_wc1)
    full, st = nid.solve_pyramid_jobs(ctxs, pose0[None])
    arrays = levels_np(p.depth0, p.im0, p.im1, p.intr, levels_n)
    depth = float(np.median(p.depth0))
    pose_in = pose0
    for l in range(levels_n - 1, -1, -1):
        out, st_l = nid.solve_pyramid_jobs(ctxs, pose0[None], max_iters=[0] * l + [10] * (levels_n - l))
        d, a, b, k = arrays[l]
        P = orc.Problem(a, d, b, p.T_wc0, k, max(1, cell >> l), bins, threads=8)
        P.set_quirks(0, 0)
        P.prepare(pose_in)
        poseo, its, _, counts = P.optimize(pose_in, 10, DELTA)
        assert its == st[0, l, 0] == st_l[0, l, 0] and counts[0] == st[0, l, 1]
        assert np.max(np.abs(out[0, :3] - poseo[:3])) < NS_TRANS * depth
        assert 2 * np.max(np.abs(out[0, 3:6] - poseo[3:6])) < NS_ROT
        pose_in = out[0]
    assert np.array_equal(pose_in, full[0])


# ---------------------------------------------------------------------------------------------- 7: no active cell
@pytest.mark.parametrize("n", [1, 5])
def test_level_without_active_cells_hands_the_pose_down_unchanged(nid, orc, make_pair, n):
    """Cells of 5x5 at 60x80 hold 192 pixels, under NID_MIN_CELL_POINTS: chi2 is 0 and the Gauss-Newton system is zero
    there, the first trial brings no decrease and the schedule stops after it (stats {1, 1, 1}); the pose is unchanged."""
    ps = [make_pair(1000 + i, 240, 320) for i in range(n)]
    ctxs = _pyramid(nid, ps, 3, lambda l: 5, 16)
    pose0 = np.stack([orc.reference_perturbation(p.T_wc1) for p in ps])
    nc, href = ctxs[2].prepare_pairs(0, np.stack([orc.se3_to_mat16(q) for q in pose0]))
    assert np.all(nc < 300) and np.all(np.isnan(href))
    out, st = nid.solve_pyramid_jobs(ctxs, pose0, max_iters=[0, 0, 10])
    assert np.array_equal(out, pose0)
    assert np.all(st[:, 2] == [1, 1, 1]) and np.all(st[:, :2] == 0)
    # the next level starts from it as if the coarse level were absent
    a, sa = nid.solve_pyramid_jobs(ctxs, pose0, max_iters=[0, 10, 10])
    b, sb = nid.solve_pyramid_jobs(ctxs, pose0, max_iters=[0, 10, 0])
    assert np.array_equal(a, b) and np.array_equal(sa[:, 1], sb[:, 1])


# ---------------------------------------------------------------------------------------------- 8: the app
def test_pose_estimation_binary_with_pyramid_levels(nid, orc, synth, tmp_path):
    if not os.path.exists(os.path.join(ROOT, "nid-pose-estimation_b200", "libnid_b200.so")):
        pytest.skip("libnid_b200.so not built")
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "apps")], stdout=subprocess.DEVNULL)
    ds = str(tmp_path / "ds")
    subprocess.check_call([sys.executable, os.path.join(ROOT, "tools", "gen_synth.py"), ds, "--rows", "240", "--cols", "320",
                           "--cell", "4", "--bins", "16"], stdout=subprocess.DEVNULL)
    with open(os.path.join(ds, "config.yaml"), "a") as f:
        f.write("pyramid_levels: 2\n")
    r = subprocess.run([os.path.join(ROOT, "bin", "NID_pose_estimation"), os.path.join(ds, "config.yaml")], cwd=str(tmp_path),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    out = r.stdout
    final = np.array([float(v) for v in out.split("the final error is \n")[1].splitlines()[0].split()])
    csv = open(tmp_path / "nid_error.csv").read().strip().split(",")
    assert len(csv) == 8 and csv[6:] == ["0", "1"]
    np.testing.assert_allclose([float(v) for v in csv[:6]], final, rtol=1e-5)
    assert "iteration= 0\t chi2= " in r.stderr
    # the same two levels through the Python mirror
    e = np.load(os.path.join(ds, "expected_inputs.npz"))
    depth = e["depth_u16"].astype(np.float64) * (1.0 / 5000)
    c0 = nid.Context(240, 320, 4, 16)
    c0.set_option("task_px", 16)
    c0.set_pair(0, depth, e["im0"], e["im1"], e["T_wc0"], e["intr"])
    c1 = nid.Context(120, 160, 2, 16)
    c1.set_option("task_px", 16)
    c1.set_pairs_downsampled(0, c0, 0)
    pose0 = orc.reference_perturbation(e["T_wc1"])
    pose, st = nid.solve_pyramid_jobs([c0, c1], pose0[None])
    assert f"pyramid level 1 (120x160): outer iterations {st[0, 1, 0]}\n" in out
    gt = orc.se3_from_mat16(synth.mat16_inverse(e["T_wc1"]))
    np.testing.assert_allclose(final, (gt - pose[0])[:6], rtol=1e-5, atol=2e-6)   # printed with 6 significant digits
