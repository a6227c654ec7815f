"""A context owns every CUDA resource it holds -- device and pinned buffers, streams, events, gather arrays and their
textures, the latency-mode graph -- and releases all of them: in nid_destroy, whatever the context reached, and in a
nid_create that fails half way. nid_live_resources counts the resources held by all contexts of the process."""
import ctypes as C
import gc

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ERR_CUDA = -1
_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)


def _d(a):
    return a.ctypes.data_as(_dp)


def _live(nid):
    gc.collect()  # (contexts of earlier tests that are no longer referenced release their resources now)
    return nid.live_resources()


def _poses(orc, pairs):
    return [orc.reference_perturbation(p.T_wc1) for p in pairs]


def test_counter_follows_a_context(nid):
    before = _live(nid)
    ctx = nid.Context(120, 160, 4, 16)
    held = nid.live_resources()
    assert held > before
    ctx.event_record(0)  # the stopwatch events are created on first use
    assert nid.live_resources() == held + 1
    ctx.close()
    assert nid.live_resources() == before


def test_failed_create_releases_what_it_acquired(nid, orc, make_pair):
    """8 x 65535 pixels pass the argument checks, but a gather array 65535 texels wide exceeds the device's limit
    (maxTexture2DGather, 32768 on current GPUs): nid_create fails after its stream and the first device buffers."""
    L = nid.lib()
    before = _live(nid)
    for _ in range(3):
        h = C.c_void_p()
        rc = L.nid_create(C.byref(h), 0, 8, 65535, 1, 16, 3, 1, 1)
        if rc == 0:
            L.nid_destroy(h)
            pytest.skip("this device allows gather arrays 65535 texels wide")
        assert rc == ERR_CUDA
        assert b"gather textures" in L.nid_last_error()
        assert not h.value
        assert nid.live_resources() == before
    # the runtime is still usable
    p = make_pair(1000, 120, 160)
    ctx = nid.Context(120, 160, 4, 16)
    ctx.set_pair(0, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
    M0 = orc.se3_to_mat16(_poses(orc, [p])[0])
    ctx.prepare(0, M0)
    Ht, Hj, J = ctx.eval(0, M0, True)
    assert np.isfinite(Ht).any() and np.isfinite(J).any()
    ctx.close()
    assert nid.live_resources() == before


def test_sorted_lifecycle_releases_everything(nid, orc, make_pair):
    """Contexts that reach every lazily created resource of the sorted path, closed: the count returns to its value
    before they were created."""
    L = nid.lib()
    pairs = [make_pair(1000, 120, 160), make_pair(1001, 120, 160)]
    pose0 = _poses(orc, pairs)
    M = np.stack([orc.se3_to_mat16(q) for q in pose0])
    before = _live(nid)
    A = nid.Context(120, 160, 4, 16, n_pairs=2, max_jobs=8)
    created = nid.live_resources()
    # u16 set-up (raw depth plane, pinned arena), batched prepare (pixel store, result buffer)
    keep = A.set_pairs_u16(0, np.stack([p.depth0_u16 for p in pairs]), np.stack([p.im0 for p in pairs]),
                           np.stack([p.im1 for p in pairs]), np.stack([p.T_wc0 for p in pairs]),
                           np.stack([p.intr for p in pairs]))
    A.prepare_pairs(0, M)
    del keep
    A.ref_weights(0)
    A.set_option("keep_hist", 1)
    A.set_option("time_kernels", 1)
    A.eval_jobs(M, [0, 1], True)
    A.set_option("task_px", 8)  # more tasks per pair: the next evaluation regrows the per-job partials
    A.prepare_pairs(0, M)
    A.eval_jobs(M, [0, 1], True)
    A.set_option("time_kernels", 0)
    A.solve_jobs(np.stack([pose0[j % 2] for j in range(8)]), [j % 2 for j in range(8)])  # lock-step, two streams
    A.solve(0, pose0[0])  # latency mode with its graph
    A.warp_sample_jobs(M, [0, 1])
    A.warp_sample(0, M[0])
    A.warp_sample_f64(0, M[0])
    A.event_record(0)
    A.event_record(1)
    A.event_elapsed_ms()
    B = nid.Context(60, 80, 4, 16)
    B.set_pairs_downsampled(0, A, 0)
    B.sync()
    A.hard_eval_jobs(M, [0, 1])
    pts = np.ascontiguousarray(A.points3d(0))
    assert nid.live_resources() > created
    B.close()
    A.close()
    assert nid.live_resources() == before
    # caller-supplied world points (a context holding them refuses the u16 set-up, kernel 1 and downsampling)
    p = pairs[0]
    P = nid.Context(120, 160, 4, 16)
    f0, f1 = p.im0.astype(np.float64), p.im1.astype(np.float64)
    assert L.nid_set_pair_points(P._h, 0, _d(pts), _d(f0), _d(f1), _d(np.ascontiguousarray(p.intr))) == 0
    P.prepare(0, M[0])
    P.eval(0, M[0], True)
    P.close()
    assert nid.live_resources() == before


def test_natural_path_lifecycle_releases_everything(nid, orc, make_pair):
    """48 bins: the natural-order kernels, their per-job partials and the lock-step LM lists."""
    p = make_pair(1000, 120, 160)
    pose0 = _poses(orc, [p])[0]
    M0 = orc.se3_to_mat16(pose0)
    before = _live(nid)
    ctx = nid.Context(120, 160, 4, 48, max_jobs=2)
    ctx.set_option("keep_hist", 1)
    ctx.set_pair(0, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
    ctx.prepare(0, M0)
    ctx.eval(0, M0, True)
    ctx.debug_hist(0, 0)
    ctx.solve(0, pose0)
    ctx.close()
    assert nid.live_resources() == before


def test_shim_contexts_are_released_by_reset(nid, orc, make_pair):
    L = nid.lib()
    L.nid_shim_reset()
    p = make_pair(1000, 120, 160)
    rows, cols, cell, bins = p.rows, p.cols, 4, 16
    N, nc = rows * cols, cell * cell
    depth = p.depth0.reshape(-1).copy()
    Twc0, intr = p.T_wc0.copy(), p.intr.copy()
    points = np.zeros(3 * N)
    im0 = p.im0.astype(np.float64).reshape(-1).copy()
    im1 = p.im1.astype(np.float64).reshape(-1).copy()
    M0 = orc.se3_to_mat16(_poses(orc, [p])[0])
    bs_value, bs_index = np.zeros(4 * N), np.zeros(N, dtype=np.int32)
    bs_counter, Href = np.zeros(nc, dtype=np.int32), np.zeros(nc)
    Ht, Hj, der = np.zeros(nc), np.zeros(nc), np.zeros(6 * nc)
    before = _live(nid)
    L.nid_shim_Calculate3Dpoint(_d(depth), _d(Twc0), _d(points), _d(intr), rows, cols)
    L.nid_shim_CudaComputeHref(_d(im0), _d(points), _d(M0), _d(intr), bins, 3, cell, rows, cols, _d(bs_value),
                               bs_index.ctypes.data_as(_ip), bs_counter.ctypes.data_as(_ip), _d(Href))
    L.nid_shim_CudaComputeH(1, _d(im0), _d(im1), _d(points), bs_counter.ctypes.data_as(_ip), _d(bs_value),
                            bs_index.ctypes.data_as(_ip), _d(M0), _d(intr), bins, 3, cell, rows, cols, _d(Href),
                            None, None, _d(Ht), _d(Hj), _d(der))
    assert np.isfinite(Ht).any()
    assert nid.live_resources() > before
    L.nid_shim_reset()
    assert nid.live_resources() == before
