"""Three-way check on the GPU: the reference's own CUDA code vs the CPU oracle vs this library. The reference's side
is the stored outputs in tests/golden/ref_gpu_*.npz (oracle/gen_ref_golden.py ran the upstream kernels, compiled
unmodified, on a B200), so the check needs nothing outside this repository. They were taken at the one image geometry
for which the unguarded reference kernels are memory-safe on a 148-SM part (see oracle/ref_gpu.py); the oracle and
this library recompute the same seeded pairs and poses here."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.mark.parametrize("cell,bins", [(4, 10), (16, 10), (8, 8), (4, 6), (4, 12), (4, 14), (1, 8)])
def test_reference_cuda_vs_oracle_vs_ours(nid, orc, synth, cell, bins):
    g = np.load(os.path.join(GOLDEN, f"ref_gpu_c{cell}_b{bins}.npz"))
    p = synth.make_pair(int(g["seed"]), int(g["rows"]), int(g["cols"]))
    assert int(p.im0.astype(np.int64).sum()) == int(g["im0_sum"]) and int(p.im1.astype(np.int64).sum()) == int(g["im1_sum"])
    pose0 = g["pose0"]
    P = orc.Problem(p.im0, p.depth0, p.im1, p.T_wc0, p.intr, cell, bins, threads=4)
    P.set_quirks(1, 1)  # the reference CUDA code tests `u+3<=cols` in the Jacobian too (computeH.cu:164)
    nc, href = P.prepare(pose0)
    # a1: Calculate3Dpoint
    # (nvcc fuses the reference's multiply-adds, the oracle and this library do not: last-bit agreement)
    ctx = nid.Context(p.rows, p.cols, cell, bins)
    ctx.set_pair(0, p.depth0, p.im0, p.im1, p.T_wc0, p.intr)
    pts = ctx.points3d(0)
    assert np.array_equal(pts, P.points3d(), equal_nan=True)
    assert int(np.isnan(pts).sum()) == int(g["pts_nan"])
    sub = pts.reshape(-1, 3)[::97]
    assert np.array_equal(np.isnan(sub), np.isnan(g["pts_sub"]))
    np.testing.assert_allclose(sub, g["pts_sub"], rtol=4e-16, atol=1e-15)
    nc2, href2 = ctx.prepare(0, orc.se3_to_mat16(pose0))
    assert np.array_equal(nc, nc2) and np.array_equal(nc2, g["ref_n_c"])
    act = ~np.isnan(g["ref_href"])
    assert np.array_equal(act, ~np.isnan(href))
    for k, xi in enumerate(g["xis"]):
        pose = orc.se3_mul(orc.se3_exp(xi), pose0)
        M = g["poses"][k]
        Ht_r, Hj_r, J_r = g["Ht"][k], g["Hj"][k], g["der"][k]
        P.set_quirks(1, 1)
        Ht_o, Hj_o, _, J_o = P.eval(pose, True)
        np.testing.assert_allclose(Ht_r[act], Ht_o[act], rtol=1e-10)
        np.testing.assert_allclose(Hj_r[act], Hj_o[act], rtol=1e-10)
        scale = np.abs(J_o[act]).max(axis=1, keepdims=True)
        assert np.max(np.abs(J_r[act] - J_o[act]) / scale) < 1e-7
        # ours follows the CPU edge's Jacobian bound (cols-1); compare entropies exactly and J loosely here,
        # tightly against the oracle in CPU-quirk mode
        Ht, Hj, J = ctx.eval(0, M, True)
        np.testing.assert_allclose(Ht[act], Ht_r[act], rtol=1e-10)
        np.testing.assert_allclose(Hj[act], Hj_r[act], rtol=1e-10)
        P.set_quirks(0, 1)
        _, _, _, J_cpu = P.eval(pose, True)
        assert np.max(np.abs(J[act] - J_cpu[act]) / scale) < 1e-8
    ctx.close()
