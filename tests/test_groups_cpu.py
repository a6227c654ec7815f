"""CPU tier of joint (group) pose solves: the host pieces nid_solve_groups runs (adjoint, block transform and combination,
rigidity check in host/nid_host_math.hpp) against the oracle's restatement, the oracle's group LM against orc_optimize, and
the rig / keyframe generators. No GPU involved."""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np
import pytest

import group_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WRAPPER = r'''
#include "nid_host_math.hpp"
using namespace nidhost;
extern "C" {
void hm_adjoint6(const double* E, double* Ad) { adjoint6(E, Ad); }
void hm_to_body(const double* Ad, const double* in, double* out) { gn_block_to_body(Ad, in, out); }
void hm_combine(int n, const double* blocks, const double* Ad, double* out) { gn_combine(n, blocks, Ad, out); }
int hm_is_rigid(const double* m) { return is_rigid(m) ? 1 : 0; }
void hm_mat16_mul(const double* a, const double* b, double* out) { mat16_mul(a, b, out); }
}
'''

_dp = C.POINTER(C.c_double)


@pytest.fixture(scope="module")
def hm(tmp_path_factory):
    d = tmp_path_factory.mktemp("hostmath_groups")
    src = d / "wrap.cpp"
    src.write_text(WRAPPER)
    so = d / "libhmg.so"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", os.path.join(ROOT, "nid-pose-estimation_b200", "host"),
                           "-o", str(so), str(src)])
    L = C.CDLL(str(so))
    L.hm_combine.argtypes = [C.c_int, _dp, _dp, _dp]
    L.hm_is_rigid.restype = C.c_int
    return L


def _p(a):
    return a.ctypes.data_as(_dp)


def _rigid(rng, rot_scale=1.0, t_scale=0.1):
    from oracle import binding as orc
    return orc.se3_to_mat16(orc.se3_exp(np.concatenate([rng.uniform(-1, 1, 3) * rot_scale, rng.uniform(-1, 1, 3) * t_scale])))


def test_adjoint_matches_the_oracle_and_conjugates_exp(hm, orc):
    rng = np.random.default_rng(21)
    for _ in range(100):
        E = _rigid(rng)
        Ad = np.zeros(36)
        hm.hm_adjoint6(_p(E), _p(Ad))
        Ad = Ad.reshape(6, 6)
        np.testing.assert_allclose(Ad, group_oracle.adjoint6(E), rtol=0, atol=1e-15)
        xi = rng.uniform(-1, 1, 6) * rng.choice([1e-6, 1e-2, 0.5])
        lhs = orc.se3_to_mat16(orc.se3_exp(Ad @ xi))
        E7 = orc.se3_from_mat16(E)
        rhs = orc.se3_to_mat16(orc.se3_mul(orc.se3_mul(E7, orc.se3_exp(xi)), orc.se3_inverse(E7)))
        np.testing.assert_allclose(lhs, rhs, rtol=0, atol=1e-12)


def test_block_transform_and_combination(hm):
    rng = np.random.default_rng(22)
    n = 4
    blocks = rng.normal(size=(n, 44))
    for i in range(n):
        A = rng.normal(size=(6, 6))
        blocks[i, 1:37] = (A @ A.T).reshape(36)
    Es = [_rigid(rng) for _ in range(n)]
    Ads = np.stack([group_oracle.adjoint6(E) for E in Es])
    want = np.zeros(44)
    for i in range(n):
        H = blocks[i, 1:37].reshape(6, 6)
        want[0] += blocks[i, 0]
        want[1:37] += (Ads[i].T @ H @ Ads[i]).reshape(36)
        want[37:43] += Ads[i].T @ blocks[i, 37:43]
        want[43] += blocks[i, 43]
        one = np.zeros(44)
        hm.hm_to_body(_p(np.ascontiguousarray(Ads[i])), _p(np.ascontiguousarray(blocks[i])), _p(one))
        np.testing.assert_allclose(one[1:37], (Ads[i].T @ H @ Ads[i]).reshape(36), rtol=1e-12, atol=1e-12)
        assert one[0] == blocks[i, 0] and one[43] == blocks[i, 43]
    out = np.zeros(44)
    hm.hm_combine(n, _p(np.ascontiguousarray(blocks)), _p(np.ascontiguousarray(Ads)), _p(out))
    np.testing.assert_allclose(out, want, rtol=1e-12, atol=1e-11)
    # without adjoints: plain sums in job order, and a group of one is its job's block bit for bit (signed zeros too)
    out = np.zeros(44)
    hm.hm_combine(n, _p(np.ascontiguousarray(blocks)), None, _p(out))
    seq = blocks[0].copy()
    for i in range(1, n):
        seq = seq + blocks[i]
    assert np.array_equal(out, seq)
    single = blocks[:1].copy()
    single[0, 5] = -0.0
    hm.hm_combine(1, _p(single), None, _p(out))
    assert out.tobytes() == single[0].tobytes()


def test_rigidity_check(hm):
    rng = np.random.default_rng(23)
    E = _rigid(rng)
    assert hm.hm_is_rigid(_p(E)) == 1
    assert hm.hm_is_rigid(_p(np.eye(4).reshape(16).copy())) == 1
    bad = []
    m = E.copy(); m[3] = 1e-12; bad.append(m)             # bottom row
    m = E.copy(); m[15] = 2.0; bad.append(m)
    m = E.copy(); m[0] *= 1 + 1e-6; bad.append(m)          # not orthonormal
    m = E.copy(); m[0:3] *= 2.0; bad.append(m)
    m = E.copy(); m[0:3] = -m[0:3]; bad.append(m)          # a reflection
    m = E.copy(); m[12] = np.nan; bad.append(m)
    for m in bad:
        assert hm.hm_is_rigid(_p(m)) == 0
    C16 = np.zeros(16)
    A, B = _rigid(rng), _rigid(rng)
    hm.hm_mat16_mul(_p(A), _p(B), _p(C16))
    np.testing.assert_allclose(C16.reshape(4, 4).T, A.reshape(4, 4).T @ B.reshape(4, 4).T, rtol=0, atol=1e-15)


def _problem(orc, p, cell, bins):
    P = orc.Problem(p.im0, p.depth0, p.im1, p.T_wc0, p.intr, cell, bins)
    P.set_quirks(0, 1)
    return P


def test_group_of_one_equals_orc_optimize_bit_for_bit(orc, make_pair):
    p = make_pair(1000, 120, 160)
    pose0 = orc.reference_perturbation(p.T_wc1)
    P = _problem(orc, p, 4, 16)
    P.prepare(pose0)
    want_pose, want_its, want_trace, want_counts = P.optimize(pose0, 10)
    pose, its, trace, counts = group_oracle.optimize_group([P], None, pose0, 10)
    assert its == want_its
    assert pose.tobytes() == want_pose.tobytes()
    assert trace.tobytes() == want_trace.tobytes()
    assert np.array_equal(counts, want_counts)


def test_rig_group_cost_decreases(orc, synth):
    rig = synth.make_rig(3, 2, 120, 160)
    T_bw1 = orc.se3_from_mat16(synth.mat16_inverse(rig.T_wb1))
    pose0 = orc.reference_perturbation(rig.T_wb1)
    probs = []
    for g, p in enumerate(rig.pairs):
        P = _problem(orc, p, 4, 16)
        P.prepare(orc.se3_mul(orc.se3_from_mat16(rig.T_cb[g]), pose0))
        probs.append(P)
    pose, its, trace, counts = group_oracle.optimize_group(probs, rig.T_cb, pose0, 10)
    assert its >= 2
    E7 = [orc.se3_from_mat16(E) for E in rig.T_cb]
    chi0 = sum(float(np.nansum(np.minimum(P.eval(orc.se3_mul(E7[g], pose0), False)[2] ** 2, 1e9))) for g, P in enumerate(probs))
    assert trace[-1, 0] < 0.9 * chi0
    assert np.all(np.diff(trace[:, 0]) <= 0)
    # the joint solve moves the body pose towards the truth
    err0 = np.linalg.norm(pose0[:3] - T_bw1[:3])
    assert np.linalg.norm(pose[:3] - T_bw1[:3]) < err0


def _digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def test_existing_generators_are_unchanged(synth):
    p = synth.make_pair(1000, 120, 160)
    assert _digest(p.im0, p.im1, p.depth0_u16, p.T_wc0, p.T_wc1) == "458c32492cfab62ec0799da35a67293b46d3a63eed12a91a7500431512b8b41e"
    p = synth.make_pair(1003, 48, 64)
    assert _digest(p.im0, p.im1, p.depth0_u16, p.T_wc0, p.T_wc1) == "64d0d85076c6274e1d6c14e94b3649da1e29a4dd54e7f94f2b430f2a4fa495fd"
    q = synth.make_sequence(5, 3, 48, 64)
    assert _digest(*[a for x in q for a in (x.im0, x.im1)]) == "44c724c0efa7c86068df4eb16d7de2c40b9450cd4d8224a34b93d53ef60916c1"


def test_rig_and_keyframe_generators(synth):
    rig = synth.make_rig(4, 3, 60, 80)
    assert len(rig.pairs) == 3 and rig.T_cb.shape == (3, 16)
    assert np.array_equal(rig.T_cb[0], np.eye(4).reshape(16))
    sub = synth.make_rig(4, 2, 60, 80)  # the first cameras of a larger rig are the smaller rig
    assert np.array_equal(sub.pairs[1].im1, rig.pairs[1].im1) and np.array_equal(sub.T_cb, rig.T_cb[:2])
    Twb1 = rig.T_wb1.reshape(4, 4).T
    for g, p in enumerate(rig.pairs):
        Tcb = rig.T_cb[g].reshape(4, 4).T
        np.testing.assert_allclose(p.T_wc1.reshape(4, 4).T, Twb1 @ np.linalg.inv(Tcb), atol=1e-14)
        R = Tcb[:3, :3]
        if g > 0:
            tilt = np.degrees(np.arccos(np.clip(R[2, 2], -1, 1)))
            assert 15 <= tilt <= 40
        assert np.all(p.depth0_u16 > 0)
    kf = synth.make_keyframes(4, 3, 60, 80)
    assert len(kf) == 3
    assert all(np.array_equal(kf[0].im1, k.im1) and np.array_equal(kf[0].T_wc1, k.T_wc1) for k in kf)
    assert not np.array_equal(kf[0].T_wc0, kf[1].T_wc0)
    # a camera tilted by 20 degrees: the straight-down Newton start of render() does not converge, the bracketed cast does
    sc = synth._Scene(np.random.default_rng(5))
    T = np.eye(4)
    T[:3, :3] = synth._rot(np.deg2rad(20), np.deg2rad(-20), 0.05)
    intr = (synth.FX / 8, synth.FY / 8, (synth.CX + 0.5) / 8 - 0.5, (synth.CY + 0.5) / 8 - 0.5)
    _, _, res = sc.render_bracketed(T, 60, 80, intr)
    assert res < synth.RENDER_TOL
