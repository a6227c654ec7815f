"""Joint LM solve over several frame pairs that share one pose, on top of the CPU oracle (oracle/binding.py): the reference's
optimize(max_iters) schedule (optimization_algorithm_levenberg.cpp:61-250, as oracle/nid_oracle.cpp's orc_optimize states it)
over the unary NID edges of all problems on one SE3 vertex, in g2o's edge order: problem 0's cells, then problem 1's.

Problem i's edges are evaluated at E_i * T (E_i column-major rigid camera-from-body, or the identity) and its Jacobians
taken w.r.t. the body update T <- exp(xi) * T: J_body = J_cam * Ad(E_i), Ad = [[R, 0], [t^ R, R]] for xi = (omega, upsilon).
The per-edge arithmetic is the oracle's (orc_eval for errors and Jacobians, orc_huber, orc_ldlt6_solve, orc_se3_*), summed in
the order of its build_system and robust_chi2; for one problem without E the result equals orc_optimize bit for bit
(tests/test_groups_cpu.py holds it to that). TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import ctypes as C
import math

import numpy as np

from oracle import binding as orc

_dp = C.POINTER(C.c_double)


def adjoint6(E16):
    """6x6 adjoint of a rigid column-major 4x4 for xi = (omega, upsilon)."""
    M = np.asarray(E16, dtype=np.float64).reshape(4, 4).T
    R, t = M[:3, :3], M[:3, 3]
    tx = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]])
    Ad = np.zeros((6, 6))
    Ad[:3, :3] = R
    Ad[3:, 3:] = R
    Ad[3:, :3] = tx @ R
    return Ad


def _edges(problems, E7, Ads, pose7, want_jac):
    """Per problem (err [cells], J_body [cells][6] as Python floats or None) at the body pose."""
    out = []
    for i, P in enumerate(problems):
        p = pose7 if E7 is None else orc.se3_mul(E7[i], pose7)
        _, _, err, J = P.eval(p, want_jac)
        Jb = None
        if want_jac:
            Jb = J.tolist()
            if Ads is not None:
                Ad = Ads[i].tolist()
                for c in range(len(Jb)):
                    row = Jb[c]
                    nb = []
                    for j in range(6):
                        s = 0.0
                        for k in range(6):
                            s += row[k] * Ad[k][j]
                        nb.append(s)
                    Jb[c] = nb
        out.append((err.tolist(), Jb))
    return out


def _chi2(edges, delta):
    chi = 0.0
    for err, _ in edges:
        for e in err:
            if math.isnan(e):
                continue
            chi += orc.huber(e * e, delta)[0]
    return chi


def _system(edges, delta):
    H = [0.0] * 36
    b = [0.0] * 6
    for err, J in edges:
        for c, e in enumerate(err):
            if math.isnan(e):
                continue
            r1 = orc.huber(e * e, delta)[1]
            Jc = J[c]
            for i in range(6):
                b[i] -= r1 * Jc[i] * 1.0 * e
            for i in range(6):
                for j in range(6):
                    H[i * 6 + j] += Jc[i] * r1 * Jc[j]
    return H, b


def optimize_group(problems, E16, pose7, max_iters=10, delta=math.sqrt(0.95)):
    """The reference's LM over the edges of `problems` (oracle Problems, prepared) at one pose. E16: [n][16] or None.
    Returns (pose7, outer iterations, trace [its][10] as orc_optimize writes it, counts {jac_evals, cost_evals}); the cost
    count includes orc_optimize's re-evaluation at the end of every outer iteration."""
    E7 = None if E16 is None else [orc.se3_from_mat16(E) for E in np.asarray(E16, dtype=np.float64).reshape(-1, 16)]
    Ads = None if E16 is None else [adjoint6(E) for E in np.asarray(E16, dtype=np.float64).reshape(-1, 16)]
    L = orc.lib()
    est = np.array(pose7, dtype=np.float64)
    lam, ni, nBad = -1.0, 2.0, 0
    tau, goodUp, goodLo, maxTrials = 1e-5, 2.0 / 3.0, 1.0 / 3.0, 10
    jac_evals = cost_evals = 0
    x = np.zeros(6)
    trace = []
    it, ok = 0, True
    while it < max_iters and ok:
        edges = _edges(problems, E7, Ads, est, True)
        currentChi = _chi2(edges, delta)
        iniChi = currentChi
        jac_evals += 1
        H, b = _system(edges, delta)
        if it == 0:
            md = 0.0
            for j in range(6):
                md = max(abs(H[j * 6 + j]), md)
            lam = tau * md
            ni, nBad = 2.0, 0
        rho, qmax = 0.0, 0
        while True:
            backup = est.copy()
            Hl = np.array(H)
            for j in range(6):
                Hl[j * 6 + j] += lam
            bb = np.array(b)
            ok2 = L.orc_ldlt6_solve(Hl.ctypes.data_as(_dp), bb.ctypes.data_as(_dp), x.ctypes.data_as(_dp))
            est = orc.se3_mul(orc.se3_exp(x), est)
            cost_evals += 1
            tempChi = _chi2(_edges(problems, E7, Ads, est, False), delta)
            if not ok2:
                tempChi = np.finfo(np.float64).max
            rho = currentChi - tempChi
            scale = 0.0
            xl = x.tolist()
            for j in range(6):
                scale += xl[j] * (lam * xl[j] + b[j])
            scale += 1e-3
            rho /= scale
            if rho > 0 and math.isfinite(tempChi):
                alpha = 1.0 - math.pow(2 * rho - 1, 3)
                alpha = min(alpha, goodUp)
                lam *= max(goodLo, alpha)
                ni = 2.0
                currentChi = tempChi
            else:
                lam *= ni
                ni *= 2
                est = backup
            qmax += 1
            if not (rho < 0 and qmax < maxTrials):
                break
        terminate = qmax == maxTrials or rho == 0
        if not terminate:
            nBad = nBad + 1 if (iniChi - currentChi) * 1e3 < iniChi else 0
            terminate = nBad >= 3
        ok = not terminate
        # orc_optimize re-evaluates at the current estimate here (the verbose block of SparseOptimizer::optimize); the
        # oracle is deterministic, so that chi2 is currentChi: counted, not recomputed
        cost_evals += 1
        trace.append([currentChi, lam, qmax, *est.tolist()])
        it += 1
    return est, it, np.array(trace).reshape(-1, 10), np.array([jac_evals, cost_evals], dtype=np.int32)
