"""The diagonal-Hessian interior point (option use_diag_hessian) in numpy
(tests/diag_hessian_oracle.py): the problem's evalHessianDiag replaces the quasi-Newton
approximation, the KKT Hessian block is diag(h) + qn_sigma.  C3 is separable (its Hessian
is diag(lam)), so there the option is Newton's method; tests/test_gpu_diag_hessian.py
holds the library to this oracle."""
import numpy as np
import pytest

from oracle.ip_oracle import InteriorPointOracle, Vars
from oracle.problems import SepQuad
from paropt_b200 import configs
from tests.diag_hessian_oracle import DiagHessianOracle, DiagSepQuad


def _run(cfg, diag=False, **options):
    cls, prob = (DiagHessianOracle, DiagSepQuad) if diag else (InteriorPointOracle, SepQuad)
    ip = cls(prob(**cfg["problem"]), dict(cfg["options"], **options))
    assert ip.optimize() == 0
    return ip


def test_newton_on_c3_reaches_the_l_bfgs_optimum_in_fewer_iterations(capsys):
    """C3-small is strictly convex, so both runs approach the one optimum; at
    abs_res_tol = 1e-10 the diagonal-Hessian run converges on the tolerance test and its
    x agrees with L-BFGS's final x to 1e-8 relative (measured 1.9e-9: L-BFGS stops on its
    no-improvement test with max_prime = 4e-9).  Iterations: 34 against 76."""
    cfg = configs.small("C3")
    lbfgs = _run(cfg, abs_res_tol=1e-10)
    newton = _run(cfg, diag=True, abs_res_tol=1e-10)
    assert newton.converged == "tolerance"
    assert lbfgs.converged is not None
    x0, x1 = lbfgs.variables.x, newton.variables.x
    rel = np.linalg.norm(x1 - x0) / np.linalg.norm(x0)
    assert rel <= 1e-8, rel
    assert newton.niter < lbfgs.niter, (newton.niter, lbfgs.niter)
    assert all(r["qn_size"] == 0 and r["qn_b0"] == 0.0 for r in newton.history)
    with capsys.disabled():
        print("\nC3-small iterations: L-BFGS %d, diagonal Hessian %d (|dx|/|x| = %.1e)"
              % (lbfgs.niter, newton.niter, rel))


def test_householder_diagonal_is_the_diagonal_of_the_hessian():
    """sepquad with the reflector: evalHessianDiag returns diag(P diag(lam) P)."""
    prob = DiagSepQuad(ntotal=40, ncon=1, householder=1, lam_min=1.0, lam_max=10.0)
    P = np.eye(40) - 2.0 * np.outer(prob.vh, prob.vh) / prob.vtv
    H = P @ np.diag(prob.lam) @ P
    h = np.zeros(40)
    assert prob.evalHessianDiag(np.zeros(40), np.zeros(1), np.zeros(0), h) == 0
    np.testing.assert_allclose(h, np.diag(H), rtol=1e-13, atol=0)


def _dense_kkt(ip, v, h):
    """The Newton matrix K of the residual computeKKTRes, with the Hessian block
    diag(h) + qn_sigma, built entry by entry (unknowns ordered x, zl, zu, z, s, t, zs, zt,
    zw, sw, tw, zsw, ztw)."""
    n, c, w = ip.nvars, ip.ncon, ip.nwcon
    sizes = [n, n, n, c, c, c, c, c, w, w, w, w, w]
    off = np.concatenate([[0], np.cumsum(sizes)])
    X, ZL, ZU, Z, S, T, ZS, ZT, ZW, SW, TW, ZSW, ZTW = [slice(off[i], off[i + 1])
                                                       for i in range(13)]
    K = np.zeros((off[-1], off[-1]))
    A = np.array(ip.Ac)  # c x n
    Aw = np.zeros((w, n))
    for i in range(w):  # Aw^T e_i
        e = np.zeros(w)
        e[i] = 1.0
        col = np.zeros(n)
        ip.w.add_jac_t(1.0, e, col)
        Aw[i] = col
    mbv = ip.opt["max_bound_value"]
    I_n, I_c, I_w = np.eye(n), np.eye(c), np.eye(w)
    # x row: (diag(h) + sigma) px - A^T pz - pzl + pzu - Aw^T pzw
    K[X, X] = np.diag(h + ip.opt["qn_sigma"])
    K[X, Z] = -A.T
    K[X, ZL] = -I_n
    K[X, ZU] = I_n
    K[X, ZW] = -Aw.T
    # bound rows (identity where the bound is absent: the step's entry is zero there)
    ml, mu = ip.lb > -mbv, ip.ub < mbv
    K[ZL, X] = np.diag(np.where(ml, v.zl, 0.0))
    K[ZL, ZL] = np.diag(np.where(ml, v.x - ip.lb, 1.0))
    K[ZU, X] = np.diag(np.where(mu, -v.zu, 0.0))
    K[ZU, ZU] = np.diag(np.where(mu, ip.ub - v.x, 1.0))
    # dense constraint rows
    K[Z, X] = A
    K[Z, S] = -I_c
    K[Z, T] = I_c
    K[S, ZS] = -I_c
    K[S, Z] = I_c
    K[T, ZT] = -I_c
    K[T, Z] = -I_c
    K[ZS, S] = np.diag(v.zs)
    K[ZS, ZS] = np.diag(v.s)
    K[ZT, T] = np.diag(v.zt)
    K[ZT, ZT] = np.diag(v.t)
    # weighting rows
    K[ZW, X] = Aw
    K[ZW, SW] = -I_w
    K[ZW, TW] = I_w
    K[SW, ZSW] = -I_w
    K[SW, ZW] = I_w
    K[TW, ZTW] = -I_w
    K[TW, ZW] = -I_w
    K[ZSW, SW] = np.diag(v.zsw)
    K[ZSW, ZSW] = np.diag(v.sw)
    K[ZTW, TW] = np.diag(v.ztw)
    K[ZTW, ZTW] = np.diag(v.tw)
    return K


def _flat(b):
    return np.concatenate([b.x, b.zl, b.zu, b.z, b.s, b.t, b.zs, b.zt,
                           b.zw, b.sw, b.tw, b.zsw, b.ztw])


@pytest.mark.parametrize("sigma", [0.0, 0.5])
def test_one_kkt_solve_solves_the_dense_newton_system(sigma):
    """Three iterations into C3 (n = 256, 32 weighting rows, lower bounds on some
    variables only), one KKT solve with its refinement step: |r - K p| <= 1e-12 |r| with
    K built densely from diag(h) + qn_sigma."""
    cfg = configs.get("C3", 256)
    ip = DiagHessianOracle(DiagSepQuad(**cfg["problem"]),
                           dict(cfg["options"], qn_sigma=sigma, max_major_iters=3))
    assert ip.optimize() == 0
    v, mu = ip.variables, ip.barrier_param
    n, nw, c = ip.nvars, ip.nwcon, ip.ncon
    res, upd, ref = Vars(n, nw, c), Vars(n, nw, c), Vars(n, nw, c)
    ip.computeKKTRes(v, mu, res)
    ip.setUpKKTDiagSystem(v, 1)
    ip.setUpKKTSystem(v, 1)
    ip.computeKKTStep(v, res, upd, 1)
    ip.computeKKTRes(v, mu, res)
    ip.addKKTResStep(v, upd, res)
    ip.computeKKTStep(v, res, ref, 1)
    upd.add(ref)
    ip.computeKKTRes(v, mu, res)
    r = _flat(res)
    K = _dense_kkt(ip, v, ip.hdiag)
    err = r - K @ _flat(upd)
    assert np.max(np.abs(r)) > 0.0
    assert np.max(np.abs(err)) <= 1e-12 * np.max(np.abs(r)), np.max(np.abs(err))
    # and addKKTResStep forms the same residual
    ip.addKKTResStep(v, upd, res)
    np.testing.assert_allclose(_flat(res), err, rtol=0, atol=1e-12 * np.max(np.abs(r)))
