"""The diagonal-Hessian interior point (option use_diag_hessian) in numpy -- TEST
INFRASTRUCTURE ONLY, the reference the device is held to.

The problem supplies evalHessianDiag(x, z, zw, h), the diagonal of the Hessian of the
Lagrangian, and the optimizer takes B = diag(h) where the quasi-Newton approximation
stood (IP.cpp:1464, 1842, 3811, 4458).  DiagHessianOracle runs the unmodified major
loop of oracle/ip_oracle.py with that B in the place of its quasi-Newton object, so
every statement of the loop keeps its order and meaning:

  * D0 = h + qn_sigma + zl/(x - lb) + zu/(ub - x)  wherever the loop takes the
    Hessian (use_qn); a step without it (the sequential linear step) has D0 without h;
  * the compact correction is absent (no Z: q = 0, m = c);
  * addKKTResStep: rx -= h p_x (then the qn_sigma term);
  * evalMeritInitDeriv: p^T B p = sum h p^2;
  * a "reset" or "update" of B changes nothing (h comes from the problem), and the
    loop reports resets as it does for a quasi-Newton object;
  * evalHessianDiag runs once after every evalObjConGradient (start, accepted points)
    with the multipliers of that point.
"""
import numpy as np

from oracle.ip_oracle import InteriorPointOracle
from oracle.problems import SepQuad


class DiagonalHessian:
    """B = diag(h) behind the quasi-Newton interface the loop calls (ParOptCompactQuasiNewton)."""

    b0 = 0.0  # the history's qn_b0 / qn_size columns: no compact form
    Z = []

    def __init__(self, h):
        self.h = h

    def compact(self):
        # (b0, d0, M, Z).  The loop forms D0 = np.full(n, b0 + qn_sigma) + bound terms
        # (IP.cpp:1864-1910), which with the vector b0 = h is h + qn_sigma + bound terms.
        return self.h, np.zeros(0), np.zeros((0, 0)), []

    def mult(self, x):
        return self.h * x

    def mult_add(self, alpha, x, y):
        y += alpha * (self.h * x)

    def reset(self):
        pass

    def update(self, s, y):
        return 0


class _WithHessianDiag:
    """The problem, with evalHessianDiag called right after each evalObjConGradient at
    the optimizer's current multipliers (the loop calls the gradient at variables.x,
    after the step has updated z and zw)."""

    def __init__(self, problem, oracle):
        self._p = problem
        self._oracle = oracle

    def __getattr__(self, name):
        return getattr(self._p, name)

    def evalObjConGradient(self, x, g, Ac):
        fail = self._p.evalObjConGradient(x, g, Ac)
        ora = self._oracle
        v = ora.variables
        assert x is v.x
        fail = fail or self._p.evalHessianDiag(v.x, v.z, v.zw, ora.hdiag)
        return fail


class DiagHessianOracle(InteriorPointOracle):
    """InteriorPointOracle with use_diag_hessian: the options are the loop's (qn_type
    is ignored), the problem must define evalHessianDiag."""

    def __init__(self, problem, options=None, comm=None):
        super().__init__(_WithHessianDiag(problem, self), options, comm)
        self.hdiag = np.zeros(self.nvars)
        self.qn = DiagonalHessian(self.hdiag)


class DiagSepQuad(SepQuad):
    """oracle.problems.SepQuad with its exact diagonal Hessian: lam, or with the
    Householder reflector diag(P diag(lam) P) = lam - 4 v^2 lam / s + 4 v^2 (v^T lam v) / s^2,
    s = v^T v (the constraints are linear: z and zw add nothing)."""

    def evalHessianDiag(self, x, z, zw, hdiag):
        if self.p["householder"]:
            vlv = self._sum([np.dot(self.vh * self.lam, self.vh)])[0]
            v2 = self.vh * self.vh
            hdiag[:] = (self.lam - (4.0 / self.vtv) * (v2 * self.lam)) + \
                (4.0 * vlv / (self.vtv * self.vtv)) * v2
        else:
            hdiag[:] = self.lam
        return 0
