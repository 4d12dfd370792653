"""Drop-in namespace for `from paropt import ParOpt` on the interior-point path
(SURVEY.md section 8f-2): the classes and helpers of paropt/ParOpt.pyx that the
hot path needs, served by libparopt_b200.so instead of the Cython extension --
no mpi4py, no MPI.  Where the reference takes an MPI communicator this module
takes a `Context` (one per GPU / rank); `ParOpt.Problem(None, ...)` opens GPU 0.

    from paropt_b200 import ParOpt
    class Quadratic(ParOpt.Problem): ...            # same callbacks as the reference
    opt = ParOpt.Optimizer(problem, {"algorithm": "ip", "qn_type": "bfgs"})
    opt.optimize(); x, z, zw, zl, zu = opt.getOptimizedPoint()

`algorithm = "ip"` and `algorithm = "tr"` (SL1QP trust region, penalty method) are built;
the MMA front end is not.

`Problem` callbacks see numpy views of host mirrors: the iterate and the gradients
cross PCIe on every call.  A problem already written in torch subclasses
`TorchProblem` instead: the same callbacks on float64 CUDA tensors that view the
optimizer's own device memory, run on the optimizer's stream, with no host copies
but the objective and constraint values.  `AutogradProblem` needs only `objcon(x)
-> (f, c)` in torch and takes the gradients and Hessian-vector products
(`use_hvec_product`) from autograd.

A `Problem` or `TorchProblem` subclass that defines `evalHessianDiag(x, z, zw,
hdiag)` -- the diagonal of the Hessian of the Lagrangian, written into `hdiag` --
can run with the option `use_diag_hessian`: the interior point then takes
`diag(hdiag) + qn_sigma` as its Hessian in place of a quasi-Newton approximation
(an exact Newton method where the Hessian is diagonal).  It runs with the monotone
barrier, one refinement step and 1 to 32 dense constraints; other settings, the
trust region and `AutogradProblem` are refused.

    class Model(ParOpt.TorchProblem):
        def evalObjConGradient(self, x, g, A): g.copy_(...); A[0].copy_(...)
"""
import numpy as np

from . import api
from .api import AutogradProblem, Context, PVec, QuasiDefBlockMat, TorchProblem  # noqa: F401

# ParOptQuasiNewton.h:18-30 enumerations, by the option strings the library takes
SKIP_NEGATIVE_CURVATURE = "skip_negative_curvature"
DAMPED_UPDATE = "damped_update"
YTY_OVER_YTS = "yty_over_yts"
YTS_OVER_STS = "yts_over_sts"

_default_ctx = None


def _context(comm):
    global _default_ctx
    if isinstance(comm, Context):
        return comm
    if _default_ctx is None:
        _default_ctx = Context(0)
    return _default_ctx


class Problem(api.Problem):
    """ParOpt.Problem (ParOpt.pyx:787-907): subclass and implement
    getVarsAndBounds(x, lb, ub), evalObjCon(x) -> (fail, fobj, con),
    evalObjConGradient(x, g, A) -> fail.  The sparse constraints are the weighting
    rows of `weighting=` (nwblock = 1) instead of the four sparse callbacks."""

    def __init__(self, comm=None, nvars=0, ncon=0, nwcon=0, nwblock=1, ninequality=-1,
                 nwinequality=-1, use_lower=True, use_upper=True, weighting=None):
        if nwcon and not weighting:
            raise ValueError("nwcon > 0 needs weighting=dict(nwcon, wstart, nw, wstride, coef0, "
                             "coef_rest, wconst): general sparse constraints are not built")
        if nwcon and nwblock != 1:
            raise ValueError("only nwblock = 1 is built")
        super().__init__(_context(comm), nvars, ncon, ninequality=ninequality,
                         nwinequality=nwinequality, use_lower=use_lower, use_upper=use_upper,
                         weighting=weighting)

    def createDesignVec(self):
        return PVec(self.ctx, self.nvars)

    def createConstraintVec(self):
        return PVec(self.ctx, int(self._w.nwcon))


class InteriorPoint(api.InteriorPoint):
    """ParOpt.InteriorPoint (ParOpt.pyx:1189-1365)."""

    def getOptimizedSlacks(self):
        d = self.get_dense()
        return d["s"], d["t"]

    def getIterationCounters(self):
        return self.counters()


class LBFGS(api.QuasiNewton):
    """ParOpt.LBFGS (ParOpt.pyx): LBFGS(problem, subspace=10)."""

    def __init__(self, problem, subspace=10, update_type=SKIP_NEGATIVE_CURVATURE,
                 diag_type=YTY_OVER_YTS):
        super().__init__(problem.ctx, problem.nvars, "bfgs", subspace)
        self.set_option("qn_update_type", update_type)
        self.set_option("qn_diag_type", diag_type)


class LSR1(api.QuasiNewton):
    """ParOpt.LSR1 (ParOpt.pyx): LSR1(problem, subspace=10)."""

    def __init__(self, problem, subspace=10):
        super().__init__(problem.ctx, problem.nvars, "sr1", subspace)


class TrustRegion(api.TrustRegion):
    """ParOpt.TrustRegion (ParOptTrustRegion.h) over the built-in quadratic subproblem."""


class Optimizer:
    """ParOpt.Optimizer (ParOptOptimizer.cpp:27-175): algorithm = "ip" runs the
    interior-point optimizer on the problem, algorithm = "tr" the trust-region front
    end (quadratic model with the compact quasi-Newton Hessian of the qn_* options,
    ParOptOptimizer.cpp:102-175).  The reference's default is "tr"
    (ParOptOptimizer.cpp:41)."""

    def __init__(self, problem, options=None):
        self.problem = problem
        self.options = dict(options or {})
        self.algorithm = self.options.pop("algorithm", "tr")
        if self.algorithm not in ("ip", "tr"):
            raise ValueError("algorithm=%r is not built ('ip' and 'tr' are)" % self.algorithm)
        self.ip = None
        self.tr = None

    def optimize(self):
        if self.algorithm == "ip":
            if self.ip is None:
                self.ip = InteriorPoint(self.problem, self.options)
            self.ip.optimize()
        else:
            if self.tr is None:
                self.tr = TrustRegion(self.problem, self.options)
            self.tr.optimize()

    def getOptimizedPoint(self):
        return (self.ip if self.algorithm == "ip" else self.tr).getOptimizedPoint()

    def setTrustRegionSubproblem(self, subproblem):
        raise NotImplementedError("user-defined trust-region subproblems are not built; the "
                                  "quadratic subproblem of ParOptOptimizer is")


def unpack_output(filename):
    """Columns of the interior-point text log (option `output_file`), as
    (names, arrays) like ParOpt.unpack_output (ParOpt.pyx:61-136).  The rows are
    the reference's fixed-width format (IP.cpp:4777-4801): four %4d then %7.1e /
    %12.5e fields, each followed by one blank."""
    names = ["iter", "nobj", "ngrd", "nhvc", "alpha", "alphx", "alphz", "fobj", "|opt|",
             "|infes|", "|dual|", "mu", "comp", "dmerit", "rho"]
    widths = [4, 4, 4, 4, 7, 7, 7, 12, 7, 7, 7, 7, 7, 8, 7]
    cols = [[] for _ in names]
    with open(filename) as fp:
        for line in fp:
            head = line.split()
            if len(head) < len(names) or not head[0].isdigit() or not head[1].isdigit():
                continue
            off = 0
            for k, w in enumerate(widths):
                field = line[off:off + w]
                off += w + 1
                try:
                    cols[k].append(int(field) if k < 4 else float(field))
                except ValueError:
                    cols[k].append(0 if k < 4 else 0.0)
    return names, [np.array(c, dtype=np.int32 if k < 4 else float) for k, c in enumerate(cols)]
