"""The synthetic workloads of oracle/problems.py as TorchProblem / AutogradProblem
subclasses: the inputs come from the oracle's numpy generators (same seeds, same
rank partition), are uploaded once, and every callback is torch arithmetic on the
device.  Used by tests/test_gpu_torch_problem.py, scripts/torch_problem_bench.py and
scripts/torch_problem_mgpu.py."""
import numpy as np
import torch

from oracle.problems import Rosenbrock, SepQuad
from paropt_b200.api import AutogradProblem, TorchProblem


def weighting_dict(w):
    """oracle.ip_oracle.Weighting -> the weighting= dict of the Python problem classes."""
    return dict(nwcon=w.nwcon, wstart=w.start, nw=w.nw, wstride=w.stride,
                coef0=float(w.coef[0]), coef_rest=float(w.coef[-1]), wconst=w.const)


class _CtxComm:
    """The oracle's `comm` (rank, size, allreduce) over a Context."""

    def __init__(self, ctx):
        self.ctx, self.rank, self.size = ctx, ctx.rank, ctx.size

    def allreduce(self, vals, op):
        return self.ctx.allreduce_sum(vals)


class _SepQuadData:
    """Uploads the seeded inputs of oracle.problems.SepQuad for this rank."""

    def _load(self, ctx, params):
        ref = SepQuad(comm=_CtxComm(ctx) if ctx.size > 1 else None, **params)
        n = ref.nvars
        dev = torch.device("cuda", ctx.device)
        x0, lb, ub = np.empty(n), np.empty(n), np.empty(n)
        ref.getVarsAndBounds(x0, lb, ub)

        def up(a):
            return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device=dev)

        self.hh = bool(ref.p["householder"])
        self.data = dict(lam=up(ref.lam), b=up(ref.b), x0=up(x0), lb=up(lb), ub=up(ub),
                         vh=up(ref.vh) if self.hh else None)
        self.A = [up(a) for a in ref.A]
        self.vtv = float(ref.vtv)
        self.beta = ref.beta.copy()
        self.beta_dev = up(ref.beta)
        weighting = weighting_dict(ref.weighting) if ref.nwcon > 0 else None
        return ref, weighting

    def _sums(self, parts):
        """Sum over the ranks of a list of 0-d tensors: stays on the device on one rank."""
        v = torch.stack(parts)
        return self.ctx.allreduce_sum(v) if self.ctx.size > 1 else v

    def _applyP(self, x):
        if not self.hh:
            return x
        vh = self.data["vh"]
        vx = self._sums([torch.dot(vh, x)])[0]
        return x - (2.0 * vx / self.vtv) * vh


class TorchSepQuad(_SepQuadData, TorchProblem):
    """oracle.problems.SepQuad with explicit torch derivatives."""

    def __init__(self, ctx, **params):
        self.ctx = ctx
        ref, weighting = self._load(ctx, params)
        super().__init__(ctx, ref.nvars, ref.ncon, ninequality=ref.ncon,
                         nwinequality=ref.nwcon, weighting=weighting)

    def getVarsAndBounds(self, x, lb, ub):
        x.copy_(self.data["x0"])
        lb.copy_(self.data["lb"])
        ub.copy_(self.data["ub"])

    def evalObjCon(self, x):
        d = self.data
        y = self._applyP(x)
        f = 0.5 * torch.dot(d["lam"] * y, y) + torch.dot(d["b"], x)
        s = self._sums([f] + [torch.dot(a, x) for a in self.A])
        beta = self.beta_dev if torch.is_tensor(s) else self.beta
        return 0, s[0], beta + s[1:]

    def _hess(self, p, out):
        """out = P diag(lam) P p."""
        d = self.data
        torch.mul(d["lam"], self._applyP(p), out=out)
        if self.hh:
            vw = self._sums([torch.dot(d["vh"], out)])[0]
            out.sub_((2.0 * vw / self.vtv) * d["vh"])

    def evalObjConGradient(self, x, g, A):
        self._hess(x, g)
        g.add_(self.data["b"])
        for j, a in enumerate(self.A):
            A[j].copy_(a)
        return 0

    def evalHvecProduct(self, x, z, zw, px, hvec):
        self._hess(px, hvec)
        return 0


class AutogradSepQuad(_SepQuadData, AutogradProblem):
    """oracle.problems.SepQuad with only objcon written out (one rank)."""

    def __init__(self, ctx, **params):
        self.ctx = ctx
        ref, weighting = self._load(ctx, params)
        super().__init__(ctx, ref.nvars, ref.ncon, ninequality=ref.ncon,
                         nwinequality=ref.nwcon, weighting=weighting)

    getVarsAndBounds = TorchSepQuad.getVarsAndBounds

    def objcon(self, x):
        d = self.data
        y = self._applyP(x)
        f = 0.5 * torch.dot(d["lam"] * y, y) + torch.dot(d["b"], x)
        return f, self.beta_dev + torch.stack([torch.dot(a, x) for a in self.A])


class TorchRosenbrock(TorchProblem):
    """oracle.problems.Rosenbrock (examples/rosenbrock/rosenbrock.cpp) with the
    weighting rows; configs "C1" has n = nvars + 1 = 1000."""

    def __init__(self, ctx, n=1000):
        ref = Rosenbrock(nvars=int(n) - 1)
        super().__init__(ctx, ref.nvars, ref.ncon, ninequality=ref.ninequality,
                         nwinequality=ref.nwinequality, weighting=weighting_dict(ref.weighting))

    def getVarsAndBounds(self, x, lb, ub):
        x.fill_(-1.0)
        lb.fill_(-2.0)
        ub.fill_(1.0)

    def evalObjCon(self, x):
        d = x[1:] - x[:-1] ** 2
        f = torch.sum((1.0 - x[:-1]) ** 2 + 100.0 * d * d)
        return 0, f, torch.stack([0.25 - torch.sum(x * x), 10.0 + torch.sum(x[::2])])

    def evalObjConGradient(self, x, g, A):
        d = x[1:] - x[:-1] ** 2
        g.zero_()
        g[:-1] += -2.0 * (1.0 - x[:-1]) + 200.0 * d * (-2.0 * x[:-1])
        g[1:] += 200.0 * d
        torch.mul(x, -2.0, out=A[0])
        A[1].zero_()
        A[1][::2] = 1.0
        return 0


def make(ctx, cfg, autograd=False):
    """The torch problem of a named workload (configs.py / golden `config`)."""
    if cfg["kind"] == "rosenbrock":
        return TorchRosenbrock(ctx, **cfg["problem"])
    return (AutogradSepQuad if autograd else TorchSepQuad)(ctx, **cfg["problem"])
