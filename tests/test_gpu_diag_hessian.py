"""The diagonal-Hessian interior point on the device (option use_diag_hessian): the
problem's evalHessianDiag replaces the quasi-Newton approximation, the KKT Hessian block
is diag(h) + qn_sigma, and the default iteration's route (DiagRhsHF -> Gram -> dense
kernel -> Pass2SVHF) runs with q = 0 columns of quasi-Newton vectors.  Held to the numpy
oracle (tests/diag_hessian_oracle.py, tests/test_oracle_diag_hessian.py) at the
tolerances of tests/parity.py."""
import ctypes as C

import numpy as np
import pytest

from paropt_b200 import configs
from tests.parity import compare_histories

pytestmark = pytest.mark.gpu

VARS, RES, UPD = 0, 1, 2
DIAG = dict(use_diag_hessian=1)


@pytest.fixture(scope="module")
def ctx():
    from paropt_b200.api import Context
    c = Context(0)
    yield c
    c.close()


def run(prob, options, history_level=2):
    from paropt_b200.api import InteriorPoint
    ip = InteriorPoint(prob, dict(options, history_level=history_level))
    try:
        ip.optimize()
        return dict(history=ip.history(), status=ip.status(), counters=ip.counters())
    finally:
        ip.free()


def oracle_run(cfg, **extra):
    from tests.diag_hessian_oracle import DiagHessianOracle, DiagSepQuad
    ref = DiagHessianOracle(DiagSepQuad(**cfg["problem"]), dict(cfg["options"], **extra))
    assert ref.optimize() == 0
    return ref


class HostDiagSepQuad:
    """The host-array sepquad (numpy callbacks) with its exact diagonal (C3: no
    reflector, h = lam)."""

    @staticmethod
    def make(ctx, params):
        from paropt_b200.host_problems import HostSepQuad

        class P(HostSepQuad):
            def evalHessianDiag(self, x, z, zw, hdiag):
                hdiag[:] = self.lam
                return 0
        return P(ctx, **params)


def torch_diag_sepquad(ctx, params, fail_at=None):
    from tests.torch_problems import TorchSepQuad

    class P(TorchSepQuad):
        calls = 0

        def evalHessianDiag(self, x, z, zw, hdiag):
            P.calls += 1
            if fail_at is not None and P.calls >= fail_at:
                return 1
            hdiag.copy_(self.data["lam"])
            return 0
    return P(ctx, **params)


@pytest.mark.parametrize("name,extra", [("C3", {}), ("C2", {}),
                                        ("C3", dict(hessian_reset_freq=5))],
                         ids=["C3", "C2", "C3-reset5"])
def test_full_history_matches_oracle(ctx, name, extra):
    """C3-small: exact diagonal, weighting constraints.  C2-small: the Householder
    reflector (h is the diagonal of P diag(lam) P, not the Hessian), 10 dense
    constraints, affine start.  C3-small with hessian_reset_freq = 5: the resets of the
    loop, reported (resetH) and without effect on diag(h).  Whole runs: iteration count,
    status, evaluation counts and info tags identical, every row within RTOL = 1e-10."""
    from paropt_b200.api import problem_from_config
    cfg = configs.small(name)
    cfg["options"].update(extra)
    prob = problem_from_config(ctx, cfg)
    try:
        out = run(prob, dict(cfg["options"], **DIAG))
    finally:
        prob.free()
    ref = oracle_run(cfg)
    n, worst, first = compare_histories(ref.history, out["history"], cfg=cfg)
    assert first is None, (first, worst)
    assert len(out["history"]) == len(ref.history)
    assert out["counters"] == (ref.niter, ref.neval, ref.ngeval)
    assert out["status"] == ref.converged == "tolerance"
    for row, rec in zip(ref.log, out["history"]):
        assert row["info"] == rec["info"], (row, rec["iter"])
    assert all(rec["qn_size"] == 0 and rec["qn_b0"] == 0.0 for rec in out["history"])


@pytest.mark.parametrize("kind", ["host", "torch"])
def test_python_problems_match_the_builtin_problem(ctx, kind):
    """The C3-small history through a numpy Problem (host arrays, one host->device copy of
    h per evaluation) and through a TorchProblem (device tensors) agrees with the built-in
    problem's to 1e-12."""
    from paropt_b200.api import problem_from_config
    cfg = configs.small("C3")
    opts = dict(cfg["options"], **DIAG)
    builtin = problem_from_config(ctx, cfg)
    try:
        ref = run(builtin, opts)
    finally:
        builtin.free()
    prob = (HostDiagSepQuad.make(ctx, cfg["problem"]) if kind == "host"
            else torch_diag_sepquad(ctx, cfg["problem"]))
    try:
        out = run(prob, opts)
    finally:
        prob.free()
    n, worst, first = compare_histories(ref["history"], out["history"], cfg=cfg, rtol=1e-12)
    assert first is None, (first, worst)
    assert n == len(ref["history"]) == len(out["history"])
    assert out["status"] == ref["status"] and out["counters"] == ref["counters"]
    for a, b in zip(ref["history"], out["history"]):
        assert a["info"] == b["info"]


def launches_per_iteration(ctx, cfg, extra, iters=3, warmup=2):
    from paropt_b200.api import InteriorPoint, problem_from_config
    prob = problem_from_config(ctx, cfg)
    ip = InteriorPoint(prob, dict(cfg["options"], max_major_iters=1000000, **extra))
    try:
        ip.begin()
        ip.iterate(warmup)
        ctx.profile(2)
        ip.iterate(iters)
        ctx.profile(0)
        counts = {}
        for name, (_, cnt) in ctx.profile_totals().items():
            base = name.split("<")[0]
            counts[base] = counts.get(base, 0) + cnt
    finally:
        ctx.profile(0)
        ip.free()
        prob.free()
    return {k: v / iters for k, v in counts.items()}


@pytest.mark.parametrize("n,staged", [(8 * 5003, True), (None, False)])
def test_launch_composition_of_an_iteration(ctx, n, staged):
    """C3 with the option: per iteration no quasi-Newton update kernel, one Gram pass, one
    dense-kernel launch and one pass of the Pass2SVF family (Pass2SVHF) -- with the
    bulk-copy staged kernels forced on at a small size and at the full size.  (With the
    staged kernels forced at the small size the Gram pass takes two launches, the same as
    in the L-BFGS iteration there: the staged kernel and the general kernel for the rows
    it leaves.)"""
    cfg = configs.get("C3", n)
    if staged:
        ctx.set_param("tma_min_tiles", 1)
        ctx.set_param("tma_grid", 7)
    try:
        per_it = launches_per_iteration(ctx, cfg, DIAG)
        lbfgs = launches_per_iteration(ctx, cfg, {})
    finally:
        ctx.set_param("tma_min_tiles", 0)
        ctx.set_param("tma_grid", 0)
    print(per_it, lbfgs)
    assert not any(k.startswith(("Update2", "sr1_pairs")) for k in per_it), per_it
    assert per_it.get("gram_kernel", 0) == lbfgs.get("gram_kernel"), (per_it, lbfgs)
    if not staged:
        assert per_it.get("gram_kernel", 0) == 1, per_it
    assert per_it.get("dense_kernel", 0) == 1, per_it
    assert per_it.get("Pass2SVHF", 0) == 1, per_it
    assert per_it.get("Pass2SVF", 0) == 0 and per_it.get("Pass2SF", 0) == 0, per_it
    assert per_it.get("Pass2R1F", 0) == 0, per_it
    assert per_it.get("DiagRhsHF", 0) == 1 and per_it.get("DiagRhsF", 0) == 0, per_it


@pytest.mark.parametrize("on_device", [1, 0])
def test_kkt_solve_solves_the_linearised_system(ctx, on_device):
    """At n = 64M, 4 iterations in: one KKT solve (dense algebra on the device, or on the
    host) leaves r - K p at <= 1e-9 of r in the x, dual and infeasibility norms, K with the
    Hessian block diag(h) + qn_sigma (addKKTResStep with rx -= h p_x)."""
    from paropt_b200.api import InteriorPoint, problem_from_config
    cfg = configs.get("C3")
    prob = problem_from_config(ctx, cfg)
    ip = InteriorPoint(prob, dict(cfg["options"], max_major_iters=1000000, **DIAG))
    try:
        ip.begin()
        ip.iterate(4)
        mu = ip.getBarrierParameter()
        lib, h = ip.lib, ip.h

        def norms():
            v = [C.c_double() for _ in range(4)]
            assert lib.pcu_ip_res_norm(h, *[C.byref(a) for a in v]) == 0
            return [a.value for a in v]

        assert lib.pcu_ip_kkt_res(h, VARS, mu, RES) == 0
        r0 = norms()
        assert lib.pcu_ip_kkt_solve(h, RES, UPD, on_device) == 0
        assert lib.pcu_ip_kkt_res(h, VARS, mu, RES) == 0
        assert lib.pcu_ip_add_kkt_res_step(h, UPD, RES) == 0
        r1 = norms()
        assert max(r0[:3]) > 0.0
        assert max(r1[:3]) <= 1e-9 * max(r0[:3]), (r0, r1)
    finally:
        ip.free()
        prob.free()


def test_full_c3_run_reaches_the_l_bfgs_point(ctx):
    """C3 at n = 64M to convergence (abs_res_tol = 1e-8) with the diagonal Hessian and with
    L-BFGS: the final points agree to 1e-6 relative; the Newton run takes fewer
    iterations."""
    from paropt_b200.api import InteriorPoint, problem_from_config
    cfg = configs.get("C3")
    xs, iters = [], []
    for extra in ({}, DIAG):
        prob = problem_from_config(ctx, cfg)
        ip = InteriorPoint(prob, dict(cfg["options"], abs_res_tol=1e-8, history_level=0,
                                      **extra))
        try:
            ip.optimize()
            assert ip.status() is not None
            xs.append(ip.getOptimizedPoint()[0].to_numpy())
            iters.append(ip.counters()[0])
        finally:
            ip.free()
            prob.free()
    rel = np.linalg.norm(xs[1] - xs[0]) / np.linalg.norm(xs[0])
    print("C3 n=64M iterations: L-BFGS %d, diagonal Hessian %d, |dx|/|x| = %.2e"
          % (iters[0], iters[1], rel))
    assert rel <= 1e-6, rel
    assert iters[1] < iters[0], iters


REFUSED = [
    ("no_callback", None),
    ("autograd", None),
    ("use_hvec_product", dict(use_hvec_product=1)),
    ("set_quasi_newton", None),
    ("mehrotra", dict(barrier_strategy="mehrotra")),
    ("mpc", dict(barrier_strategy="mehrotra_predictor_corrector")),
    ("comp_fraction", dict(barrier_strategy="complementarity_fraction")),
    ("no_refinement", dict(iterative_refinement_steps=0)),
    ("two_refinements", dict(iterative_refinement_steps=2)),
    ("slm", dict(sequential_linear_method=1)),
    ("no_dense_constraint", None),
]


@pytest.mark.parametrize("case,options", REFUSED, ids=[c for c, _ in REFUSED])
def test_refused_combinations(ctx, case, options):
    """Each combination outside the covered route: pcu_ip_begin returns non-zero, and the
    Python optimizer raises."""
    from paropt_b200.api import InteriorPoint, QuasiNewton, problem_from_config
    cfg = configs.get("C3", 8 * 512)
    if case == "no_callback":
        prob = problem_from_config(ctx, configs.small("C1"))  # no evalHessianDiag
    elif case == "autograd":
        from tests.torch_problems import AutogradSepQuad
        prob = AutogradSepQuad(ctx, **cfg["problem"])
    elif case == "no_dense_constraint":
        prob = problem_from_config(ctx, configs.get("C3", 8 * 512, ncon=0))
    else:
        prob = problem_from_config(ctx, cfg)
    opts = dict(cfg["options"], **DIAG)
    opts.update(options or {})
    qn = None
    for attempt in ("c", "python"):
        ip = InteriorPoint(prob, opts)
        try:
            if case == "set_quasi_newton":
                qn = QuasiNewton(ctx, prob.nvars)
                ip.setQuasiNewton(qn)
            if attempt == "c":
                assert ip.lib.pcu_ip_begin(ip.h) != 0
                assert ip.lib.pcu_ip_optimize(ip.h) != 0
            else:
                with pytest.raises(RuntimeError):
                    ip.optimize()
        finally:
            ip.free()
            if qn is not None:
                qn.free()
                qn = None
    prob.free()


def test_trust_region_refuses_the_option(ctx):
    from paropt_b200.api import TrustRegion, problem_from_config
    prob = problem_from_config(ctx, configs.get("C3", 8 * 512))
    tr = TrustRegion(prob)
    try:
        assert tr.lib.pcu_tr_set_option_int(tr.h, b"use_diag_hessian", 1) != 0
        with pytest.raises(ValueError):
            tr.setOption("use_diag_hessian", 1)
    finally:
        tr.free()
        prob.free()


def test_failed_diagonal_is_a_failed_gradient_evaluation(ctx):
    """evalHessianDiag reporting a failure at the starting point stops the run, as a
    failed initial gradient evaluation does."""
    from paropt_b200.api import InteriorPoint
    cfg = configs.small("C3")
    prob = torch_diag_sepquad(ctx, cfg["problem"], fail_at=1)
    ip = InteriorPoint(prob, dict(cfg["options"], **DIAG))
    try:
        assert ip.lib.pcu_ip_optimize(ip.h) != 0
    finally:
        ip.free()
        prob.free()
