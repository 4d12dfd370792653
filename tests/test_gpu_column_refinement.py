"""The default iteration's KKT solve (one iterative-refinement step, at most 32 columns
[A|Z]) does its refinement in the column space of [A|Z] (pcu_dense.cuh:
pcu_dense_solve): after the Gram pass and one dense-kernel launch, a single pass
(Pass2SVF) applies the refined step and takes its statistics.  Parity of that route
with the oracle, the elementwise two-pass refinement (PCU_NO_FUSE21) and the host's
dense algebra (PCU_NO_CHAIN) is held by tests/test_gpu_gram_paths.py; here: the launch
structure, and that the one-sweep step solves the linearised system."""
import ctypes as C

import pytest

from paropt_b200 import configs

pytestmark = pytest.mark.gpu

VARS, RES, UPD = 0, 1, 2


@pytest.fixture(scope="module")
def ctx():
    from paropt_b200.api import Context
    c = Context(0)
    yield c
    c.close()


def launches_per_iteration(ctx, cfg, iters=3, warmup=2):
    from paropt_b200.api import InteriorPoint, problem_from_config
    prob = problem_from_config(ctx, cfg)
    ip = InteriorPoint(prob, dict(cfg["options"], max_major_iters=1000000))
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
def test_one_pass_applies_the_refined_step(ctx, n, staged):
    """C3 (c = 1, L-BFGS m = 10): per iteration no Pass2R1F, no Pass2SF, one Pass2SVF
    and one dense-kernel launch -- with the bulk-copy staged kernels forced on at a
    small size (every CTA wraps its stage ring) and at the full size."""
    cfg = configs.get("C3", n)
    if staged:
        ctx.set_param("tma_min_tiles", 1)
        ctx.set_param("tma_grid", 7)
    try:
        per_it = launches_per_iteration(ctx, cfg)
    finally:
        ctx.set_param("tma_min_tiles", 0)
        ctx.set_param("tma_grid", 0)
    assert per_it.get("Pass2R1F", 0) == 0, per_it
    assert per_it.get("Pass2SF", 0) == 0, per_it
    assert per_it.get("Pass2SVF", 0) == 1, per_it
    assert per_it.get("dense_kernel", 0) == 1, per_it


@pytest.mark.parametrize("on_device", [1, 0])
def test_column_space_refinement_solves_the_linearised_system(ctx, on_device):
    """At n = 64M, 4 iterations in (quasi-Newton pairs present): the step of the
    default route (dense algebra on the device, or on the host) leaves r - K p
    (addKKTResStep) at <= 1e-9 of r in the x, dual and infeasibility norms, the bound
    of test_kkt_step_solves_the_linearised_system_at_full_size."""
    from paropt_b200.api import InteriorPoint, problem_from_config
    cfg = configs.get("C3")
    prob = problem_from_config(ctx, cfg)
    ip = InteriorPoint(prob, dict(cfg["options"], max_major_iters=1000000))
    try:
        ip.begin()
        ip.iterate(4)
        mu = ip.getBarrierParameter()
        lib, h = ip.lib, ip.h

        def norms():
            v = [C.c_double() for _ in range(4)]
            assert lib.pcu_ip_res_norm(h, *[C.byref(a) for a in v]) == 0
            return [a.value for a in v]

        qn = C.c_int()
        assert lib.pcu_ip_qn_compact(h, None, C.byref(qn), None, None) == 0
        assert qn.value > 0
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
