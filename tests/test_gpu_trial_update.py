"""The line search's first trial point is taken by the update pass itself (TrialUpdateF =
Update1FT<1, 1>, pcu_kernels.cuh): it writes the new point and multipliers into the
trial buffers, takes TrialF's merit sums, and on acceptance the buffers are exchanged
with the variables instead of running TrialF and then Update1FT.  PCU_NO_TRIALUPD
selects the separate TrialF + Update1FT sequence, the reference of these tests."""
import os

import numpy as np
import pytest

from paropt_b200 import configs
from tests.parity import compare_histories, load_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from paropt_b200.api import Context
    c = Context(0)
    yield c
    c.close()


def launches_per_iteration(ctx, cfg, iters=3, warmup=2):
    """Launches per iteration by full kernel name (Update1FT<1, 0> and TrialUpdateF
    apart)."""
    from paropt_b200.api import InteriorPoint, problem_from_config
    prob = problem_from_config(ctx, cfg)
    ip = InteriorPoint(prob, dict(cfg["options"], max_major_iters=1000000))
    try:
        ip.begin()
        ip.iterate(warmup)
        ctx.profile(2)
        ip.iterate(iters)
        ctx.profile(0)
        counts = dict((name, cnt) for name, (_, cnt) in ctx.profile_totals().items())
    finally:
        ctx.profile(0)
        ip.free()
        prob.free()
    return {k: v / iters for k, v in counts.items()}


@pytest.mark.parametrize("n,staged", [(8 * 5003, True), (None, False)])
def test_update_pass_replaces_the_first_trial(ctx, n, staged):
    """C3 (every first trial accepted): per iteration one TrialUpdateF and one Pass2SVF,
    no TrialF and no stand-alone Update1FT -- with the bulk-copy staged kernels forced
    on at a small size and at the full size."""
    cfg = configs.get("C3", n)
    if staged:
        ctx.set_param("tma_min_tiles", 1)
        ctx.set_param("tma_grid", 7)
    try:
        per_it = launches_per_iteration(ctx, cfg)
    finally:
        ctx.set_param("tma_min_tiles", 0)
        ctx.set_param("tma_grid", 0)
    assert per_it.get("TrialUpdateF", 0) == 1, per_it
    assert per_it.get("Pass2SVF", 0) == 1, per_it
    assert per_it.get("TrialF", 0) == 0, per_it
    assert not any(k.startswith("Update1FT") for k in per_it), per_it


def run(ctx, cfg, iters, separate, extra=None):
    from paropt_b200.api import InteriorPoint, problem_from_config
    if separate:
        os.environ["PCU_NO_TRIALUPD"] = "1"
    try:
        prob = problem_from_config(ctx, cfg)
        opts = dict(cfg["options"], history_level=2, **(extra or {}))
        if iters is not None:
            opts["max_major_iters"] = iters
        ip = InteriorPoint(prob, opts)
        ip.optimize()
        x, z, zw, zl, zu = ip.getOptimizedPoint()
        out = dict(history=ip.history(), status=ip.status(), counters=ip.counters(),
                   point=[x.to_numpy(), np.asarray(z), zw.to_numpy(), zl.to_numpy(),
                          zu.to_numpy()])
        ip.free()
        prob.free()
    finally:
        os.environ.pop("PCU_NO_TRIALUPD", None)
    return out


# C1 (Rosenbrock) and its back-tracking variant reject first trials: the update pass's
# results are dropped, the later trials run TrialF and the accepted point the stand-alone
# Update1FT, and the next first trial is TrialF too.  C4: L-SR1, reproducible for 11
# iterations.
@pytest.mark.parametrize("name,iters,extra", [
    ("C1_small", None, None), ("C1_var_backtrack", None, None), ("C2_small", None, None),
    ("C3_small", None, None), ("C3_small", None, dict(use_diag_hessian=1)),
    ("C4_small", 12, None)])
def test_history_matches_separate_trial_and_update(ctx, name, iters, extra):
    """Same point, same multipliers, same statistics; the merit sums are taken over
    other tiles (last-bit differences): the two histories agree to 1e-12 with the same
    evaluation counts and line-search flags, and so do the final points."""
    cfg = load_golden(name)["config"]
    fused = run(ctx, cfg, iters, False, extra)
    sep = run(ctx, cfg, iters, True, extra)
    if name.startswith("C1"):
        # the rejection path is exercised: some line search evaluated more than one trial
        nev = [h["neval"] for h in sep["history"]]
        assert any(b - a > 1 for a, b in zip(nev, nev[1:])), nev
    nh = len(sep["history"]) if iters is None else iters - 1
    cnt, worst, first = compare_histories(sep["history"], fused["history"], max_iters=nh,
                                          cfg=cfg, rtol=1e-12)
    assert cnt == nh and first is None, (first, worst)
    for a, b in list(zip(fused["history"], sep["history"]))[:nh]:
        assert a["info"] == b["info"] and a["neval"] == b["neval"], (a["iter"], a["info"], b["info"])
    if iters is None:
        assert fused["status"] == sep["status"] and fused["counters"] == sep["counters"]
        for a, b in zip(fused["point"], sep["point"]):
            np.testing.assert_allclose(a, b, rtol=1e-12, atol=0.0)


def test_final_point_through_exchanged_buffers_is_bit_identical(ctx):
    """C3_small, every first trial accepted: x, zl, zu, zw live in the exchanged trial
    buffers at the end, and read through pcu_ip_get_point they equal the separate
    sequence's bit for bit (same step_clip expressions, same operands)."""
    cfg = load_golden("C3_small")["config"]
    fused = run(ctx, cfg, 20, False)
    sep = run(ctx, cfg, 20, True)
    for a, b in zip(fused["point"], sep["point"]):
        assert np.array_equal(a, b)
