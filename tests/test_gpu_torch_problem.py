"""Python problems on the device: TorchProblem / AutogradProblem (paropt_b200/api.py)
whose callbacks are torch code on zero-copy views of the optimizer's vectors, run on
the optimizer's stream.  The problems are the workloads of oracle/problems.py
(tests/torch_problems.py); histories are compared with the unmodified reference's
(tests/golden) under tests/parity.py (RTOL = 1e-10)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.parity import compare_histories, load_golden

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ctx():
    from paropt_b200.api import Context
    c = Context(0)
    yield c
    c.close()


def run_ip(prob, cfg, **extra):
    from paropt_b200.api import InteriorPoint
    ip = InteriorPoint(prob, dict(cfg["options"], history_level=2, **extra))
    ip.optimize()
    out = dict(history=ip.history(), status=ip.status(), counters=ip.counters())
    ip.free()
    return out


def check_full(gold, out):
    n, worst, first = compare_histories(gold["history"], out["history"], cfg=gold["config"])
    assert first is None, (first, worst)
    assert n == len(gold["history"]) == len(out["history"])
    niter, neval, ngeval = out["counters"]
    assert (niter, neval, ngeval) == (gold["final"]["niter"], gold["final"]["neval"],
                                      gold["final"]["ngeval"])
    assert out["status"] == gold["status"]
    for row, rec in zip(gold["log"], out["history"]):
        assert row["info"] == rec["info"], (row, rec["iter"])


def test_rosenbrock_matches_reference_without_host_copies(ctx):
    from tests.torch_problems import make
    gold = load_golden("C1_small")
    prob = make(ctx, gold["config"])
    out = run_ip(prob, gold["config"])
    check_full(gold, out)
    assert prob.h2d_bytes == 0 and prob.d2h_bytes == 0
    assert prob.callback_ms() > 0.0
    prob.free()


@pytest.mark.parametrize("name", ["C2_small", "C3_small"])
def test_sepquad_matches_reference(ctx, name):
    from tests.torch_problems import make
    gold = load_golden(name)
    prob = make(ctx, gold["config"])
    out = run_ip(prob, gold["config"])
    check_full(gold, out)
    assert prob.transfer_bytes() == (0, 0)
    prob.free()


@pytest.mark.parametrize("autograd", [False, True])
def test_hessian_vector_products_match_reference(ctx, autograd):
    """Inexact-Newton GMRES steps (use_hvec_product) with the torch problem's
    evalHvecProduct: written out, or the double backward of AutogradProblem."""
    from tests.torch_problems import make
    gold = load_golden("C2_var_gmres")
    prob = make(ctx, gold["config"], autograd=autograd)
    out = run_ip(prob, gold["config"])
    prob.free()
    check_full(gold, out)
    assert [r["nhvec"] for r in gold["history"]] == [r["nhvec"] for r in out["history"]]
    assert out["history"][-1]["nhvec"] > 0


def test_autograd_problem_matches_reference_and_explicit_gradients(ctx):
    import torch
    from tests.torch_problems import make
    gold = load_golden("C2_small")
    cfg = gold["config"]
    prob = make(ctx, cfg, autograd=True)
    out = run_ip(prob, cfg)
    check_full(gold, out)
    # the gradients at the starting point against the explicit ones
    explicit = make(ctx, cfg)
    n, c = prob.nvars, prob.ncon
    dev = prob.device
    x = prob.data["x0"].clone()
    got = [torch.empty(n, dtype=torch.float64, device=dev) for _ in range(c + 1)]
    ref = [torch.empty(n, dtype=torch.float64, device=dev) for _ in range(c + 1)]
    assert prob.evalObjConGradient(x, got[0], got[1:]) == 0
    assert explicit.evalObjConGradient(x, ref[0], ref[1:]) == 0
    for k, (a, b) in enumerate(zip(got, ref)):
        err = float(torch.max(torch.abs(a - b))) / float(torch.max(torch.abs(b)))
        assert err <= 1e-13, (k, err)
    # the objective and constraints agree too
    _, f0, c0 = prob.evalObjCon(x)
    _, f1, c1 = explicit.evalObjCon(x)
    assert abs(float(f0) - float(f1)) <= 1e-13 * abs(float(f1))
    assert torch.allclose(c0, c1, rtol=1e-13, atol=0.0)
    explicit.free()
    prob.free()


def test_trust_region_matches_reference(ctx):
    """ParOpt.Optimizer with algorithm = "tr" on the torch Rosenbrock, compared as
    tests/test_gpu_tr.py compares the built-in one."""
    from paropt_b200 import ParOpt
    from tests.test_gpu_tr import CENTRE_RTOL
    from tests.torch_problems import make
    gold = load_golden("C1_tr")
    prob = make(ctx, gold["config"])
    opt = ParOpt.Optimizer(prob, dict(gold["config"]["options"], algorithm="tr",
                                      tr_write_output_frequency=1))
    opt.optimize()
    hist = opt.tr.history()
    assert opt.tr.converged()
    assert len(hist) == len(gold["log"]) == len(gold["centres"])
    for k, (h, row, c) in enumerate(zip(hist, gold["log"], gold["centres"])):
        assert h["info"] == row["info"], (k, h["info"], row["info"])
        for key in ("xsum", "xnorm", "xmaxabs"):
            err = abs(h[key] - c[key]) / max(abs(c[key]), c["xnorm"], 1e-300)
            assert err <= CENTRE_RTOL, (k, key, h[key], c[key], err)
    x = opt.getOptimizedPoint()[0].to_numpy()
    final = gold["final"]
    assert abs(float(np.sum(x)) - final["xsum"]) <= CENTRE_RTOL * max(abs(final["xsum"]),
                                                                     final["xnorm"])
    assert prob.transfer_bytes() == (0, 0)
    opt.tr.free()
    prob.free()


def test_write_output_and_quasi_newton_correction_hooks(ctx):
    from tests.torch_problems import TorchSepQuad
    gold = load_golden("C2_small")
    cfg = gold["config"]
    freq = 4

    class Hooked(TorchSepQuad):
        def __init__(self, *a, **k):
            self.seen, self.corrections = [], 0
            super().__init__(*a, **k)

        def writeOutput(self, it, x):
            self.seen.append((it, float(x.sum())))

        def computeQuasiNewtonUpdateCorrection(self, x, z, zw, s, y):
            assert len(z) == self.ncon and zw.numel() == 0
            self.corrections += 1
            return 0

    prob = Hooked(ctx, **cfg["problem"])
    out = run_ip(prob, cfg, write_output_frequency=freq)
    check_full(gold, out)
    hist = {r["iter"]: r for r in out["history"]}
    its = [it for it, _ in prob.seen]
    assert its == [k for k in sorted(hist) if k % freq == 0], its
    for it, xsum in prob.seen:
        ref = hist[it]["xsum"]
        assert abs(xsum - ref) <= 1e-12 * max(abs(ref), hist[it]["xnorm"]), (it, xsum, ref)
    # one correction per quasi-Newton update: one per gradient after the first
    assert prob.corrections == out["counters"][2] - 1, (prob.corrections, out["counters"])
    prob.free()


def test_callbacks_wait_for_the_callers_stream(ctx):
    """Problem data rewritten on torch's default stream right before optimize(),
    without a synchronisation: the callbacks on the optimizer's stream see the new
    values (the fill is held back by a spin kernel so that it is still running when
    the first callback starts)."""
    import torch
    from paropt_b200.api import InteriorPoint
    from tests.torch_problems import TorchSepQuad
    gold = load_golden("C3_small")
    cfg = gold["config"]
    prob = TorchSepQuad(ctx, **cfg["problem"])
    ip = InteriorPoint(prob, dict(cfg["options"], history_level=2))
    good = {k: v.clone() for k, v in prob.data.items() if v is not None}
    good_A = [a.clone() for a in prob.A]
    for v in list(prob.data.values()) + prob.A:
        if v is not None:
            v.fill_(0.5)
    torch.cuda.synchronize()
    default = torch.cuda.default_stream(prob.device)
    with torch.cuda.stream(default):
        torch.cuda._sleep(50_000_000)  # ~25 ms of spinning ahead of the fill
        for k, v in good.items():
            prob.data[k].copy_(v)
        for a, v in zip(prob.A, good_A):
            a.copy_(v)
        assert not default.query()  # the fill is still pending
        ip.optimize()
    out = dict(history=ip.history(), status=ip.status(), counters=ip.counters())
    ip.free()
    prob.free()
    check_full(gold, out)


def test_callback_exception_raises_and_context_stays_usable(ctx):
    from paropt_b200.api import InteriorPoint
    from tests.torch_problems import TorchRosenbrock, make
    gold = load_golden("C1_small")

    class Broken(TorchRosenbrock):
        it = 0

        def writeOutput(self, it, x):
            self.it = it

        def evalObjCon(self, x):
            if self.it >= 3:
                raise ValueError("objective not available at iteration %d" % self.it)
            return super().evalObjCon(x)

    prob = Broken(ctx, **gold["config"]["problem"])
    ip = InteriorPoint(prob, dict(gold["config"]["options"], write_output_frequency=1,
                                  history_level=1))
    with pytest.raises(RuntimeError, match="ValueError"):
        ip.optimize()
    assert ip.history()[-1]["iter"] <= 4
    ip.free()
    prob.free()
    prob = make(ctx, gold["config"])
    out = run_ip(prob, gold["config"])
    prob.free()
    check_full(gold, out)


def test_first_iterations_match_reference_at_full_size(ctx):
    import torch
    from tests.torch_problems import make
    if torch.cuda.get_device_properties(0).total_memory < 60e9:
        pytest.skip("needs a 64 GB+ GPU")
    gold = load_golden("C3_full")
    cfg = gold["config"]
    iters = 12
    prob = make(ctx, cfg)
    out = run_ip(prob, cfg, max_major_iters=iters + 1)
    prob.free()
    n, worst, first = compare_histories(gold["history"], out["history"], max_iters=iters, cfg=cfg)
    assert n == iters and first is None, (first, worst)
    for row, rec in zip(gold["log"][:iters], out["history"]):
        assert row["info"] == rec["info"], (row, rec["iter"])


def test_two_gpu_history_matches_reference():
    import json
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    port = 29700 + (os.getpid() % 1000)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(ROOT, "scripts", "torch_problem_mgpu.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [ln for ln in out.stdout.splitlines() if ln.startswith("TORCH_MGPU ")][-1]
    verdict = json.loads(line[len("TORCH_MGPU "):])
    assert verdict["world"] == 2 and verdict["compared"] == verdict["rows"]
    assert verdict["first_violation"] is None, verdict
    assert verdict["transfer_bytes"] == [0, 0]
