"""The drop-in boundary, compiled and run: the UNMODIFIED reference
ParOptInteriorPoint (objects of oracle/_ref, built from the upstream ParOpt sources
that PAROPT_REF names) drives the adapter classes of tests/adapters/paropt_cuda_adapters.h --
ParOptCudaVec : ParOptVec, ParOptCudaQuasiDefBlockMat : ParOptQuasiDefMat,
ParOptCudaCompactQN : ParOptCompactQuasiNewton -- injected through the reference's
own factories (createDesignVec / createConstraintVec / createQuasiDefMat,
src/ParOptProblem.h:58,65,72, and setQuasiNewton, IP.cpp:1193).  Every vector
operation, reduction, block-matrix factor / solve and quasi-Newton update / product
of that run executes in libparopt_b200.so on the GPU; the reference's raw-pointer
loops see the same storage through unified memory (pcu_vec_host_ptr).  The history
must follow the reference's own host run (tests/golden) under tests/parity.py."""
import json
import os
import subprocess

import pytest

from tests.parity import compare_histories, load_golden

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER = os.path.join(ROOT, "oracle", "_ref", "adapter_driver")


def run_adapter_driver(cfg, tmp_path):
    from oracle.make_golden import driver_args, parse_log
    hist = str(tmp_path / "hist.jsonl")
    log = str(tmp_path / "paropt.out")
    env = dict(os.environ, OPENBLAS_NUM_THREADS="1", PCU_SHIM_NP="1")
    out = subprocess.run([DRIVER] + driver_args(cfg) + ["hist=" + hist, "log=" + log],
                         env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    recs = [json.loads(line) for line in open(hist)]
    rows, status = parse_log(log)
    return ([r for r in recs if "iter" in r], [r for r in recs if "final" in r][0], rows,
            status, out.stderr)


# C3_nb2_small: two sparse constraints per block -- the reference's ParOptQuasiDefBlockMat
# with nwblock = 2 (packed-upper dpptrf / dpptrs) against pcu_blockmat_create_blocks.
# S1_small: a ParOptSparseProblem (general CSR sparse constraints, SURVEY.md section 8f-3) --
# the reference's ParOptQuasiDefSparseMat + sparse Cholesky against pcu_sparsemat
# (ParOptCudaQuasiDefSparseMat in oracle/ref_driver.cpp), the CSR products on the device.
@pytest.mark.parametrize("name,iters", [("C1_small", None), ("C2_small", None),
                                        ("C3_small", None), ("C4_small", 11),
                                        ("C3_nb2_small", 39), ("S1_small", None)])
def test_reference_interior_point_runs_on_cuda_vectors(tmp_path, name, iters):
    if not os.path.exists(DRIVER):
        pytest.skip("oracle/_ref/adapter_driver not built (build() needs PAROPT_REF = the "
                    "upstream ParOpt sources)")
    gold = load_golden(name)
    cfg = gold["config"]
    if iters is not None:
        cfg = dict(cfg, options=dict(cfg["options"], max_major_iters=iters + 1))
    hist, final, rows, status, err = run_adapter_driver(cfg, tmp_path)
    assert "reference ParOptInteriorPoint on ParOptCudaVec vectors" in err, err[-500:]
    launched = [int(ln.split()[1]) for ln in err.splitlines()
                if ln.startswith("adapter_driver:") and "kernels of libparopt_b200" in ln]
    assert launched and launched[0] > 100, err[-500:]
    n, worst, first = compare_histories(gold["history"], hist, max_iters=iters, cfg=gold["config"])
    assert first is None, (first, worst)
    if iters is None:  # full history: iteration count, counters, status, log tags
        assert n == len(gold["history"])
        for key in ("niter", "neval", "ngeval"):
            assert final[key] == gold["final"][key], key
        assert status == gold["status"]
        for a, b in zip(gold["log"], rows):
            assert a["info"] == b["info"], (a, b)
    else:
        assert n == iters
