"""CPU-side tests: the C ABI library loads and exports every symbol declared in
include/paropt_b200.h (no compute calls without a GPU), the host-side partition
logic, and the multi-rank host path over gloo (world_size 2)."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "paropt_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    names = set(re.findall(r"\b(pcu_[a-z0-9_]+)\s*\(", text))
    # typedef'd callback struct members are not exported symbols
    return sorted(n for n in names if not n.endswith("_callbacks"))


def test_library_exports_every_declared_symbol():
    from paropt_b200 import build
    lib_path = build.build()  # builds if stale (nvcc cross-compiles without a GPU)
    lib = ctypes.CDLL(lib_path)
    missing = [n for n in declared_symbols() if not hasattr(lib, n)]
    assert not missing, missing
    from paropt_b200 import _lib
    unbound = [n for n in declared_symbols() if n not in _lib.SIGNATURES]
    assert not unbound, unbound
    _lib.load()


def test_wide_gram_partition_covers_the_tile_triangle_once():
    """Host side of gram_wide_kernel (pcu_gram.cu, gram_wide_deal): for every width the
    kernel takes, the segments dealt to the consumer warps cover each pair of 8-column tiles
    (ti >= tj) exactly once, every warp holds n2u two-pair segments plus at most two optional
    ones, the loads differ by at most two pairs, and a last column alone in its tile
    (m = 8 k + 1) becomes a side column instead of a tile row (C4: m = 121 -> 15 tile rows,
    120 tile pairs, ten per warp)."""
    from paropt_b200 import _lib
    lib = _lib.load()
    I = ctypes.c_int
    taken = 0
    for m in range(41, 161):
        nt, n2u, side, warps, slots = I(), I(), I(), I(), I()
        probe = lib.pcu_gram_wide_plan(m, nt, n2u, side, warps, slots, None, None, None)
        assert warps.value > 0 and slots.value > 0
        if probe != 0:
            continue
        taken += 1
        size = warps.value * slots.value
        ti = (ctypes.c_ubyte * size)()
        tj = (ctypes.c_ubyte * size)()
        npairs = (ctypes.c_ubyte * size)()
        assert lib.pcu_gram_wide_plan(m, nt, n2u, side, warps, slots, ti, tj, npairs) == 0
        assert side.value == (1 if m % 8 == 1 else 0)
        assert nt.value == ((m - 1) // 8 if side.value else (m + 7) // 8)
        seen = set()
        loads = []
        for w in range(warps.value):
            load = 0
            for s_ in range(slots.value):
                k = w * slots.value + s_
                if npairs[k] == 0:
                    continue
                assert s_ < n2u.value + 2
                if s_ < n2u.value:
                    assert npairs[k] == 2
                for q in range(npairs[k]):
                    pair = (ti[k], tj[k] + q)
                    assert pair[1] <= pair[0] < nt.value, (m, pair)
                    assert pair not in seen, (m, pair)
                    seen.add(pair)
                load += npairs[k]
            loads.append(load)
        assert len(seen) == nt.value * (nt.value + 1) // 2, (m, len(seen))
        assert max(loads) - min(loads) <= 2, (m, loads)
        if m == 121:
            assert nt.value == 15 and loads == [10] * warps.value
    assert taken == 120  # every width from 41 to 160 columns


def test_library_is_sm100a_only():
    from paropt_b200 import build
    cuobjdump = os.path.join(os.path.dirname(build.NVCC), "cuobjdump")  # the toolkit that built it
    out = subprocess.run([cuobjdump, "-lelf", build.LIB], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_no_cuda_device_fails_loudly():
    """There is no CPU fallback: without a device context creation raises."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from paropt_b200.api import Context
    with pytest.raises(RuntimeError):
        Context(0)


def test_partition_matches_reference_block_rows():
    from oracle.problems import partition
    for ntotal, nw, size in [(1000, 0, 3), (16000, 8, 2), (64 * 1024 * 1024, 8, 8), (1001, 0, 4)]:
        off = 0
        tot_w = 0
        for rank in range(size):
            o, n, nwc = partition(ntotal, nw, rank, size)
            assert o == off
            if nw:
                assert o % nw == 0 and (n % nw == 0 or rank == size - 1)
            off += n
            tot_w += nwc
        assert off == ntotal
        assert tot_w == (ntotal // nw if nw else 0)


def test_generator_is_partition_independent():
    from oracle.problems import SepQuad

    class FakeComm:
        def __init__(self, rank, size):
            self.rank, self.size = rank, size

        def allreduce(self, arr, op="sum"):
            return np.asarray(arr, dtype=np.float64)

    full = SepQuad(ntotal=4096, ncon=2, nw=8)
    parts = [SepQuad(comm=FakeComm(r, 2), ntotal=4096, ncon=2, nw=8) for r in range(2)]
    np.testing.assert_array_equal(full.lam, np.concatenate([p.lam for p in parts]))
    np.testing.assert_array_equal(full.A[1], np.concatenate([p.A[1] for p in parts]))
    x, lb, ub = (np.zeros(4096) for _ in range(3))
    full.getVarsAndBounds(x, lb, ub)
    xs = []
    for p in parts:
        a, b, c = (np.zeros(p.nvars) for _ in range(3))
        p.getVarsAndBounds(a, b, c)
        xs.append(a)
    np.testing.assert_array_equal(x, np.concatenate(xs))


WORKER = r"""
import json, os, sys
sys.path.insert(0, %(root)r)
import torch.distributed as dist
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%(port)d",
                        rank=int(sys.argv[1]), world_size=2)
from oracle.ip_oracle import InteriorPointOracle, TorchComm
from oracle.problems import SepQuad
from tests.parity import load_golden
gold = load_golden(%(name)r)
comm = TorchComm()
cfg = gold["config"]
ip = InteriorPointOracle(SepQuad(comm=comm, **cfg["problem"]),
                         dict(cfg["options"], max_major_iters=%(iters)d), comm=comm)
ip.optimize()
if comm.rank == 0:
    json.dump(ip.history, open(%(out)r, "w"))
dist.destroy_process_group()
"""


@pytest.mark.parametrize("name,iters", [("C2_small", 12), ("C3_small", 12)])
def test_two_rank_gloo_oracle_matches_reference(tmp_path, name, iters):
    """Host-side multi-rank logic (block-row partition, rank-local weighting
    constraints, small allreduces) over torch.distributed/gloo, world_size 2,
    against the reference run with 2 ranks (golden *_np2) and with 1 rank."""
    import json
    from tests.parity import compare_histories, load_golden
    out = tmp_path / "hist.json"
    port = 29500 + (os.getpid() % 2000)
    script = tmp_path / "worker.py"
    script.write_text(WORKER % dict(root=ROOT, port=port, name=name, iters=iters + 1,
                                    out=str(out)))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)]) for r in range(2)]
    for p in procs:
        assert p.wait(timeout=600) == 0
    hist = json.load(open(out))
    for gname in (name + "_np2", name):
        gold = load_golden(gname)
        n, worst, first = compare_histories(gold["history"], hist, max_iters=iters, cfg=gold["config"])
        assert n == iters and first is None, (gname, first, worst)


def test_unpack_output_reads_the_fixed_width_log(tmp_path):
    """paropt_b200.ParOpt.unpack_output parses the reference's iteration rows
    (IP.cpp:4777-4801: four %4d, then %7.1e / %12.5e columns, one blank between)."""
    ParOpt = pytest.importorskip("paropt_b200.ParOpt")
    rows = [(0, 1, 1, 0, 0.0, 0.0, 0.0, 1.234567e+03, 1.2e+01, 3.4e-02, 5.6e+00, 1.0e-01, 9.9e-01,
             -1.2e+00, 0.0),
            (1, 2, 2, 0, 1.0, 9.5e-01, 8.1e-01, -7.65432e-01, 2.2e+00, 1.4e-03, 6.6e-01, 1.0e-01,
             8.8e-01, -3.4e-01, 1.5e+02)]
    path = tmp_path / "paropt.out"
    with open(path, "w") as fp:
        fp.write("ParOpt: Parameter summary\n\n")
        fp.write("iter nobj ngrd nhvc   alpha   alphx   alphz         fobj   |opt| |infes|  |dual|      mu"
                 "    comp   dmerit     rho info\n")
        for r in rows:
            fp.write("%4d %4d %4d %4d %7.1e %7.1e %7.1e %12.5e %7.1e %7.1e %7.1e %7.1e %7.1e %8.1e %7.1e %s\n"
                     % (r + ("skipH",)))
    names, cols = ParOpt.unpack_output(str(path))
    assert names[7] == "fobj" and len(cols) == 15
    assert list(cols[0]) == [0, 1] and list(cols[2]) == [1, 2]
    assert abs(cols[7][0] - 1.23457e+03) < 1e-2 and abs(cols[7][1] + 7.65432e-01) < 1e-6
    assert abs(cols[13][1] + 3.4e-01) < 1e-9 and abs(cols[14][1] - 1.5e+02) < 1e-9


def test_header_is_plain_c(tmp_path):
    """The drop-in boundary is a C ABI: include/paropt_b200.h must compile as C99
    (no C++ or CUDA types in the signatures) and every prototype must link."""
    import subprocess
    src = tmp_path / "abi.c"
    src.write_text('#include "paropt_b200.h"\n'
                   "int main(void) { return pcu_version() == 0; }\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-fsyntax-only",
                    "-I", os.path.join(root, "include"), str(src)], check=True)


def test_adapter_driver_links_against_the_product_library():
    """oracle/_ref/adapter_driver (the reference running on the CUDA adapter classes,
    tests/adapters/paropt_cuda_adapters.h) is linked against libparopt_b200.so and
    resolves the C-ABI symbols the adapters call -- no compute here (no GPU)."""
    drv = os.path.join(ROOT, "oracle", "_ref", "adapter_driver")
    if not os.path.exists(drv):
        pytest.skip("adapter_driver not built (build() needs PAROPT_REF = the upstream ParOpt "
                    "sources)")
    out = subprocess.run(["ldd", drv], capture_output=True, text=True).stdout
    assert "libparopt_b200.so" in out and "not found" not in out, out
    syms = subprocess.run(["nm", "-D", "--undefined-only", drv], capture_output=True,
                          text=True).stdout
    for name in ("pcu_vec_host_ptr", "pcu_vec_mdot", "pcu_blockmat_factor", "pcu_qn_update",
                 "pcu_qn_compact", "pcu_ctx_set_param"):
        assert name in syms, name
