#!/usr/bin/env python
"""Interior-point iterations/s of one workload through three kinds of problem, timed
in alternation in one process:

  builtin  the library's CUDA sepquad (pcu_problem_create_sepquad)
  torch    the same problem as a TorchProblem (tests/torch_problems.py: torch
           callbacks on zero-copy views of the optimizer's vectors, its stream)
  numpy    the same problem as a numpy api.Problem (oracle/problems.py callbacks on
           the library's pinned host mirrors) -- a reference point, a few iterations

    python scripts/torch_problem_bench.py --out RESULT.json [--config C3] [--n NTOTAL]
        [--iters 20] [--rounds 2] [--numpy-iters 3]

Per arm: iterations/s from CUDA events on the context's stream around a window of
`iters` iterations after the L-BFGS memory is full (the numpy arm: after two
iterations), callback ms per iteration (events around the callbacks), bytes moved
between host and device per iteration, and the card's name, power limit and SM clock
read around the timed windows.  Writes the JSON result to --out (outside the source
tree, e.g. a run's output directory) and prints it."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from paropt_b200 import configs  # noqa: E402

QN_WARMUP = 12  # iterations until the L-BFGS memory (m = 10) is full


def card(index=0):
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=" + q,
                              "--format=csv,noheader,nounits"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        name, power, sm, sm_max = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit_w": float(power), "sm_mhz": float(sm),
                "sm_max_mhz": float(sm_max)}
    except Exception as e:  # the numbers are reported without the card, never silently
        return {"error": "nvidia-smi query failed: %s" % e}


def numpy_problem(ctx, ref, weighting):
    from paropt_b200.api import Problem

    class NumpySepQuad(Problem):
        def getVarsAndBounds(self, x, lb, ub):
            ref.getVarsAndBounds(x, lb, ub)

        def evalObjCon(self, x):
            return ref.evalObjCon(x)

        def evalObjConGradient(self, x, g, A):
            return ref.evalObjConGradient(x, g, A)

        def transfer_bytes(self):
            return self.h2d_bytes, self.d2h_bytes

    return NumpySepQuad(ctx, ref.nvars, ref.ncon, ninequality=ref.ncon,
                        nwinequality=ref.nwcon, weighting=weighting)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--config", default="C3")
    ap.add_argument("--n", type=int, default=None, help="global number of variables")
    ap.add_argument("--iters", type=int, default=20, help="timed iterations per window")
    ap.add_argument("--rounds", type=int, default=2, help="alternations of the arms")
    ap.add_argument("--numpy-iters", type=int, default=3,
                    help="timed iterations of the numpy arm (0: leave it out)")
    ap.add_argument("--out", required=True, help="path of the JSON result file")
    args = ap.parse_args()

    cfg = configs.get(args.config, args.n)
    if cfg["kind"] != "sepquad":
        raise SystemExit("the torch_problem benchmark runs the sepquad workloads")
    # host-side inputs first: the seeded generators of oracle/problems.py
    from oracle.problems import SepQuad
    from tests.torch_problems import weighting_dict
    ref = SepQuad(**cfg["problem"])
    weighting = weighting_dict(ref.weighting) if ref.nwcon > 0 else None
    print("workload %s: n = %d, ncon = %d, nwcon = %d" % (args.config, ref.nvars, ref.ncon,
                                                          ref.nwcon), file=sys.stderr)

    from paropt_b200.api import BuiltinProblem, Context, InteriorPoint
    from tests.torch_problems import TorchSepQuad
    ctx = Context(0)
    arms = {"builtin": BuiltinProblem(ctx, "sepquad", **cfg["problem"]),
            "torch": TorchSepQuad(ctx, **cfg["problem"])}
    if args.numpy_iters > 0:
        arms["numpy"] = numpy_problem(ctx, ref, weighting)
    ips, res = {}, {}
    for name, prob in arms.items():
        ip = InteriorPoint(prob, dict(cfg["options"], max_major_iters=1000000, history_level=1))
        ip.begin()
        ip.iterate(QN_WARMUP if name != "numpy" else 2)
        ips[name] = ip
        res[name] = {"iters": 0, "ms": 0.0, "callback_ms": 0.0, "h2d_bytes": 0, "d2h_bytes": 0,
                     "windows": []}
    cards = [card()]
    for r in range(args.rounds):
        for name, prob in arms.items():
            if name == "numpy" and r > 0:
                continue
            ip = ips[name]
            steps = args.numpy_iters if name == "numpy" else args.iters
            h0 = prob.transfer_bytes() if hasattr(prob, "transfer_bytes") else (0, 0)
            i0 = ip.counters()[0]
            t0 = len(ip.iter_times())
            ctx.timer_start()
            ip.iterate(steps)
            ms = ctx.timer_stop()
            done = ip.counters()[0] - i0
            h1 = prob.transfer_bytes() if hasattr(prob, "transfer_bytes") else (0, 0)
            cb = sum(t[1] for t in ip.iter_times()[t0:])
            a = res[name]
            a["iters"] += done
            a["ms"] += ms
            a["callback_ms"] += cb
            a["h2d_bytes"] += h1[0] - h0[0]
            a["d2h_bytes"] += h1[1] - h0[1]
            a["windows"].append({"iters": done, "iters_per_s": done / (ms / 1e3) if ms else 0.0})
        cards.append(card())
    out = {"workload": args.config, "nvars": ref.nvars, "ncon": ref.ncon, "nwcon": ref.nwcon,
           "card": cards, "arms": {}}
    for name, a in res.items():
        n = max(a["iters"], 1)
        out["arms"][name] = {
            "iters_per_s": a["iters"] / (a["ms"] / 1e3) if a["ms"] else 0.0,
            "ms_per_iter": a["ms"] / n, "callback_ms_per_iter": a["callback_ms"] / n,
            "h2d_bytes_per_iter": a["h2d_bytes"] // n, "d2h_bytes_per_iter": a["d2h_bytes"] // n,
            "timed_iters": a["iters"], "windows": a["windows"]}
    out["arms"]["torch"]["transfer_bytes_total"] = list(arms["torch"].transfer_bytes())
    for ip in ips.values():
        ip.free()
    for prob in arms.values():
        prob.free()
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fp:
        json.dump(out, fp, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
