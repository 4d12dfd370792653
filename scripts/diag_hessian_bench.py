#!/usr/bin/env python
"""The interior point on one sepquad workload with L-BFGS and with its exact diagonal
Hessian (use_diag_hessian), each run to convergence, the two arms alternating in one
process:

    python scripts/diag_hessian_bench.py --out RESULT.json [--config C3] [--n NTOTAL]
        [--rounds 2]

Per run: iterations, status, the time to solution (CUDA events on the context's stream
around optimize(): starting point + every iteration + the callbacks), ms per iteration
(the mean of the per-iteration CUDA-event times) and the KKT-solve ms per iteration.
The card's name, power limit and SM clocks are read before and after every run.  Both
arms use the workload's options; the objective and the final x of each run are reported
with the relative distance between the arms' final points.  Writes the JSON result to
--out (outside the source tree, e.g. a run's output directory) and prints it."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from paropt_b200 import configs  # noqa: E402


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


ARMS = {"lbfgs": {}, "diag_hessian": {"use_diag_hessian": 1}}


def one_run(ctx, cfg, extra):
    import numpy as np
    from paropt_b200.api import InteriorPoint, problem_from_config
    prob = problem_from_config(ctx, cfg)
    ip = InteriorPoint(prob, dict(cfg["options"], history_level=1, **extra))
    try:
        before = card()
        ctx.timer_start()
        ip.optimize()
        total_ms = ctx.timer_stop()
        after = card()
        niter = ip.counters()[0]
        times = ip.iter_times()
        hist = ip.history()
        x = ip.getOptimizedPoint()[0].to_numpy()
        return {
            "iterations": niter, "status": ip.status(), "fobj": hist[-1]["fobj"],
            "time_to_solution_ms": total_ms,
            "ms_per_iter": float(np.mean([t[0] for t in times])) if times else None,
            "kkt_ms_per_iter": float(np.mean([t[2] for t in times])) if times else None,
            "callback_ms_per_iter": float(np.mean([t[1] for t in times])) if times else None,
            "card_before": before, "card_after": after}, x
    finally:
        ip.free()
        prob.free()


def main():
    import numpy as np
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--config", default="C3")
    ap.add_argument("--n", type=int, default=None, help="global number of variables")
    ap.add_argument("--rounds", type=int, default=2, help="alternations of the two arms")
    ap.add_argument("--out", required=True, help="path of the JSON result file")
    args = ap.parse_args()
    cfg = configs.get(args.config, args.n)
    if cfg["kind"] != "sepquad":
        raise SystemExit("the built-in sepquad problems have the exact diagonal")
    from paropt_b200.api import Context
    ctx = Context(0)
    runs = {k: [] for k in ARMS}
    final = {}
    for r in range(args.rounds):
        for name, extra in ARMS.items():
            rec, x = one_run(ctx, cfg, extra)
            rec["round"] = r
            runs[name].append(rec)
            final[name] = x
            print("%-13s round %d: %4d iterations (%s), %.1f ms to solution, %.3f ms/iter"
                  % (name, r, rec["iterations"], rec["status"], rec["time_to_solution_ms"],
                     rec["ms_per_iter"]), file=sys.stderr)
    ctx.close()
    x0, x1 = final["lbfgs"], final["diag_hessian"]
    out = {"workload": args.config, "problem": cfg["problem"], "options": cfg["options"],
           "runs": runs,
           "final_x_rel_distance": float(np.linalg.norm(x1 - x0) / np.linalg.norm(x0))}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fp:
        json.dump(out, fp, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
