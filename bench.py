#!/usr/bin/env python
"""bench.py -- interior-point iterations/s and KKT-solve ms at n = 64M (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--config C3] [--n NTOTAL] [--dump-outputs DIR]

A "step" is one pass of the interior-point major loop (IP.cpp:4607-5329) on the
named synthetic workload (default: configs[2] of BASELINE.json -- multi-material
topology-style problem, n = 64M, nwcon = 8M, 1 dense constraint, L-BFGS m = 10).
Multi-GPU runs shard the design vector exactly as the reference shards it over
MPI ranks (strong scaling: the global n stays 64M).

Prints ONE JSON line (rank 0).  Extra keys: `roofline` (dominant kernel, measured
live with CUDA events on the launching stream), `cpu_baseline` (the unmodified
reference compiled in oracle/_ref, timed on a bounded sample on the host cores),
`e2e` (same metric through the host-callback API: the iterate goes device->host
and the gradients host->device through pinned buffers on every callback),
`kkt_solve_ms`, `iter_roofline_frac`, `clocks`, `gpu_launches`.

--dump-outputs DIR writes the optimizer's point after the last timed step as
DIR/<name>.npy (float64): x, zl, zu, zw, sw, tw (at DUMP_SAMPLE sorted indices drawn
with a fixed seed when longer) and the dense z, s, t, zs, zt, c.  The
workloads are seeded, so two builds run with the same arguments can be compared
output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from
# stdout carries exactly one JSON line: libraries that write to file descriptor 1
# (NCCL prints its version banner there) are sent to stderr, the line goes to the
# saved descriptor
_REAL_STDOUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(line):
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


from paropt_b200 import configs  # noqa: E402

METRIC = "interior_point_iterations_per_sec"
UNIT = "iterations/s"
QN_WARMUP = 12  # iterations until the L-BFGS memory (m = 10) is full


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fp:
            return float(json.load(fp)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def measured_fp64_tflops():
    """cuBLAS DGEMM burst peak measured on this pool's B200 (scripts/measure_fp64_peak.py):
    the denominator of the FP64-tensor roofline of the Gram pass (MEASURED_PEAKS.json has
    no fp64 figure)."""
    path = os.path.join(ROOT, "profiles", "r2b_fp64_peak.json")
    try:
        with open(path) as fp:
            return float(json.load(fp)["fp64_dgemm_tflops_burst"]), "measured (profiles/r2b_fp64_peak.json, cuBLAS DGEMM 8192^3)"
    except Exception:
        return 40.0, "fallback (nominal B200 fp64 tensor peak)"


# ---------------------------------------------------------------- clocks
class ClockSampler:
    """Samples nvidia-smi while the timed region runs (B200_PROFILING.md)."""

    def __init__(self, index=0):
        self.index = index
        self.lines = []
        self.proc = None
        self.thread = None

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                smax = float(parts[2])
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        med = sm[len(sm) // 2] if sm else None
        return {"sm_mhz": med, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------ algorithmic traffic
def kernel_words(name, N, W, c, q):
    """Algorithmic fp64 words per launch of each kernel (DESIGN.md section 4)."""
    m = c + q
    table = {
        "ResF": (9 + c) * N + 10 * W,
        "DiagF": 6 * N + 5 * W,
        "DiagRhsF": (8 + c) * N + 7 * W,                    # DiagF + d1, d2 of the first solve
        "Pass1F": 9 * N + 11 * W,
        "Pass1RF": (8 + m) * N + 11 * W,
        "Pass1VF": (9 + c + m) * N + 7 * W,
        "Pass2F": (12 + m) * N + 15 * W + 3 * N + 5 * W,   # the accumulating refinement solve
        "Pass2RF": (16 + m) * N + 30 * W,                   # pass 2 + refinement residual
        "Pass2R1F": (14 + m) * N + 30 * W,                  # ... + first half of the next solve
        "Pass2SF": (16 + m) * N + 20 * W,                   # accumulating pass 2 + step statistics (g)
        "Pass2R1W": (15 + m) * N,                           # Pass2R1F on the column-split staged kernel (+ A p_z)
        "Pass2SW": (17 + m) * N,                            # Pass2SF likewise
        "StatsF": 9 * N + 8 * W,
        "TrialF": 5 * N + 6 * W,
        "Update1F": (10 + c) * N + 15 * W,
        "Update2F": (5 + c) * N + W,
        "Update1FT": (10 + c) * N + 15 * W,                 # <1>: + next iteration's statistics, no extra traffic
        "Update2FT": (7 + c) * N + W,                       # <1>: + zl, zu for |rx| of the next iteration
        "dense_kernel": None,
        "gram_kernel": (m + 2) * N + 2 * W,                 # [A|Z|d1] columns + Dinv; Cw, d2
        "mdot_kernel": None,  # (1 + columns of the chunk) N, see below
    }
    name = name.split("<")[0]
    if name == "ResFT":  # ResF with has_step / norm_type fixed at compile time
        name = "ResF"
    return table.get(name)


def iteration_words(N, W, c, q):
    """BASELINE.md section 4: algorithmic words per interior-point iteration."""
    return (200 + 16 * c + 9 * q) * N + 238 * W


def kkt_words(N, W, c, q):
    return (51 + 5 * c + 3 * q) * N + 62 * W


# ------------------------------------------------------------------ outputs
DUMP_SAMPLE = 1 << 20  # entries kept per vector: six vectors stay below 64 MB in float64


def dump_outputs(ip, outdir):
    """Writes the optimizer's current point (getOptimizedPoint / getOptimizedSlacks)
    as outdir/<name>.npy, float64 (see the module docstring)."""
    import ctypes as C

    import numpy as np
    from paropt_b200.api import PVec

    os.makedirs(outdir, exist_ok=True)
    handles = [C.c_void_p() for _ in range(6)]
    ip.lib.pcu_ip_get_point(ip.h, *[C.byref(h) for h in handles])
    arrays = ip.get_dense()
    for name, h in zip(("x", "zw", "zl", "zu", "sw", "tw"), handles):
        if not h.value:
            continue
        a = PVec(ip.ctx, handle=h.value).to_numpy()
        if a.size > DUMP_SAMPLE:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))]
        arrays[name] = a
    for name, a in arrays.items():
        np.save(os.path.join(outdir, name + ".npy"), np.asarray(a, dtype=np.float64))


# ---------------------------------------------------------------- reference
def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_ref_driver(cfg, nranks, timeout=1200):
    """Runs the unmodified reference (oracle/_ref/ref_driver) and returns the
    per-iteration records (with wall-clock stamps) and the final record."""
    sys.path.insert(0, ROOT)
    from oracle.make_golden import DRIVER, driver_args  # checker side (cpu baseline leg)

    if not os.path.exists(DRIVER):
        return None, None
    env = dict(os.environ)
    env["OPENBLAS_NUM_THREADS"] = "1"
    env["PCU_SHIM_NP"] = str(nranks)
    with tempfile.TemporaryDirectory() as tmp:
        hist = os.path.join(tmp, "hist.jsonl")
        cmd = [DRIVER] + driver_args(cfg) + ["hist=" + hist, "log=/dev/null"]
        subprocess.run(cmd, check=True, env=env, stdout=subprocess.DEVNULL, timeout=timeout)
        recs = [json.loads(line) for line in open(hist)]
    return [r for r in recs if "iter" in r], [r for r in recs if "final" in r][0]


def reference_full_size(cfg_name, ntotal, warmup, steps, timed_budget_s=150.0,
                        total_budget_s=420.0):
    """The reference arm at the metric's OWN configuration: the unmodified reference
    (oracle/_ref/ref_driver) at the full `ntotal`, one shim rank per host core.  The
    driver stamps every major iteration with its wall clock; the run is stopped once
    `steps` iterations after the warm-up are on record, or -- so that the arm ends
    within a few minutes on any host -- once the timed region has lasted
    `timed_budget_s` (at least 3 timed iterations are always taken)."""
    import signal
    from oracle.make_golden import DRIVER, driver_args  # checker side (reference arm)

    if not os.path.exists(DRIVER):
        return None
    cores = host_cores()
    nranks = max(1, min(cores, 64))
    if ntotal >= (1 << 20):
        nranks = max(1, min(nranks, ntotal // (1 << 16)))
    cfg = configs.get(cfg_name, ntotal)
    cfg["options"] = dict(cfg["options"], max_major_iters=warmup + steps + 1)
    env = dict(os.environ, OPENBLAS_NUM_THREADS="1", PCU_SHIM_NP=str(nranks))
    t_start = time.time()
    with tempfile.TemporaryDirectory() as tmp:
        hist = os.path.join(tmp, "hist.jsonl")
        cmd = [DRIVER] + driver_args(cfg) + ["hist=" + hist, "log=/dev/null"]
        proc = subprocess.Popen(cmd, env=env, stdout=subprocess.DEVNULL,
                                stderr=subprocess.DEVNULL, start_new_session=True)
        walls = []
        stopped = "completed"

        def read():
            out = []
            try:
                for line in open(hist):
                    try:
                        r = json.loads(line)
                    except ValueError:
                        break  # partial last line
                    if "iter" in r:
                        out.append(r["wall"])
            except OSError:
                pass
            return out

        while proc.poll() is None:
            time.sleep(0.5)
            walls = read()
            timed = len(walls) - 1 - warmup
            if timed >= steps:
                stopped = "all steps on record"
                break
            if timed >= 3 and walls[-1] - walls[warmup] >= timed_budget_s:
                stopped = "timed-region budget of %.0f s" % timed_budget_s
                break
            if time.time() - t_start > total_budget_s and timed >= 1:
                stopped = "total budget of %.0f s" % total_budget_s
                break
        if proc.poll() is None:
            try:
                os.killpg(proc.pid, signal.SIGKILL)
            except OSError:
                pass
            proc.wait()
        walls = read() or walls
    if len(walls) < 3:
        return None
    k0 = min(warmup, len(walls) - 2)
    k1 = min(len(walls) - 1, k0 + steps)
    dt = walls[k1] - walls[k0]
    rate = (k1 - k0) / dt
    return {
        "value": rate, "unit": UNIT, "cores": nranks, "kind": "reference",
        "sample": ("unmodified reference ParOptInteriorPoint (oracle/_ref) at the full size "
                   "n=%d, %d shim ranks (one per host core), major iterations %d..%d timed "
                   "(%.1f s, the driver's own wall-clock stamps); run stopped: %s"
                   % (ntotal, nranks, k0, k1, dt, stopped)),
        "sample_n": ntotal, "steps": k1 - k0, "warmup": k0, "same_config": True,
        "seconds_per_iteration": dt / (k1 - k0), "wall_s": time.time() - t_start,
    }


def reference_rate(cfg_name, ntotal, warmup, steps, budget_s=25.0):
    """Iterations/s of the reference's CPU implementation at `ntotal` variables,
    measured on a bounded sample (smaller n, linear scaling in n) with one shim
    rank per host core."""
    cores = host_cores()
    nranks = max(1, min(cores, 64))
    iters = warmup + steps

    def cfg_for(n):
        cfg = configs.get(cfg_name, n)
        cfg["options"] = dict(cfg["options"], max_major_iters=iters + 1)
        return cfg

    unit = 8 * nranks
    n_probe = max(unit * 64, (1 << 18) // unit * unit)
    t0 = time.time()
    hist, fin = run_ref_driver(cfg_for(n_probe), nranks)
    if hist is None:
        return None
    probe_s = time.time() - t0
    n_s = int(n_probe * min(64.0, max(1.0, budget_s / max(probe_s, 1e-3))))
    n_s = max(unit, n_s // unit * unit)
    n_s = min(n_s, ntotal)
    if n_s > n_probe:
        hist, fin = run_ref_driver(cfg_for(n_s), nranks)
    else:
        n_s = n_probe
    k0 = min(warmup, len(hist) - 2)
    k1 = len(hist) - 1
    dt = hist[k1]["wall"] - hist[k0]["wall"]
    rate_sample = (k1 - k0) / dt
    return {
        "value": rate_sample * (float(n_s) / float(ntotal)),
        "unit": UNIT,
        "cores": nranks,
        "kind": "reference",
        "sample": ("unmodified reference ParOptInteriorPoint (oracle/_ref), %d shim "
                   "ranks, n=%d, iterations %d..%d timed (%.2f s); scaled by n/%d "
                   "(O(n) work per iteration)" % (nranks, n_s, k0, k1, dt, ntotal)),
        "sample_iterations_per_sec": rate_sample,
        "sample_n": n_s,
    }


# --------------------------------------------------------------------- ours
def iterate_exactly(ip, n):
    """Runs n major iterations.  The default workload converges after ~96 iterations; a
    run that converges first starts over from its starting point (begin), so that n is
    always the number of steps.  Returns (iterations run, restarts)."""
    done = restarts = 0
    while True:
        k0 = ip.counters()[0]
        converged = ip.iterate(n - done)
        done += ip.counters()[0] - k0
        if done >= n or not converged:
            return done, restarts
        ip.begin()
        restarts += 1


def run_ours(args):
    import torch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:
        raise SystemExit("bench: --dump-outputs writes the point of one process; use --gpus 1")
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from paropt_b200.api import BuiltinProblem, Context, InteriorPoint, problem_from_config
    from paropt_b200.host_problems import HostSepQuad

    ctx = Context(local_rank)
    if world > 1:
        ctx.init_distributed()

    cfg = configs.get(args.config, args.n)
    weak = bool(cfg.get("per_gpu")) and args.n is None
    if weak:  # configs[4]: the named size is per GPU
        cfg["problem"]["ntotal"] = cfg["problem"]["ntotal"] * world
    ntotal = cfg["problem"]["ntotal"]
    c = cfg["problem"]["ncon"]
    msub = cfg["options"].get("qn_subspace_size", 10)
    q = 2 * msub if cfg["options"].get("qn_type", "bfgs") == "bfgs" else msub
    warmup = max(args.warmup, QN_WARMUP)
    steps = args.steps

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def barrier():
        ctx.sync()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- parity across the N ranks before anything is timed ------------------
    # The small named workloads, partitioned over the ranks of THIS run exactly as
    # the timed workload is, against the histories of the unmodified reference
    # (tests/golden, the rule of tests/parity.py).
    parity = None
    if not args.no_parity:
        from tests.parity import checked, compare_histories, load_golden

        parity = {"world": world, "first_violation": None, "worst": 0.0, "cases": {},
                  "rule": "tests/parity.py (RTOL 1e-10); goldens = unmodified reference"}
        for gname, giters in (("C2_small", 41), ("C3_small", 50)):
            gold = load_golden(gname)
            gcfg = gold["config"]
            gp = problem_from_config(ctx, gcfg)
            gip = InteriorPoint(gp, dict(gcfg["options"], history_level=2,
                                         max_major_iters=giters + 1))
            gip.optimize()
            ghist = gip.history()
            gip.free()
            gp.free()
            n_cmp, worst, first = compare_histories(gold["history"], ghist, max_iters=giters,
                                                    cfg=gcfg)
            chk = checked(worst)
            w = max(chk.values())
            parity["cases"][gname] = {"compared": n_cmp, "worst": float("%.3e" % w),
                                      "worst_key": max(chk, key=chk.get),
                                      "residual_norms_rel": float("%.3e" % max(
                                          [v for k, v in worst.items() if k.startswith("rel:")]
                                          + [0.0])),
                                      "first_violation": first}
            parity["worst"] = max(parity["worst"], float("%.3e" % w))
            if first is not None and parity["first_violation"] is None:
                parity["first_violation"] = dict(first, case=gname)

    # ---- device-resident run: `value` --------------------------------------
    prob = problem_from_config(ctx, cfg)
    N, W = prob.nvars, prob.nwcon
    opts = dict(cfg["options"], max_major_iters=1000000, history_level=1)
    ip = InteriorPoint(prob, opts)
    ip.begin()
    iterate_exactly(ip, warmup)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # Per-kernel CUDA events (two records per launch) cost ~55 us per iteration: 0.4 % of a
    # 1-GPU step, 3 % of an 8-GPU one (scripts/launch_overhead_probe.py).  On one GPU --
    # the line the roofline is quoted on -- they cover the timed region itself; on several
    # GPUs the timed region runs without them and the kernel table comes from the same
    # number of steps run right after it.
    events_in_timed = (not args.no_kernel_profile) and world == 1
    if events_in_timed:
        ctx.profile(2)
    launches0 = ctx.kernel_launches()
    ctx.timer_start()
    done, restarts = iterate_exactly(ip, steps)
    ms = ctx.timer_stop()
    barrier()
    ctx.profile(0)
    clocks = sampler.stop() if rank == 0 else None
    launches = ctx.kernel_launches() - launches0
    times = ip.iter_times()[-done:] if done else []
    if args.dump_outputs:
        dump_outputs(ip, args.dump_outputs)
    prof_ms = None
    if not args.no_kernel_profile and not events_in_timed:
        barrier()  # rank 0 has just joined its clock sampler
        ctx.profile(2)
        ctx.timer_start()
        try:
            ip.iterate(steps)  # (stops early, on every rank alike, if the run converges)
        except RuntimeError as exc:  # the timed region is already in hand
            sys.stderr.write("bench: kernel-table pass stopped: %s\n" % exc)
        prof_ms = max_over_ranks(ctx.timer_stop())
        barrier()
        ctx.profile(0)
    ms = max_over_ranks(ms)
    kkt_ms = max_over_ranks(sum(t[2] for t in times) / max(len(times), 1))
    cb_ms = max_over_ranks(sum(t[1] for t in times) / max(len(times), 1))
    prof = ctx.profile_totals()
    hist = ip.history()
    qn_size = hist[-1]["qn_size"] if hist else q
    ip.free()
    prob.free()
    value = done / (ms / 1e3) if ms > 0 else 0.0
    ms_per_step = ms / max(done, 1)

    # dominant kernel of the timed region and its roofline
    peak, peak_src = measured_peak_gbs()
    roof = None
    if prof:
        name = max(prof, key=lambda k: prof[k][0])
        tot_ms, cnt = prof[name]
        words = kernel_words(name, N, W, c, qn_size)
        if name == "mdot_kernel":
            # launches of 8-column chunks: average columns per launch from totals
            m = c + qn_size
            chunks = -(-m // 8)
            words = (m / chunks + 1) * N
        avg_ms = tot_ms / cnt
        achieved = words * 8 / (avg_ms * 1e-3) / 1e9 if words else None
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        # ncu DRAM bytes of the kernel at the 1-GPU size of the metric (C3): they say
        # nothing about a rank's share at N > 1 or about another workload
        if os.path.exists(tpath) and world == 1 and args.config == "C3" and args.n is None:
            try:
                traffic = json.load(open(tpath)).get(name.split("<")[0].replace("ResFT", "ResF"))
            except Exception:
                traffic = None
        roof = {"bound": "hbm", "kernel": name, "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
                "traffic": traffic, "peak_source": peak_src,
                "avg_launch_ms": avg_ms, "launches": cnt,
                "share_of_step": tot_ms / (prof_ms or ms) if ms else None,
                "events_over": ("the timed region" if events_in_timed else
                                "%d more steps right after the timed region (%.3f ms/step "
                                "with the events)" % (steps, (prof_ms or 0.0) / max(steps, 1))),
                "algorithmic_bytes_per_launch": words * 8 if words else None,
                "kernels": {k: {"ms": round(v[0], 3), "launches": v[1]}
                            for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}}
    if roof and roof["kernel"] == "gram_kernel" and words:
        # the Gram pass S = V^T D0^-1 V over mcol = c + q (+ 1: right-hand side) columns:
        # (mcol)(mcol + 1) N flops on the lower triangle the kernel computes; tensor-bound
        # when its arithmetic intensity exceeds the ridge of the two measured peaks
        tf_peak, tf_src = measured_fp64_tflops()
        mcol = c + qn_size + 1
        flops = float(mcol) * (mcol + 1) * N
        ai = flops / (words * 8.0)
        if ai > tf_peak * 1e12 / (peak * 1e9):
            ach = flops / (roof["avg_launch_ms"] * 1e-3) / 1e12
            roof.update({"bound": "tensor", "achieved": ach, "peak": tf_peak, "unit": "TFLOP/s",
                         "frac": ach / tf_peak, "peak_source": tf_src,
                         "algorithmic_flops_per_launch": flops,
                         "arithmetic_intensity_flop_per_byte": ai})
    iter_bytes = 8.0 * iteration_words(N, W, c, qn_size)
    user_ms = cb_ms
    solver_ms = max(ms_per_step - user_ms, 1e-9)
    iter_frac = iter_bytes / (solver_ms * 1e-3) / 1e9 / peak
    kkt_frac = 8.0 * kkt_words(N, W, c, qn_size) / (max(kkt_ms, 1e-9) * 1e-3) / 1e9 / peak

    # ---- end to end through the host-callback API: `e2e` --------------------
    e2e = None
    if not args.no_e2e:
        def allreduce(a):
            if world == 1:
                return a
            t = torch.tensor(a, dtype=torch.float64, device="cuda")
            dist.all_reduce(t)
            return t.cpu().numpy()

        if args.e2e_python:
            hp = HostSepQuad(ctx, allreduce=allreduce, **cfg["problem"])
            e_kind = ("python callbacks (torch-CPU threaded numpy views) on the library's "
                      "pinned host arrays")
        else:
            hp = BuiltinProblem(ctx, "sepquad", host=True, nthreads=host_cores() // world,
                                **cfg["problem"])
            e_kind = ("C++ host callbacks over host arrays (pcu_problem_create_host), "
                      "%d host threads" % max(1, host_cores() // world))
        hip = InteriorPoint(hp, dict(cfg["options"], max_major_iters=1000000,
                                     history_level=1))
        e_warm, e_steps = max(args.e2e_warmup, QN_WARMUP), args.e2e_steps
        hip.begin()
        hip.iterate(e_warm)
        barrier()
        h2d0, d2h0 = hp.transfer_bytes()
        ht0 = hp.host_times() if hasattr(hp, "host_times") else None
        i0 = hip.counters()[0]
        ctx.timer_start()
        hip.iterate(e_steps)
        e_ms = max_over_ranks(ctx.timer_stop())
        barrier()
        h2d1, d2h1 = hp.transfer_bytes()
        e_done = hip.counters()[0] - i0
        host_ms = None
        if hasattr(hp, "host_times"):
            ht1 = hp.host_times()
            host_ms = {"d2h": (ht1[0] - ht0[0]) / max(e_done, 1),
                       "user": (ht1[1] - ht0[1]) / max(e_done, 1),
                       "h2d_if_PCU_HOST_TIMING": (ht1[2] - ht0[2]) / max(e_done, 1)}
        e_times = hip.iter_times()[-e_done:] if e_done else []
        e2e = {"value": e_done / (e_ms / 1e3) if e_ms > 0 else 0.0, "unit": UNIT,
               "h2d_bytes_per_step": (h2d1 - h2d0) // max(e_done, 1),
               "d2h_bytes_per_step": (d2h1 - d2h0) // max(e_done, 1),
               "steps": e_done, "warmup": e_warm, "ms_per_step": e_ms / max(e_done, 1),
               "callback_ms_per_step": sum(t[1] for t in e_times) / max(len(e_times), 1),
               "host_ms_per_step": host_ms,
               "note": "same loop through the host-array problem API: " + e_kind +
                       "; per callback the iterate is copied device->host and the "
                       "gradients host->device (pinned buffers) inside the timed region; "
                       "callback_ms = user code + copies"}
        hip.free()
        hp.free()

    # ---- CPU baseline (rank 0, single-GPU runs only) -------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            cpu = reference_rate(args.config, ntotal, QN_WARMUP, 6)
        except Exception as exc:  # the checker must never sink the bench line
            cpu = {"value": None, "unit": UNIT, "cores": host_cores(), "kind": "reference",
                   "sample": "failed: %r" % (exc,)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world,
            "steps": done, "restarts": restarts, "warmup": warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak" if weak else "strong",
            "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(args.config, cfg, ntotal),
                "n_per_gpu": N, "partition": "block-row over %d GPU(s)" % world,
                "l2_note": "every pass streams >= 0.5 GB per vector (>> 126 MB L2)",
                "warmup_note": "warm-up raised to %d so the L-BFGS memory is full" % QN_WARMUP},
            "kkt_solve_ms": kkt_ms, "kkt_roofline_frac": kkt_frac,
            "callback_ms_per_step": cb_ms, "iter_roofline_frac": iter_frac,
            "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "parity": parity,
            "gpu_launches": launches, "clocks": clocks,
        }
        emit(line)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def workload_name(cfg_name, cfg, ntotal):
    c = cfg["problem"]["ncon"]
    return "%s: %s n=%d ncon=%d nwcon=%d qn=%s m=%d" % (
        cfg_name, cfg["kind"], ntotal, c, ntotal // 8 if cfg["problem"].get("nw") else 0,
        cfg["options"].get("qn_type", "bfgs"), cfg["options"].get("qn_subspace_size", 10))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    cfg = configs.get(args.config, args.n)
    if bool(cfg.get("per_gpu")) and args.n is None:
        cfg["problem"]["ntotal"] = cfg["problem"]["ntotal"] * world
    ntotal = cfg["problem"]["ntotal"]
    warmup = max(args.warmup, QN_WARMUP)
    t0 = time.time()
    if args.ref_sample:
        res = reference_rate(args.config, ntotal, warmup, args.steps)
    else:
        res = reference_full_size(args.config, ntotal, warmup, args.steps)
    if res is None:
        emit({"impl": "reference",
              "unavailable": "oracle/_ref/ref_driver has not been built"})
        return
    steps = res.get("steps", args.steps)
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT,
        "n_gpus": world, "steps": steps,
        "warmup": res.get("warmup", warmup), "ms_per_step": 1e3 / res["value"],
        "higher_is_better": True,
        "scaling": "weak" if cfg.get("per_gpu") and args.n is None else "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.config, cfg, ntotal),
                   "reference_arm": ("CPU, the metric's own size" if res.get("same_config")
                                     else "CPU sample n=%d, linear in n" % res["sample_n"]),
                   "steps_requested": args.steps},
        "cpu_baseline": res,
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "wall_s": time.time() - t0,
    }
    emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed interior-point iterations (a run that converges restarts)")
    ap.add_argument("--warmup", type=int, default=QN_WARMUP)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C3")
    ap.add_argument("--n", type=int, default=None, help="global number of design variables")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--e2e-warmup", type=int, default=QN_WARMUP)
    ap.add_argument("--e2e-python", action="store_true",
                    help="drive the end-to-end leg through the Python Problem class")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-kernel-profile", action="store_true",
                    help="no per-kernel CUDA events in the timed region (roofline = null)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true",
                    help="skip the golden-history comparisons before the timed region")
    ap.add_argument("--ref-sample", action="store_true",
                    help="--impl reference on a bounded smaller-n sample (scaled by n) "
                         "instead of the full size")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the optimizer's point after the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
