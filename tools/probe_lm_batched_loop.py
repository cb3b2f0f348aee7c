"""Measure the batched alternating LM loop (csrc/lm_loop_batched.cu) against one loop per seed.

    python tools/probe_lm_batched_loop.py --out profiles/r07_lm_batched_loop.json

1. Loop timing on fetch__circle, seeds from the stand-in candidate generator, N in --ns, the planner's non-anytime
   arguments (20 steps, return when valid, no convergence test):
   - wall time per loop and per iteration (host clock around the call, which ends in a stream synchronisation);
   - device time per iteration of the decision and compaction kernels, from torch.profiler in a separate pass;
   - up to N = 32 the same seeds through cppflow_lm_alternating_loss_many (one job, stream and host poll per seed;
     32 is the number of distinct streams torch.cuda.Stream() hands out per device).
2. Planner latency and valid-plan count over the 13 benchmark problems for lm_seeds in --lm_seeds
   (LatentIkCandidateGenerator(seed=3), k = 175).
The card's name and power limit are read in the same run and stored with the numbers."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cppflow_b200.data_type_utils import ALL_PROBLEM_FILENAMES, problem_from_filename  # noqa: E402
from cppflow_b200.data_types import PlannerSettings  # noqa: E402
from cppflow_b200.optimization import run_lm_optimization_batched, run_lm_optimization_many  # noqa: E402
from cppflow_b200.planners import CppFlowPlanner, LatentIkCandidateGenerator, LmIkCandidateGenerator  # noqa: E402

DEV = "cuda:0"
KW = dict(max_n_steps=20, return_if_valid_after_n_steps=0, convergence_threshold=1e6)
MANY_MAX_JOBS = 32  # distinct streams torch.cuda.Stream() hands out per device (see loop_timing)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def timed(fn, reps):
    ts = []
    out = None
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts), min(ts), out


def kernel_times(fn):
    """Device time (us) per launch of the batched loop's own kernels, from one profiled call."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    acc = {}
    for ev in prof.events():
        name = ev.name
        for key in ("lmb_decide_kernel", "lmb_compact_kernel", "lmb_gather_kernel", "path_metrics_kernel"):
            if key in name:
                t = getattr(ev, "device_time", None)
                if t is None:
                    t = ev.cuda_time
                a = acc.setdefault(key, [0.0, 0])
                a[0] += t
                a[1] += 1
    return {k: {"us_per_launch": v[0] / v[1], "launches": v[1]} for k, v in acc.items()}


def loop_timing(ns, reps):
    problem = problem_from_filename(None, "fetch__circle", device=DEV)
    seeds_all = LmIkCandidateGenerator(seed=1)(problem, max(ns)).contiguous()
    rows = []
    for n in ns:
        seeds = seeds_all[:n].contiguous()
        run = lambda: run_lm_optimization_batched(problem, seeds, 60.0, **KW)  # noqa: E731
        run()  # warm-up: workspaces, kernel attributes
        med, best, res = timed(run, reps)
        iters = max(r.n_steps_taken for r in res) + 1
        row = {"N": n, "T": problem.n_timesteps, "iterations": iters, "loop_ms_median": med * 1e3, "loop_ms_min": best * 1e3,
               "iteration_us_median": med / iters * 1e6, "valid_seeds": sum(r.is_valid for r in res),
               "differencing_steps": sum(r.schedule.count("d") for r in res),
               "pose_steps": sum(r.schedule.count("p") for r in res)}
        row["kernels"] = kernel_times(run)
        if n <= MANY_MAX_JOBS:
            # one job, stream and host poll per seed.  torch.cuda.Stream() hands out the streams of a pool of 32 per
            # device, and ops.lm_alternating_loss_many keys each job's workspace and pinned buffer by its stream: two
            # jobs on one stream would overwrite each other's iterates and tags.  So at most 32 jobs.
            streams = [torch.cuda.Stream(DEV) for _ in range(n)]
            assert len({s.cuda_stream for s in streams}) == n, "two jobs on one CUDA stream"
            singles = [s.contiguous() for s in seeds]
            cur = torch.cuda.current_stream(DEV)

            def many():
                for s in streams:
                    s.wait_stream(cur)
                out = run_lm_optimization_many([problem] * n, singles, streams, 60.0, **KW)
                for s in streams:
                    cur.wait_stream(s)
                return out

            many()
            med_m, best_m, res_m = timed(many, reps)
            iters_m = max(r.n_steps_taken for r in res_m) + 1
            row["many_iterations"] = iters_m
            row["many_loop_ms_median"] = med_m * 1e3
            row["many_loop_ms_min"] = best_m * 1e3
            row["many_iteration_us_median"] = med_m / iters_m * 1e6
            row["many_equals_batched"] = all(torch.equal(a.x_opt, b.x_opt) and a.schedule == b.schedule
                                             for a, b in zip(res, res_m))
        print(json.dumps(row), flush=True)
        rows.append(row)
    return rows


def planner(lm_seeds_list):
    settings = PlannerSettings(k=175, tmax_sec=30.0, anytime_mode_enabled=False, verbosity=0)
    problems = [problem_from_filename(None, n, device=DEV) for n in ALL_PROBLEM_FILENAMES]
    out = []
    for n in lm_seeds_list:
        lat, valid, used = [], [], []
        for p in problems:
            pl = CppFlowPlanner(settings, p.robot, LatentIkCandidateGenerator(seed=3), lm_seeds=n)
            pl.generate_plan(p)  # warm-up
            pl = CppFlowPlanner(settings, p.robot, LatentIkCandidateGenerator(seed=3), lm_seeds=n)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = pl.generate_plan(p)
            torch.cuda.synchronize()
            lat.append(time.perf_counter() - t0)
            valid.append(bool(r.plan.is_valid))
            used.append(r.debug_info.get("lm_seed_index", 0))
        row = {"lm_seeds": n, "valid_plans": sum(valid), "problems": len(problems),
               "plan_ms_median": statistics.median(lat) * 1e3, "plan_ms_max": max(lat) * 1e3,
               "per_problem": [{"problem": name, "valid": v, "ms": t * 1e3, "seed_used": u}
                               for name, v, t, u in zip(ALL_PROBLEM_FILENAMES, valid, lat, used)]}
        print(json.dumps({k: v for k, v in row.items() if k != "per_problem"}), flush=True)
        out.append(row)
    return out


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--ns", default="1,16,32,64,175,1024,8192")
    ap.add_argument("--lm_seeds", default="1,16,64")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="JSON file for the results")
    args = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this probe measures the GPU and has no CPU fallback")
    res = {"card": card(), "loop": loop_timing([int(v) for v in args.ns.split(",")], args.reps),
           "planner": planner([int(v) for v in args.lm_seeds.split(",")])}
    res["card_after"] = card()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    return res


if __name__ == "__main__":
    main()
