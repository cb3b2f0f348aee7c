#!/usr/bin/env python
"""Benchmark of the path-refinement hot path (BASELINE.json metric: waypoint FK+Jac+collision+LM evals/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config 5, SURVEY.md 8d): synthetic P = 8192 candidate paths x T = 300 waypoints of the 8-dof Fetch, the four
fetch__circle cuboids as obstacles, seeds = smooth joint path + N(0, 0.05^2).  One "step" = ONE fused LM iteration
with every residual term on (pose + joint differencing + virtual configs + capsule self- and env-collisions) followed
by clamp_to_joint_limits, over all P*T waypoints; one waypoint evaluation = FK + 6xD Jacobian + 28 capsule-pair and
40 capsule-cuboid distances + its share of the block-tridiagonal normal-equation assembly and solve.
Multi-GPU: weak scaling - every rank refines its own shard of P paths, no collective in the data path; after the
timed steps every rank reduces its per-path costs to one packed key on the device and the keys are all-gathered over
NCCL (inside the timed region; the host reads the result after the closing event).  Extra keys of the same line:
`strong` (the SAME 8192 paths split P/N per GPU), `quality` (the reference's alternating step sequence on a
collision-free variant of the workload, cost argmin over valid paths), per-kernel times and roofline fractions.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

import torch

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

# algorithmic FLOPs per waypoint evaluation (SURVEY.md 8d formula, Fetch instance; DESIGN.md "Roofline")
F_ASSEMBLE = 581 + 96 + 90 + 624 + 2520 + 4800 + 63  # FK, Jacobian, pose error, normal equations, self, env, extra frames
F_SOLVE = 1451                                       # block-tridiagonal factor/solve share: (7/3) D^3 + 4 D^2
F_STEP_SURVEY = 9100                                 # the per-eval figure SURVEY.md 8d quotes for the fused iteration
BYTES_PER_EVAL = 64                                  # read q once, write x_new once (8 dof * 4 B * 2)
F_POSE_STEP = 581 + 96 + 90 + 624 + 315              # pose-only LM step: FK, Jacobian, error, normal equations, D x D solve
F_FLAGS = 581 + 63 + 2520 + 4800                     # collision flags: all-link FK + 28 pair + 40 capsule-cuboid distances
SOLVE_WS_PASSES = 3                                  # block solve: read A, write (-S^-1, u), read them back


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed LM iterations (20 = the reference's max_n_steps, planners.py:416)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--paths", type=int, default=8192)
    ap.add_argument("--waypoints", type=int, default=300)
    ap.add_argument("--chunks", type=int, default=0, help="path chunks (streams) of the pipelined LM iterations (0: ResidentPipeline's choice)")
    ap.add_argument("--cpu-sample-paths", type=int, default=24)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (rank 0's shard; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the GPU path: use it with --impl ours")
    return args


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int, period: float = 0.01):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._halt = threading.Event()
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._halt.set()
        self.join(timeout=1.0)
        return {
            "sm_mhz": statistics.median(self.samples) if self.samples else None,
            "sm_max_mhz": self.max_mhz,
            "reasons": sorted(self.reasons),
            "samples": len(self.samples),
        }


def physical_gpu_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


# ------------------------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the oracle port of the reference's dense torch path on the host cores


def cpu_reference_step_rate(T: int, sample_paths: int, steps: int, warmup: int):
    """evals/s of the reference's CPU path (oracle/ port; the reference itself needs jrl and cannot be imported):
    per path, dense LmResidualFns.get_r_and_J with every term on + _lm_full_step (dense (T*D)^2 Cholesky) + clamp."""
    from oracle import robots as OR, lm as OL
    from oracle.workloads import synthetic_problem as oracle_problem, cuboid_tensors, FETCH_CIRCLE_OBSTACLES

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    model, target, x0 = oracle_problem("fetch", sample_paths, T, seed=0)
    cuboids, Tcuboids = cuboid_tensors(FETCH_CIRCLE_OBSTACLES)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        OL.run_fixed_schedule(model, x0, target, "a", Tcuboids, cuboids)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    mean_dt = sum(times) / len(times)
    return sample_paths * T / mean_dt, mean_dt, cores


def run_reference(args, rank: int):
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    # a step of the reference arm is a bounded sample of the workload: sized so that steps + warmup end within minutes
    budget_paths = int(max(2, min(args.cpu_sample_paths, 600.0 / (0.065 * (steps + warmup)))))
    args.cpu_sample_paths = budget_paths
    rate, dt, cores = cpu_reference_step_rate(args.waypoints, args.cpu_sample_paths, steps, warmup)
    sample = (f"{args.cpu_sample_paths} of {args.paths} paths x {args.waypoints} waypoints per step (dense get_r_and_J + "
              f"_lm_full_step, all terms on), fp32, torch {torch.__version__}, {cores} threads; evals/s is size-independent "
              f"per path so the sample rate is the full-workload rate")
    line = {
        "impl": "reference",
        "metric": "waypoint FK+Jac+collision+LM evals/s",
        "value": rate,
        "unit": "waypoint-evals/s",
        "n_gpus": args.gpus,
        "steps": steps,
        "warmup": warmup,
        "ms_per_step": dt * 1e3,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic",
        "config": workload_config(args, args.gpus),
        "cpu_baseline": {"value": rate, "unit": "waypoint-evals/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": "waypoint-evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------------------------------
# second half of BASELINE.json's metric: plan latency on fetch__circle (config 2): collision flags of k = 175 candidate
# paths -> dp_search -> run_lm_optimization (the reference's non-anytime call: max 20 steps, return once valid)


def plan_latency_gpu(dev, k=175, reps=10):
    from cppflow_b200.collision_detection import qpaths_batched_collisions
    from cppflow_b200.data_type_utils import problem_from_filename
    from cppflow_b200.optimization import run_lm_optimization
    from cppflow_b200.planners import LmIkCandidateGenerator
    from cppflow_b200.search import dp_search

    problem = problem_from_filename(None, "fetch__circle", device=dev)
    qs = LmIkCandidateGenerator(seed=1)(problem, k).contiguous()

    def plan():
        self_v, env_v = qpaths_batched_collisions(problem, qs)
        best = dp_search(problem.robot, qs, self_v, env_v, verbosity=0).to(dev)
        return run_lm_optimization(problem, best, max_n_steps=20, tmax_sec=30.0, return_if_valid_after_n_steps=0,
                                   convergence_threshold=1e6, verbosity=0)

    for _ in range(2):
        res = plan()
    torch.cuda.synchronize(dev)
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        res = plan()
        torch.cuda.synchronize(dev)
        times.append((time.perf_counter() - t0) * 1e3)
    return {
        "problem": "fetch__circle", "k": k, "waypoints": problem.n_timesteps, "unit": "ms",
        "value": statistics.median(times), "min": min(times), "reps": reps,
        "lm_steps": res.n_steps_taken + 1, "schedule": res.schedule, "valid": bool(res.is_valid),
        "what": "host wall clock, candidates resident on the GPU: capsule collision flags -> dp_search -> "
                "run_lm_optimization(max_n_steps=20, return once valid); one 8-float device->host read per LM step",
        "candidates": "stand-in LM-IK generator (IKFlow weights unavailable offline), excluded from the timing",
    }, problem, qs.cpu()


def plan_all_problems_gpu(dev, k=175, reps=5):
    """BASELINE config 4: the 13 benchmark problems (candidate generation included), one after the other and
    in one batched run (planners.plan_many: one CUDA stream per problem, stages phase by phase, LM loops in lock step).  Host wall clock, median."""
    from cppflow_b200.data_type_utils import ALL_PROBLEM_FILENAMES, problem_from_filename
    from cppflow_b200.data_types import PlannerSettings
    from cppflow_b200.planners import CppFlowPlanner, LmIkCandidateGenerator, plan_many

    problems = [problem_from_filename(None, name, device=dev) for name in ALL_PROBLEM_FILENAMES]

    def factory(problem):
        return CppFlowPlanner(PlannerSettings(k=k, tmax_sec=30.0, anytime_mode_enabled=False, verbosity=0), problem.robot,
                              LmIkCandidateGenerator(seed=1))

    def sequential():
        return [factory(p).generate_plan(p) for p in problems]

    def batched():
        return plan_many(factory, problems)

    out = {}
    for name, fn in (("sequential_ms", sequential), ("batched_ms", batched)):
        fn()
        torch.cuda.synchronize(dev)
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            res = fn()
            torch.cuda.synchronize(dev)
            ts.append((time.perf_counter() - t0) * 1e3)
        out[name] = statistics.median(ts)
    out.update({"problems": len(problems), "k": k, "waypoints_total": sum(p.n_timesteps for p in problems),
                "valid_plans": sum(bool(r.plan.is_valid) for r in res),
                "what": "CppFlowPlanner.generate_plan on all 13 benchmark problems: stand-in candidate generation + "
                        "collision flags + dp_search + alternating LM loop (max 20 steps, return once valid)"})
    return out


def plan_latency_cpu(problem, qs, schedule):
    """The same plan through the oracle port of the reference's torch path on the host cores (the LM loop replays the
    step types the GPU run took; the reference's per-step klampt validity check is not included)."""
    from oracle import robots as OR, lm as OL, search as OS

    torch.set_num_threads(os.cpu_count() or 1)
    model = OR.get_model("fetch")
    cuboids = [c.detach().float().cpu() for c in problem.obstacles_cuboids]
    Tcuboids = [t.detach().float().cpu() for t in problem.obstacles_Tcuboids]
    target = problem.target_path.detach().float().cpu()
    t0 = time.perf_counter()
    self_v = OS.qpaths_batched_self_collisions(model, qs)
    env_v = OS.qpaths_batched_env_collisions(model, qs, cuboids, Tcuboids)
    t1 = time.perf_counter()
    best = OS.dp_search(model, qs, self_v, env_v)[0]
    t2 = time.perf_counter()
    OL.run_fixed_schedule(model, best, target, schedule, Tcuboids, cuboids)
    t3 = time.perf_counter()
    return {"value": (t3 - t0) * 1e3, "unit": "ms", "flags_ms": (t1 - t0) * 1e3, "dp_search_ms": (t2 - t1) * 1e3,
            "lm_ms": (t3 - t2) * 1e3, "schedule": schedule, "cores": os.cpu_count(), "kind": "port"}


def workload_config(args, n_gpus):
    if not args.chunks:  # ResidentPipeline's own choice (the reference arm reports the same configuration)
        args.chunks = 6 if args.paths >= 6144 else 1 if args.paths >= 3072 else 2 if args.paths >= 1536 else 4
    return {
        "workload": f"synthetic {args.paths} paths x {args.waypoints} waypoints Fetch 8-DOF, one fused LM iteration "
                    "(pose + differencing + virtual configs + self/env capsule collisions) + clamp; 4 fetch__circle cuboids",
        "paths_per_gpu": args.paths,
        "waypoints": args.waypoints,
        "robot": "fetch",
        "parallelism": f"paths sharded over {n_gpus} GPU(s), no data-path collective; per GPU the K iterations run as "
                       f"{args.chunks} independent path chunks on {args.chunks} streams (solve of one chunk under the assembly "
                       "of another), every chunk doing all K iterations",
        "chunks_per_gpu": args.chunks,
        "l2": "no flush: each step streams ~1.9 GB (q, x_new, 433 MB block workspace written+read twice) >> 126 MB L2",
    }


DUMP_BYTES = 60_000_000  # --dump-outputs stays under 64 MB: past that, a sample of the paths drawn with a fixed seed


def dump_outputs(out_dir, x_out, metrics, best, P, T, D):
    """What a caller of the timed path receives from its last step, as .npy files in `out_dir`:
    x_out.npy [n, T, D] float32 refined joint paths and path_metrics.npy [n, 8] float32 (the per-path metrics the
    cost argmin ranks, ops.METRIC_NAMES + tag) of n paths - all P, or a sorted sample drawn with seed 0 when they do not
    fit DUMP_BYTES -, path_index.npy [n] float64 which paths those are, and argmin.npy float64 [cost, global index,
    n_valid, valid, trajectory length] of the argmin over all paths.  The timed path computes sign-only metrics: its
    min_self / min_env columns are the exact minimum distance when negative and an unspecified non-negative value
    (+inf when every capsule pair was culled) otherwise, so they are written as min(d, 0): 0 = no collision, else the
    exact depth.  The inputs are seeded, so two builds can be compared file by file.  Every array is written; the names
    of those holding a NaN or inf are returned (and reported on stderr and in the result line)."""
    import numpy as np
    from cppflow_b200.ops import METRIC_NAMES

    n = min(P, DUMP_BYTES // ((T * D + metrics.shape[1]) * 4))
    idx = np.arange(P) if n == P else np.sort(np.random.default_rng(0).choice(P, n, replace=False))
    sel = torch.from_numpy(idx).to(x_out.device)
    path_metrics = metrics.index_select(0, sel)
    for col in (METRIC_NAMES.index("min_self"), METRIC_NAMES.index("min_env")):
        path_metrics[:, col].clamp_(max=0.0)
    arrays = {
        "x_out": x_out.view(P, T, D).index_select(0, sel).cpu().numpy(),
        "path_metrics": path_metrics.cpu().numpy(),
        "path_index": idx.astype(np.float64),
        "argmin": np.array([best.cost, best.global_index, best.n_valid, best.valid, best.trajectory_length], np.float64),
    }
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    non_finite = [name for name, a in arrays.items() if not np.isfinite(a).all()]
    if non_finite:
        print(f"--dump-outputs: the timed path produced NaN or inf in {non_finite}", file=sys.stderr)
    return non_finite


# ------------------------------------------------------------------------------------------------------------------


def emit(line: dict):
    """The ONE JSON line goes to the real stdout; everything else printed to fd 1 (NCCL's version banner, library
    chatter) was redirected to stderr by main()."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


_GRAPHS = {}


def time_pipeline(rpipe, x_in, x_out, steps, barrier, metrics=None, tail=None):
    """K pipelined steps (+ optionally each chunk's metrics and a tail enqueued on the current stream) between two CUDA
    events with a barrier + device synchronisation on both sides.  -> (ms total, whatever `tail` returned).
    The K x chunks x (assemble, solve) launches (+ the metrics) are captured once into a CUDA graph and replayed: one
    launch per timed region instead of hundreds of Python -> ctypes calls (with 8 ranks on 16 host cores the enqueue
    loop's jitter otherwise shows up as skew in front of the all-gather)."""

    def enqueue():
        for _ in range(steps):
            rpipe.enqueue_step(x_in, x_out)
        if metrics is not None:
            rpipe.enqueue_metrics(x_out, metrics)

    key = (id(rpipe), x_in.data_ptr(), x_out.data_ptr(), steps, None if metrics is None else metrics.data_ptr())
    if key not in _GRAPHS:
        rpipe.begin(); enqueue(); rpipe.end()  # eager once: first calls set kernel attributes
        torch.cuda.synchronize()
        _GRAPHS[key] = (rpipe, rpipe.capture(enqueue))  # (the pipeline is kept alive with its graph)
    graph = _GRAPHS[key][1]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    graph.replay()
    pending = tail() if tail is not None else None
    e1.record()
    barrier()
    return e0.elapsed_time(e1), pending


def main():
    global _REAL_STDOUT
    args = parse()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from cppflow_b200 import ops, _lib
    from cppflow_b200.robot import get_robot
    from cppflow_b200.synthetic import synthetic_problem, synthetic_seeds_host, FEASIBLE
    from cppflow_b200.lm_hyper_parameters import all_terms_parameters, ALT_LOSS_V2_1_DIFF, ALT_LOSS_V2_1_POSE
    from cppflow_b200.distributed import enqueue_argmin, shard_range
    from cppflow_b200.pipeline import ResidentPipeline, HostPipeline, numa_local
    import ctypes

    lib = _lib.load()
    robot = get_robot("fetch")
    P, T, D = args.paths, args.waypoints, robot.ndof
    problem = synthetic_problem(robot, T, seed=0, device=dev)
    with numa_local(dev):  # page-locked buffers on the GPU's own NUMA node
        _, x_host = synthetic_seeds_host(robot, P, T, seed=0, shard=rank, pin=True)
    x0 = x_host.to(dev)
    x_out = torch.empty_like(x0)
    prm = ops.make_params(all_terms_parameters())
    ob = problem.obstacle_tables
    rid = robot.robot_id
    evals_per_step = P * T
    steps, warmup = args.steps, max(args.warmup, 3)

    def step(src=x0, dst=x_out):
        return ops.lm_full_step(rid, D, prm, src, None, problem.target_path, P, T, ob, True, out=dst)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    # the K timed iterations run chunk-pipelined: the path set is cut into `--chunks` chunks with one stream each, and
    # the block solve of one chunk runs under the assembly of another (pipeline.ResidentPipeline, CPPFLOW_LM_OVERLAP)
    rpipe = ResidentPipeline(problem, P, all_terms_parameters(), n_chunks=args.chunks or None)
    args.chunks = len(rpipe.chunks)
    metrics = torch.empty((P, 8), device=dev, dtype=torch.float32)

    def argmin_tail():
        # every rank: packed (invalid, TL, global index) key of its best path -> ONE all-gather of 3 int64 per rank
        return enqueue_argmin(metrics, problem.constraints, rank * P, world)

    for _ in range(warmup):
        step()
    # warm-up of the pipelined steps AND of the once-per-job tail (metrics kernel, NCCL all-gather): first calls load modules
    time_pipeline(rpipe, x0, x_out, warmup, barrier, metrics, argmin_tail)[1].result()

    # ---- headline: K steps + the cost argmin, inputs resident in HBM, CUDA events, max over ranks
    sampler = ClockSampler(physical_gpu_index(local_rank), period=float(os.environ.get("BENCH_CLOCK_PERIOD", "0.005")))
    sampler.start()
    ms_total, pending = time_pipeline(rpipe, x0, x_out, steps, barrier, metrics, argmin_tail)
    timed_outputs = (x_out.clone(), metrics.clone()) if args.dump_outputs and rank == 0 else None
    # a 20-step region is ~10 ms: keep the sampler running over a few more identical regions so that it sees load
    for _ in range(3):
        time_pipeline(rpipe, x0, x_out, steps, barrier, metrics, argmin_tail)
    clocks = sampler.stop()
    best = pending.result()
    dumped = None
    if timed_outputs is not None:
        dumped = {"dir": args.dump_outputs, "non_finite": dump_outputs(args.dump_outputs, *timed_outputs, best, P, T, D)}
        del timed_outputs
    ms_total = max_over_ranks(ms_total)
    ms_per_step = ms_total / steps
    value = world * evals_per_step / (ms_per_step * 1e-3)
    # the same K steps without the tail: what the tail costs
    ms_steps_only = max_over_ranks(time_pipeline(rpipe, x0, x_out, steps, barrier)[0]) / steps

    # ---- strong scaling: the SAME P paths split over the ranks (P / N per GPU), K steps, no tail
    strong = None
    sizes = sorted({max(16, P // n) for n in (2, 4, 8)} | ({max(16, P // world)} if world > 1 else set()), reverse=True)
    per_size, per_size_twisted, seg_of = {}, {}, {}
    for n_paths in sizes:
        s0, _ = shard_range(P, rank % max(1, P // n_paths), max(1, P // n_paths))
        xs = x0[s0 * T:(s0 + n_paths) * T]
        # few paths per GPU: the solve's chain of T dependent steps is most of the iteration -> the segmented
        # (parallel-in-time) solve, chosen by path count (pipeline.ResidentPipeline segments="auto"); the twisted solve's
        # time at the same size is reported beside it
        for seg, dst in (("auto", per_size), (0, per_size_twisted)):
            if seg == 0 and seg_of.get(n_paths) == 0:
                dst[n_paths] = per_size[n_paths]  # "auto" already was the twisted solve
                continue
            pipe_s = ResidentPipeline(problem, n_paths, all_terms_parameters(), segments=seg)
            seg_of.setdefault(n_paths, pipe_s.segments)
            time_pipeline(pipe_s, xs, x_out[: n_paths * T], warmup, barrier)
            dst[n_paths] = max_over_ranks(time_pipeline(pipe_s, xs, x_out[: n_paths * T], steps, barrier)[0]) / steps
    if world > 1:
        ms_strong = per_size[max(16, P // world)]
        strong = {"paths_total": P, "paths_per_gpu": max(16, P // world), "ms_per_step": ms_strong,
                  "evals_per_s": evals_per_step / (ms_strong * 1e-3),
                  "efficiency": ms_steps_only / (world * ms_strong),
                  "solve_segments": seg_of[max(16, P // world)],
                  "ms_per_step_twisted_solve": per_size_twisted[max(16, P // world)],
                  "efficiency_twisted_solve": ms_steps_only / (world * per_size_twisted[max(16, P // world)]),
                  "what": "same 8192 x 300 workload split P/N per GPU, K pipelined steps, max over ranks; efficiency = "
                          "t(P paths on one GPU, measured in this run) / (N * t(P/N paths per GPU))"}
    strong_preview = {
        "what": "per-GPU step time with P/n paths resident (paths are independent and no data-path collective exists, so "
                "this is the n-GPU strong-scaling step time); efficiency = t(P) / (n * t(P/n))",
        "ms_per_step": {str(n): per_size[n] for n in sizes},
        "solve_segments": {str(n): seg_of[n] for n in sizes},
        "ms_per_step_twisted_solve": {str(n): per_size_twisted[n] for n in sizes},
        "efficiency": {f"1/{P // n}": ms_steps_only / ((P // n) * per_size[n]) for n in sizes},
    }

    # ---- e2e: host buffers in, host buffers out, through the public API, copies inside the timed region
    pipe = HostPipeline(problem, P, all_terms_parameters())
    with numa_local(dev):
        out_hosts = [torch.empty_like(x_host).pin_memory() for _ in range(pipe.depth)]
    out_host = out_hosts[0]
    e2e_steps = steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(2 * pipe.depth):
        pipe.refine_async(x_host, out_hosts[i % pipe.depth])
    barrier()
    # every step is an independent job (host paths in, refined host paths out) submitted with refine_async: a step's
    # copy-in runs under the copy-out of the step before it (two slots of device buffers); the region ends when the
    # last step's result is in host memory
    t0 = time.perf_counter()
    e0.record()
    done = [pipe.refine_async(x_host, out_hosts[i % pipe.depth]) for i in range(e2e_steps)]
    for ev in done:
        torch.cuda.current_stream(dev).wait_event(ev)
    e1.record()
    barrier()
    wall = time.perf_counter() - t0
    e2e_ms = max_over_ranks(max(e0.elapsed_time(e1), 0.0))
    e2e_value = world * evals_per_step / (e2e_ms / e2e_steps * 1e-3)
    # the same job one call at a time (each refine joins the caller's stream before the next starts): its latency
    for _ in range(2):
        pipe.refine(x_host, out_host)
    barrier()
    e0.record()
    for _ in range(e2e_steps):
        pipe.refine(x_host, out_host)
    e1.record()
    barrier()
    e2e_serial_ms = max_over_ranks(e0.elapsed_time(e1)) / e2e_steps
    h2d = x_host.numel() * 4
    d2h = out_host.numel() * 4
    # the box's own floor for that traffic: the same two pinned buffers copied in and out at once on two streams, no
    # kernels (every rank at the same time: the ranks share the host's memory system) - the e2e figure is PCIe-bound and
    # moves with the box (1.64 to 2.2 ms seen), so the line carries its denominator
    s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    d_in, d_out = torch.empty_like(x0), torch.empty_like(x0)

    def raw_copies(n):
        for _ in range(n):
            with torch.cuda.stream(s_in):
                d_in.copy_(x_host, non_blocking=True)
            with torch.cuda.stream(s_out):
                out_host.copy_(d_out, non_blocking=True)
        torch.cuda.current_stream(dev).wait_stream(s_in)
        torch.cuda.current_stream(dev).wait_stream(s_out)

    raw_copies(2)
    barrier()
    s_in.wait_stream(torch.cuda.current_stream(dev))
    s_out.wait_stream(torch.cuda.current_stream(dev))
    e0.record()
    s_in.wait_event(e0)
    s_out.wait_event(e0)
    raw_copies(e2e_steps)
    e1.record()
    barrier()
    raw_copy_ms = max_over_ranks(e0.elapsed_time(e1)) / e2e_steps
    del d_in, d_out

    # ---- the same iteration on ONE stream (assembly and solve back to back), for comparison
    n_single = steps
    barrier()
    e0.record()
    for _ in range(n_single):
        step()
    e1.record()
    torch.cuda.synchronize(dev)
    ms_single = e0.elapsed_time(e1) / n_single

    # ---- per-kernel durations (live, CUDA events on the launching stream) for the roofline
    n_prof = steps
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(n_prof)]
    ws = ops._workspace(dev, lib.cppflow_lm_full_workspace_bytes(rid, P, T), "lm_full")
    cu, tc, no = ops._obs(ob)
    st = _lib.stream_ptr(dev)
    for i in range(n_prof):
        ev[i][0].record()
        _lib.check(lib.cppflow_lm_full_assemble(rid, prm, _lib.ptr(x0), None, _lib.ptr(problem.target_path), P, T, cu, tc,
                                                no, _lib.ptr(ws), ws.numel(), st))
        ev[i][1].record()
        _lib.check(lib.cppflow_lm_full_solve(rid, prm, _lib.ptr(x0), P, T, 1, _lib.ptr(ws), ws.numel(), _lib.ptr(x_out), st))
        ev[i][2].record()
    torch.cuda.synchronize(dev)
    ms_assemble = statistics.mean(ev[i][0].elapsed_time(ev[i][1]) for i in range(n_prof))
    ms_solve = statistics.mean(ev[i][1].elapsed_time(ev[i][2]) for i in range(n_prof))

    def timed(fn, reps=10):
        fn()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize(dev)
        return a.elapsed_time(b) / reps

    # the other kernels of the path at the headline size (8192 x 300 configurations each)
    prm_pose, prm_diff = ops.make_params(ALT_LOSS_V2_1_POSE), ops.make_params(ALT_LOSS_V2_1_DIFF)
    ms_pose = timed(lambda: ops.lm_pose_step(rid, D, prm_pose, x0, problem.target_path, True, out=x_out))
    ms_flags = timed(lambda: ops.collision_flags(rid, D, x0, ob))
    ms_metrics = timed(lambda: ops.path_metrics(rid, D, x0, problem.target_path, P, T, ob))
    ms_diff = timed(lambda: ops.lm_full_step(rid, D, prm_diff, x0, None, problem.target_path, P, T, ob, True, out=x_out))

    # ---- FP32 peak measured live (MEASURED_PEAKS.json has no FP32 entry)
    scratch = torch.zeros(16, device=dev)
    flops = ctypes.c_double(0.0)
    blocks, iters = 148 * 2 * 4, 4096
    for _ in range(2):
        _lib.check(lib.cppflow_fp32_probe(blocks, iters, _lib.ptr(scratch), ctypes.byref(flops), st))
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pe0.record()
    for _ in range(5):
        _lib.check(lib.cppflow_fp32_probe(blocks, iters, _lib.ptr(scratch), ctypes.byref(flops), st))
    pe1.record()
    torch.cuda.synchronize(dev)
    fp32_peak_tflops = 5 * flops.value / (pe0.elapsed_time(pe1) * 1e-3) / 1e12

    peaks = {}
    try:
        with open(os.path.join(REPO, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    hbm_src = "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    traffic = None
    try:
        with open(os.path.join(REPO, "profiles", "traffic.json")) as f:
            traffic = json.load(f)
    except Exception:
        pass

    achieved_tflops = F_ASSEMBLE * evals_per_step / (ms_assemble * 1e-3) / 1e12
    ws_bytes = lib.cppflow_lm_full_workspace_bytes(rid, P, T)
    roofline = {
        "kernel": "lm_assemble_kernel<Fetch> (FK + Jacobian + pose error + capsule distances + normal-equation blocks)",
        "bound": "fp32",
        "achieved": achieved_tflops,
        "peak": fp32_peak_tflops,
        "unit": "TFLOP/s",
        "frac": achieved_tflops / fp32_peak_tflops,
        "peak_source": "measured live: cppflow_fp32_probe (8 independent FMA chains/thread, 148x8 CTAs x 1024 thr)",
        "flop_per_eval": F_ASSEMBLE,
        "evals_per_launch": evals_per_step,
        "ms_per_launch": ms_assemble,
        "traffic": (traffic or {}).get("lm_assemble_kernel"),
    }
    solve_bytes = SOLVE_WS_PASSES * ws_bytes + 2 * x0.numel() * 4  # block passes over the workspace; read q, write x
    roofline_solve = {
        "kernel": "lm_block_solve_kernel<Fetch> (twisted block-Thomas sweep, TMA bulk-copy block loads)",
        "bound": "hbm",
        "achieved": solve_bytes / (ms_solve * 1e-3) / 1e9,
        "peak": hbm_peak,
        "unit": "GB/s",
        "frac": solve_bytes / (ms_solve * 1e-3) / 1e9 / hbm_peak,
        "peak_source": hbm_src,
        "bytes_per_launch": solve_bytes,
        "ms_per_launch": ms_solve,
        "traffic": (traffic or {}).get("lm_block_solve_kernel"),
    }
    step_tflops = F_STEP_SURVEY * evals_per_step / (ms_per_step * 1e-3) / 1e12
    roofline_step = {
        "what": "whole fused iteration (the K timed steps INCLUDING the cost-argmin tail), SURVEY 8d figure of 9.1 kFLOP per evaluation",
        "bound": "fp32", "achieved": step_tflops, "peak": fp32_peak_tflops, "unit": "TFLOP/s",
        "frac": step_tflops / fp32_peak_tflops,
        "frac_steps_only": F_STEP_SURVEY * evals_per_step / (ms_steps_only * 1e-3) / 1e12 / fp32_peak_tflops,
        "hbm_algorithmic_gbs": BYTES_PER_EVAL * evals_per_step / (ms_per_step * 1e-3) / 1e9,
        "hbm_peak_gbs": hbm_peak,
    }

    def frac_fp32(flop_per_eval, ms):
        return flop_per_eval * evals_per_step / (ms * 1e-3) / 1e12 / fp32_peak_tflops

    rooflines_other = {
        "lm_pose_step_kernel": {"bound": "fp32", "flop_per_eval": F_POSE_STEP, "ms_per_launch": ms_pose,
                                "frac": frac_fp32(F_POSE_STEP, ms_pose),
                                "hbm_frac": BYTES_PER_EVAL * evals_per_step / (ms_pose * 1e-3) / 1e9 / hbm_peak},
        "collision_flags_kernel": {"bound": "fp32", "flop_per_eval": F_FLAGS, "ms_per_launch": ms_flags,
                                   "frac": frac_fp32(F_FLAGS, ms_flags)},
        "path_metrics_kernel": {"bound": "fp32", "flop_per_eval": F_FLAGS + 90, "ms_per_launch": ms_metrics,
                                "frac": frac_fp32(F_FLAGS + 90, ms_metrics)},
        "differencing_step (assemble + solve, ALT_LOSS_V2_1_DIFF)": {"ms_per_step": ms_diff},
    }

    # ---- quality: the reference's alternating step sequence on the collision-free variant of the workload; the cost
    # argmin then has valid paths to choose from (the headline workload's target path runs through a cuboid)
    def quality():
        sched = "pppddppdppp"
        prob_f = synthetic_problem(robot, T, device=dev, **FEASIBLE)
        _, xf_host = synthetic_seeds_host(robot, P, T, shard=rank, **FEASIBLE)
        xf = xf_host.to(dev)
        bufs = [torch.empty_like(xf), torch.empty_like(xf)]
        mq = torch.empty((P, 8), device=dev, dtype=torch.float32)

        def run():
            src = xf
            for i, c in enumerate(sched):
                dst = bufs[i % 2]
                if c == "p":
                    ops.lm_pose_step(rid, D, prm_pose, src, prob_f.target_path, True, out=dst)
                else:
                    ops.lm_full_step(rid, D, prm_diff, src, None, prob_f.target_path, P, T, prob_f.obstacle_tables, True, out=dst)
                src = dst
            _lib.check(lib.cppflow_path_metrics(rid, _lib.ptr(src), _lib.ptr(prob_f.target_path), P, T,
                                                *ops._obs(prob_f.obstacle_tables), _lib.ptr(mq), st))
            return enqueue_argmin(mq, prob_f.constraints, rank * P, world)

        run().result()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a.record()
        pend = run()
        b.record()
        barrier()
        ms = max_over_ranks(a.elapsed_time(b))
        bq = pend.result()
        assert bq.valid and bq.cost < 1e9, f"no valid path after {sched}: best cost {bq.cost}"
        return {"schedule": sched, "workload": f"same shape, collision-free reference path (seed {FEASIBLE['seed']}, amplitude {FEASIBLE['amp']})",
                "ms_total": ms, "evals_per_s": world * evals_per_step * len(sched) / (ms * 1e-3),
                "n_valid": bq.n_valid, "n_paths": world * P, "best_cost": bq.cost, "best_rank": bq.rank, "best_path": bq.index}

    def guarded(fn, *a, **kw):
        # the extra keys below must never cost the headline its line: a failure is reported in place
        try:
            return fn(*a, **kw)
        except Exception as e:  # noqa: BLE001
            import traceback

            traceback.print_exc(file=sys.stderr)
            return {"error": f"{type(e).__name__}: {e}"}

    quality_res = guarded(quality) if world == 1 else quality()  # collective inside: every rank must take part

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    plan = None
    plan_all = None
    dp_ms = None
    if world == 1:
        plan_all = guarded(plan_all_problems_gpu, dev)
        got = guarded(plan_latency_gpu, dev)
        if isinstance(got, tuple):
            plan, plan_problem, plan_qs = got
            if not args.no_cpu_baseline:
                plan["cpu_baseline"] = guarded(plan_latency_cpu, plan_problem, plan_qs, plan["schedule"])

            def dp_times():
                out = {}
                from cppflow_b200.collision_detection import qpaths_batched_collisions
                from cppflow_b200.planners import LmIkCandidateGenerator

                for k in (175, 300):
                    qs = plan_qs.to(dev) if k == 175 else LmIkCandidateGenerator(seed=2)(plan_problem, k).contiguous()
                    sv, evf = qpaths_batched_collisions(plan_problem, qs)
                    ms = timed(lambda: ops.dp_search(rid, D, qs, sv, evf))
                    n_t = qs.shape[1]
                    out[f"k{k}"] = {"ms": ms, "us_per_step": ms * 1e3 / (n_t - 1), "waypoints": n_t,
                                    "flags_ms": timed(lambda: qpaths_batched_collisions(plan_problem, qs))}
                return out

            dp_ms = guarded(dp_times)
        else:
            plan = got

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        rate, dt, cores = cpu_reference_step_rate(T, args.cpu_sample_paths, 2, 1)
        cpu_baseline = {
            "value": rate, "unit": "waypoint-evals/s", "cores": cores, "kind": "port",
            "sample": f"{args.cpu_sample_paths} of {P} paths x {T} waypoints, 2 timed steps ({dt:.2f} s each) of the oracle "
                      f"port of the reference's dense torch path (get_r_and_J all terms + _lm_full_step), fp32, "
                      f"torch {torch.__version__}",
        }

    line = {
        "metric": "waypoint FK+Jac+collision+LM evals/s",
        "value": value,
        "unit": "waypoint-evals/s",
        "n_gpus": world,
        "steps": steps,
        "warmup": warmup,
        "ms_per_step": ms_per_step,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic",
        "config": workload_config(args, world),
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "waypoint-evals/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms / e2e_steps, "wall_ms_per_step": wall / e2e_steps * 1e3, "steps": e2e_steps,
                "api": "cppflow_b200.pipeline.HostPipeline.refine_async(host x -> host x_new), pinned host buffers, "
                       "independent steps two deep in flight",
                "ms_per_step_one_at_a_time": e2e_serial_ms,
                "raw_duplex_copy_ms_per_step": raw_copy_ms, "frac_of_raw_copy": raw_copy_ms / (e2e_ms / e2e_steps)},
        "gpu_launches": steps * 2 * len(rpipe.chunks) + len(rpipe.chunks) + 1,  # K x (assemble + solve) per chunk, metrics per chunk, key + argmin
        "ms_per_step_without_tail": ms_steps_only,
        "single_stream_ms_per_step": ms_single,
        "roofline": roofline,
        "roofline_solve": roofline_solve,
        "roofline_step": roofline_step,
        "rooflines_other": rooflines_other,
        "kernel_ms": {"lm_assemble_kernel": ms_assemble, "lm_block_solve_kernel": ms_solve, "lm_pose_step_kernel": ms_pose,
                      "collision_flags_kernel": ms_flags, "path_metrics_kernel": ms_metrics, "dp_search": dp_ms},
        "strong": strong,
        "strong_preview": strong_preview,
        "quality": quality_res,
        "cpu_baseline": cpu_baseline,
        "plan_latency": plan,
        "plan_all_problems": plan_all,
        "argmin": {"cost": best.cost, "rank": best.rank, "path": best.index, "n_valid": best.n_valid,
                   "trajectory_length": best.trajectory_length,
                   "note": "headline workload: the reference joint path runs through a cuboid, so no path can be valid; "
                           "invalid paths are ranked by trajectory length (see `quality` for the feasible variant)"},
    }
    if dumped is not None:
        line["dump_outputs"] = dumped
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
