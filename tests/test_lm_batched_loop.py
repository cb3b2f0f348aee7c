"""The batched alternating LM loop (csrc/lm_loop_batched.cu, optimization.run_lm_optimization_batched) against the
single-seed native loop, seed by seed and bit for bit; its C ABI's argument checks; the DP backtrack from chosen
terminals; and the planner's `lm_seeds` option against `lm_seeds = 1` on the same candidates."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda:0"
gpu = pytest.mark.gpu

# the argument sets of the planner's two call patterns and a single step (test_native_alternating_loop_equals_python_loop)
LOOP_ARGS = (
    dict(max_n_steps=20, return_if_valid_after_n_steps=0, convergence_threshold=1e6),
    dict(max_n_steps=30, return_if_valid_after_n_steps=int(1e8), convergence_threshold=0.005),
    dict(max_n_steps=1, return_if_valid_after_n_steps=0, convergence_threshold=1e6),
)
PROBLEMS = ("fetch__circle", "fetch_arm__s", "panda__2cubes", "fetch__hello")


def _problem(name):
    from cppflow_b200.data_type_utils import problem_from_filename

    return problem_from_filename(None, name, device=DEV)


def _seed_set(problem):
    """dp_search's path, 48 stand-in candidates and a seed with a mid-path flip: [50, T, ndof]."""
    from cppflow_b200.collision_detection import qpaths_batched_collisions
    from cppflow_b200.planners import LmIkCandidateGenerator
    from cppflow_b200.search import dp_search

    T = problem.n_timesteps
    qs = LmIkCandidateGenerator(seed=1)(problem, 64).contiguous()
    self_v, env_v = qpaths_batched_collisions(problem, qs)
    best = dp_search(problem.robot, qs, self_v, env_v, verbosity=0).to(DEV).contiguous()
    bad = best.clone()
    bad[T // 2:] = bad[T // 2:].flip(0)
    return torch.cat([best[None], qs[:48], bad[None]], dim=0).contiguous()


def _assert_seedwise_equal(problem, seeds, batched, tmax_sec, idx=None, **kw):
    from cppflow_b200.optimization import run_lm_optimization

    idx = range(seeds.shape[0]) if idx is None else idx
    for i in idx:
        b = batched[i]
        a = run_lm_optimization(problem, seeds[i].contiguous(), tmax_sec=tmax_sec, verbosity=0, native=True, **kw)
        assert b.parallel_seed_idx == i
        assert b.schedule == a.schedule, (i, kw, a.schedule, b.schedule)
        assert b.n_steps_taken == a.n_steps_taken and b.is_valid == a.is_valid, (i, kw)
        assert torch.equal(b.x_opt, a.x_opt), (i, kw)


# ---------------------------------------------------------------------------------------------------------------- CPU


def test_header_declares_the_batched_entry_points():
    from cppflow_b200 import _lib

    h = open(os.path.join(REPO, "include", "cppflow_b200.h")).read()
    for name in ("cppflow_lm_alternating_batched_workspace_bytes", "cppflow_lm_alternating_loss_batched",
                 "cppflow_dp_backtrack"):
        assert re.search(r"\b" + name + r"\(", h), name
        assert name in _lib.EXPORTED_SYMBOLS, name
    m = re.search(r"#define CPPFLOW_LM_BATCHED_PINNED_BYTES (\d+)", h)
    assert m and int(m.group(1)) == _lib.LM_BATCHED_PINNED_BYTES
    assert _lib.LM_BATCHED_PINNED_BYTES >= 3 * 4  # two counts and the completion tag


def test_evaluate_rejects_bad_lm_seeds():
    import sys

    sys.path.insert(0, os.path.join(REPO, "tools"))
    try:
        import evaluate
    finally:
        sys.path.pop(0)
    with pytest.raises(SystemExit):
        evaluate.main(["--lm_seeds", "0"])
    with pytest.raises(SystemExit):
        evaluate.main(["--lm_seeds", "4", "--planner", "PlannerSearcher"])


# ---------------------------------------------------------------------------------------------------------------- GPU


@gpu
@pytest.mark.parametrize("name", PROBLEMS)
def test_batched_loop_equals_single_seed_loops(name):
    """Every seed of the batched loop takes the steps, decisions and bits of the single-seed native loop on that seed
    alone: the dp path, 48 candidates and a flipped seed (which take different schedules; some stay invalid)."""
    from cppflow_b200.optimization import run_lm_optimization_batched

    problem = _problem(name)
    seeds = _seed_set(problem)
    outcomes = set()
    for kw in LOOP_ARGS:
        batched = run_lm_optimization_batched(problem, seeds, 30.0, **kw)
        assert len(batched) == seeds.shape[0]
        _assert_seedwise_equal(problem, seeds, batched, 30.0, **kw)
        outcomes |= {(kw["max_n_steps"], r.n_steps_taken, r.is_valid, r.schedule) for r in batched}
    print(f"{name}: {len(outcomes)} distinct (budget, n_steps_taken, is_valid, schedule) outcomes over the seeds")


@gpu
def test_batched_loop_one_seed():
    from cppflow_b200.optimization import run_lm_optimization_batched

    problem = _problem("fetch_arm__s")
    seeds = _seed_set(problem)[:1].contiguous()
    for kw in LOOP_ARGS:
        _assert_seedwise_equal(problem, seeds, run_lm_optimization_batched(problem, seeds, 30.0, **kw), 30.0, **kw)


def _metrics_cluster_size(T):
    """Cluster size path_metrics gives one path of T waypoints (k_metrics.cu: G lanes per waypoint, <= 8 CTAs)."""
    G = 4 if T <= 256 else (2 if T <= 512 else 1)
    per_cta = 128 // G
    return min((T + per_cta - 1) // per_cta, 8)


def _native_runs(problem, seeds, tmax_sec, **kw):
    """(batched, singles) through the ops layer: lists of (x_opt, n_steps_taken, is_valid, schedule, last_metrics)."""
    from cppflow_b200 import ops
    from cppflow_b200.lm_hyper_parameters import ALT_LOSS_V2_1_DIFF, ALT_LOSS_V2_1_POSE

    rob = problem.robot
    args = (rob.robot_id, rob.ndof, ops.make_params(ALT_LOSS_V2_1_DIFF), ops.make_params(ALT_LOSS_V2_1_POSE),
            problem.constraints)
    tail = (problem.obstacle_tables, kw["max_n_steps"], tmax_sec, kw["return_if_valid_after_n_steps"],
            kw["convergence_threshold"])
    batched = ops.lm_alternating_loss_batched(*args, seeds, problem.target_path, *tail)
    singles = [ops.lm_alternating_loss(*args, s.contiguous(), problem.target_path, problem.n_timesteps, *tail)
               for s in seeds]
    return batched, singles


def _assert_native_equal(batched, singles):
    """Every field of every seed, the seven metric columns of the last iterate bit for bit (column 7 is no metric: the
    single loop leaves its completion tag there, the batched loop 0)."""
    for i, (b, a) in enumerate(zip(batched, singles)):
        assert b[3] == a[3], (i, a[3], b[3])
        assert b[1] == a[1] and b[2] == a[2], i
        assert torch.equal(b[0], a[0]), i
        assert b[4][:7] == a[4][:7], (i, a[4], b[4])
        assert b[4][7] == 0.0, i


@gpu
def test_batched_loop_keeps_the_single_path_metrics_kernel_for_many_differencing_seeds():
    """path_metrics takes one CTA per path once paths x cluster size > 296 CTAs, and that kernel adds the trajectory
    length in another order.  300 seeds that are pose-valid after their first step take their differencing step in the
    SAME iteration, well above the switch: the batched loop must still give every seed the single loop's metrics (the
    trajectory length bit for bit) and decisions."""
    from cppflow_b200 import ops
    from cppflow_b200.optimization import run_lm_optimization

    problem = _problem("fetch__circle")
    rob, T = problem.robot, problem.n_timesteps
    csize = _metrics_cluster_size(T)
    n_switch = 296 // csize + 1  # the fewest paths for which path_metrics switches kernels
    base = run_lm_optimization(problem, _seed_set(problem)[0].contiguous(), tmax_sec=30.0, verbosity=0,
                               max_n_steps=20, return_if_valid_after_n_steps=0, convergence_threshold=1e6)
    assert base.is_valid
    g = torch.Generator(device=DEV).manual_seed(0)
    noise = 1e-4 * torch.randn((300, T, rob.ndof), generator=g, device=DEV)
    seeds = (base.x_opt[None] + noise).contiguous()  # a refined path, slightly disturbed: pose-valid after one step
    for kw in LOOP_ARGS[:2]:
        batched, singles = _native_runs(problem, seeds, 60.0, **kw)
        _assert_native_equal(batched, singles)
        per_iteration = [sum(1 for r in batched if len(r[3]) > j and r[3][j] == "d")
                         for j in range(max(len(r[3]) for r in batched))]
        assert max(per_iteration) >= n_switch, (per_iteration, n_switch)
    # the switch does change the trajectory length of these paths: dropping the one-path kernel would be caught
    final = torch.stack([r[0] for r in batched]).reshape(-1, rob.ndof)
    many = ops.path_metrics(rob.robot_id, rob.ndof, final, problem.target_path, 300, T, problem.obstacle_tables)
    one = torch.stack([ops.path_metrics(rob.robot_id, rob.ndof, r[0], problem.target_path, 1, T,
                                        problem.obstacle_tables)[0] for r in batched])
    n_diff = int((many[:, 4] != one[:, 4]).sum())
    print(f"{n_diff} of 300 trajectory lengths differ between the one-path and the many-path metrics kernel")
    assert n_diff > 0


@gpu
def test_batched_loop_long_paths_take_the_unfused_pose_step():
    """T > 1024: the pose step is not fused with the metrics (gathered lm_pose_step over all pose seeds, then the
    metrics of every gathered path), as in the single loop.  fetch__circle's target path with every pose repeated 4x."""
    import dataclasses

    base = _problem("fetch__circle")
    seeds = _seed_set(base)
    rep = 4
    problem = dataclasses.replace(base, target_path=base.target_path.repeat_interleave(rep, dim=0).contiguous())
    assert problem.n_timesteps > 1024
    idx = [0, 1, 2, 3, 10, 20, 30, 49]
    long_seeds = seeds[idx].repeat_interleave(rep, dim=1).contiguous()
    outcomes = set()
    for kw in LOOP_ARGS:
        batched, singles = _native_runs(problem, long_seeds, 120.0, **kw)
        _assert_native_equal(batched, singles)
        outcomes |= {r[3] for r in batched}
    assert any("p" in s for s in outcomes), outcomes
    print(f"long paths: schedules {sorted(outcomes)}")


@gpu
def test_batched_loop_2048_seeds():
    from cppflow_b200.optimization import run_lm_optimization_batched
    from cppflow_b200.planners import LmIkCandidateGenerator

    problem = _problem("fetch__circle")
    seeds = LmIkCandidateGenerator(seed=2)(problem, 2048).contiguous()
    kw = dict(max_n_steps=6, return_if_valid_after_n_steps=int(1e8), convergence_threshold=0.005)
    batched = run_lm_optimization_batched(problem, seeds, 60.0, **kw)
    idx = np.random.default_rng(0).choice(2048, size=16, replace=False).tolist()
    _assert_seedwise_equal(problem, seeds, batched, 60.0, idx=idx, **kw)


@gpu
def test_batched_loop_edge_cases():
    from cppflow_b200.optimization import run_lm_optimization_batched

    problem = _problem("panda__2cubes")
    seeds = _seed_set(problem)[:12].contiguous()
    # no step: the seeds come back unchanged
    for r, s in zip(run_lm_optimization_batched(problem, seeds, 30.0, 0, 0, 1e6), seeds):
        assert r.n_steps_taken == 0 and not r.is_valid and r.schedule == ""
        assert torch.equal(r.x_opt, s)
    kw = dict(max_n_steps=1, return_if_valid_after_n_steps=0, convergence_threshold=1e6)
    _assert_seedwise_equal(problem, seeds, run_lm_optimization_batched(problem, seeds, 30.0, **kw), 30.0, **kw)
    # tmax_sec = 0: both loops stop after the decisions of iteration 0
    kw = dict(max_n_steps=20, return_if_valid_after_n_steps=0, convergence_threshold=1e6)
    batched = run_lm_optimization_batched(problem, seeds, 0.0, **kw)
    assert all(r.n_steps_taken == 0 and len(r.schedule) == 1 for r in batched)
    _assert_seedwise_equal(problem, seeds, batched, 0.0, **kw)
    # tmax_sec / max_n_steps = None as in run_lm_alternating_loss
    kw = dict(max_n_steps=3, return_if_valid_after_n_steps=0, convergence_threshold=1e6)
    _assert_seedwise_equal(problem, seeds, run_lm_optimization_batched(problem, seeds, None, **kw), None, **kw)


@gpu
def test_batched_loop_truncates_long_schedules_like_the_single_loop():
    """300 iterations (no convergence: threshold 0) record CPPFLOW_LM_SCHEDULE_MAX - 1 = 255 step types in both loops."""
    from cppflow_b200.optimization import run_lm_optimization_batched

    problem = _problem("fetch__circle")
    seeds = _seed_set(problem)[:3].contiguous()
    kw = dict(max_n_steps=300, return_if_valid_after_n_steps=int(1e8), convergence_threshold=0.0)
    batched = run_lm_optimization_batched(problem, seeds, 120.0, **kw)
    assert all(r.n_steps_taken == 299 and len(r.schedule) == 255 for r in batched)
    _assert_seedwise_equal(problem, seeds, batched, 120.0, **kw)


@gpu
def test_batched_loop_argument_errors():
    from cppflow_b200 import _lib, ops
    from cppflow_b200.lm_hyper_parameters import ALT_LOSS_V2_1_DIFF, ALT_LOSS_V2_1_POSE

    lib = _lib.load()
    problem = _problem("fetch__circle")
    rob, T = problem.robot, problem.n_timesteps
    N = 4
    seeds = _seed_set(problem)[:N].contiguous()
    target = problem.target_path.contiguous()
    need = lib.cppflow_lm_alternating_batched_workspace_bytes(rob.robot_id, N, T)
    assert need > 0
    assert lib.cppflow_lm_alternating_batched_workspace_bytes(rob.robot_id, 2 * N, T) > need
    ws = torch.empty(need + 512, dtype=torch.uint8, device=DEV)
    base = ws.data_ptr() + (-ws.data_ptr()) % 256
    pinned = torch.zeros(_lib.LM_BATCHED_PINNED_BYTES // 4, dtype=torch.int32).pin_memory()
    out = torch.empty_like(seeds)
    res = (_lib.LmLoopResultC * N)()
    pd, pp = ops.make_params(ALT_LOSS_V2_1_DIFF), ops.make_params(ALT_LOSS_V2_1_POSE)
    c = problem.constraints
    cons = _lib.ConstraintsC(c.max_allowed_position_error_cm, c.max_allowed_rotation_error_deg, c.max_allowed_mjac_deg,
                             c.max_allowed_mjac_cm)
    ob = problem.obstacle_tables
    cu, tc, no = ops._obs(ob)
    stream = _lib.stream_ptr(DEV)

    def call(n=N, x=seeds.data_ptr(), wsp=base, wsb=need, pin=pinned.data_ptr(), results=res):
        return lib.cppflow_lm_alternating_loss_batched(rob.robot_id, pd, pp, cons, C.c_void_p(x), C.c_void_p(target.data_ptr()),
                                                       n, T, cu, tc, no, 5, 30.0, 0, 1e6, C.c_void_p(wsp), wsb,
                                                       C.c_void_p(pin), C.c_void_p(out.data_ptr()), results, stream)

    E_INVALID, E_WORKSPACE = -1, -3
    assert call(wsb=need - 1) == E_WORKSPACE
    assert call(wsp=base + 16, wsb=need) == E_INVALID
    assert call(x=0) == E_INVALID
    assert call(pin=0) == E_INVALID
    assert call(results=None) == E_INVALID
    assert call(n=-1) == E_INVALID
    out.fill_(-7.0)
    assert call(n=0, x=0, wsp=0, wsb=0, pin=0, results=None) == 0  # nothing to do, nothing touched
    torch.cuda.synchronize()
    assert bool((out == -7.0).all())
    assert call() == 0  # and a good call still works after the refused ones
    torch.cuda.synchronize()


@gpu
def test_dp_backtrack_from_every_terminal():
    """k = 175 fetch__circle search: the backtrack from every terminal equals a CPU backtrack of memo, bit for bit;
    the argmin terminal gives dp_search's path."""
    from cppflow_b200 import ops
    from cppflow_b200.collision_detection import qpaths_batched_collisions
    from cppflow_b200.planners import LatentIkCandidateGenerator
    from cppflow_b200.search import dp_search

    problem = _problem("fetch__circle")
    qs = LatentIkCandidateGenerator(seed=3)(problem, 175).contiguous()
    k, T, D = qs.shape
    self_v, env_v = qpaths_batched_collisions(problem, qs)
    best, memo, costs, _ = dp_search(problem.robot, qs, self_v, env_v, verbosity=0, return_details=True)
    terminals = torch.arange(k, dtype=torch.int32, device=DEV)
    paths = ops.dp_backtrack(qs, memo, terminals).cpu()
    q_cpu, memo_cpu = qs.cpu(), memo.cpu()
    for j in range(k):
        i = j
        ref = torch.empty((T, D))
        for t in range(T - 1, -1, -1):  # oracle/search.py:71-75
            ref[t] = q_cpu[i, t]
            i = int(memo_cpu[i, t])
        assert torch.equal(paths[j], ref), j
    last = costs[:, T - 1].cpu()
    i_best = int(torch.argmin(last))  # first index on ties, as torch.min
    assert torch.equal(paths[i_best], best.cpu())
    with pytest.raises(ValueError):
        ops.dp_backtrack(qs, memo, torch.tensor([k], dtype=torch.int32))


def _settings():
    from cppflow_b200.data_types import PlannerSettings

    return PlannerSettings(k=175, tmax_sec=30.0, anytime_mode_enabled=False, verbosity=0)


def _compare_planners(names, make_generator, n_seeds):
    from cppflow_b200.planners import CppFlowPlanner

    one, many = {}, {}
    for name in names:
        problem = _problem(name)
        a = CppFlowPlanner(_settings(), problem.robot, make_generator()).generate_plan(problem)
        b = CppFlowPlanner(_settings(), problem.robot, make_generator(), lm_seeds=n_seeds).generate_plan(problem)
        one[name], many[name] = a, b
        assert "lm_seed_index" not in a.debug_info
        idx = b.debug_info["lm_seed_index"]
        assert 0 <= idx < n_seeds
        if a.plan.is_valid:
            assert b.plan.is_valid, name
        if idx == 0:  # seed 0 is dp_search's own path: the same refinement as lm_seeds = 1
            assert b.plan.is_valid == a.plan.is_valid, name
            assert torch.equal(a.plan.q_path, b.plan.q_path), name
            assert a.debug_info["n_optimization_steps"] == b.debug_info["n_optimization_steps"], name
    n1 = sum(r.plan.is_valid for r in one.values())
    nn = sum(r.plan.is_valid for r in many.values())
    print(f"valid plans: lm_seeds=1: {n1}/{len(names)}, lm_seeds={n_seeds}: {nn}/{len(names)}")
    assert nn >= n1
    return one, many


@gpu
def test_planner_lm_seeds_never_loses_a_valid_plan():
    from cppflow_b200.data_type_utils import ALL_PROBLEM_FILENAMES
    from cppflow_b200.planners import LatentIkCandidateGenerator

    _compare_planners(ALL_PROBLEM_FILENAMES, lambda: LatentIkCandidateGenerator(seed=3), 16)


@gpu
def test_planner_lm_seeds_on_flappy_bird_with_the_stand_in_generator():
    """Records whether the DP's next-best paths turn panda__flappy_bird valid with the stand-in candidates; only the
    monotonicity is asserted."""
    from cppflow_b200.planners import LmIkCandidateGenerator

    for n in (16, 64):
        one, many = _compare_planners(["panda__flappy_bird"], lambda: LmIkCandidateGenerator(seed=1), n)
        print(f"panda__flappy_bird: lm_seeds=1 valid={one['panda__flappy_bird'].plan.is_valid}, "
              f"lm_seeds={n} valid={many['panda__flappy_bird'].plan.is_valid} "
              f"(seed {many['panda__flappy_bird'].debug_info['lm_seed_index']})")


@gpu
def test_plan_many_runs_lm_seeds_planners_one_by_one():
    from cppflow_b200.planners import CppFlowPlanner, LmIkCandidateGenerator, plan_many

    names = ["fetch_arm__s", "panda__1cube"]
    problems = [_problem(n) for n in names]

    def factory(problem):
        return CppFlowPlanner(_settings(), problem.robot, LmIkCandidateGenerator(seed=1), lm_seeds=8)

    seq = [factory(p).generate_plan(p) for p in problems]
    con = plan_many(factory, problems)
    for name, a, b in zip(names, seq, con):
        assert a.plan.is_valid == b.plan.is_valid, name
        assert torch.equal(a.plan.q_path, b.plan.q_path), name
        assert a.debug_info["lm_seed_index"] == b.debug_info["lm_seed_index"], name
