"""The Levenberg-Marquardt refinement loop with the reference's call surface (cppflow/optimization.py).

  levenberg_marquardt_only_pose  :61-92    -> csrc/k_pose.cu (one fused kernel: FK, Jacobian, error, solve)
  levenberg_marquardt_full       :116-144  -> csrc/k_lm_full.cu (implicit block-tridiagonal assembly + block Cholesky)
  run_lm_alternating_loss        :147-373  same control flow; one device->host read of 8 floats per iteration
  run_lm_optimization            :376-426
Unlike the reference (`assert parallel_count == 1`, :128) the full step handles `parallel_count` stacked paths in
one launch; `run_lm_fixed_schedule` runs a data-independent step sequence over thousands of paths (SURVEY 8d, config 5);
`run_lm_optimization_batched` runs the alternating loop, with its per-path decisions, over many seeds of one problem.
"""
from dataclasses import dataclass
from time import time
from typing import Dict, List, Optional
import warnings

import torch

from . import ops
from .config import ENV_COLLISIONS_IGNORED, SELF_COLLISIONS_IGNORED
from .data_types import Constraints, Problem
from .lm_hyper_parameters import ALT_LOSS_V2_1_DIFF, ALT_LOSS_V2_1_POSE, OptimizationParameters, all_terms_parameters
from .optimization_utils import LmResidualFns, clamp_to_joint_limits, path_metrics, x_is_valid


@dataclass
class OptimizationProblem:
    problem: Problem
    constraints: Constraints
    seed: torch.Tensor
    target_path: torch.Tensor
    verbosity: int
    parallel_count: int
    results_df: Optional[Dict]

    @property
    def robot(self):
        return self.problem.robot

    @property
    def n_timesteps(self):
        return self.problem.n_timesteps


@dataclass
class OptimizationState:
    x: torch.Tensor
    n_steps: int
    t0: float


@dataclass
class OptimizationResult:
    x_opt: torch.Tensor
    n_steps_taken: int
    is_valid: bool
    parallel_seed_idx: int
    schedule: str = ""  # not in the reference: the step types taken, 'p' = pose-only, 'd' = differencing


def levenberg_marquardt_only_pose(opt_problem: OptimizationProblem, opt_state: OptimizationState,
                                  opt_params: OptimizationParameters, return_residual: bool = False,
                                  clamp: bool = False):
    """x + dx with (J^T J + lambda I) dx = J^T e per waypoint; does not mutate opt_state.x.  With
    return_residual=True also returns the alpha-scaled J [n,6,ndof] and e [n,6,1] like the reference."""
    robot = opt_problem.robot
    target = opt_problem.problem.target_path  # row i of x uses target row i % T
    return ops.lm_pose_step(robot.robot_id, robot.ndof, ops.make_params(opt_params), opt_state.x, target, clamp,
                            return_residual=return_residual)


def levenberg_marquardt_full(opt_problem: OptimizationProblem, opt_state: OptimizationState,
                             opt_params: OptimizationParameters, return_residual: bool = False, clamp: bool = False):
    """x + dx with (J^T J + lambda I) dx = J^T r over the whole path(s).  With return_residual=True the dense
    LmJacobian / LmResidual of the (single) path are built as well - debugging only."""
    robot = opt_problem.robot
    problem = opt_problem.problem
    xv = opt_params.virtual_configs if opt_params.use_virtual_configs else None
    if xv is not None and xv.numel() == 0:
        xv = None
    # one path: the solve's dependent chain is the whole step -> the segmented solve, as in the native loop
    x_new = ops.lm_full_step(robot.robot_id, robot.ndof, ops.make_params(opt_params), opt_state.x, xv,
                             problem.target_path, opt_problem.parallel_count, problem.n_timesteps,
                             problem.obstacle_tables, clamp,
                             segments=ops.LOOP_SEGMENTS if opt_problem.parallel_count == 1 else 0)
    if return_residual:
        assert opt_problem.parallel_count == 1, "dense residuals are only built for a single path"
        jac, res = LmResidualFns.get_r_and_J(opt_params, robot, opt_state.x, problem.target_path,
                                             Tcuboids=problem.obstacles_Tcuboids, cuboids=problem.obstacles_cuboids)
        return x_new, jac, res
    return x_new


def run_lm_fixed_schedule(problem: Problem, x_seed: torch.Tensor, schedule: str, parallel_count: int = 1,
                          params_pose: OptimizationParameters = ALT_LOSS_V2_1_POSE,
                          params_diff: OptimizationParameters = ALT_LOSS_V2_1_DIFF,
                          params_all: Optional[OptimizationParameters] = None) -> torch.Tensor:
    """Run a fixed step sequence over `parallel_count` stacked paths with no host synchronisation:
    'p' = pose-only step, 'd' = differencing step (virtual configs = current x, optimization.py:253),
    'a' = all residual terms on.  Every step is followed by clamp_to_joint_limits (fused into the kernels)."""
    robot = problem.robot
    T = problem.n_timesteps
    assert x_seed.shape == (T * parallel_count, robot.ndof)
    x = x_seed
    prm_pose, prm_diff = ops.make_params(params_pose), ops.make_params(params_diff)
    prm_all = ops.make_params(params_all if params_all is not None else all_terms_parameters())
    for step in schedule:
        if step == "p":
            x = ops.lm_pose_step(robot.robot_id, robot.ndof, prm_pose, x, problem.target_path, True)
        elif step in ("d", "a"):
            x = ops.lm_full_step(robot.robot_id, robot.ndof, prm_diff if step == "d" else prm_all, x, None,
                                 problem.target_path, parallel_count, T, problem.obstacle_tables, True)
        else:
            raise ValueError(f"unknown step '{step}' in schedule (use 'p', 'd', 'a')")
    return x


def run_lm_alternating_loss(opt_problem: OptimizationProblem, opt_state: OptimizationState,
                            params_diff: OptimizationParameters, params_pose: OptimizationParameters,
                            return_residuals: bool, tmax_sec: float, max_n_steps: int,
                            return_if_valid_after_n_steps: int, convergence_threshold: float, verbosity: int = 0,
                            save_images: bool = False, results_df: Optional[Dict] = None, mesh_validator=None,
                            native: bool = True):
    """Control flow of optimization.py:147-373 for ONE path (parallel_count == 1).  Without a mesh validator the loop
    runs inside the library (csrc/lm_loop.cu: same decisions, ~10 us of host time per iteration);
    `run_lm_alternating_loss_python` is the same loop in Python, kept for the mesh-validator callback, for
    verbosity > 1 and as the cross-check of the native loop (tests/test_gpu_planner.py)."""
    assert opt_problem.parallel_count == 1, "the alternating loop is per path; batch with run_lm_fixed_schedule"
    if save_images or return_residuals:
        raise NotImplementedError("save_images / return_residuals (debug outputs of the reference's loop) are not reproduced")
    if results_df is not None:
        # the reference logs every iterate through Problem.write_qpath_to_results_df, which itself raises
        # NotImplementedError (data_types.py:419-420): passing a results_df fails there too, it is never silently ignored
        raise NotImplementedError("results_df logging is not available (Problem.write_qpath_to_results_df raises in the "
                                  "reference as well, data_types.py:419-420)")
    if tmax_sec is None:
        assert (max_n_steps is not None) and (return_if_valid_after_n_steps is not None)
        assert return_if_valid_after_n_steps <= max_n_steps
        tmax_sec = float("inf")
    if max_n_steps is None:
        assert tmax_sec is not None
        max_n_steps = int(1e9)
    if native and mesh_validator is None and verbosity <= 1 and not (SELF_COLLISIONS_IGNORED or ENV_COLLISIONS_IGNORED):
        problem, robot = opt_problem.problem, opt_problem.robot
        x_opt, n_steps, is_valid, schedule, _ = ops.lm_alternating_loss(
            robot.robot_id, robot.ndof, ops.make_params(params_diff), ops.make_params(params_pose),
            opt_problem.constraints, opt_state.x, problem.target_path, problem.n_timesteps, problem.obstacle_tables,
            min(max_n_steps, 2 ** 31 - 1), tmax_sec, min(return_if_valid_after_n_steps, 2 ** 31 - 1), convergence_threshold)
        return OptimizationResult(x_opt=x_opt, n_steps_taken=n_steps, is_valid=is_valid, parallel_seed_idx=0,
                                  schedule=schedule)
    return run_lm_alternating_loss_python(opt_problem, opt_state, params_diff, params_pose, tmax_sec, max_n_steps,
                                          return_if_valid_after_n_steps, convergence_threshold, verbosity, mesh_validator)


def run_lm_alternating_loss_python(opt_problem: OptimizationProblem, opt_state: OptimizationState,
                                   params_diff: OptimizationParameters, params_pose: OptimizationParameters,
                                   tmax_sec: float, max_n_steps: int, return_if_valid_after_n_steps: int,
                                   convergence_threshold: float, verbosity: int = 0, mesh_validator=None):
    problem = opt_problem.problem

    def printc(*args, **kwargs):
        if verbosity > 1:
            print(*args, **kwargs)

    params_diff = OptimizationParameters(**params_diff.__dict__)  # copies: virtual_configs is reassigned below
    params_pose = OptimizationParameters(**params_pose.__dict__)

    tls_post_differencing = []
    last_valid = None
    last_valid_idx = -1
    pose_pos_valid = True  # the reference starts (True, False): the first step is pose-only (:219-220)
    pose_rot_valid = False
    converged = False
    i = 0
    schedule = ""
    t0 = time()
    for i in range(max_n_steps):
        if pose_pos_valid and pose_rot_valid:
            # virtual configs = current solution (:253) -> their residual is identically 0: pass xv = None
            params_diff.virtual_configs = torch.tensor([])
            printc("  ----> differencing")
            x_new = levenberg_marquardt_full(opt_problem, opt_state, params_diff, clamp=True)
            was_differencing = True
            schedule += "d"
        else:
            printc("  --> only pose")
            x_new = levenberg_marquardt_only_pose(opt_problem, opt_state, params_pose, clamp=True)
            was_differencing = False
            schedule += "p"
        opt_state.x = x_new  # clamp_to_joint_limits is fused into both kernels (:259)

        metrics = path_metrics(problem, opt_state.x, 1).cpu()  # one sync: TL (:268) and the validity inputs (:318)
        tl_new = float(metrics[0, 4])
        if was_differencing:
            if not converged and len(tls_post_differencing) > 0:
                diff = abs(tl_new - tls_post_differencing[-1])
                if diff < convergence_threshold:
                    converged = True
                    if last_valid_idx == i - 1:
                        break
            tls_post_differencing.append(tl_new)

        x_sol, _, (pose_pos_valid, pose_rot_valid, _mr, _mp, _sc, _ec) = x_is_valid(
            problem, opt_problem.constraints, opt_problem.target_path, opt_state.x, parallel_count=1,
            verbosity=verbosity, mesh_validator=mesh_validator, metrics=metrics,
        )
        if x_sol is not None:
            last_valid_idx = i
            last_valid = opt_state.x.clone()
            if converged:
                break
        if time() - t0 > tmax_sec:
            if last_valid is not None:
                opt_state.x = last_valid.clone()
            break
        if last_valid is not None:
            if i > return_if_valid_after_n_steps:
                break
            if i > max_n_steps:
                break
    x_return = last_valid if last_valid is not None else opt_state.x
    return OptimizationResult(x_opt=x_return, n_steps_taken=i, is_valid=last_valid is not None, parallel_seed_idx=0,
                              schedule=schedule)


def run_lm_optimization(problem: Problem, x_seed: torch.Tensor, tmax_sec: float, max_n_steps: int,
                        return_if_valid_after_n_steps: int, convergence_threshold: float, parallel_count: int = 1,
                        results_df: Optional[Dict] = None, verbosity: int = 1, mesh_validator=None,
                        native: bool = True) -> OptimizationResult:
    """Optimise a trajectory (optimization.py:376-426)."""
    if SELF_COLLISIONS_IGNORED:
        warnings.warn("robot-robot are collisions will be ignored during LM optimization")
    if ENV_COLLISIONS_IGNORED:
        warnings.warn("environment-robot collisions will be ignored during LM optimization")
    stacked_target_path = (
        problem.target_path if parallel_count == 1 else torch.vstack([problem.target_path] * parallel_count)
    )
    assert stacked_target_path.shape == (problem.n_timesteps * parallel_count, 7)
    assert stacked_target_path.shape[0] == x_seed.shape[0]
    assert x_seed.shape[1] == problem.robot.ndof
    assert isinstance(max_n_steps, int), f"error: max_n_steps must be int, is {type(max_n_steps)}"
    if parallel_count > 1:
        # the reference stacks `parallel_count` seeds but its full LM step asserts parallel_count == 1 (:128); here
        # every seed runs its own alternating loop (all of them in the library's batched loop) and the first valid one
        # (lowest seed index) is returned - the first seed's last iterate if none is valid
        assert mesh_validator is None, "parallel seeds run inside the library: no mesh callback"
        T = problem.n_timesteps
        results = run_lm_optimization_batched(problem, x_seed.reshape(parallel_count, T, problem.robot.ndof), tmax_sec,
                                              max_n_steps, return_if_valid_after_n_steps, convergence_threshold)
        return next((r for r in results if r.is_valid), results[0])
    opt_problem = OptimizationProblem(problem, problem.constraints, x_seed, stacked_target_path, verbosity,
                                      parallel_count, results_df)
    opt_state = OptimizationState(x_seed.clone(), 0, time())
    return run_lm_alternating_loss(
        opt_problem, opt_state, ALT_LOSS_V2_1_DIFF, ALT_LOSS_V2_1_POSE, return_residuals=False, verbosity=verbosity,
        tmax_sec=tmax_sec, max_n_steps=max_n_steps, return_if_valid_after_n_steps=return_if_valid_after_n_steps,
        convergence_threshold=convergence_threshold, save_images=False, results_df=results_df,
        mesh_validator=mesh_validator, native=native,
    )


def run_lm_optimization_batched(problem: Problem, x_seeds: torch.Tensor, tmax_sec: Optional[float],
                                max_n_steps: Optional[int], return_if_valid_after_n_steps: int,
                                convergence_threshold: float) -> List[OptimizationResult]:
    """run_lm_optimization for N seed paths x_seeds [N, T, ndof] of one problem at once (csrc/lm_loop_batched.cu): every
    kernel launch of an iteration covers all unfinished seeds and the host reads the iteration's outcome once, whatever
    N.  Result i (parallel_seed_idx = i) is bit for bit that of run_lm_optimization(problem, x_seeds[i]); the time limit
    is checked once per iteration for all seeds.  tmax_sec / max_n_steps = None as in run_lm_alternating_loss."""
    robot = problem.robot
    assert x_seeds.dim() == 3 and x_seeds.shape[1:] == (problem.n_timesteps, robot.ndof), \
        f"x_seeds must be [N, {problem.n_timesteps}, {robot.ndof}], is {tuple(x_seeds.shape)}"
    if tmax_sec is None:
        assert (max_n_steps is not None) and (return_if_valid_after_n_steps is not None)
        assert return_if_valid_after_n_steps <= max_n_steps
        tmax_sec = float("inf")
    if max_n_steps is None:
        assert tmax_sec is not None
        max_n_steps = int(1e9)
    out = ops.lm_alternating_loss_batched(
        robot.robot_id, robot.ndof, ops.make_params(ALT_LOSS_V2_1_DIFF), ops.make_params(ALT_LOSS_V2_1_POSE),
        problem.constraints, x_seeds, problem.target_path, problem.obstacle_tables, max_n_steps, tmax_sec,
        return_if_valid_after_n_steps, convergence_threshold)
    return [OptimizationResult(x_opt=x, n_steps_taken=n, is_valid=v, parallel_seed_idx=i, schedule=s)
            for i, (x, n, v, s, _) in enumerate(out)]


def run_lm_optimization_many(problems, x_seeds, streams, tmax_sec: float, max_n_steps: int,
                             return_if_valid_after_n_steps: int, convergence_threshold: float):
    """run_lm_optimization for several independent problems in lock step: problem i's kernels run on streams[i] and the
    library takes every loop's decisions after having enqueued the next step of all of them.  Same results as one
    run_lm_optimization call per problem.  -> list of OptimizationResult."""
    jobs = []
    for problem, x_seed, stream in zip(problems, x_seeds, streams):
        robot = problem.robot
        assert x_seed.shape == (problem.n_timesteps, robot.ndof)
        jobs.append(dict(rid=robot.robot_id, ndof=robot.ndof, params_diff=ops.make_params(ALT_LOSS_V2_1_DIFF),
                         params_pose=ops.make_params(ALT_LOSS_V2_1_POSE), constraints=problem.constraints, x_seed=x_seed,
                         target=problem.target_path, ob=problem.obstacle_tables, max_n_steps=max_n_steps, tmax_sec=tmax_sec,
                         return_if_valid_after_n_steps=return_if_valid_after_n_steps,
                         convergence_threshold=convergence_threshold, stream=stream))
    return [OptimizationResult(x_opt=x, n_steps_taken=n, is_valid=v, parallel_seed_idx=0, schedule=s)
            for x, n, v, s, _ in ops.lm_alternating_loss_many(jobs)]
