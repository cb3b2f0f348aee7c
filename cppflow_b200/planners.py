"""Planner front-end with the reference's control flow (cppflow/planners.py: Planner._run_pipeline :191-292,
PlannerSearcher :301-336, CppFlowPlanner.generate_plan :345-468).

IKFlow (the conditional normalising flow that proposes the k candidate joint paths, planners.py:116-172) runs on the
CUDA path as `IkflowCandidateGenerator` (cppflow_b200/ikflow.py) with a checkpoint's state dict or seeded random
weights; its pretrained weights are not available offline.  The candidate generator is a pluggable callable
`(problem, k) -> [k, T, ndof]`.  The default, `LatentIkCandidateGenerator`, keeps the reference's latent plumbing (one
latent per path, tiled over the waypoints; sampling around the latent of an initial configuration) on top of
`LatentIkSolver`, which traces one inverse-kinematics branch per latent by coarse-to-fine numerical continuation with
the pose-only LM steps of the CUDA kernel (SURVEY.md 8f, row f2)."""
from time import time
from typing import Callable, Dict, Optional, Tuple

import torch

from .collision_detection import qpaths_batched_collisions
from .config import DEVICE, OPTIMIZATION_CONVERGENCE_THRESHOLD, SUCCESS_THRESHOLD_initial_q_norm_dist
from .data_types import PathReport, PlannerResult, PlannerSettings, Problem, TimingData
from .evaluation_utils import get_mjacs
from .optimization import run_lm_optimization
from .optimization_utils import path_metrics
from .search import dp_search
from . import ops
from .lm_hyper_parameters import ALT_LOSS_V2_1_POSE

DEFAULT_RERUN_NEW_K = 125  # planners.py:47

CandidateGenerator = Callable[[Problem, int], torch.Tensor]


class LmIkCandidateGenerator:
    """k candidate paths = k random joint configurations, each copied to every waypoint and pulled onto that waypoint's
    target pose by pose-only LM steps of the CUDA kernel (csrc/k_pose.cu) with a decreasing damping schedule
    (lambda 1e-1 -> 1e-6: from a far seed the reference's lambda = 1e-6 is a Gauss-Newton step and converges on only
    ~15-30 % of the waypoints in 6 steps; the damped schedule reaches 80-90 % on the 7-dof arms).  Every waypoint is
    solved on its own from the same far seed - the first stand-in; `LatentIkSolver` below replaces it."""

    LAMBDAS = (1e-1,) * 4 + (3e-2,) * 4 + (1e-2,) * 4 + (1e-3,) * 3 + (1e-4, 1e-5, 1e-6, 1e-6, 1e-6)

    def __init__(self, n_steps: Optional[int] = None, seed: int = 0):
        self.lambdas = self.LAMBDAS if n_steps is None else self.LAMBDAS[-n_steps:] if n_steps <= len(self.LAMBDAS) \
            else (self.LAMBDAS[0],) * (n_steps - len(self.LAMBDAS)) + self.LAMBDAS
        self.gen = torch.Generator().manual_seed(seed)
        self._prm = ops.make_params(ALT_LOSS_V2_1_POSE)

    def __call__(self, problem: Problem, k: int) -> torch.Tensor:
        robot, T = problem.robot, problem.n_timesteps
        dev = problem.target_path.device
        lim = torch.tensor(robot.actuated_joints_limits, dtype=torch.float32)
        mid, half = lim.mean(dim=1), (lim[:, 1] - lim[:, 0]) / 2
        base = mid + 0.6 * half * (2 * torch.rand((k, 1, robot.ndof), generator=self.gen) - 1)
        x = base.expand(k, T, robot.ndof).reshape(k * T, robot.ndof).contiguous().to(dev)
        ops.lm_pose_steps_(robot.robot_id, robot.ndof, self._prm, self.lambdas, x, problem.target_path, True)
        return x.reshape(k, T, robot.ndof)


class LatentIkSolver:
    """Stands where `IKFlowSolver` stands in the reference (planners.py:75-82, :165-171): a map
    (end-effector pose path, latent) -> joint configurations in which ONE latent picks ONE smooth inverse-kinematics
    branch along the whole path.  IKFlow gets that from a conditional normalising flow with pretrained weights (not
    available offline); here the latent IS a seed configuration in normalised joint coordinates (`network_width` =
    ndof, latent 0 = the middle of every joint range, +-1 = +-60 % of the half range), and the branch is traced by
    numerical continuation on the CUDA pose-step kernel (csrc/k_pose.cu), coarse to fine:

      1. waypoint 0 of every path: damped LM steps from the seed (lambda 1e-1 -> 1e-6, the far-seed schedule);
      2. every `stride`-th waypoint in sequence, each started from the previous coarse waypoint's solution;
      3. the gaps are halved level by level: a new waypoint starts from the joint-space interpolation of its two solved
         neighbours (all new waypoints of a level in ONE launch) and takes a few lightly damped steps;
      4. two undamped polishing steps over all k * T waypoints.

    Solving every waypoint independently from the same far seed (the first stand-in, `LmIkCandidateGenerator`) reached
    the target on ~30 % of the Fetch waypoints and the branches of neighbouring waypoints did not match; continuation
    converges wherever the branch exists and gives dp_search paths that are already smooth."""

    FAR = (1e-1,) * 4 + (3e-2,) * 4 + (1e-2,) * 4 + (1e-3,) * 3 + (1e-4, 1e-5, 1e-6, 1e-6, 1e-6)
    NEAR = (1e-2, 1e-3, 1e-3, 1e-4, 1e-5, 1e-6, 1e-6, 1e-6)
    FILL = (1e-4, 1e-5, 1e-6, 1e-6)
    POLISH = (1e-6, 1e-6)
    LATENT_TO_HALF_RANGE = 0.6

    def __init__(self, robot, stride: int = 16):
        self.robot = robot
        self.network_width = robot.ndof
        self.stride = max(1, int(stride))
        self._prm = ops.make_params(ALT_LOSS_V2_1_POSE)
        lim = torch.tensor(robot.actuated_joints_limits, dtype=torch.float32)
        self._mid, self._half = lim.mean(dim=1), (lim[:, 1] - lim[:, 0]) / 2
        self._schedules: Dict = {}
        self._donors: Dict = {}
        self.last_converged: Optional[torch.Tensor] = None

    # latent <-> seed configuration (the role of the flow's forward / reverse pass, planners.py:174-189)
    def latent_to_configuration(self, latent: torch.Tensor) -> torch.Tensor:
        mid, half = self._mid.to(latent.device), self._half.to(latent.device)
        return mid + self.LATENT_TO_HALF_RANGE * half * latent.clamp(-1.0 / self.LATENT_TO_HALF_RANGE, 1.0 / self.LATENT_TO_HALF_RANGE)

    def configuration_to_latent(self, q: torch.Tensor) -> torch.Tensor:
        mid, half = self._mid.to(q.device), self._half.to(q.device)
        return (q - mid) / (self.LATENT_TO_HALF_RANGE * half)

    def _steps(self, x: torch.Tensor, targets: torch.Tensor, lambdas) -> torch.Tensor:
        """len(lambdas) pose-only LM steps in place on x [n, ndof]; row i tracks targets[i % len(targets)]"""
        return ops.lm_pose_steps_(self.robot.robot_id, self.robot.ndof, self._prm, lambdas, x, targets, True)

    def _schedule(self, T: int, dev):
        """Coarse waypoints and, per refinement level, (new waypoints, left / right solved neighbours, interpolation
        weights) as device index tensors - built once per (T, device)."""
        key = (T, str(dev))
        if key not in self._schedules:
            coarse = list(range(0, T, self.stride))
            if coarse[-1] != T - 1:
                coarse.append(T - 1)
            solved, levels = list(coarse), []
            while True:
                new, left, right = [], [], []
                for a, b in zip(solved[:-1], solved[1:]):
                    if b - a > 1:
                        new.append((a + b) // 2); left.append(a); right.append(b)
                if not new:
                    break
                ni, li, ri = (torch.tensor(v, device=dev) for v in (new, left, right))
                levels.append((ni, li, ri, ((ni - li).float() / (ri - li).float())[None, :, None]))
                solved = sorted(solved + new)
            self._schedules[key] = (coarse, levels)
        return self._schedules[key]

    def _converged(self, x: torch.Tensor, targets: torch.Tensor) -> torch.Tensor:
        """bool [n]: pose error inside the plan constraints (0.1 mm, 0.1 deg; scripts/evaluate.py:51-56)"""
        err, _ = ops.pose_errors(self.robot.robot_id, self.robot.ndof, x, targets)
        return (err[:, 3:].norm(dim=1) < 1e-4) & (err[:, :3].norm(dim=1) < 1.745e-3)

    def _donor_scores(self, k: int, dev) -> torch.Tensor:
        """Fixed random preference matrix [k, k] (row p: which converged path p continues on when its own branch ends),
        drawn once per k from a seeded host generator: candidate sets are reproducible run to run."""
        key = (k, str(dev))
        if key not in self._donors:
            self._donors[key] = torch.rand((k, k), generator=torch.Generator().manual_seed(20240613)).to(dev)
        return self._donors[key]

    def solve_paths(self, ee_path: torch.Tensor, latents: torch.Tensor, generator: Optional[torch.Generator] = None,
                    n_restarts: int = 3) -> torch.Tensor:
        """ee_path [T, 7], latents [k, network_width] -> [k, T, ndof]; `self.last_converged` = bool [k, T].
        Nothing here synchronises with the host."""
        T, k, D = ee_path.shape[0], latents.shape[0], self.robot.ndof
        dev = ee_path.device
        ee_path = ee_path.contiguous()
        x = torch.empty((k, T, D), device=dev, dtype=torch.float32)
        coarse, levels = self._schedule(T, dev)
        # every random number of the call in ONE host -> device copy: fresh seeds for the restarts at waypoint 0 and at
        # every coarse waypoint (a per-waypoint copy from pageable memory would serialise host and device each time)
        fresh = (torch.rand((n_restarts + len(coarse) - 1, k, self.network_width), generator=generator) * 2 - 1).to(dev)
        alts = self.latent_to_configuration(fresh)
        cur = self.latent_to_configuration(latents.to(dev).float()).contiguous()
        self._steps(cur, ee_path[0:1], self.FAR)
        # a damped LM descent with joint-limit clamping gets stuck on ~40 % of random Fetch seeds: the seeds that did
        # not reach the first pose are redrawn (the converged ones keep their latent's branch)
        for r in range(n_restarts):
            ok = self._converged(cur, ee_path[0:1])
            alt = alts[r].contiguous()
            self._steps(alt, ee_path[0:1], self.FAR)
            cur = torch.where(ok[:, None], cur, alt)
        x[:, 0] = cur
        for j, t in enumerate(coarse[1:]):
            cur = cur.clone()
            self._steps(cur, ee_path[t:t + 1], self.NEAR)
            # a branch that ended (joint limit, singularity) restarts from a fresh seed at this waypoint; if that fails
            # too it is continued on a converged path's branch, drawn at random (per path: the argmax of a random score
            # over the converged paths)
            ok = self._converged(cur, ee_path[t:t + 1])
            alt = alts[n_restarts + j].contiguous()
            self._steps(alt, ee_path[t:t + 1], self.FAR)
            ok_alt = self._converged(alt, ee_path[t:t + 1])
            cur = torch.where(ok[:, None], cur, alt)
            ok = ok | ok_alt
            donor = (self._donor_scores(k, dev) * ok[None, :]).argmax(dim=1)
            cur = torch.where(ok[:, None], cur, cur[donor])
            x[:, t] = cur
        for ni, li, ri, w in levels:
            sub = (x[:, li] * (1 - w) + x[:, ri] * w).reshape(k * ni.numel(), D).contiguous()
            self._steps(sub, ee_path[ni].contiguous(), self.FILL)
            x[:, ni] = sub.reshape(k, ni.numel(), D)
        flat = x.reshape(k * T, D)
        self._steps(flat, ee_path, self.POLISH)
        self.last_converged = self._converged(flat, ee_path).reshape(k, T)
        return flat.reshape(k, T, D)

    def generate_ik_solutions(self, ee_path_tiled: torch.Tensor, latent: torch.Tensor, clamp_to_joint_limits: bool = True):
        """IKFlowSolver.generate_ik_solutions' call shape (planners.py:165-171): ee_path_tiled [k*T, 7] = the pose path
        repeated k times, latent [k*T, width] = one latent per path repeated T times (`_sample_latents`) -> [k*T, ndof].
        The joint-limit clamp is part of every LM step, so `clamp_to_joint_limits` is always in force."""
        assert ee_path_tiled.shape[0] == latent.shape[0]
        n = latent.shape[0]
        # rows of one path share their latent: the first change of latent marks T
        T = n if n < 2 else int((latent[1:] != latent[:-1]).any(dim=1).nonzero()[0, 0]) + 1 if bool((latent[1:] != latent[:-1]).any()) else n
        assert n % T == 0
        k = n // T
        return self.solve_paths(ee_path_tiled[:T], latent.reshape(k, T, -1)[:, 0]).reshape(n, self.robot.ndof)


class LatentIkCandidateGenerator:
    """`(problem, k) -> [k, T, ndof]` through the reference's latent plumbing (planners.py:116-172, :191-216): one
    latent per path (`_sample_latents`, uniform or gaussian with `latent_vector_scale`, tiled over the T waypoints as
    [k*T, width]), sampled around the latent of `problem.initial_configuration` when there is one
    (`_get_configuration_corresponding_latent` + `_sample_latents_near`, whose first path keeps the centre latent)."""

    def __init__(self, seed: int = 0, latent_distribution: str = "uniform", latent_vector_scale: float = 2.0, stride: int = 16):
        assert latent_distribution in {"uniform", "gaussian"}
        self.gen = torch.Generator().manual_seed(seed)
        self.latent_distribution, self.latent_vector_scale, self.stride = latent_distribution, latent_vector_scale, stride
        self._solvers: Dict[str, LatentIkSolver] = {}
        self.last_converged: Optional[torch.Tensor] = None  # bool [k, T] of the last call: pose reached per waypoint

    def solver(self, robot) -> LatentIkSolver:
        if robot.name not in self._solvers:
            self._solvers[robot.name] = LatentIkSolver(robot, self.stride)
        return self._solvers[robot.name]

    def _sample_latents(self, k: int, n_timesteps: int, width: int) -> torch.Tensor:
        """planners.py:116-134"""
        if self.latent_distribution == "gaussian":
            latents = torch.randn((k, width), generator=self.gen) * self.latent_vector_scale
        else:
            w = self.latent_vector_scale
            latents = torch.rand((k, width), generator=self.gen) * w - (w / 2)
        return torch.repeat_interleave(latents, n_timesteps, dim=0)

    def _sample_latents_near(self, k: int, n_timesteps: int, center_latent: torch.Tensor) -> torch.Tensor:
        """planners.py:136-153"""
        width = center_latent.numel()
        w = self.latent_vector_scale
        latents = torch.rand((k, width), generator=self.gen) * w - (w / 2) + center_latent.reshape(1, width).cpu()
        latents[0] = center_latent.reshape(width).cpu()
        return torch.repeat_interleave(latents, n_timesteps, dim=0)

    def _get_configuration_corresponding_latent(self, robot, qs: torch.Tensor, ee_pose: torch.Tensor) -> torch.Tensor:
        """planners.py:174-189 (the flow run in reverse): here the latent of a configuration is the configuration itself
        in normalised joint coordinates; the pose it reaches plays no role."""
        return self.solver(robot).configuration_to_latent(qs.reshape(1, robot.ndof).float().cpu())

    def _get_k_ikflow_qpaths(self, robot, ee_path: torch.Tensor, batched_latent: torch.Tensor, k: int) -> torch.Tensor:
        """planners.py:155-172 -> stacked [k, T, ndof]"""
        n = ee_path.shape[0]
        assert batched_latent.shape[0] == k * n, "one latent row per (path, waypoint), as _sample_latents lays them out"
        # == generate_ik_solutions(ee_path.repeat((k, 1)), batched_latent) without materialising the tiled pose path
        solver = self.solver(robot)
        qs = solver.solve_paths(ee_path, batched_latent.reshape(k, n, -1)[:, 0], generator=self.gen)
        self.last_converged = solver.last_converged
        return qs

    def __call__(self, problem: Problem, k: int, initial_q_latent: Optional[torch.Tensor] = None) -> torch.Tensor:
        robot, T = problem.robot, problem.n_timesteps
        if problem.initial_configuration is not None and initial_q_latent is None:
            initial_q_latent = self._get_configuration_corresponding_latent(robot, problem.initial_configuration,
                                                                            problem.target_path[0])
        if initial_q_latent is not None:
            batched = self._sample_latents_near(k, T, initial_q_latent)
        else:
            batched = self._sample_latents(k, T, self.solver(robot).network_width)
        return self._get_k_ikflow_qpaths(robot, problem.target_path, batched, k)


class IkflowCandidateGenerator(LatentIkCandidateGenerator):
    """`(problem, k) -> [k, T, ndof]` from IKFlow's network (cppflow_b200/ikflow.py, csrc/k_flow.cu), as the reference
    does it (planners.py:116-189): the latent sampling of `LatentIkCandidateGenerator` at the flow's `network_width`,
    the reverse pass with the joint-limit clamp, and the forward pass for the latent of an initial configuration.
    `solver_or_factory` is an `IkflowSolver` or a callable `robot -> IkflowSolver` (called once per robot).  Every
    IKFlow sample is close to its target pose, so `last_converged` stays None: dp_search gets the collision flags only,
    as in the reference."""

    def __init__(self, solver_or_factory, seed: int = 0, latent_distribution: str = "uniform",
                 latent_vector_scale: float = 2.0):
        super().__init__(seed, latent_distribution, latent_vector_scale)
        self._factory = solver_or_factory if callable(solver_or_factory) else None
        self._fixed = None if callable(solver_or_factory) else solver_or_factory

    def solver(self, robot):
        if self._fixed is not None:
            assert self._fixed.robot.name == robot.name, f"the IKFlow solver is for {self._fixed.robot.name}, not {robot.name}"
            return self._fixed
        if robot.name not in self._solvers:
            self._solvers[robot.name] = self._factory(robot)
        return self._solvers[robot.name]

    def _get_configuration_corresponding_latent(self, robot, qs: torch.Tensor, ee_pose: torch.Tensor) -> torch.Tensor:
        """planners.py:174-189: the forward pass of the flow at (qs, ee_pose)"""
        return self.solver(robot).configuration_to_latent(qs.reshape(1, robot.ndof), ee_pose.reshape(1, 7))

    def _get_k_ikflow_qpaths(self, robot, ee_path: torch.Tensor, batched_latent: torch.Tensor, k: int) -> torch.Tensor:
        """planners.py:155-172 -> stacked [k, T, ndof]"""
        n = ee_path.shape[0]
        assert batched_latent.shape[0] == k * n, "one latent row per (path, waypoint), as _sample_latents lays them out"
        solver = self.solver(robot)
        latents = batched_latent.reshape(k, n, -1)[:, 0].to(ee_path.device)
        self.last_converged = None
        return solver.solve_paths(ee_path, latents, clamp_to_joint_limits=True)


def _with_unreached_waypoints(env_v: torch.Tensor, generator) -> torch.Tensor:
    """IKFlow's samples all lie close to the target pose; the stand-in generator's do not where its LM descent got
    stuck.  Such waypoints (generator.last_converged == False) are handed to dp_search as violations (the K_COLLISION_COST
    penalty of search.py:15), so the search prefers candidates that actually reach the pose - it cannot see pose errors."""
    conv = getattr(generator, "last_converged", None)
    if conv is None or conv.shape != env_v.shape:
        return env_v
    return env_v | ~conv


def report_from_qpath(qpath: torch.Tensor, problem: Problem) -> PathReport:
    """Capsule-based stand-in for plan_from_qpath (data_type_utils.py:244-276; its klampt mesh checks are out of scope)."""
    m = path_metrics(problem, qpath.contiguous(), 1).cpu()[0].tolist()
    c = problem.constraints
    valid = (m[0] < c.max_allowed_position_error_cm and m[1] < c.max_allowed_rotation_error_deg
             and m[2] < c.max_allowed_mjac_deg and m[3] < c.max_allowed_mjac_cm and m[5] >= 0 and m[6] >= 0)
    dist = 0.0
    if problem.initial_configuration is not None:  # part of Plan.is_valid in the reference (data_types.py:245)
        dist = float(torch.norm(problem.initial_configuration.to(qpath.device) - qpath[0]))
        valid = valid and dist < SUCCESS_THRESHOLD_initial_q_norm_dist
    return PathReport(qpath, m[0], m[1], m[2], m[3], m[4], m[5], m[6], bool(valid), dist)


class Planner:
    def __init__(self, settings: PlannerSettings, robot, candidate_generator: Optional[CandidateGenerator] = None):
        self._cfg = settings
        self._robot = robot
        self._candidates = candidate_generator if candidate_generator is not None else LatentIkCandidateGenerator()

    def set_settings(self, settings: PlannerSettings):
        self._cfg = settings

    @property
    def robot(self):
        return self._robot

    @property
    def name(self) -> str:
        return str(self.__class__.__name__)

    def _run_pipeline(self, problem: Problem, **kwargs) -> Tuple[torch.Tensor, bool, TimingData, Dict, Tuple]:
        """Candidates -> collision flags -> dp_search (planners.py:191-292)."""
        existing_q_data = kwargs.get("rerun_data")
        t0 = time()
        k = self._cfg.k if existing_q_data is None else DEFAULT_RERUN_NEW_K
        qs = self._candidates(problem, k)  # [k, T, ndof]
        time_ikflow = time() - t0
        if self._cfg.return_only_1st_plan:
            return qs[0], False, TimingData(-1, time_ikflow, 0.0, 0.0, 0.0, 0.0), {}, (qs[0], None, None)

        t0 = time()
        k_current = qs.shape[0]
        self_v, env_v = qpaths_batched_collisions(problem, qs)  # one launch for both flag sets
        pct = torch.stack([self_v.sum(), env_v.sum()]).float().cpu() / (k_current * problem.n_timesteps) * 100  # one sync
        env_v = _with_unreached_waypoints(env_v, self._candidates)
        assert pct[0] < 95.0, f"too many self collisions: {pct[0]} %"
        assert pct[1] < 95.0, f"too many env collisions: {pct[1]} %"
        if existing_q_data is not None:
            qs_prev, self_prev, env_prev = existing_q_data
            qs = torch.cat([qs_prev, qs], dim=0)
            self_v = torch.cat([self_prev, self_v], dim=0)
            env_v = torch.cat([env_prev, env_v], dim=0)
        if problem.initial_configuration is not None:
            qs[:, 0, :] = problem.initial_configuration.to(qs.device)
            self_v[:, 0] = False
            env_v[:, 0] = False
        time_coll = time() - t0

        t0 = time()
        qpath_search = dp_search(self.robot, qs, self_v, env_v, verbosity=0)
        q_data = (qs, self_v, env_v)
        time_dp = time() - t0
        return qpath_search, False, TimingData(-1, time_ikflow, time_coll, 0.0, time_dp, 0.0), {}, q_data

    def generate_plan(self, problem: Problem, **kwargs) -> PlannerResult:
        raise NotImplementedError()


class PlannerSearcher(Planner):
    """dp_search only (planners.py:301-336)."""

    def generate_plan(self, problem: Problem, **kwargs) -> PlannerResult:
        assert problem.robot.name == self.robot.name
        t0 = time()
        qpath_search, _, td, debug_info, _ = self._run_pipeline(problem, **kwargs)
        return PlannerResult(report_from_qpath(qpath_search, problem),
                             TimingData(time() - t0, td.ikflow, td.coll_checking, td.batch_opt, td.dp_search, 0.0), [], [],
                             debug_info)


class CppFlowPlanner(Planner):
    """dp_search followed by LM optimisation (planners.py:339-468)."""

    def generate_plan(self, problem: Problem, **kwargs) -> PlannerResult:
        t0 = kwargs.get("t0", time())
        rerun_data = kwargs.get("rerun_data")
        search_qpath, is_valid, td, debug_info, q_data = self._run_pipeline(problem, **kwargs)

        def time_is_exceeded():
            return time() - t0 > self._cfg.tmax_sec

        def return_(qpath):
            return PlannerResult(report_from_qpath(qpath, problem),
                                 TimingData(time() - t0, td.ikflow, td.coll_checking, td.batch_opt, td.dp_search, td.optimizer),
                                 [], [], debug_info)

        if self._cfg.return_only_1st_plan:
            return return_(search_qpath)
        if self._cfg.do_rerun_if_large_dp_search_mjac:
            mjac_deg, mjac_cm = get_mjacs(problem.robot, search_qpath)
            if mjac_deg > self._cfg.rerun_mjac_threshold_deg or mjac_cm > self._cfg.rerun_mjac_threshold_cm:
                kwargs["rerun_data"] = q_data
                search_qpath, is_valid, td, debug_info, q_data = self._run_pipeline(problem, **kwargs)
        if time_is_exceeded():
            return return_(search_qpath)
        if (not self._cfg.anytime_mode_enabled) and is_valid:
            return return_(search_qpath)

        t0_opt = time()
        if self._cfg.anytime_mode_enabled:
            result = run_lm_optimization(problem, search_qpath, max_n_steps=75, tmax_sec=self._cfg.tmax_sec - (time() - t0),
                                         return_if_valid_after_n_steps=int(1e8),
                                         convergence_threshold=OPTIMIZATION_CONVERGENCE_THRESHOLD,
                                         verbosity=self._cfg.verbosity)
        else:
            result = run_lm_optimization(problem, search_qpath, max_n_steps=20, tmax_sec=self._cfg.tmax_sec - (time() - t0),
                                         return_if_valid_after_n_steps=0, convergence_threshold=1e6,
                                         verbosity=self._cfg.verbosity)
        td.optimizer = time() - t0_opt
        debug_info["n_optimization_steps"] = result.n_steps_taken
        if result.is_valid:
            return self._result_from_optimization(problem, result, td, debug_info, t0)
        if self._cfg.do_rerun_if_optimization_fails and (rerun_data is None) and (not time_is_exceeded()):
            kwargs["rerun_data"] = q_data
            kwargs["t0"] = t0
            return self.generate_plan(problem, **kwargs)
        return return_(result.x_opt.detach())

    def _result_from_optimization(self, problem: Problem, result, td: TimingData, debug_info: Dict, t0: float) -> PlannerResult:
        """The plan returned after the LM loop (planners.py:426-452): the optimised path, with the requested initial
        configuration swapped in when that keeps the plan valid."""

        def return_(qpath):
            return PlannerResult(report_from_qpath(qpath, problem),
                                 TimingData(time() - t0, td.ikflow, td.coll_checking, td.batch_opt, td.dp_search, td.optimizer),
                                 [], [], debug_info)

        x_opt = result.x_opt.detach()
        if result.is_valid and problem.initial_configuration is not None:
            init = problem.initial_configuration.to(x_opt.device)
            if torch.norm(init - x_opt[0]) < SUCCESS_THRESHOLD_initial_q_norm_dist:
                return return_(x_opt)
            x_opt_swapped = torch.cat((init, x_opt[1:]), dim=0)
            if report_from_qpath(x_opt_swapped, problem).is_valid:
                return return_(x_opt_swapped)
        return return_(x_opt)


_STREAM_POOL: Dict[str, list] = {}


def plan_many(planner_factory: Callable[[Problem], Planner], problems):
    """Plan several independent problems in one batched run (BASELINE config 4: the 13 benchmark problems).

    A single plan is a chain of small dependent launches with one host round trip per LM iteration (~1-3 ms at a few %
    of the GPU).  Here every problem gets its own CUDA stream and scratch buffers and the stages run phase by phase:
      1. candidates -> collision flags -> dp_search of every problem are enqueued without any host synchronisation;
      2. one host read per problem for the reference's "< 95 % colliding" asserts (planners.py:237,247);
      3. the alternating LM loops of all problems advance in lock step inside the library
         (cppflow_lm_alternating_loss_many: the next step of every unfinished loop is enqueued before the host waits);
      4. the plan reports.
    Results equal those of one `generate_plan` call per problem.  Planners with a rerun option or
    `return_only_1st_plan` set (and non-CppFlowPlanner planners) are run one after the other instead.
    (Host threads do not help here: the stages are Python-bound and serialise on the GIL - 13 threads were 1.5x slower
    than the sequential loop.)  -> list of PlannerResult in order."""
    from .optimization import run_lm_optimization_many

    problems = list(problems)
    planners = [planner_factory(p) for p in problems]
    if not problems:
        return []
    batchable = all(isinstance(pl, CppFlowPlanner) and not pl._cfg.return_only_1st_plan
                    and not pl._cfg.do_rerun_if_large_dp_search_mjac and not pl._cfg.do_rerun_if_optimization_fails
                    and pl._cfg.anytime_mode_enabled == planners[0]._cfg.anytime_mode_enabled for pl in planners)
    if not batchable:
        return [pl.generate_plan(p) for pl, p in zip(planners, problems)]
    t0 = time()
    device = problems[0].target_path.device
    cur = torch.cuda.current_stream(device)
    pool = _STREAM_POOL.setdefault(str(device), [])  # the same streams every call: their allocator pools and the
    while len(pool) < len(problems):                   # per-stream scratch buffers (ops._workspace) are reused
        pool.append(torch.cuda.Stream(device))
    streams = pool[: len(problems)]
    staged = []
    for pl, p, s in zip(planners, problems, streams):
        with torch.cuda.stream(s):
            s.wait_stream(cur)
            qs = pl._candidates(p, pl._cfg.k)
            self_v, env_v = qpaths_batched_collisions(p, qs)
            counts = torch.stack([self_v.sum(), env_v.sum()]).float()
            env_v = _with_unreached_waypoints(env_v, pl._candidates)
            if p.initial_configuration is not None:
                qs[:, 0, :] = p.initial_configuration.to(qs.device)
                self_v[:, 0] = False
                env_v[:, 0] = False
            search = dp_search(pl.robot, qs, self_v, env_v, verbosity=0).contiguous()
            staged.append((qs, counts, search))
    for p, s, (qs, counts, _) in zip(problems, streams, staged):
        with torch.cuda.stream(s):
            pct = counts.cpu() / (qs.shape[0] * p.n_timesteps) * 100
        assert pct[0] < 95.0, f"too many self collisions: {pct[0]} %"
        assert pct[1] < 95.0, f"too many env collisions: {pct[1]} %"
    t_search = time() - t0
    cfg = planners[0]._cfg
    tmax = min(pl._cfg.tmax_sec for pl in planners) - (time() - t0)
    t0_opt = time()
    if cfg.anytime_mode_enabled:
        results = run_lm_optimization_many(problems, [st[2] for st in staged], streams, tmax, 75, int(1e8),
                                           OPTIMIZATION_CONVERGENCE_THRESHOLD)
    else:
        results = run_lm_optimization_many(problems, [st[2] for st in staged], streams, tmax, 20, 0, 1e6)
    t_opt = time() - t0_opt
    out = []
    for pl, p, s, res in zip(planners, problems, streams, results):
        with torch.cuda.stream(s):
            td = TimingData(-1, 0.0, t_search, 0.0, 0.0, t_opt)
            out.append(pl._result_from_optimization(p, res, td, {"n_optimization_steps": res.n_steps_taken}, t0))
        cur.wait_stream(s)
    return out
