"""Exact IK from flow samples: the per-row stopping rule of cppflow_ik_refine and the select rule of cppflow_ik_select
(TEST INFRASTRUCTURE - see oracle/__init__.py).

ikflow's IKFlowSolver.generate_exact_ik_solutions samples the flow, runs batched Levenberg-Marquardt IK on the
samples and resamples the targets that did not converge, with more samples per round.  That description is restated
from memory of ikflow's public code; it was not checked against it.  The LM step itself is the reference's
levenberg_marquardt_only_pose + clamp_to_joint_limits (oracle/lm.py), the error the reference's get_6d_pose_errors.
Dtype-generic: float64 for a ground truth.
"""
from dataclasses import replace
from typing import Optional, Sequence, Tuple

import torch

from . import geometry as G
from . import lm as L
from .robots import RobotModel


def pose_error_norms(model: RobotModel, x: torch.Tensor, targets: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """(|e_pos| [n] in m, |e_rot| [n] in rad) of get_6d_pose_errors (row i against targets[i])."""
    e, _ = L.get_6d_pose_errors(model, x, targets)
    return e[:, 3:, 0].norm(dim=1), e[:, :3, 0].norm(dim=1)


def converged(model: RobotModel, x: torch.Tensor, targets: torch.Tensor, pos_tol: float, rot_tol: float,
              check_self_collision: bool = False) -> torch.Tensor:
    """The stopping rule: |e_pos| < pos_tol and |e_rot| < rot_tol (strict), and with `check_self_collision` every
    capsule self pair at distance > 0."""
    p, r = pose_error_norms(model, x, targets)
    ok = (p < pos_tol) & (r < rot_tol)
    if check_self_collision:
        ok = ok & (G.self_collision_distances(model, x) > 0).all(dim=1)
    return ok


def refine(model: RobotModel, x: torch.Tensor, targets: torch.Tensor, lambdas: Sequence[float], pms: L.LmParams,
           pos_tol: float, rot_tol: float, check_self_collision: bool = False, early_exit: bool = True,
           clamp: bool = True) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """Row i: before step s (and after the last one) check the stopping rule; a row that meets it stops, the others
    take levenberg_marquardt_only_pose with lm_lambda = lambdas[s] (+ the clamp).  Without `early_exit` every row takes
    every step.  -> (x [n, D], status bool [n], steps taken int64 [n])."""
    x = x.clone()
    n = x.shape[0]
    active = torch.ones(n, dtype=torch.bool)
    steps = torch.zeros(n, dtype=torch.int64)
    for lam in lambdas:
        if early_exit:
            active &= ~converged(model, x, targets, pos_tol, rot_tol, check_self_collision)
        idx = active.nonzero()[:, 0]
        if idx.numel() == 0:
            break
        xs = L.levenberg_marquardt_only_pose(model, x[idx], targets[idx], replace(pms, lm_lambda=float(lam)))
        if clamp:
            L.clamp_to_joint_limits(model, xs)
        x[idx] = xs
        steps[idx] += 1
    return x, converged(model, x, targets, pos_tol, rot_tol, check_self_collision), steps


def select(status: torch.Tensor, unsolved: torch.Tensor, solutions: Optional[torch.Tensor] = None,
           valid: Optional[torch.Tensor] = None, q: Optional[torch.Tensor] = None) -> torch.Tensor:
    """The select rule of one round: status bool [n, rep] of the samples of targets unsolved [n].  For each target the
    converged sample with the smallest j (sample 0 when none converged) goes to solutions[target], and valid[target]
    says whether one converged (both updated in place when given, from q [n * rep, D]).  -> the targets still unsolved,
    in list order."""
    n, rep = status.shape
    found = status.any(dim=1)
    pick = torch.where(found, status.to(torch.int64).argmax(dim=1), torch.zeros_like(found, dtype=torch.int64))
    if solutions is not None:
        rows = torch.arange(n, device=status.device) * rep + pick
        solutions[unsolved.long()] = q[rows]
        valid[unsolved.long()] = found
    return unsolved[~found]
