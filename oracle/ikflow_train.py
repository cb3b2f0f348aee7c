"""IKFlow's training definition over oracle/ikflow.py's network (TEST INFRASTRUCTURE - see oracle/__init__.py).

What ikflow's `train.py` computes.  It is restated from memory of the public code because that code is not available
offline: the loss, softflow, the padding and the hyperparameter defaults of cppflow_b200/ikflow_training.py are
unverified.  The CUDA training step (cppflow_b200/csrc/k_flow_train.cu) is pinned to these functions.

  * `forward_with_logdet(net, x, cond)` is `net`'s forward pass (x -> z) with log|det dz/dx|: the sum over every
    half-coupling of the clamped s, plus logDetM of the joint scale; permutations add 0.  `cond` is the full
    [n, dim_cond] condition, softflow scale included (`Glow.forward` takes [n, 7] poses and sets the scale to 0).
  * `nll(z, log_det) = mean(0.5 |z|^2 - log_det)`, the negative log-likelihood under N(0, I) without the constant
    0.5 width log(2 pi), which ikflow drops too.
  * `training_batch` builds a batch from data and noise passed in; `sample_training_data` draws the data.

`bf16=True` rounds where `Glow(..., bf16=True)` does (oracle/ikflow.py's module docstring)."""
from typing import Optional

import torch

from .ikflow import GLOWCouplingBlock, Glow


def _block_forward_with_logdet(block: GLOWCouplingBlock, x: torch.Tensor, c: torch.Tensor, bf16: bool):
    """GLOWCouplingBlock.forward(x, c) (x -> z) and the per-row sum of the clamped s of both half-couplings"""
    x1, x2 = x[:, : block.len1], x[:, block.len1:]
    s2, t2 = block._st(block.subnet2, x2, c, block.len1, bf16)
    y1 = torch.exp(s2) * x1 + t2
    s1, t1 = block._st(block.subnet1, y1, c, block.len2, bf16)
    y2 = torch.exp(s1) * x2 + t1
    return torch.cat([y1, y2], dim=1), s2.sum(dim=1) + s1.sum(dim=1)


def forward_with_logdet(net: Glow, x: torch.Tensor, cond: torch.Tensor, bf16: bool = False):
    """x [n, width], cond [n, dim_cond] (poses and softflow scale) -> (z, log|det dz/dx| [n]), in x.dtype"""
    c = cond.to(x.dtype)
    lin, blocks = net.module_list[0], list(net.module_list[1:])
    m = torch.diagonal(lin.M).to(x.dtype)
    x = x * m
    # logDetM, evaluated in x.dtype (the module's fp32 buffer would cap an fp64 check at fp32 accuracy)
    log_det = torch.zeros(x.shape[0], dtype=x.dtype, device=x.device) + m.abs().log().sum()
    for i in range(0, len(blocks), 2):
        x, ld = _block_forward_with_logdet(blocks[i + 1], x[:, blocks[i].perm], c, bf16)
        log_det = log_det + ld
    return x, log_det


def nll(z: torch.Tensor, log_det: torch.Tensor) -> torch.Tensor:
    """ikflow's training loss: mean(0.5 |z|^2 - log_det) (the constant 0.5 width log(2 pi) dropped)"""
    return (0.5 * (z * z).sum(dim=1) - log_det).mean()


def sample_training_data(model, n: int, generator: Optional[torch.Generator] = None):
    """jrl's sample_joint_angles_and_poses(n, only_non_self_colliding=True) with this repository's capsule model
    standing in for jrl's: q uniform within the joint limits, rows with a capsule self-collision dropped (so fewer
    than n may come back), poses FK(q) as [x, y, z, qw, qx, qy, qz].  `model` is an oracle.robots.RobotModel."""
    from . import geometry as G, kinematics as K

    lim = torch.tensor(model.actuated_joints_limits, dtype=torch.float64)
    q = lim[:, 0] + torch.rand((n, model.ndof), generator=generator, dtype=torch.float64) * (lim[:, 1] - lim[:, 0])
    keep = G.self_collision_distances(model, q).min(dim=1).values >= 0
    q = q[keep]
    return q, K.forward_kinematics(model, q)


def training_batch(q: torch.Tensor, poses: torch.Tensor, idx: torch.Tensor, c: torch.Tensor, eps: torch.Tensor,
                   flip: torch.Tensor, width: int, dim_cond: int, softflow_noise_scale: float):
    """One training batch from data and externally drawn noise, in q.dtype.

    Row r takes sample idx[r] of (q [N, ndof], poses [N, 7]).  x = [q | 0 ...] (the padding columns ndof..width are 0)
    plus, with softflow (dim_cond 8), softflow_noise_scale * c[r] * eps[r] (c ~ U(0, 1) per row, eps ~ N(0, I_width)),
    and cond = [pose | c].  At inference the scale column is 0 (Glow.condition).  The quaternion of the pose is negated
    where flip[r] is true (a fair coin): forward kinematics emits the hemisphere with the largest component positive
    (csrc/kinematics.cuh: rotmat_to_quat) but target paths carry either sign, so training sees both.  Without softflow
    c and eps are unused and width must equal ndof (the padding would have no density)."""
    n, ndof = idx.shape[0], q.shape[1]
    x = torch.zeros((n, width), dtype=q.dtype, device=q.device)
    x[:, :ndof] = q[idx]
    pose = poses[idx].clone()
    pose[:, 3:] = torch.where(flip.bool()[:, None], -pose[:, 3:], pose[:, 3:])
    if dim_cond == 7:
        assert width == ndof, "width > ndof needs softflow (dim_cond 8)"
        return x, pose
    x = x + (softflow_noise_scale * c.to(q.dtype))[:, None] * eps.to(q.dtype)
    return x, torch.cat([pose, c.to(q.dtype)[:, None]], dim=1)
