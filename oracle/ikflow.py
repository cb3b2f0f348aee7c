"""IKFlow's conditional GLOW network, restated in torch (TEST INFRASTRUCTURE - see oracle/__init__.py).

What ikflow 0.2 builds in `ikflow/model.py: glow_cNF_model` from FrEIA modules, for a robot with `ndof` joints:

  * input width `dim_latent_space` (>= ndof), condition `[x, y, z, qw, qx, qy, qz]` plus a softflow scale of 0 when
    softflow is enabled (dim_cond 8, else 7);
  * `FixedLinearTransform` with diagonal M: 1 / max(|lower_i|, |upper_i|) for joint i < ndof, 1 for the padding
    dimensions, b = 0 (x -> x M + b forward, (y - b) M^-1 reverse);
  * then `nb_nodes` times `PermuteRandom(seed=i)` (x -> x[:, perm]) followed by `GLOWCouplingBlock(clamp=rnvp_clamp)`
    conditioned on the condition.  The split is len1 = width // 2, len2 = width - len1.  Subnet 1 maps
    [half 1 | cond] to [s | t] for half 2, subnet 2 maps [half 2 | cond] to [s | t] for half 1; each is
    (Linear -> LeakyReLU(0.01)) x coeff_fn_config at width coeff_fn_internal_size, then a final Linear.  The scale is
    exp(clamp * 0.636 * atan(s / clamp)).  Forward (x -> z): half 1 from subnet 2 of half 2, then half 2 from subnet 1
    of the new half 1.  Reverse (z -> x): half 2 from subnet 1 of half 1, then half 1 from subnet 2 of the new half 2.

Parameter names are those of FrEIA's `GraphINN` (`module_list.0.M`, `module_list.{2b+1}.perm`,
`module_list.{2b+2}.subnet1.{j}.weight`, ...), so `Glow.state_dict()` is the weight format
`cppflow_b200.ikflow.IkflowSolver` loads.

CAVEAT: this is restated from the public ikflow / FrEIA sources.  Neither package is available offline, so this module
is the definition the CUDA path (cppflow_b200/csrc/k_flow.cu) is pinned to.  Loading a real IKFlow checkpoint stays
unverified until someone with one tries it.

`bf16=True` rounds to bfloat16 exactly where the CUDA path does: every subnet input [half | cond], the weights of the
tensor-core layers (all but the last Linear of a subnet) and their outputs after bias + LeakyReLU.  Everything else
(accumulation, the last Linear with its fp32 weights, the coupling arithmetic) is computed in the dtype of the input.
"""
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch
from torch import nn

LEAKY_SLOPE = 0.01
ATAN_SCALE = 0.636


def split_lengths(width: int) -> Tuple[int, int]:
    return width // 2, width - width // 2


def permutation(seed: int, width: int) -> np.ndarray:
    """PermuteRandom(seed=seed): np.random.seed(seed); np.random.permutation(width)"""
    return np.random.RandomState(seed).permutation(width)


def joint_scale(limits: Sequence[Tuple[float, float]], width: int) -> torch.Tensor:
    """Diagonal of FixedLinearTransform's M (fp64)."""
    m = torch.ones(width, dtype=torch.float64)
    for i, (lo, hi) in enumerate(limits):
        m[i] = 1.0 / max(abs(lo), abs(hi))
    return m


def _bf16(x: torch.Tensor) -> torch.Tensor:
    return x.to(torch.bfloat16).to(x.dtype)


def subnet(c_in: int, c_out: int, internal: int, n_layers: int) -> nn.Sequential:
    """ikflow's subnet_constructor: (Linear, LeakyReLU) x n_layers, Linear"""
    assert n_layers in (1, 2, 3, 4)
    mods: List[nn.Module] = []
    for i in range(n_layers):
        mods += [nn.Linear(c_in if i == 0 else internal, internal), nn.LeakyReLU(LEAKY_SLOPE)]
    mods.append(nn.Linear(internal, c_out))
    return nn.Sequential(*mods)


def run_subnet(net: nn.Sequential, u: torch.Tensor, bf16: bool) -> torch.Tensor:
    linears = [m for m in net if isinstance(m, nn.Linear)]
    h = _bf16(u) if bf16 else u
    for lin in linears[:-1]:
        w, b = lin.weight.to(u.dtype), lin.bias.to(u.dtype)
        if bf16:
            w = _bf16(w)
        h = torch.nn.functional.leaky_relu(h @ w.T + b, LEAKY_SLOPE)
        if bf16:
            h = _bf16(h)
    return h @ linears[-1].weight.to(u.dtype).T + linears[-1].bias.to(u.dtype)


class FixedLinearTransform(nn.Module):
    def __init__(self, m_diag: torch.Tensor):
        super().__init__()
        M = torch.diag(m_diag.float())
        self.register_buffer("M", M.t().contiguous())
        self.register_buffer("M_inv", M.t().inverse().contiguous())
        self.register_buffer("b", torch.zeros(m_diag.numel()))
        self.register_buffer("logDetM", torch.slogdet(M)[1])


class PermuteRandom(nn.Module):
    def __init__(self, seed: int, width: int):
        super().__init__()
        p = permutation(seed, width)
        inv = np.zeros_like(p)
        inv[p] = np.arange(width)
        self.register_buffer("perm", torch.as_tensor(p, dtype=torch.int64))
        self.register_buffer("perm_inv", torch.as_tensor(inv, dtype=torch.int64))


class GLOWCouplingBlock(nn.Module):
    def __init__(self, width: int, dim_cond: int, internal: int, n_layers: int, clamp: float):
        super().__init__()
        self.len1, self.len2 = split_lengths(width)
        self.clamp = clamp
        self.subnet1 = subnet(self.len1 + dim_cond, 2 * self.len2, internal, n_layers)
        self.subnet2 = subnet(self.len2 + dim_cond, 2 * self.len1, internal, n_layers)

    def _st(self, net, u, c, n_out, bf16):
        a = run_subnet(net, torch.cat([u, c], dim=1), bf16)
        s, t = a[:, :n_out], a[:, n_out:]
        return self.clamp * ATAN_SCALE * torch.atan(s / self.clamp), t

    def forward(self, x: torch.Tensor, c: torch.Tensor, rev: bool = False, bf16: bool = False) -> torch.Tensor:
        x1, x2 = x[:, : self.len1], x[:, self.len1:]
        if not rev:
            s2, t2 = self._st(self.subnet2, x2, c, self.len1, bf16)
            y1 = torch.exp(s2) * x1 + t2
            s1, t1 = self._st(self.subnet1, y1, c, self.len2, bf16)
            y2 = torch.exp(s1) * x2 + t1
        else:
            s1, t1 = self._st(self.subnet1, x1, c, self.len2, bf16)
            y2 = (x2 - t1) * torch.exp(-s1)
            s2, t2 = self._st(self.subnet2, y2, c, self.len1, bf16)
            y1 = (x1 - t2) * torch.exp(-s2)
        return torch.cat([y1, y2], dim=1)


class Glow(nn.Module):
    """glow_cNF_model.  `module_list` holds [FixedLinearTransform, (PermuteRandom, GLOWCouplingBlock) x nb_nodes]."""

    def __init__(self, limits: Sequence[Tuple[float, float]], width: int, nb_nodes: int, internal: int, n_layers: int,
                 clamp: float, softflow: bool = True):
        super().__init__()
        assert width >= len(limits)
        self.ndof, self.width, self.dim_cond = len(limits), width, 8 if softflow else 7
        mods: List[nn.Module] = [FixedLinearTransform(joint_scale(limits, width))]
        for i in range(nb_nodes):
            mods += [PermuteRandom(i, width), GLOWCouplingBlock(width, self.dim_cond, internal, n_layers, clamp)]
        self.module_list = nn.ModuleList(mods)

    def condition(self, poses: torch.Tensor) -> torch.Tensor:
        """[n, 7] poses -> [n, dim_cond] conditions (softflow scale 0)"""
        if self.dim_cond == 7:
            return poses
        return torch.cat([poses, torch.zeros((poses.shape[0], 1), dtype=poses.dtype, device=poses.device)], dim=1)

    def forward(self, x: torch.Tensor, poses: torch.Tensor, rev: bool = False, bf16: bool = False) -> torch.Tensor:
        """x -> z (rev=False) or z -> x (rev=True), computed in x.dtype; poses [n, 7]"""
        c = self.condition(poses.to(x.dtype))
        lin, blocks = self.module_list[0], list(self.module_list[1:])
        m = torch.diagonal(lin.M).to(x.dtype)
        if not rev:
            x = x * m
            for i in range(0, len(blocks), 2):
                x = blocks[i + 1](x[:, blocks[i].perm], c, False, bf16)
            return x
        for i in reversed(range(0, len(blocks), 2)):
            x = blocks[i + 1](x, c, True, bf16)[:, blocks[i].perm_inv]
        return x / m


def random_glow(limits, width: int, nb_nodes: int, internal: int, n_layers: int, clamp: float = 2.5,
                softflow: bool = True, seed: int = 0) -> Glow:
    """A Glow with nn.Linear's default initialisation drawn from a seeded generator."""
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(seed)
        return Glow(limits, width, nb_nodes, internal, n_layers, clamp, softflow)
