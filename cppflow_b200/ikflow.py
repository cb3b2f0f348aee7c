"""IKFlow on the CUDA path: the conditional GLOW network that proposes the reference's candidate joint paths
(cppflow/planners.py:116-189; ikflow's `IKFlowSolver`), run by csrc/k_flow.cu.

`IkflowSolver` packs a state dict in the format of FrEIA's `GraphINN` (`module_list.0.M`,
`module_list.{2b+1}.perm`, `module_list.{2b+2}.subnet1.{j}.weight`, ...; the network is defined in
oracle/ikflow.py) onto the device once; every call is then one library call on the current stream.  Without a
state dict it draws seeded random weights with nn.Linear's default initialisation: the role of the reference's
`Planner(..., is_mock=True)`.  Pretrained IKFlow weights are not bundled; loading a real checkpoint is unverified."""
from dataclasses import dataclass
from typing import Dict, Optional

import numpy as np
import torch

from . import _lib, ops
from .config import DEVICE

SUBNET_IN_WIDTH = 64  # first-layer input of the packed tables (zero-padded [half | cond])
OUT_ROWS = 16  # rows of the packed last Linear


@dataclass
class IkflowModelParameters:
    """The fields of ikflow's IkflowModelParameters that shape the network (ikflow/model.py)."""

    coupling_layer: str = "glow"
    nb_nodes: int = 12
    dim_latent_space: int = 9
    coeff_fn_config: int = 3
    coeff_fn_internal_size: int = 1024
    rnvp_clamp: float = 2.5
    softflow_enabled: bool = True


def _split(width: int):
    return width // 2, width - width // 2


def params_from_state_dict(sd: Dict[str, torch.Tensor], rnvp_clamp: float = 2.5) -> IkflowModelParameters:
    """The IkflowModelParameters a GraphINN state dict was built with, read from its shapes (the clamp is not stored
    in the state dict: it is an argument)."""
    W = sd["module_list.0.M"].shape[0]
    nb = sum(1 for k in sd if k.endswith(".perm"))
    pre = "module_list.2.subnet1"
    L = sum(1 for k in sd if k.startswith(pre + ".") and k.endswith(".weight")) - 1
    H, c_in = sd[pre + ".0.weight"].shape
    return IkflowModelParameters(nb_nodes=nb, dim_latent_space=W, coeff_fn_config=L, coeff_fn_internal_size=H,
                                 rnvp_clamp=rnvp_clamp, softflow_enabled=c_in - W // 2 == 8)


def random_state_dict(robot, params: IkflowModelParameters, seed: int = 0) -> Dict[str, torch.Tensor]:
    """Seeded weights in GraphINN's format: nn.Linear's default init (uniform +-1/sqrt(fan_in) for weight and bias),
    the FixedLinearTransform of the robot's joint limits and PermuteRandom(seed=b)."""
    W, H, L = params.dim_latent_space, params.coeff_fn_internal_size, params.coeff_fn_config
    dc = 8 if params.softflow_enabled else 7
    len1, len2 = _split(W)
    g = torch.Generator().manual_seed(seed)
    m = torch.ones(W, dtype=torch.float64)
    for i, (lo, hi) in enumerate(robot.actuated_joints_limits):
        m[i] = 1.0 / max(abs(lo), abs(hi))
    M = torch.diag(m.float())
    sd = {"module_list.0.M": M, "module_list.0.M_inv": M.inverse(), "module_list.0.b": torch.zeros(W),
          "module_list.0.logDetM": torch.slogdet(M)[1]}

    def uniform(shape, fan_in):
        bound = 1.0 / np.sqrt(fan_in)
        return (torch.rand(shape, generator=g) * 2 - 1) * bound

    for b in range(params.nb_nodes):
        p = np.random.RandomState(b).permutation(W)
        inv = np.zeros_like(p)
        inv[p] = np.arange(W)
        sd[f"module_list.{2 * b + 1}.perm"] = torch.as_tensor(p, dtype=torch.int64)
        sd[f"module_list.{2 * b + 1}.perm_inv"] = torch.as_tensor(inv, dtype=torch.int64)
        for name, c_in, c_out in (("subnet1", len1 + dc, 2 * len2), ("subnet2", len2 + dc, 2 * len1)):
            dims = [c_in] + [H] * L + [c_out]
            for j in range(L + 1):
                pre = f"module_list.{2 * b + 2}.{name}.{2 * j}"
                sd[pre + ".weight"] = uniform((dims[j + 1], dims[j]), dims[j])
                sd[pre + ".bias"] = uniform((dims[j + 1],), dims[j])
    return sd


def pack_fp32(p: IkflowModelParameters, sd: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    """A GraphINN state dict -> the packed tables of include/cppflow_b200.h (cppflow_flow_desc), all FP32 on the CPU
    but the int32 permutations."""
    W, H, L, nb = p.dim_latent_space, p.coeff_fn_internal_size, p.coeff_fn_config, p.nb_nodes
    dim_cond = 8 if p.softflow_enabled else 7
    len1, len2 = _split(W)
    w_in = torch.zeros((nb, 2, H, SUBNET_IN_WIDTH))
    w_hidden = torch.zeros((nb, 2, max(L - 1, 0), H, H))
    b_hidden = torch.zeros((nb, 2, L, H))
    w_out = torch.zeros((nb, 2, OUT_ROWS, H))
    b_out = torch.zeros((nb, 2, OUT_ROWS))
    perm = torch.zeros((nb, W), dtype=torch.int32)
    perm_inv = torch.zeros((nb, W), dtype=torch.int32)
    M = sd["module_list.0.M"]
    if tuple(M.shape) != (W, W):
        raise ValueError(f"module_list.0.M is {tuple(M.shape)}, expected ({W}, {W})")
    scale = torch.diagonal(M).float().clone()
    for b in range(nb):
        key = f"module_list.{2 * b + 1}.perm"
        pb = sd[key].to(torch.int64) if key in sd else torch.as_tensor(np.random.RandomState(b).permutation(W))
        if sorted(pb.tolist()) != list(range(W)):
            raise ValueError(f"{key} is not a permutation of {W} elements")
        perm[b] = pb.to(torch.int32)
        perm_inv[b, pb] = torch.arange(W, dtype=torch.int32)
        for s, (name, c_in, c_out) in enumerate((("subnet1", len1 + dim_cond, 2 * len2),
                                                 ("subnet2", len2 + dim_cond, 2 * len1))):
            pre = f"module_list.{2 * b + 2}.{name}"
            dims = [c_in] + [H] * L + [c_out]
            for j in range(L + 1):
                w, bias = sd[f"{pre}.{2 * j}.weight"].float(), sd[f"{pre}.{2 * j}.bias"].float()
                if tuple(w.shape) != (dims[j + 1], dims[j]) or tuple(bias.shape) != (dims[j + 1],):
                    raise ValueError(f"{pre}.{2 * j}: weight {tuple(w.shape)} / bias {tuple(bias.shape)}, expected "
                                     f"({dims[j + 1]}, {dims[j]}) / ({dims[j + 1]},)")
                if j == 0:
                    w_in[b, s, :, :c_in] = w
                elif j < L:
                    w_hidden[b, s, j - 1] = w
                if j < L:
                    b_hidden[b, s, j] = bias
                else:
                    w_out[b, s, :c_out] = w
                    b_out[b, s, :c_out] = bias
    return {"w_in": w_in, "w_hidden": w_hidden, "b_hidden": b_hidden, "w_out": w_out, "b_out": b_out, "scale": scale,
            "perm": perm, "perm_inv": perm_inv}


class IkflowSolver:
    """(end-effector poses, latents) -> joint configurations through IKFlow's network on the CUDA path.

    network_width = params.dim_latent_space.  `state_dict` (GraphINN names, see the module docstring) is packed once:
    BF16 [out, in] tables for the tensor-core layers, FP32 for the biases, last Linears and joint scale, int32
    permutations."""

    def __init__(self, robot, params: Optional[IkflowModelParameters] = None, state_dict: Optional[Dict] = None,
                 seed: int = 0, device=DEVICE):
        params = params if params is not None else IkflowModelParameters()
        if params.coupling_layer != "glow":
            raise ValueError(f"coupling_layer '{params.coupling_layer}' is not supported (only 'glow')")
        self.robot, self.params = robot, params
        self.network_width = params.dim_latent_space
        self.dim_cond = 8 if params.softflow_enabled else 7
        self.device = torch.device(device)
        self.state_dict = {k: v.detach().cpu() for k, v in
                           (state_dict if state_dict is not None else random_state_dict(robot, params, seed)).items()}
        self._tables = self._pack(self.state_dict)
        t = self._tables
        self.desc = _lib.FlowDescC(
            robot.robot_id, self.network_width, robot.ndof, self.dim_cond, params.nb_nodes, params.coeff_fn_config,
            params.coeff_fn_internal_size, float(params.rnvp_clamp), t["w_in"].data_ptr(),
            t["w_hidden"].data_ptr() if t["w_hidden"] is not None else None, t["b_hidden"].data_ptr(),
            t["w_out"].data_ptr(), t["b_out"].data_ptr(), t["scale"].data_ptr(), t["perm"].data_ptr(),
            t["perm_inv"].data_ptr())

    def _pack(self, sd: Dict[str, torch.Tensor]) -> Dict[str, Optional[torch.Tensor]]:
        t = pack_fp32(self.params, sd)
        dev, L = self.device, self.params.coeff_fn_config
        return {"w_in": t["w_in"].to(torch.bfloat16).to(dev),
                "w_hidden": t["w_hidden"].to(torch.bfloat16).to(dev) if L > 1 else None,
                "b_hidden": t["b_hidden"].to(dev), "w_out": t["w_out"].to(dev), "b_out": t["b_out"].to(dev),
                "scale": t["scale"].to(dev), "perm": t["perm"].to(dev), "perm_inv": t["perm_inv"].to(dev)}

    def run(self, x: torch.Tensor, cond: torch.Tensor, reverse: bool, clamp: bool = False) -> torch.Tensor:
        """The network over x [n, network_width]; row i conditioned on cond[i % len(cond)] (poses [m, 7])."""
        return ops.flow_run(self.desc, x.to(self.device), cond.to(self.device), reverse, clamp)

    def generate_ik_solutions(self, ee_path_tiled: torch.Tensor, latent: torch.Tensor,
                              clamp_to_joint_limits: bool = True) -> torch.Tensor:
        """IKFlowSolver.generate_ik_solutions' call shape (planners.py:165-171): poses [n, 7], latents
        [n, network_width] -> [n, ndof]."""
        assert ee_path_tiled.shape[0] == latent.shape[0], "one pose per latent row"
        return self.run(latent, ee_path_tiled, True, clamp_to_joint_limits)[:, : self.robot.ndof]

    def solve_paths(self, ee_path: torch.Tensor, latents: torch.Tensor, clamp_to_joint_limits: bool = True) -> torch.Tensor:
        """ee_path [T, 7], latents [k, network_width] -> [k, T, ndof]: path p is the reverse pass of latent p at every
        waypoint (== generate_ik_solutions(ee_path.repeat((k, 1)), latents.repeat_interleave(T, 0)), without tiling
        the poses).  Nothing here synchronises with the host."""
        T, k = ee_path.shape[0], latents.shape[0]
        z = latents.to(self.device, torch.float32).repeat_interleave(T, dim=0)
        q = self.run(z, ee_path, True, clamp_to_joint_limits)
        return q[:, : self.robot.ndof].reshape(k, T, self.robot.ndof)

    def configuration_to_latent(self, q: torch.Tensor, pose: torch.Tensor) -> torch.Tensor:
        """The forward pass of the reference's _get_configuration_corresponding_latent (planners.py:174-189):
        q [m, ndof] zero-padded to network_width, poses [m, 7] or [1, 7] -> latents [m, network_width]."""
        q = q.to(self.device, torch.float32).reshape(-1, self.robot.ndof)
        x = torch.cat([q, torch.zeros((q.shape[0], self.network_width - self.robot.ndof), device=self.device)], dim=1)
        return self.run(x, pose.reshape(-1, 7), False)
