"""Training IKFlow on the device (csrc/k_flow_train.cu): the conditional GLOW network of cppflow_b200/ikflow.py fitted to
a robot's joint configurations by maximum likelihood, as ikflow's `train.py` does.

`IkflowTrainer` keeps FP32 master weights and Adam moments in the packed layout of `IkflowSolver._pack`, a
device-resident dataset of self-collision-free configurations and their poses, and runs every step as two library
calls on the current stream (draw the batch, then forward + loss + backward + Adam), optionally replayed as one CUDA
graph.  `state_dict()` is in FrEIA's GraphINN format: it loads into `oracle.ikflow.Glow`, `IkflowSolver` and
`IkflowCandidateGenerator` without conversion.

The defaults are ikflow's `train.py` defaults as far as they are known without its source at hand, and are UNVERIFIED:
batch 512, lr 5e-4, Adam betas (0.9, 0.999), weight decay 1.8e-5 (L2, added to the gradient as torch.optim.Adam
does), ExponentialLR gamma 0.9794 stepped once per 2.5 M samples, softflow noise scale 1e-3.  Adam's eps is torch's
default 1e-8.  The training definition (loss, softflow, padding, quaternion signs) is oracle/ikflow_train.py's."""
from dataclasses import asdict
from typing import Dict, Optional

import numpy as np
import torch

from . import _lib, ops
from .config import DEVICE
from .ikflow import OUT_ROWS, SUBNET_IN_WIDTH, IkflowModelParameters, _split, pack_fp32, random_state_dict

_TABLES = ("w_in", "w_hidden", "b_hidden", "w_out", "b_out")


def table_shapes(p: IkflowModelParameters) -> Dict[str, tuple]:
    """Shapes of the FP32 tables, in the order they are concatenated in the parameter vector."""
    nb, H, L = p.nb_nodes, p.coeff_fn_internal_size, p.coeff_fn_config
    return {"w_in": (nb, 2, H, SUBNET_IN_WIDTH), "w_hidden": (nb, 2, L - 1, H, H), "b_hidden": (nb, 2, L, H),
            "w_out": (nb, 2, OUT_ROWS, H), "b_out": (nb, 2, OUT_ROWS)}


def split_tables(flat: torch.Tensor, p: IkflowModelParameters) -> Dict[str, torch.Tensor]:
    """Views of a packed parameter (or gradient) vector as its tables."""
    shapes = table_shapes(p)
    sizes = [int(np.prod(s)) for s in shapes.values()]
    if flat.numel() != sum(sizes):
        raise ValueError(f"vector of {flat.numel()} floats, the network has {sum(sizes)}")
    return {name: t.view(shape) for (name, shape), t in zip(shapes.items(), torch.split(flat, sizes))}


def unpack(tables: Dict[str, torch.Tensor], p: IkflowModelParameters) -> Dict[str, torch.Tensor]:
    """Packed FP32 tables -> the subnet entries of a GraphINN state dict (the inverse of ikflow.pack_fp32 on them)."""
    W, L, nb = p.dim_latent_space, p.coeff_fn_config, p.nb_nodes
    dim_cond = 8 if p.softflow_enabled else 7
    len1, len2 = _split(W)
    sd = {}
    for b in range(nb):
        for s, (name, c_in, c_out) in enumerate((("subnet1", len1 + dim_cond, 2 * len2),
                                                 ("subnet2", len2 + dim_cond, 2 * len1))):
            pre = f"module_list.{2 * b + 2}.{name}"
            for j in range(L + 1):
                if j == 0:
                    w = tables["w_in"][b, s, :, :c_in]
                elif j < L:
                    w = tables["w_hidden"][b, s, j - 1]
                else:
                    w = tables["w_out"][b, s, :c_out]
                bias = tables["b_hidden"][b, s, j] if j < L else tables["b_out"][b, s, :c_out]
                sd[f"{pre}.{2 * j}.weight"] = w.detach().cpu().clone()
                sd[f"{pre}.{2 * j}.bias"] = bias.detach().cpu().clone()
    return sd


def sample_dataset(robot, n: int, seed: int, device=DEVICE):
    """jrl's sample_joint_angles_and_poses(n, only_non_self_colliding=True) on the device (oracle/ikflow_train.py:
    sample_training_data): q uniform within the joint limits, self-colliding rows (the capsule model's
    collision flags, no obstacles) dropped, poses = forward kinematics.  Returns (q [m, ndof], poses [m, 7]), m <= n."""
    g = torch.Generator().manual_seed(seed)
    q = robot.sample_joint_angles(n, generator=g).to(device)
    self_flags, _ = ops.collision_flags(robot.robot_id, robot.ndof, q, None, want_self=True, want_env=False)
    q = q[self_flags == 0].contiguous()
    return q, robot.forward_kinematics(q).contiguous()


def sample_errors(solver, poses: torch.Tensor, k: int = 16, seed: int = 0):
    """The flow as an IK sampler: k reverse-pass samples (z ~ N(0, I), joints clamped to the limits) per pose of
    poses [m, 7] -> position (m) and rotation (rad, sign-invariant) errors [m k] of their forward kinematics."""
    from .evaluation_utils import positional_errors, rotational_errors

    g = torch.Generator(device=solver.device).manual_seed(seed)
    target = poses.to(solver.device).repeat_interleave(k, 0).contiguous()
    z = torch.randn((target.shape[0], solver.network_width), generator=g, device=solver.device)
    q = solver.run(z, target, True, clamp=True)[:, : solver.robot.ndof].contiguous()
    reached = solver.robot.forward_kinematics(q)
    return positional_errors(target, reached), rotational_errors(target, reached)


def sample_accuracy(solver, poses: torch.Tensor, k: int = 16, seed: int = 0) -> Dict[str, float]:
    """Mean and median of sample_errors."""
    pos, rot = sample_errors(solver, poses, k, seed)
    return {"pos_mean_m": pos.mean().item(), "pos_median_m": pos.median().item(), "rot_mean_rad": rot.mean().item(),
            "rot_median_rad": rot.median().item()}


class IkflowTrainer:
    """Trains IKFlow's network for `robot` on one GPU.

    robot, params (the network's shape), seed (initial weights, dataset and batch draws), batch_size (a multiple of
    128), lr, betas, eps, weight_decay, lr_decay (gamma of the exponential decay), lr_decay_samples (samples between
    two decays), softflow_noise_scale, n_data (configurations drawn for the dataset before self-colliding ones are
    dropped), state_dict (initial weights in GraphINN format; seeded nn.Linear initialisation otherwise), use_graph
    (replay steps after the first as one CUDA graph), history (capacity of the loss ring buffer).  See the module
    docstring for which defaults are unverified."""

    def __init__(self, robot, params: Optional[IkflowModelParameters] = None, seed: int = 0, batch_size: int = 512,
                 lr: float = 5e-4, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 1.8e-5,
                 lr_decay: float = 0.9794, lr_decay_samples: int = 2_500_000, softflow_noise_scale: float = 1e-3,
                 n_data: int = 1_000_000, state_dict: Optional[Dict] = None, use_graph: bool = False,
                 history: int = 1 << 16, device=DEVICE):
        params = params if params is not None else IkflowModelParameters()
        if params.coupling_layer != "glow":
            raise ValueError(f"coupling_layer '{params.coupling_layer}' is not supported (only 'glow')")
        if batch_size < 128 or batch_size % 128 != 0:
            raise ValueError(f"batch_size {batch_size} is not a positive multiple of 128")
        if params.dim_latent_space > robot.ndof and not params.softflow_enabled:
            raise ValueError("dim_latent_space > ndof needs softflow_enabled: the padding has no density without it")
        self.robot, self.params, self.seed, self.batch_size = robot, params, seed, batch_size
        self.softflow_noise_scale = float(softflow_noise_scale)
        self.n_data, self.use_graph = n_data, use_graph
        self.hyper = dict(lr=lr, beta1=betas[0], beta2=betas[1], eps=eps, weight_decay=weight_decay, lr_decay=lr_decay,
                          lr_decay_steps=max(1, round(lr_decay_samples / batch_size)))
        self.device = torch.device(device)
        self.dim_cond = 8 if params.softflow_enabled else 7
        dev, W, B = self.device, params.dim_latent_space, batch_size

        sd = state_dict if state_dict is not None else random_state_dict(robot, params, seed)
        packed = pack_fp32(params, {k: v.detach().cpu() for k, v in sd.items()})
        self.params_flat = torch.cat([packed[k].reshape(-1) for k in _TABLES]).to(dev)
        self.adam_m = torch.zeros_like(self.params_flat)
        self.adam_v = torch.zeros_like(self.params_flat)
        self.counters = torch.zeros(3, dtype=torch.int64, device=dev)
        self.scale, self.perm, self.perm_inv = packed["scale"].to(dev), packed["perm"].to(dev), packed["perm_inv"].to(dev)
        self.tables = split_tables(self.params_flat, params)
        self._refresh_bf16()

        self.data_q, self.data_poses = sample_dataset(robot, n_data, seed, dev)
        self.x = torch.empty((B, W), device=dev)
        self.cond = torch.empty((B, self.dim_cond), device=dev)
        self.loss = torch.zeros(1, device=dev)
        self._hist = torch.full((history,), float("nan"), device=dev)
        self._build_desc()
        self.workspace = torch.empty(ops.flow_train_workspace_bytes(self.desc, B), dtype=torch.uint8, device=dev)
        self.steps_issued = 0
        self._graph = None

    # ---------------------------------------------------------------------------------------------- tables
    def _refresh_bf16(self):
        """The BF16 inference tables and the transposed copies from the FP32 master weights (the step's optimizer
        rewrites them the same way after every update)."""
        t, L = self.tables, self.params.coeff_fn_config
        w_in = t["w_in"].to(torch.bfloat16)
        w_hidden = t["w_hidden"].to(torch.bfloat16) if L > 1 else None
        w_out_t = torch.zeros((*t["w_out"].shape[:2], t["w_out"].shape[3], SUBNET_IN_WIDTH), dtype=torch.bfloat16,
                              device=self.device)
        w_out_t[..., :OUT_ROWS] = t["w_out"].to(torch.bfloat16).transpose(-1, -2)
        self.bf16 = {"w_in": w_in, "w_hidden": w_hidden, "w_in_t": w_in.transpose(-1, -2).contiguous(),
                     "w_hidden_t": w_hidden.transpose(-1, -2).contiguous() if L > 1 else None, "w_out_t": w_out_t}
        if hasattr(self, "desc"):
            self._build_desc()

    def _build_desc(self):
        p, t, b = self.params, self.tables, self.bf16

        def addr(x):
            return x.data_ptr() if x is not None else None

        flow = _lib.FlowDescC(
            self.robot.robot_id, p.dim_latent_space, self.robot.ndof, self.dim_cond, p.nb_nodes, p.coeff_fn_config,
            p.coeff_fn_internal_size, float(p.rnvp_clamp), addr(b["w_in"]), addr(b["w_hidden"]), addr(t["b_hidden"]),
            addr(t["w_out"]), addr(t["b_out"]), addr(self.scale), addr(self.perm), addr(self.perm_inv))
        h = self.hyper
        self.desc = _lib.FlowTrainDescC(
            flow, addr(self.params_flat), addr(self.adam_m), addr(self.adam_v), addr(b["w_in_t"]), addr(b["w_hidden_t"]),
            addr(b["w_out_t"]), addr(self.counters), h["lr"], h["beta1"], h["beta2"], h["eps"], h["weight_decay"],
            h["lr_decay"], h["lr_decay_steps"])

    # ----------------------------------------------------------------------------------------------- steps
    def draw_batch(self, idx: Optional[torch.Tensor] = None, noise: Optional[torch.Tensor] = None):
        """The batch of the current step into self.x / self.cond (idx / noise: see ops.flow_train_batch)."""
        ops.flow_train_batch(self.desc, self.data_q, self.data_poses, self.seed, self.softflow_noise_scale, self.x,
                             self.cond, idx, noise)

    def _issue(self):
        self.draw_batch()
        ops.flow_train_step(self.desc, self.x, self.cond, self.workspace, self.loss)
        slot = torch.remainder(self.counters[2:3] - 1, self._hist.numel())
        self._hist.index_copy_(0, slot, self.loss)

    def step(self, n: int = 1):
        """n training steps on the current stream, without a host synchronisation (graph mode: the capture after
        the first step synchronises once)."""
        for _ in range(n):
            if self.use_graph and self.steps_issued >= 1:
                if self._graph is None:
                    self._graph = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(self._graph):
                        self._issue()
                self._graph.replay()
            else:
                self._issue()
            self.steps_issued += 1

    def loss_and_grad(self, x: torch.Tensor, cond: torch.Tensor):
        """(mean NLL [1], packed FP32 gradient [P]) of the batch x [n, width], cond [n, dim_cond]; no update."""
        n = x.shape[0]
        ws = self.workspace
        need = ops.flow_train_workspace_bytes(self.desc, n)
        if need > ws.numel():
            ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        loss = torch.zeros(1, device=self.device)
        grad = torch.empty_like(self.params_flat)
        ops.flow_train_step(self.desc, x.contiguous(), cond.contiguous(), ws, loss, grad, update=False)
        return loss, grad

    def loss_history(self) -> torch.Tensor:
        """Losses of the steps taken, oldest first (the last `history` of them); reading it synchronises."""
        taken = int(self.counters[2].item())
        cap = self._hist.numel()
        if taken <= cap:
            return self._hist[:taken].clone()
        k = taken % cap
        return torch.cat([self._hist[k:], self._hist[:k]])

    @property
    def steps_skipped(self) -> torch.Tensor:
        """Device counter of the steps whose update was skipped for a non-finite gradient."""
        return self.counters[1]

    # ------------------------------------------------------------------------------------------ weights out
    def state_dict(self) -> Dict[str, torch.Tensor]:
        """The current weights in GraphINN format (names and shapes of oracle.ikflow.Glow.state_dict())."""
        p, W = self.params, self.params.dim_latent_space
        m = self.scale.detach().cpu().double()
        M = torch.diag(m.float())
        sd = {"module_list.0.M": M, "module_list.0.M_inv": torch.diag((1.0 / m).float()), "module_list.0.b": torch.zeros(W),
              "module_list.0.logDetM": torch.slogdet(M)[1]}
        perm, perm_inv = self.perm.cpu().long(), self.perm_inv.cpu().long()
        for b in range(p.nb_nodes):
            sd[f"module_list.{2 * b + 1}.perm"] = perm[b].clone()
            sd[f"module_list.{2 * b + 1}.perm_inv"] = perm_inv[b].clone()
        sd.update(unpack(self.tables, p))
        return sd

    def solver(self):
        """An IkflowSolver on the current weights."""
        from .ikflow import IkflowSolver

        return IkflowSolver(self.robot, self.params, state_dict=self.state_dict(), device=self.device)

    # ------------------------------------------------------------------------------------- checkpointing
    def save(self, path: str):
        """Weights, Adam moments, counters (step count and the generator's position: batches are drawn from
        (seed, step)), the loss ring buffer and the configuration."""
        torch.save({"robot": self.robot.name, "model": asdict(self.params), "seed": self.seed,
                    "batch_size": self.batch_size, "hyper": dict(self.hyper), "n_data": self.n_data,
                    "softflow_noise_scale": self.softflow_noise_scale, "history": self._hist.numel(),
                    "params": self.params_flat.cpu(), "adam_m": self.adam_m.cpu(), "adam_v": self.adam_v.cpu(),
                    "counters": self.counters.cpu(), "loss_ring": self._hist.cpu(), "steps_issued": self.steps_issued},
                   path)

    @classmethod
    def load(cls, path: str, use_graph: bool = False, device=DEVICE) -> "IkflowTrainer":
        """A trainer that continues the saved run exactly where it stopped."""
        from .robot import get_robot

        ck = torch.load(path, map_location="cpu", weights_only=False)
        h = ck["hyper"]
        params = IkflowModelParameters(**ck["model"])
        tr = cls(get_robot(ck["robot"]), params, seed=ck["seed"], batch_size=ck["batch_size"], lr=h["lr"],
                 betas=(h["beta1"], h["beta2"]), eps=h["eps"], weight_decay=h["weight_decay"], lr_decay=h["lr_decay"],
                 lr_decay_samples=h["lr_decay_steps"] * ck["batch_size"],
                 softflow_noise_scale=ck["softflow_noise_scale"], n_data=ck["n_data"], use_graph=use_graph,
                 history=ck["history"], device=device)
        tr.params_flat.copy_(ck["params"])
        tr.adam_m.copy_(ck["adam_m"])
        tr.adam_v.copy_(ck["adam_v"])
        tr.counters.copy_(ck["counters"])
        tr._hist.copy_(ck["loss_ring"])
        tr.steps_issued = ck["steps_issued"]
        tr._refresh_bf16()
        return tr
