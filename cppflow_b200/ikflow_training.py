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
default 1e-8.  The training definition (loss, softflow, padding, quaternion signs) is oracle/ikflow_train.py's.

Data-parallel training (IkflowTrainer's process_group and micro_batches): one global step uses S = W x M shards of B
rows, W ranks (one GPU each) of M micro-batches each.  Shard j holds rows j B ... (j + 1) B - 1 of the global batch,
whose row g is drawn from (seed, step, g).  The reduced gradient is G = (1 / S) T(g_0, ..., g_{S-1}), g_j the gradient
of shard j's mean NLL and T the balanced pairwise tree in shard order (tree_levels).  With W and M powers of two a
rank owns an aligned subtree: it sums its M gradients with the same tree (local_schedule), and the W partials are
combined by the top of the tree in rank order, on the slice of the vector each rank owns, by the library's
fixed-order reduction.  NCCL only moves bytes (all_to_all, all_gather), so G, the shard losses' mean carried in the
same vector, and every update depend on (S, B) alone: (W, M) = (8, 1), (2, 4) and (1, 8) give the same bits."""
from dataclasses import asdict
from typing import Dict, List, Optional, Tuple

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


def _is_pow2(v: int) -> bool:
    return v >= 1 and v & (v - 1) == 0


def tree_levels(S: int) -> List[List[Tuple[Tuple[int, int], Tuple[int, int]]]]:
    """The balanced pairwise tree over S (a power of two) shards in shard order, level by level: each entry is a pair
    (left, right) of half-open shard ranges whose sums are added, left + right; T(g_0, ..., g_{S-1}) is the root."""
    if not _is_pow2(S):
        raise ValueError(f"{S} shards: the tree needs a power of two")
    levels, w = [], 1
    while w < S:
        levels.append([((a, a + w), (a + w, a + 2 * w)) for a in range(0, S, 2 * w)])
        w *= 2
    return levels


def local_schedule(M: int) -> List[Tuple]:
    """A rank's M micro-batch gradients summed with the tree of tree_levels(M) while they arrive, in log2(M) + 1
    buffers used as a stack: ("grad", j, slot) computes the gradient of micro-batch j into `slot`, ("add", slot)
    replaces slot by slot + (slot + 1) (the left and right subtrees of equal size on top of the stack).  The sum ends
    in slot 0."""
    if not _is_pow2(M):
        raise ValueError(f"micro_batches {M} is not a power of two")
    ops, sizes = [], []
    for j in range(M):
        ops.append(("grad", j, len(sizes)))
        sizes.append(1)
        while len(sizes) >= 2 and sizes[-1] == sizes[-2]:
            ops.append(("add", len(sizes) - 2))
            sizes[-2:] = [2 * sizes[-1]]
    return ops


def tree_sum(values, add=lambda a, b: a + b):
    """T(values) in the order of tree_levels: the reference the library's reduction and local_schedule implement."""
    v = list(values)
    if not _is_pow2(len(v)):
        raise ValueError(f"{len(v)} values: the tree needs a power of two")
    while len(v) > 1:
        v = [add(v[i], v[i + 1]) for i in range(0, len(v), 2)]
    return v[0]


class IkflowTrainer:
    """Trains IKFlow's network for `robot` on one GPU, or data-parallel on the ranks of a process group.

    robot, params (the network's shape), seed (initial weights, dataset and batch draws), batch_size (a multiple of
    128; per shard), lr, betas, eps, weight_decay, lr_decay (gamma of the exponential decay), lr_decay_samples
    (samples between two decays; counted in global steps of S x batch_size samples), softflow_noise_scale, n_data
    (configurations drawn for the dataset before self-colliding ones are dropped; every rank draws the same),
    state_dict (initial weights in GraphINN format; seeded nn.Linear initialisation otherwise), use_graph (replay
    steps after the first as one CUDA graph, collectives included), history (capacity of the loss ring buffer),
    process_group (a torch.distributed NCCL group of W ranks, W a power of two, one GPU each; None: one GPU, W = 1),
    micro_batches (M, a power of two: shards per rank and step).  With process_group None and micro_batches 1 a step
    is the one-call step of csrc/k_flow_train.cu; otherwise it is the data-parallel step of the module docstring, and
    every rank holds bit-identical weights after it.  See the module docstring for which defaults are unverified."""

    def __init__(self, robot, params: Optional[IkflowModelParameters] = None, seed: int = 0, batch_size: int = 512,
                 lr: float = 5e-4, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 1.8e-5,
                 lr_decay: float = 0.9794, lr_decay_samples: int = 2_500_000, softflow_noise_scale: float = 1e-3,
                 n_data: int = 1_000_000, state_dict: Optional[Dict] = None, use_graph: bool = False,
                 history: int = 1 << 16, device=DEVICE, process_group=None, micro_batches: int = 1):
        params = params if params is not None else IkflowModelParameters()
        if params.coupling_layer != "glow":
            raise ValueError(f"coupling_layer '{params.coupling_layer}' is not supported (only 'glow')")
        if batch_size < 128 or batch_size % 128 != 0:
            raise ValueError(f"batch_size {batch_size} is not a positive multiple of 128")
        if params.dim_latent_space > robot.ndof and not params.softflow_enabled:
            raise ValueError("dim_latent_space > ndof needs softflow_enabled: the padding has no density without it")
        self.group = process_group
        if process_group is not None:
            import torch.distributed as dist

            self.world, self.rank = dist.get_world_size(process_group), dist.get_rank(process_group)
        else:
            self.world, self.rank = 1, 0
        if not _is_pow2(self.world):
            raise ValueError(f"{self.world} ranks: data-parallel training needs a power of two")
        if not isinstance(micro_batches, int) or not _is_pow2(micro_batches):
            raise ValueError(f"micro_batches {micro_batches} is not a power of two")
        self.micro_batches = micro_batches
        self.shards = self.world * micro_batches
        self.robot, self.params, self.seed, self.batch_size = robot, params, seed, batch_size
        self.softflow_noise_scale = float(softflow_noise_scale)
        self.n_data, self.use_graph = n_data, use_graph
        self.hyper = dict(lr=lr, beta1=betas[0], beta2=betas[1], eps=eps, weight_decay=weight_decay, lr_decay=lr_decay,
                          lr_decay_steps=max(1, round(lr_decay_samples / (self.shards * batch_size))))
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
        self._sharded = process_group is not None or micro_batches > 1
        if self._sharded:
            self._init_shards()

    def _init_shards(self):
        """Buffers of the data-parallel step: the local tree's stack of log2(M) + 1 gradients and the reduced G, each
        padded to a multiple of W x 64 floats with the shard's mean loss at index P, and the all_to_all output."""
        P, W = self.params_flat.numel(), self.world
        self._P = P
        self._Ppad = -(-(P + 1) // (64 * W)) * 64 * W
        depth = self.micro_batches.bit_length()
        self._stack = torch.zeros((depth, self._Ppad), device=self.device)
        self._G = torch.zeros(self._Ppad, device=self.device)
        self._recv = torch.empty((W, self._Ppad // W), device=self.device) if W > 1 else None

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
        if self._sharded:
            self._issue_sharded()
        else:
            self.draw_batch()
            ops.flow_train_step(self.desc, self.x, self.cond, self.workspace, self.loss)
        slot = torch.remainder(self.counters[2:3] - 1, self._hist.numel())
        self._hist.index_copy_(0, slot, self.loss)

    def _draw_shard(self, j: int):
        """Shard j of this rank's M: rows (rank M + j) B ... of the global batch, into self.x / self.cond."""
        B = self.batch_size
        ops.flow_train_batch(self.desc, self.data_q, self.data_poses, self.seed, self.softflow_noise_scale, self.x,
                             self.cond, first_row=(self.rank * self.micro_batches + j) * B)

    def _local_partial(self) -> torch.Tensor:
        """T over this rank's M shard gradients (and shard losses at index P), in self._stack[0]."""
        P = self._P
        for op in local_schedule(self.micro_batches):
            if op[0] == "grad":
                _, j, slot = op
                self._draw_shard(j)
                buf = self._stack[slot]
                ops.flow_train_step(self.desc, self.x, self.cond, self.workspace, buf[P:P + 1], buf[:P], update=False)
            else:
                ops.flow_grad_tree_reduce(self._stack[op[1]:op[1] + 2], self._stack[op[1]])
        return self._stack[0]

    def _exchange(self, partial: torch.Tensor):
        """G = (1 / S) T(partials of the W ranks in rank order) into self._G: all_to_all gives this rank slice `rank`
        of every partial, the library's tree reduces it, all_gather assembles G on every rank."""
        W, scale = self.world, 1.0 / self.shards
        if W == 1:
            ops.flow_grad_tree_reduce(partial.view(1, -1), self._G, scale)
            return
        import torch.distributed as dist

        chunk = self._Ppad // W
        dist.all_to_all_single(self._recv.view(-1), partial, group=self.group)
        mine = self._G[self.rank * chunk:(self.rank + 1) * chunk]
        ops.flow_grad_tree_reduce(self._recv, mine, scale)
        dist.all_gather_into_tensor(self._G, mine, group=self.group)

    def _issue_sharded(self):
        self._exchange(self._local_partial())
        ops.flow_train_apply(self.desc, self._G, self.batch_size, self.workspace)
        self.loss.copy_(self._G[self._P:self._P + 1])

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
        (seed, step)), the loss ring buffer and the configuration, with the shard count S and the per-shard batch B.
        Data-parallel: every rank holds the same state, and rank 0 writes it (the other ranks return)."""
        if self.rank != 0:
            return
        torch.save({"robot": self.robot.name, "model": asdict(self.params), "seed": self.seed,
                    "batch_size": self.batch_size, "shards": self.shards, "hyper": dict(self.hyper), "n_data": self.n_data,
                    "softflow_noise_scale": self.softflow_noise_scale, "history": self._hist.numel(),
                    "params": self.params_flat.cpu(), "adam_m": self.adam_m.cpu(), "adam_v": self.adam_v.cpu(),
                    "counters": self.counters.cpu(), "loss_ring": self._hist.cpu(), "steps_issued": self.steps_issued},
                   path)

    @classmethod
    def load(cls, path: str, use_graph: bool = False, device=DEVICE, process_group=None,
             micro_batches: Optional[int] = None, batch_size: Optional[int] = None) -> "IkflowTrainer":
        """A trainer that continues the saved run exactly where it stopped, bit for bit, on any W ranks of
        process_group (None: one GPU) with M = micro_batches such that W x M is the saved shard count S (None: S / W).
        batch_size, when given, must be the saved per-shard batch.  A different S or B would be another run: rejected."""
        from .robot import get_robot

        ck = torch.load(path, map_location="cpu", weights_only=False)
        h = ck["hyper"]
        S, B = ck.get("shards", 1), ck["batch_size"]
        if process_group is not None:
            import torch.distributed as dist

            W = dist.get_world_size(process_group)
        else:
            W = 1
        if micro_batches is None:
            micro_batches = S // W if S % W == 0 else 0
        if W * micro_batches != S:
            raise ValueError(f"{path} was trained with {S} shards per step; {W} ranks x {micro_batches} micro-batches "
                             "is another run")
        if batch_size is not None and batch_size != B:
            raise ValueError(f"{path} was trained with {B} rows per shard, not {batch_size}")
        params = IkflowModelParameters(**ck["model"])
        tr = cls(get_robot(ck["robot"]), params, seed=ck["seed"], batch_size=B, lr=h["lr"],
                 betas=(h["beta1"], h["beta2"]), eps=h["eps"], weight_decay=h["weight_decay"], lr_decay=h["lr_decay"],
                 lr_decay_samples=h["lr_decay_steps"] * S * B,
                 softflow_noise_scale=ck["softflow_noise_scale"], n_data=ck["n_data"], use_graph=use_graph,
                 history=ck["history"], device=device, process_group=process_group, micro_batches=micro_batches)
        tr.params_flat.copy_(ck["params"])
        tr.adam_m.copy_(ck["adam_m"])
        tr.adam_v.copy_(ck["adam_v"])
        tr.counters.copy_(ck["counters"])
        tr._hist.copy_(ck["loss_ring"])
        tr.steps_issued = ck["steps_issued"]
        tr._refresh_bf16()
        return tr
