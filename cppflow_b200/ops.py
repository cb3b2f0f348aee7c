"""Thin functional layer over the C ABI: allocates outputs with torch, checks shapes like the reference's
asserts do, passes raw pointers + the current CUDA stream.  Everything here runs on the GPU; nothing falls back."""
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import LmParamsC, ptr, stream_ptr, require_cuda, check

import functools


def _on_device(fn):
    """Make the device of the first CUDA tensor argument current for the duration of the call.  The library opts in
    to large shared-memory footprints and picks stream priorities per CURRENT device (cudaFuncSetAttribute is per
    device), and `torch.cuda.current_stream(device)` is only launchable from that device's context: without this a
    process that keeps cuda:0 current while refining tensors on cuda:1 would launch with the wrong context."""

    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        for a in args:
            if isinstance(a, torch.Tensor) and a.is_cuda:
                if a.device.index != torch.cuda.current_device():
                    with torch.cuda.device(a.device):
                        return fn(*args, **kwargs)
                break
        return fn(*args, **kwargs)

    return wrapper


ROBOT_IDS = {"fetch": 0, "fetch_arm": 1, "panda": 2}
LM_CLAMP, LM_OVERLAP, LM_FUSED = 1, 2, 4  # CPPFLOW_LM_CLAMP / _OVERLAP / _FUSED (include/cppflow_b200.h)


def loop_segments() -> int:
    """Segments of the single-path full step (the differencing step of run_lm_alternating_loss): the native loop
    (csrc/lm_loop.cu: loop_step_flags) and the Python loop must take the same solve to return the same bits.
    CPPFLOW_LOOP_SEGMENTS = 0 restores the twisted solve in both."""
    import os

    n = int(os.environ.get("CPPFLOW_LOOP_SEGMENTS", "16"))
    return min(max(n, 0), 255)


def lm_segments(n: int) -> int:
    """CPPFLOW_LM_SEGMENTS(n): the flag bits that ask for the segmented solve with n time segments (0: twisted solve)."""
    assert 0 <= n <= 255, "segments must be in [0, 255]"
    return (n & 0xFF) << 8


def _info(robot_id: int) -> _lib.RobotInfoC:
    info = _lib.RobotInfoC()
    check(_lib.load().cppflow_robot_info_get(robot_id, info))
    return info


class Obstacles:
    """Host-side copy of the cuboid tables of a Problem (obstacles_cuboids [6], obstacles_Tcuboids [4,4];
    data_type_utils.py:109-127), flattened once so every launch can pass them by value."""

    def __init__(self, cuboids: Optional[Sequence[torch.Tensor]] = None, Tcuboids: Optional[Sequence[torch.Tensor]] = None):
        cuboids = list(cuboids) if cuboids is not None else []
        Tcuboids = list(Tcuboids) if Tcuboids is not None else []
        assert len(cuboids) == len(Tcuboids), "cuboids / Tcuboids length mismatch"
        assert len(cuboids) <= 8, "at most 8 cuboid obstacles are supported"
        self.n = len(cuboids)
        cu, tc = [], []
        for c, T in zip(cuboids, Tcuboids):
            c = torch.as_tensor(c).detach().float().cpu().reshape(-1)
            T = torch.as_tensor(T).detach().float().cpu()
            assert c.numel() == 6 and T.shape == (4, 4)
            cu += c.tolist()
            tc += T.reshape(-1).tolist()
        self._cu = _lib.host_floats(cu) if self.n else None
        self._tc = _lib.host_floats(tc) if self.n else None

    @property
    def cuboids_ptr(self):
        return self._cu

    @property
    def Tcuboids_ptr(self):
        return self._tc

    def single(self, i: int) -> "Obstacles":
        o = Obstacles.__new__(Obstacles)
        o.n = 1
        o._cu = _lib.host_floats(list(self._cu[6 * i : 6 * i + 6]))
        o._tc = _lib.host_floats(list(self._tc[16 * i : 16 * i + 16]))
        return o


NO_OBSTACLES = None


def _obs(ob: Optional[Obstacles]):
    if ob is None or ob.n == 0:
        return None, None, 0
    return ob.cuboids_ptr, ob.Tcuboids_ptr, ob.n


def make_params(pms) -> LmParamsC:
    """OptimizationParameters (lm_hyper_parameters.py:14-80) -> cppflow_lm_params.  None fields (the reference's
    parameter sets leave unused alphas as None) become 0."""

    def f(v):
        return 0.0 if v is None else float(v)

    for flag in ("pose_do_scale_down_satisfied", "differencing_do_ignore_satisfied", "differencing_do_scale_satisfied"):
        if getattr(pms, flag, False):
            raise NotImplementedError(
                f"OptimizationParameters.{flag}=True: the row scaling / filtering options are implemented on the dense form "
                "(optimization_utils.LmResidualFns.get_r_and_J and its helpers), not in the block-tridiagonal CUDA solver. "
                "Both live parameter sets leave them off (lm_hyper_parameters.py:86-151) and the reference's own "
                "get_r_and_J raises AttributeError when one is on (it reads pms.constraints, optimization_utils.py:515-520)"
            )
    return LmParamsC(
        f(pms.lm_lambda), f(pms.alpha_position), f(pms.alpha_rotation), f(pms.alpha_differencing),
        f(pms.alpha_differencing_prismatic_scaling), f(pms.alpha_virtual_configs), f(pms.alpha_self_collision),
        f(pms.alpha_env_collision), int(bool(pms.use_pose)), int(bool(pms.use_differencing)),
        int(bool(pms.use_virtual_configs)), int(pms.n_virtual_configs or 0), int(bool(pms.use_self_collisions)),
        int(bool(pms.use_env_collisions)),
    )


def _check_q(q: torch.Tensor, ndof: int, name="x") -> torch.Tensor:
    q = require_cuda(q, name)
    assert q.dim() == 2 and q.shape[1] == ndof, f"{name} must be [n, {ndof}], is {tuple(q.shape)}"
    return q


@_on_device
def forward_kinematics(rid: int, ndof: int, q: torch.Tensor) -> torch.Tensor:
    q = _check_q(q, ndof)
    out = torch.empty((q.shape[0], 7), device=q.device, dtype=torch.float32)
    check(_lib.load().cppflow_forward_kinematics(rid, ptr(q), q.shape[0], ptr(out), stream_ptr(q.device)))
    return out


@_on_device
def jacobian(rid: int, ndof: int, q: torch.Tensor) -> torch.Tensor:
    q = _check_q(q, ndof)
    out = torch.empty((q.shape[0], 6, ndof), device=q.device, dtype=torch.float32)
    check(_lib.load().cppflow_jacobian(rid, ptr(q), q.shape[0], ptr(out), stream_ptr(q.device)))
    return out


@_on_device
def pose_errors(rid: int, ndof: int, q: torch.Tensor, target: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    q = _check_q(q, ndof)
    target = require_cuda(target, "target_poses")
    assert target.dim() == 2 and target.shape[1] == 7 and target.shape[0] > 0
    assert q.shape[0] % target.shape[0] == 0, "x rows must be a multiple of the target path length"
    err = torch.empty((q.shape[0], 6), device=q.device, dtype=torch.float32)
    cur = torch.empty((q.shape[0], 7), device=q.device, dtype=torch.float32)
    check(_lib.load().cppflow_pose_errors(rid, ptr(q), ptr(target), q.shape[0], target.shape[0], ptr(err), ptr(cur),
                                          stream_ptr(q.device)))
    return err, cur


@_on_device
def lm_pose_step(rid: int, ndof: int, params: LmParamsC, q: torch.Tensor, target: torch.Tensor, clamp: bool,
                 return_residual: bool = False, out: Optional[torch.Tensor] = None):
    q = _check_q(q, ndof)
    target = require_cuda(target, "target_path")
    assert target.dim() == 2 and target.shape[1] == 7 and target.shape[0] > 0
    assert q.shape[0] % target.shape[0] == 0, "x rows must be a multiple of the target path length"
    n = q.shape[0]
    x_out = torch.empty_like(q) if out is None else out
    J = torch.empty((n, 6, ndof), device=q.device, dtype=torch.float32) if return_residual else None
    e = torch.empty((n, 6, 1), device=q.device, dtype=torch.float32) if return_residual else None
    check(_lib.load().cppflow_lm_pose_step(rid, params, ptr(q), ptr(target), n, target.shape[0], int(clamp), ptr(x_out),
                                           ptr(J), ptr(e), stream_ptr(q.device)))
    if return_residual:
        return x_out, J, e
    return x_out


@_on_device
def lm_pose_steps_(rid: int, ndof: int, params: LmParamsC, lambdas, q: torch.Tensor, target: torch.Tensor,
                   clamp: bool = True) -> torch.Tensor:
    """len(lambdas) pose-only LM steps in place on q (step i with damping lambdas[i]): one library call."""
    assert q.is_cuda and q.dtype == torch.float32 and q.is_contiguous() and q.dim() == 2 and q.shape[1] == ndof
    target = require_cuda(target, "target_path")
    assert target.dim() == 2 and target.shape[1] == 7 and q.shape[0] % target.shape[0] == 0
    tmp = torch.empty_like(q)
    lam = _lib.host_floats([float(v) for v in lambdas])
    check(_lib.load().cppflow_lm_pose_steps(rid, params, lam, len(lambdas), ptr(q), ptr(tmp), ptr(target), q.shape[0],
                                            target.shape[0], int(clamp), stream_ptr(q.device)))
    return q


@_on_device
def clamp_to_joint_limits_(rid: int, ndof: int, q: torch.Tensor) -> torch.Tensor:
    assert q.is_cuda and q.dtype == torch.float32 and q.is_contiguous(), "in-place clamp needs a contiguous fp32 CUDA tensor"
    assert q.dim() == 2 and q.shape[1] == ndof
    check(_lib.load().cppflow_clamp_to_joint_limits(rid, ptr(q), q.shape[0], stream_ptr(q.device)))
    return q


@_on_device
def self_collision_distances(rid: int, ndof: int, n_pairs: int, q: torch.Tensor, with_jacobian: bool = False):
    q = _check_q(q, ndof)
    n = q.shape[0]
    d = torch.empty((n, n_pairs), device=q.device, dtype=torch.float32)
    J = torch.empty((n, n_pairs, ndof), device=q.device, dtype=torch.float32) if with_jacobian else None
    check(_lib.load().cppflow_self_collision_distances(rid, ptr(q), n, ptr(d), ptr(J), stream_ptr(q.device)))
    return (d, J) if with_jacobian else d


@_on_device
def env_collision_distances(rid: int, ndof: int, n_caps: int, q: torch.Tensor, ob: Obstacles, index: int = 0,
                            with_jacobian: bool = False):
    q = _check_q(q, ndof)
    n = q.shape[0]
    one = ob if ob.n == 1 and index == 0 else ob.single(index)
    d = torch.empty((n, n_caps), device=q.device, dtype=torch.float32)
    J = torch.empty((n, n_caps, ndof), device=q.device, dtype=torch.float32) if with_jacobian else None
    check(_lib.load().cppflow_env_collision_distances(rid, ptr(q), n, one.cuboids_ptr, one.Tcuboids_ptr, ptr(d), ptr(J),
                                                      stream_ptr(q.device)))
    return (d, J) if with_jacobian else d


@_on_device
def collision_flags(rid: int, ndof: int, q: torch.Tensor, ob: Optional[Obstacles], want_self=True, want_env=True):
    q = _check_q(q, ndof)
    n = q.shape[0]
    s = torch.empty((n,), device=q.device, dtype=torch.uint8) if want_self else None
    e = torch.empty((n,), device=q.device, dtype=torch.uint8) if want_env else None
    cu, tc, no = _obs(ob)
    check(_lib.load().cppflow_collision_flags(rid, ptr(q), n, cu, tc, no, ptr(s), ptr(e), stream_ptr(q.device)))
    return s, e


_WORKSPACES = {}


def _workspace(device, nbytes: int, key: str) -> torch.Tensor:
    """Grow-only scratch buffer per (device, current stream, purpose): the C ABI never allocates, and launches enqueued
    on different streams (planners.plan_many runs one problem per stream) must not share scratch memory."""
    k = (str(device), torch.cuda.current_stream(device).cuda_stream, key)
    buf = _WORKSPACES.get(k)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty((max(nbytes, 256),), device=device, dtype=torch.uint8)
        _WORKSPACES[k] = buf
    return buf


@_on_device
def lm_full_step(rid: int, ndof: int, params: LmParamsC, q: torch.Tensor, xv: Optional[torch.Tensor],
                 target: Optional[torch.Tensor], P: int, T: int, ob: Optional[Obstacles], clamp: bool,
                 out: Optional[torch.Tensor] = None, overlap: bool = False,
                 workspace: Optional[torch.Tensor] = None, fused: bool = False, segments: int = 0) -> torch.Tensor:
    """levenberg_marquardt_full (+ clamp) for P paths of T waypoints on the current stream.  `fused`: CPPFLOW_LM_FUSED
    (elimination inside the assembly kernel, same bits).  `segments`: CPPFLOW_LM_SEGMENTS (parallel-in-time solve for
    few paths, csrc/lm_segsolve.cuh; rounding-level differences, larger workspace).  `overlap`: launch the
    solve with CPPFLOW_LM_OVERLAP (footprint that fits next to an assembly CTA, high launch priority) - for callers that run several chunks
    of paths on several streams (pipeline.ResidentPipeline), which must also pass one `workspace` per stream."""
    q = _check_q(q, ndof)
    assert q.shape[0] == P * T, f"x must have P*T = {P * T} rows, has {q.shape[0]}"
    if xv is not None:
        xv = _check_q(xv, ndof, "virtual_configs")
        assert xv.shape == q.shape
    if target is not None:
        target = require_cuda(target, "target_path")
        assert target.shape == (T, 7), f"target_path must be [{T}, 7], is {tuple(target.shape)}"
    lib = _lib.load()
    flags = (LM_CLAMP if clamp else 0) | (LM_OVERLAP if overlap else 0) | (LM_FUSED if fused else 0) | lm_segments(segments)
    nbytes = lib.cppflow_lm_full_workspace_bytes_ex(rid, P, T, flags)
    if workspace is None:
        ws = _workspace(q.device, nbytes, "lm_full")
    else:
        ws = workspace
        assert ws.is_cuda and ws.dtype == torch.uint8 and ws.numel() >= nbytes, "workspace too small"
    x_out = torch.empty_like(q) if out is None else out
    cu, tc, no = _obs(ob)
    check(lib.cppflow_lm_full_step(rid, params, ptr(q), ptr(xv), ptr(target), P, T, cu, tc, no, flags, ptr(ws),
                                   ws.numel(), ptr(x_out), stream_ptr(q.device)))
    return x_out


@_on_device
def joint_limit_flags(rid: int, ndof: int, q2d: torch.Tensor, eps_revolute: float, eps_prismatic: float) -> torch.Tensor:
    q2d = _check_q(q2d, ndof, "qs")
    out = torch.empty((q2d.shape[0],), device=q2d.device, dtype=torch.float32)
    check(_lib.load().cppflow_joint_limit_flags(rid, ptr(q2d), q2d.shape[0], float(eps_revolute), float(eps_prismatic),
                                                ptr(out), stream_ptr(q2d.device)))
    return out


@_on_device
def dp_search(rid: int, ndof: int, q: torch.Tensor, self_flags: torch.Tensor, env_flags: torch.Tensor):
    """-> best_path [T,D], memo int32 [k,T], costs [k,T], chosen int32 [T]"""
    q = require_cuda(q, "q")
    assert q.dim() == 3 and q.shape[2] == ndof, f"q must be [k, T, {ndof}], is {tuple(q.shape)}"
    k, T, _ = q.shape
    sf = require_cuda(self_flags.to(q.device), "self_collision_violations", torch.uint8)
    ef = require_cuda(env_flags.to(q.device), "env_collision_violations", torch.uint8)
    assert sf.shape == (k, T) and ef.shape == (k, T)
    lib = _lib.load()
    ws = _workspace(q.device, lib.cppflow_dp_search_workspace_bytes(k, T), "dp_search")
    best = torch.empty((T, ndof), device=q.device, dtype=torch.float32)
    memo = torch.empty((k, T), device=q.device, dtype=torch.int32)
    costs = torch.empty((k, T), device=q.device, dtype=torch.float32)
    chosen = torch.empty((T,), device=q.device, dtype=torch.int32)
    check(lib.cppflow_dp_search(rid, ptr(q), ptr(sf), ptr(ef), k, T, ptr(ws), ws.numel(), ptr(best), ptr(memo),
                                ptr(costs), ptr(chosen), stream_ptr(q.device)))
    return best, memo, costs, chosen


METRIC_NAMES = ("max_pos_cm", "max_rot_deg", "mjac_deg", "mjac_cm", "tl", "min_self", "min_env")


METRICS_SIGN_ONLY = 1  # CPPFLOW_METRICS_SIGN_ONLY


@_on_device
def path_metrics(rid: int, ndof: int, q: torch.Tensor, target: torch.Tensor, P: int, T: int,
                 ob: Optional[Obstacles], sign_only: bool = False) -> torch.Tensor:
    """[P, 8] metrics (METRIC_NAMES).  `sign_only`: the two minimum-distance columns are exact only when negative
    (enough for x_is_valid and the cost ranking; about half the time for thousands of paths)."""
    q = _check_q(q, ndof)
    assert q.shape[0] == P * T
    target = require_cuda(target, "target_path")
    assert target.shape == (T, 7)
    out = torch.empty((P, 8), device=q.device, dtype=torch.float32)
    cu, tc, no = _obs(ob)
    check(_lib.load().cppflow_path_metrics_ex(rid, ptr(q), ptr(target), P, T, cu, tc, no, METRICS_SIGN_ONLY if sign_only else 0,
                                              ptr(out), stream_ptr(q.device)))
    return out


@_on_device
def path_key_argmin(metrics: torch.Tensor, constraints, first_index: int) -> torch.Tensor:
    """int64 [3] = (smallest ranking key, number of valid paths, first_index) of the [P, 8] metrics rows, one launch
    (distributed.path_keys is the same arithmetic in torch)."""
    metrics = require_cuda(metrics, "metrics")
    assert metrics.dtype == torch.float32 and metrics.dim() == 2 and metrics.shape[1] == 8 and metrics.is_contiguous()
    out = torch.empty((3,), device=metrics.device, dtype=torch.int64)
    cons = _lib.ConstraintsC(constraints.max_allowed_position_error_cm, constraints.max_allowed_rotation_error_deg,
                             constraints.max_allowed_mjac_deg, constraints.max_allowed_mjac_cm)
    import ctypes as C

    check(_lib.load().cppflow_path_key_argmin(ptr(metrics), metrics.shape[0], C.byref(cons), first_index, ptr(out),
                                              stream_ptr(metrics.device)))
    return out


_PINNED = {}


@_on_device
def lm_alternating_loss(rid: int, ndof: int, params_diff: LmParamsC, params_pose: LmParamsC, constraints,
                        x_seed: torch.Tensor, target: torch.Tensor, T: int, ob: Optional[Obstacles], max_n_steps: int,
                        tmax_sec: float, return_if_valid_after_n_steps: int, convergence_threshold: float):
    """run_lm_alternating_loss for one path, driven by the library's C++ loop (csrc/lm_loop.cu): the same control flow
    as optimization.run_lm_alternating_loss_python with ~10 us instead of ~55 us of host time per iteration.
    -> (x_opt [T, ndof], n_steps_taken, is_valid, schedule, last_metrics list of 8)"""
    x_seed = _check_q(x_seed, ndof, "x_seed")
    assert x_seed.shape[0] == T, "the alternating loop refines ONE path"
    target = require_cuda(target, "target_path")
    assert target.shape == (T, 7)
    lib = _lib.load()
    dev = x_seed.device
    ws = _workspace(dev, lib.cppflow_lm_alternating_workspace_bytes(rid, T) + 256, "lm_loop")
    off = (-ws.data_ptr()) % 256
    pkey = (str(dev), torch.cuda.current_stream(dev).cuda_stream)
    pinned = _PINNED.get(pkey)
    if pinned is None:
        pinned = _PINNED[pkey] = torch.empty(8, dtype=torch.float32).pin_memory()
    cons = _lib.ConstraintsC(constraints.max_allowed_position_error_cm, constraints.max_allowed_rotation_error_deg,
                             constraints.max_allowed_mjac_deg, constraints.max_allowed_mjac_cm)
    res = _lib.LmLoopResultC()
    x_out = torch.empty_like(x_seed)
    cu, tc, no = _obs(ob)
    import ctypes as C

    tmax = 1e30 if tmax_sec is None or tmax_sec == float("inf") else float(tmax_sec)
    check(lib.cppflow_lm_alternating_loss(
        rid, params_diff, params_pose, cons, ptr(x_seed), ptr(target), T, cu, tc, no, int(max_n_steps), tmax,
        int(return_if_valid_after_n_steps), float(convergence_threshold), C.c_void_p(ws.data_ptr() + off),
        ws.numel() - off, C.c_void_p(pinned.data_ptr()), ptr(x_out), C.byref(res), stream_ptr(dev)))
    return x_out, int(res.n_steps_taken), bool(res.is_valid), res.schedule.decode(), list(res.last_metrics)


def lm_alternating_loss_many(jobs):
    """The alternating loop for several independent (problem, seed path) pairs in lock step (csrc/lm_loop.cu):
    `jobs` = list of dicts with keys rid, ndof, params_diff, params_pose, constraints, x_seed [T, ndof], target [T, 7],
    ob (Obstacles or None), max_n_steps, tmax_sec, return_if_valid_after_n_steps, convergence_threshold, stream
    (torch.cuda.Stream).  -> list of (x_opt, n_steps_taken, is_valid, schedule, last_metrics)."""
    import ctypes as C

    lib = _lib.load()
    n = len(jobs)
    arr = (_lib.LmLoopJobC * n)()
    keep, outs = [], []
    for k, jb in enumerate(jobs):
        x_seed = _check_q(jb["x_seed"], jb["ndof"], "x_seed")
        T = x_seed.shape[0]
        target = require_cuda(jb["target"], "target_path")
        assert target.shape == (T, 7)
        dev = x_seed.device
        stream = jb["stream"]
        nbytes = lib.cppflow_lm_alternating_workspace_bytes(jb["rid"], T) + 256
        with torch.cuda.stream(stream):
            ws = _workspace(dev, nbytes, "lm_loop")
            x_out = torch.empty_like(x_seed)
        off = (-ws.data_ptr()) % 256
        pkey = (str(dev), stream.cuda_stream)
        pinned = _PINNED.get(pkey)
        if pinned is None:
            pinned = _PINNED[pkey] = torch.empty(8, dtype=torch.float32).pin_memory()
        c = jb["constraints"]
        cons = _lib.ConstraintsC(c.max_allowed_position_error_cm, c.max_allowed_rotation_error_deg,
                                 c.max_allowed_mjac_deg, c.max_allowed_mjac_cm)
        res = _lib.LmLoopResultC()
        cu, tc, no = _obs(jb["ob"])
        tmax = jb["tmax_sec"]
        a = arr[k]
        a.robot = jb["rid"]
        a.params_diff = C.pointer(jb["params_diff"])
        a.params_pose = C.pointer(jb["params_pose"])
        a.constraints = C.pointer(cons)
        a.d_x_seed = x_seed.data_ptr()
        a.d_target = target.data_ptr()
        a.T = T
        a.h_cuboids = C.cast(cu, _lib.c_float_p) if cu is not None else None
        a.h_Tcuboids = C.cast(tc, _lib.c_float_p) if tc is not None else None
        a.n_obstacles = no
        a.max_n_steps = int(min(jb["max_n_steps"], 2 ** 31 - 1))
        a.tmax_sec = 1e30 if tmax is None or tmax == float("inf") else float(tmax)
        a.return_if_valid_after_n_steps = int(min(jb["return_if_valid_after_n_steps"], 2 ** 31 - 1))
        a.convergence_threshold = float(jb["convergence_threshold"])
        a.d_workspace = ws.data_ptr() + off
        a.workspace_bytes = ws.numel() - off
        a.h_pinned_metrics = pinned.data_ptr()
        a.d_x_out = x_out.data_ptr()
        a.result = C.pointer(res)
        a.stream = stream.cuda_stream
        keep.append((x_seed, target, ws, pinned, cons, cu, tc))
        outs.append((x_out, res))
    check(lib.cppflow_lm_alternating_loss_many(n, arr))
    return [(x, int(r.n_steps_taken), bool(r.is_valid), r.schedule.decode(), list(r.last_metrics)) for x, r in outs]


FLOW_REVERSE, FLOW_CLAMP = 1, 2  # CPPFLOW_FLOW_REVERSE / _CLAMP (include/cppflow_b200.h)


@_on_device
def flow_run(desc: _lib.FlowDescC, x: torch.Tensor, cond: torch.Tensor, reverse: bool, clamp: bool = False,
             out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """IKFlow's GLOW network over the rows of x [n, width] (csrc/k_flow.cu): z -> x with `reverse`, x -> z otherwise.
    Row i is conditioned on cond[i % len(cond)] ([x, y, z, qw, qx, qy, qz]).  `clamp` (reverse only) clamps the
    first ndof output columns to the joint limits.  Workspace from the per-stream scratch buffer; no host sync."""
    import ctypes as C

    x = require_cuda(x, "x")
    cond = require_cuda(cond, "cond")
    assert x.dim() == 2 and x.shape[1] == desc.width, f"x must be [n, {desc.width}], is {tuple(x.shape)}"
    assert cond.dim() == 2 and cond.shape[1] == 7 and cond.shape[0] >= 1, f"cond must be [m, 7], is {tuple(cond.shape)}"
    n = x.shape[0]
    out = torch.empty_like(x) if out is None else out
    assert out.is_cuda and out.dtype == torch.float32 and out.is_contiguous() and out.shape == x.shape
    lib = _lib.load()
    nbytes = lib.cppflow_flow_workspace_bytes(C.byref(desc), n)
    if nbytes == 0:
        check(-1)
    ws = _workspace(x.device, nbytes, "flow")
    flags = (FLOW_REVERSE if reverse else 0) | (FLOW_CLAMP if clamp else 0)
    check(lib.cppflow_flow_run(C.byref(desc), ptr(x), ptr(cond), n, cond.shape[0], flags, ptr(ws), ws.numel(), ptr(out),
                               stream_ptr(x.device)))
    return out


FLOW_TRAIN_NO_UPDATE = 1  # CPPFLOW_FLOW_TRAIN_NO_UPDATE (include/cppflow_b200.h)


def flow_train_workspace_bytes(desc: _lib.FlowTrainDescC, batch: int) -> int:
    """Bytes of the workspace of flow_train_step; raises for a desc or batch the library rejects."""
    import ctypes as C

    nbytes = _lib.load().cppflow_flow_train_workspace_bytes(C.byref(desc), batch)
    if nbytes == 0:
        check(-1)
    return nbytes


def flow_train_step(desc: _lib.FlowTrainDescC, x: torch.Tensor, cond: torch.Tensor, workspace: torch.Tensor,
                    loss: torch.Tensor, grad: Optional[torch.Tensor] = None, update: bool = True) -> None:
    """One training step of IKFlow's network (csrc/k_flow_train.cu) on the current stream: x [n, width] and cond
    [n, dim_cond] (n % 128 == 0) -> loss [1] (the batch's mean NLL), the packed gradient into `grad` when given, and
    with `update` the Adam step on the tables `desc` points at.  No allocation and no host synchronisation."""
    import ctypes as C

    n = x.shape[0]
    assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous() and x.shape == (n, desc.flow.width)
    assert cond.is_cuda and cond.dtype == torch.float32 and cond.is_contiguous() and cond.shape == (n, desc.flow.dim_cond)
    assert loss.is_cuda and loss.dtype == torch.float32 and loss.numel() >= 1
    assert grad is None or (grad.is_cuda and grad.dtype == torch.float32 and grad.is_contiguous())
    flags = 0 if update else FLOW_TRAIN_NO_UPDATE
    check(_lib.load().cppflow_flow_train_step(C.byref(desc), ptr(x), ptr(cond), n, flags, ptr(workspace),
                                              workspace.numel() * workspace.element_size(), ptr(loss), ptr(grad),
                                              stream_ptr(x.device)))


def flow_train_batch(desc: _lib.FlowTrainDescC, q: torch.Tensor, poses: torch.Tensor, seed: int, noise_scale: float,
                     x: torch.Tensor, cond: torch.Tensor, idx: Optional[torch.Tensor] = None,
                     noise: Optional[torch.Tensor] = None) -> None:
    """Draws the training batch of the desc's current step counter into x [n, width] and cond [n, dim_cond] from the
    dataset q [N, ndof], poses [N, 7] (include/cppflow_b200.h: cppflow_flow_train_batch).  No host synchronisation."""
    import ctypes as C

    n = x.shape[0]
    assert q.is_cuda and q.dtype == torch.float32 and q.is_contiguous() and q.shape[1] == desc.flow.ndof
    assert poses.is_cuda and poses.dtype == torch.float32 and poses.is_contiguous() and poses.shape == (q.shape[0], 7)
    assert x.is_contiguous() and x.shape == (n, desc.flow.width) and cond.is_contiguous()
    assert cond.shape == (n, desc.flow.dim_cond)
    check(_lib.load().cppflow_flow_train_batch(C.byref(desc), ptr(q), ptr(poses), q.shape[0], n, seed & (2**64 - 1),
                                               float(noise_scale), ptr(x), ptr(cond), ptr(idx), ptr(noise),
                                               stream_ptr(x.device)))
