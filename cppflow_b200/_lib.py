"""ctypes binding of libcppflow_b200.so (include/cppflow_b200.h).

There is no CPU fallback: if the library is missing or a call fails this raises `RuntimeError`, which is also
what the reference's TimerContext turns any failure into (cppflow/utils.py:139-141)."""
import ctypes as C
import os
import threading

import torch

from . import _build

_LOCK = threading.Lock()
_LIB = None

c_float_p = C.POINTER(C.c_float)


class LmParamsC(C.Structure):
    """cppflow_lm_params"""

    _fields_ = [
        ("lm_lambda", C.c_float),
        ("alpha_position", C.c_float),
        ("alpha_rotation", C.c_float),
        ("alpha_differencing", C.c_float),
        ("alpha_differencing_prismatic_scaling", C.c_float),
        ("alpha_virtual_configs", C.c_float),
        ("alpha_self_collision", C.c_float),
        ("alpha_env_collision", C.c_float),
        ("use_pose", C.c_int32),
        ("use_differencing", C.c_int32),
        ("use_virtual_configs", C.c_int32),
        ("n_virtual_configs", C.c_int32),
        ("use_self_collisions", C.c_int32),
        ("use_env_collisions", C.c_int32),
    ]


class RobotInfoC(C.Structure):
    """cppflow_robot_info"""

    _fields_ = [
        ("ndof", C.c_int32),
        ("n_capsules", C.c_int32),
        ("n_pairs", C.c_int32),
        ("n_chain", C.c_int32),
        ("lower", C.c_float * 8),
        ("upper", C.c_float * 8),
        ("is_prismatic", C.c_int32 * 8),
        ("capsules", (C.c_float * 7) * 10),
        ("capsule_frame", C.c_int32 * 10),
        ("pairs", (C.c_int32 * 2) * 28),
        ("name", C.c_char * 16),
    ]


class ConstraintsC(C.Structure):
    """cppflow_constraints"""

    _fields_ = [
        ("max_allowed_position_error_cm", C.c_double),
        ("max_allowed_rotation_error_deg", C.c_double),
        ("max_allowed_mjac_deg", C.c_double),
        ("max_allowed_mjac_cm", C.c_double),
    ]


class LmLoopResultC(C.Structure):
    """cppflow_lm_loop_result"""

    _fields_ = [
        ("n_steps_taken", C.c_int32),
        ("is_valid", C.c_int32),
        ("last_metrics", C.c_float * 8),
        ("schedule", C.c_char * 256),
    ]


class LmLoopJobC(C.Structure):
    """cppflow_lm_loop_job"""

    _fields_ = [
        ("robot", C.c_int32),
        ("params_diff", C.POINTER(LmParamsC)),
        ("params_pose", C.POINTER(LmParamsC)),
        ("constraints", C.POINTER(ConstraintsC)),
        ("d_x_seed", C.c_void_p),
        ("d_target", C.c_void_p),
        ("T", C.c_int64),
        ("h_cuboids", c_float_p),
        ("h_Tcuboids", c_float_p),
        ("n_obstacles", C.c_int32),
        ("max_n_steps", C.c_int32),
        ("tmax_sec", C.c_double),
        ("return_if_valid_after_n_steps", C.c_int32),
        ("convergence_threshold", C.c_double),
        ("d_workspace", C.c_void_p),
        ("workspace_bytes", C.c_size_t),
        ("h_pinned_metrics", C.c_void_p),
        ("d_x_out", C.c_void_p),
        ("result", C.POINTER(LmLoopResultC)),
        ("stream", C.c_void_p),
    ]


class FlowDescC(C.Structure):
    """cppflow_flow_desc"""

    _fields_ = [
        ("robot", C.c_int32),
        ("width", C.c_int32),
        ("ndof", C.c_int32),
        ("dim_cond", C.c_int32),
        ("nb_nodes", C.c_int32),
        ("coeff_fn_config", C.c_int32),
        ("coeff_fn_internal_size", C.c_int32),
        ("rnvp_clamp", C.c_float),
        ("d_w_in", C.c_void_p),
        ("d_w_hidden", C.c_void_p),
        ("d_b_hidden", C.c_void_p),
        ("d_w_out", C.c_void_p),
        ("d_b_out", C.c_void_p),
        ("d_scale", C.c_void_p),
        ("d_perm", C.c_void_p),
        ("d_perm_inv", C.c_void_p),
    ]


class FlowTrainDescC(C.Structure):
    """cppflow_flow_train_desc"""

    _fields_ = [
        ("flow", FlowDescC),
        ("d_params", C.c_void_p),
        ("d_adam_m", C.c_void_p),
        ("d_adam_v", C.c_void_p),
        ("d_w_in_t", C.c_void_p),
        ("d_w_hidden_t", C.c_void_p),
        ("d_w_out_t", C.c_void_p),
        ("d_counters", C.c_void_p),
        ("lr", C.c_double),
        ("beta1", C.c_double),
        ("beta2", C.c_double),
        ("eps", C.c_double),
        ("weight_decay", C.c_double),
        ("lr_decay", C.c_double),
        ("lr_decay_steps", C.c_int64),
    ]


class IkRefineDescC(C.Structure):
    """cppflow_ik_refine_desc"""

    _fields_ = [
        ("lambdas", C.c_float * 32),
        ("n_steps", C.c_int32),
        ("pos_tol", C.c_float),
        ("rot_tol", C.c_float),
        ("alpha_position", C.c_float),
        ("alpha_rotation", C.c_float),
        ("flags", C.c_int32),
    ]


LM_BATCHED_PINNED_BYTES = 64  # CPPFLOW_LM_BATCHED_PINNED_BYTES

ABI_VERSION = 5  # CPPFLOW_ABI_VERSION of include/cppflow_b200.h

_VP, _I, _I64, _SZ, _F, _DBL = C.c_void_p, C.c_int, C.c_int64, C.c_size_t, C.c_float, C.c_double
_PROTOTYPES = {
    # name: (restype, argtypes)
    "cppflow_version": (C.c_char_p, []),
    "cppflow_last_error": (C.c_char_p, []),
    "cppflow_abi_info": (_I, [C.POINTER(C.c_int64), _I]),
    "cppflow_robot_info_get": (_I, [_I, C.POINTER(RobotInfoC)]),
    "cppflow_forward_kinematics": (_I, [_I, _VP, _I64, _VP, _VP]),
    "cppflow_jacobian": (_I, [_I, _VP, _I64, _VP, _VP]),
    "cppflow_pose_errors": (_I, [_I, _VP, _VP, _I64, _I64, _VP, _VP, _VP]),
    "cppflow_lm_pose_step": (_I, [_I, C.POINTER(LmParamsC), _VP, _VP, _I64, _I64, _I, _VP, _VP, _VP, _VP]),
    "cppflow_lm_pose_steps": (_I, [_I, C.POINTER(LmParamsC), c_float_p, _I, _VP, _VP, _VP, _I64, _I64, _I, _VP]),
    "cppflow_clamp_to_joint_limits": (_I, [_I, _VP, _I64, _VP]),
    "cppflow_self_collision_distances": (_I, [_I, _VP, _I64, _VP, _VP, _VP]),
    "cppflow_env_collision_distances": (_I, [_I, _VP, _I64, c_float_p, c_float_p, _VP, _VP, _VP]),
    "cppflow_collision_flags": (_I, [_I, _VP, _I64, c_float_p, c_float_p, _I, _VP, _VP, _VP]),
    "cppflow_lm_full_workspace_bytes": (_SZ, [_I, _I64, _I64]),
    "cppflow_lm_full_workspace_bytes_ex": (_SZ, [_I, _I64, _I64, _I]),
    "cppflow_lm_full_step": (_I, [_I, C.POINTER(LmParamsC), _VP, _VP, _VP, _I64, _I64, c_float_p, c_float_p, _I, _I,
                                  _VP, _SZ, _VP, _VP]),
    "cppflow_lm_full_assemble": (_I, [_I, C.POINTER(LmParamsC), _VP, _VP, _VP, _I64, _I64, c_float_p, c_float_p, _I, _VP,
                                      _SZ, _VP]),
    "cppflow_lm_full_solve": (_I, [_I, C.POINTER(LmParamsC), _VP, _I64, _I64, _I, _VP, _SZ, _VP, _VP]),
    "cppflow_lm_alternating_workspace_bytes": (_SZ, [_I, _I64]),
    "cppflow_lm_alternating_loss": (_I, [_I, C.POINTER(LmParamsC), C.POINTER(LmParamsC), C.POINTER(ConstraintsC), _VP, _VP,
                                         _I64, c_float_p, c_float_p, _I, _I, _DBL, _I, _DBL, _VP, _SZ, _VP, _VP,
                                         C.POINTER(LmLoopResultC), _VP]),
    "cppflow_lm_alternating_loss_many": (_I, [_I, C.POINTER(LmLoopJobC)]),
    "cppflow_lm_alternating_batched_workspace_bytes": (_SZ, [_I, _I64, _I64]),
    "cppflow_lm_alternating_loss_batched": (_I, [_I, C.POINTER(LmParamsC), C.POINTER(LmParamsC), C.POINTER(ConstraintsC),
                                                 _VP, _VP, _I64, _I64, c_float_p, c_float_p, _I, _I, _DBL, _I, _DBL, _VP,
                                                 _SZ, _VP, _VP, C.POINTER(LmLoopResultC), _VP]),
    "cppflow_joint_limit_flags": (_I, [_I, _VP, _I64, _F, _F, _VP, _VP]),
    "cppflow_dp_search_workspace_bytes": (_SZ, [_I64, _I64]),
    "cppflow_dp_search": (_I, [_I, _VP, _VP, _VP, _I64, _I64, _VP, _SZ, _VP, _VP, _VP, _VP, _VP]),
    "cppflow_dp_backtrack": (_I, [_VP, _VP, _I64, _I64, _I, _VP, _I64, _VP, _VP]),
    "cppflow_path_metrics": (_I, [_I, _VP, _VP, _I64, _I64, c_float_p, c_float_p, _I, _VP, _VP]),
    "cppflow_path_key_argmin": (_I, [_VP, _I64, C.POINTER(ConstraintsC), _I64, _VP, _VP]),
    "cppflow_path_metrics_ex": (_I, [_I, _VP, _VP, _I64, _I64, c_float_p, c_float_p, _I, _I, _VP, _VP]),
    "cppflow_flow_workspace_bytes": (_SZ, [C.POINTER(FlowDescC), _I64]),
    "cppflow_flow_run": (_I, [C.POINTER(FlowDescC), _VP, _VP, _I64, _I64, _I, _VP, _SZ, _VP, _VP]),
    "cppflow_flow_train_workspace_bytes": (_SZ, [C.POINTER(FlowTrainDescC), _I64]),
    "cppflow_flow_train_step": (_I, [C.POINTER(FlowTrainDescC), _VP, _VP, _I64, _I, _VP, _SZ, _VP, _VP, _VP]),
    "cppflow_flow_train_batch": (_I, [C.POINTER(FlowTrainDescC), _VP, _VP, _I64, _I64, C.c_uint64, _F, _VP, _VP, _VP, _VP,
                                      _VP]),
    "cppflow_flow_train_batch_rows": (_I, [C.POINTER(FlowTrainDescC), _VP, _VP, _I64, _I64, _I64, C.c_uint64, _F, _VP, _VP,
                                           _VP, _VP, _VP]),
    "cppflow_flow_train_apply": (_I, [C.POINTER(FlowTrainDescC), _VP, _I64, _VP, _SZ, _VP]),
    "cppflow_flow_grad_tree_reduce": (_I, [_VP, _I, _I64, _I64, _F, _VP, _VP]),
    "cppflow_ik_refine": (_I, [_I, C.POINTER(IkRefineDescC), _VP, _VP, _I64, _I64, _VP, _VP, _VP, _VP, _VP]),
    "cppflow_ik_round_inputs": (_I, [_VP, _I64, _I, _VP, C.c_uint64, _I, _I, _F, _VP, _VP, _VP]),
    "cppflow_ik_select_workspace_bytes": (_SZ, [_I64]),
    "cppflow_ik_select": (_I, [_I, _VP, _VP, _VP, _I64, _I, _VP, _VP, _VP, _VP, _VP, _SZ, _VP]),
    "cppflow_fp32_probe": (_I, [_I, _I, _VP, C.POINTER(C.c_double), _VP]),
}
EXPORTED_SYMBOLS = tuple(_PROTOTYPES)


def library_path() -> str:
    return _build.LIB


def load(build_if_missing: bool = True):
    """Load (building first when the in-tree .so is absent or stale and nvcc is available)."""
    global _LIB
    with _LOCK:
        if _LIB is not None:
            return _LIB
        path = _build.LIB
        if build_if_missing and _build.is_stale():
            try:
                _build.build()
            except Exception as e:  # a prebuilt library is still usable on a box without nvcc - IF its ABI matches,
                if not os.path.exists(path):  # which the check below establishes
                    raise RuntimeError(f"libcppflow_b200.so is missing and could not be built: {e}") from e
                import warnings

                warnings.warn(f"libcppflow_b200.so is older than its sources and could not be rebuilt ({e}); "
                              "loading it after an ABI check")
        if not os.path.exists(path):
            raise RuntimeError(
                f"{path} not found. Build it with `python -m cppflow_b200._build` (needs nvcc); there is no CPU fallback."
            )
        lib = C.CDLL(path)
        missing = [name for name in _PROTOTYPES if not hasattr(lib, name)]
        if missing:
            raise RuntimeError(f"{path} does not export {missing}: it was built from another include/cppflow_b200.h; "
                               "rebuild with `python -m cppflow_b200._build --force`")
        for name, (restype, argtypes) in _PROTOTYPES.items():
            fn = getattr(lib, name)
            fn.restype = restype
            fn.argtypes = argtypes
        got = (C.c_int64 * 6)()
        n = lib.cppflow_abi_info(got, 6)
        want = [ABI_VERSION] + [C.sizeof(t) for t in (LmParamsC, RobotInfoC, ConstraintsC, LmLoopResultC, LmLoopJobC)]
        if n != 6 or list(got) != want:
            raise RuntimeError(f"{path}: ABI mismatch (library {list(got)[:n]}, binding {want}): struct layouts differ, "
                               "refusing to call into it; rebuild with `python -m cppflow_b200._build --force`")
        _LIB = lib
        return lib


class CppflowError(RuntimeError):
    pass


def check(rc: int):
    if rc != 0:
        msg = load().cppflow_last_error().decode()
        raise CppflowError(f"cppflow_b200 native call failed (code {rc}): {msg}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(t: torch.Tensor, name: str, dtype=torch.float32) -> torch.Tensor:
    """The hot path has no CPU implementation: insist on a contiguous CUDA tensor of the right dtype."""
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(
            f"{name} is on {t.device}: cppflow_b200 runs only on CUDA (sm_100a); there is no CPU fallback"
        )
    if t.dtype != dtype:
        t = t.to(dtype)
    return t.contiguous()


def host_floats(values):
    """Small host float table -> ctypes array pointer (kept alive by the caller holding the return value)."""
    arr = (C.c_float * len(values))(*values)
    return arr
