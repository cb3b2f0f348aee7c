"""CPU: the C-ABI library loads, exports every symbol include/cppflow_b200.h declares, and its compile-time robot
tables agree with the oracle's independently written tables.  No compute calls (no GPU here)."""
import ctypes
import os
import re

import numpy as np
import pytest

from oracle import robots as R

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_functions():
    text = open(os.path.join(REPO, "include", "cppflow_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(cppflow_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_are_exported():
    from cppflow_b200 import _lib

    lib = _lib.load()
    names = declared_functions()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/cppflow_b200.h but not exported"
    assert set(names) == set(_lib.EXPORTED_SYMBOLS), set(names) ^ set(_lib.EXPORTED_SYMBOLS)
    assert b"sm_100a" in lib.cppflow_version()


def test_struct_layouts_match_header():
    from cppflow_b200 import _lib

    assert ctypes.sizeof(_lib.LmParamsC) == 8 * 4 + 6 * 4
    assert ctypes.sizeof(_lib.RobotInfoC) == 4 * 4 + 8 * 4 * 3 + 10 * 7 * 4 + 10 * 4 + 28 * 2 * 4 + 16


def test_error_codes_and_workspace_sizes_without_gpu():
    from cppflow_b200 import _lib

    lib = _lib.load()
    info = _lib.RobotInfoC()
    assert lib.cppflow_robot_info_get(7, info) == -1  # CPPFLOW_E_INVALID
    assert b"unknown robot id" in lib.cppflow_last_error()
    # blocks (paths padded to 16-path groups, rounded to 256 bytes)
    assert lib.cppflow_lm_full_workspace_bytes(0, 8192, 300) == 8192 * 300 * 44 * 4
    assert lib.cppflow_lm_full_workspace_bytes(2, 10, 20) == 16 * 20 * 36 * 4
    # segmented solve (16 segments): + factor area (= blocks) + corners (2 sides x 27 float4 per segment) + 15 separators
    base = 16 * 300 * 44 * 4
    assert lib.cppflow_lm_full_workspace_bytes_ex(0, 16, 300, 16 << 8) == (
        base + 16 * 300 * 44 * 4 + 16 * 2 * 27 * 16 * 16 + 15 * 2 * 16 * 16)
    assert lib.cppflow_lm_full_workspace_bytes_ex(0, 16, 300, 0) == base
    assert lib.cppflow_lm_full_workspace_bytes_ex(0, 16, 6, 16 << 8) == lib.cppflow_lm_full_workspace_bytes(0, 16, 6)
    assert lib.cppflow_dp_search_workspace_bytes(175, 295) >= 4 * (295 * 175 + 294 * 175 * 175)
    with pytest.raises(_lib.CppflowError):
        _lib.check(-1)


def test_lm_step_rejects_unknown_flags_without_gpu():
    """A do_clamp bit outside CLAMP | OVERLAP | SEGMENTS (4 selected a removed variant) is an invalid argument, reported
    before anything reaches the device - every other argument here would pass the checks."""
    from cppflow_b200 import _lib
    from cppflow_b200.lm_hyper_parameters import ALT_LOSS_V2_1_DIFF
    from cppflow_b200.ops import make_params

    lib = _lib.load()
    P, T = 16, 20
    nbytes = lib.cppflow_lm_full_workspace_bytes_ex(0, P, T, 4)
    assert nbytes > 0
    prm = make_params(ALT_LOSS_V2_1_DIFF)
    dummy = ctypes.c_void_p(1 << 20)  # never dereferenced: non-null and 256-byte aligned
    assert lib.cppflow_lm_full_step(0, prm, dummy, None, dummy, P, T, None, None, 0, 4, dummy, nbytes, dummy, None) == -1
    assert b"do_clamp" in lib.cppflow_last_error()
    assert lib.cppflow_lm_full_solve(0, prm, dummy, P, T, 4 | 1, dummy, nbytes, dummy, None) == -1
    assert b"do_clamp" in lib.cppflow_last_error()


@pytest.mark.parametrize("name", ["fetch", "fetch_arm", "panda"])
def test_robot_tables_match_oracle(name):
    from cppflow_b200.robot import get_robot
    from cppflow_b200 import ops

    rob = get_robot(name)
    m = R.get_model(name)
    assert rob.ndof == m.ndof and rob.name == m.name and rob.formal_robot_name == m.formal_robot_name
    assert rob.prismatic_joint_idxs == m.prismatic_joint_idxs and rob.revolute_joint_idxs == m.revolute_joint_idxs
    assert rob.actuated_joint_names == m.actuated_joint_names
    assert rob.end_effector_link_name == m.end_effector_link_name
    np.testing.assert_allclose(np.array(rob.actuated_joints_limits), np.array(m.actuated_joints_limits), atol=1e-6)
    assert rob._collision_pairs == m.pairs
    assert list(rob._collision_capsules_by_link.keys()) == [c.link for c in m.capsules]
    info = ops._info(rob.robot_id)
    for c, cap in enumerate(m.capsules):
        np.testing.assert_allclose(list(info.capsules[c]), list(cap.p1) + list(cap.p2) + [cap.radius], atol=1e-7)
        assert info.capsule_frame[c] == cap.frame
    assert info.n_chain == len(m.chain)


def test_no_cpu_fallback():
    import torch
    from cppflow_b200.robot import get_robot

    rob = get_robot("panda")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        rob.forward_kinematics(torch.zeros((3, 7)))
    with pytest.raises(NotImplementedError):
        rob.config_self_collides(None)


def test_ctypes_structs_match_the_c_header(tmp_path):
    """sizeof / offsetof of every struct of include/cppflow_b200.h, as gcc sees them, against the ctypes mirrors."""
    import shutil
    import subprocess

    from cppflow_b200 import _lib

    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    src = tmp_path / "sizes.c"
    src.write_text(
        '#include <stdio.h>\n#include <stddef.h>\n#include "cppflow_b200.h"\n'
        "int main(void) {\n"
        '  printf("%zu %zu %zu %zu %zu\\n", sizeof(cppflow_lm_params), sizeof(cppflow_robot_info), sizeof(cppflow_constraints),\n'
        "         sizeof(cppflow_lm_loop_result), sizeof(cppflow_lm_loop_job));\n"
        '  printf("%zu %zu %zu %zu %zu\\n", offsetof(cppflow_lm_loop_job, T), offsetof(cppflow_lm_loop_job, tmax_sec),\n'
        "         offsetof(cppflow_lm_loop_job, convergence_threshold), offsetof(cppflow_lm_loop_job, result),\n"
        "         offsetof(cppflow_lm_loop_result, schedule));\n"
        "  return 0;\n}\n")
    exe = tmp_path / "sizes"
    subprocess.run([gcc, "-I", os.path.join(REPO, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()
    sizes = [int(v) for v in out]
    J, R_ = _lib.LmLoopJobC, _lib.LmLoopResultC
    assert sizes == [ctypes.sizeof(_lib.LmParamsC), ctypes.sizeof(_lib.RobotInfoC), ctypes.sizeof(_lib.ConstraintsC),
                     ctypes.sizeof(R_), ctypes.sizeof(J), J.T.offset, J.tmax_sec.offset, J.convergence_threshold.offset,
                     J.result.offset, R_.schedule.offset]
