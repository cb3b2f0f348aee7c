"""Exact IK from IKFlow's samples (csrc/k_ik.cu; cppflow_b200/ikflow.py: generate_exact_ik_solutions; the refinement
option of planners.IkflowCandidateGenerator) against the fp64 oracle of the stopping and select rules
(oracle/ik_exact.py).

CPU: the struct layout matches the C header, the C ABI rejects bad arguments, and the oracle's stopping rule is
levenberg_marquardt_only_pose stopped at the first step whose error check passes.  GPU: the fused refinement equals
cppflow_lm_pose_steps bit for bit (all steps, and per group of rows with the same step count), its converged rows pass
the fp64 check, generate_exact_ik_solutions equals the same rounds written with separate launches and torch
selection, runs are deterministic and replay from a CUDA graph without host synchronisation, and the planner's
refinement reports the oracle's convergence."""
import ctypes
import os
import shutil
import subprocess
from dataclasses import replace

import pytest
import torch

from oracle import ik_exact as OX
from oracle import lm as OL
from oracle import robots as OR

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda:0"
ROBOTS = ["fetch", "fetch_arm", "panda"]
# far-seed damping schedule of planners.LmIkCandidateGenerator (20 steps), the default of generate_exact_ik_solutions
LAMBDAS = (1e-1,) * 4 + (3e-2,) * 4 + (1e-2,) * 4 + (1e-3,) * 3 + (1e-4, 1e-5, 1e-6, 1e-6, 1e-6)
# the fp64 check of a row the FP32 kernel calls converged: FK in FP32 vs fp64 differs by ~1e-7 m / 1e-6 rad
ORACLE_BAND_POS, ORACLE_BAND_ROT = 1e-6, 1e-5
SELF_BAND = 5e-6  # m: FP32 capsule distances against fp64 (tests/test_collision_culls.py uses the same band)
# exact-IK success of the random-weight IKFlow-size flow on 3000 FK targets (seed 11), defaults of
# generate_exact_ik_solutions; measured on a B200: fetch 0.855, fetch_arm 0.985, panda 0.936.  A trained flow is
# expected to do better; these floors keep a margin below the random-weight rates.
SUCCESS_FLOOR = {"fetch": 0.80, "fetch_arm": 0.95, "panda": 0.90}


def _random_q(limits, n, gen, dtype=torch.float32):
    lim = torch.tensor(limits, dtype=torch.float64)
    return (lim[:, 0] + (lim[:, 1] - lim[:, 0]) * torch.rand((n, len(limits)), generator=gen, dtype=torch.float64)).to(dtype)


# ----------------------------------------------------------------------------------------------------------- CPU


def test_ik_refine_desc_layout_matches_the_c_header(tmp_path):
    from cppflow_b200 import _lib

    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    src = tmp_path / "ik.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "cppflow_b200.h"\nint main(void) {\n'
                   '  printf("%zu %zu %zu %zu %zu %zu %zu %d\\n", sizeof(cppflow_ik_refine_desc),\n'
                   '         offsetof(cppflow_ik_refine_desc, n_steps), offsetof(cppflow_ik_refine_desc, pos_tol),\n'
                   '         offsetof(cppflow_ik_refine_desc, rot_tol), offsetof(cppflow_ik_refine_desc, alpha_position),\n'
                   '         offsetof(cppflow_ik_refine_desc, alpha_rotation), offsetof(cppflow_ik_refine_desc, flags),\n'
                   '         CPPFLOW_IK_MAX_STEPS);\n'
                   "  return 0;\n}\n")
    exe = tmp_path / "ik"
    subprocess.run([gcc, "-I", os.path.join(REPO, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    D = _lib.IkRefineDescC
    assert got == [ctypes.sizeof(D), D.n_steps.offset, D.pos_tol.offset, D.rot_tol.offset, D.alpha_position.offset,
                   D.alpha_rotation.offset, D.flags.offset, 32]


def _desc(**kw):
    from cppflow_b200 import _lib

    d = _lib.IkRefineDescC()
    d.n_steps, d.pos_tol, d.rot_tol, d.alpha_position, d.alpha_rotation, d.flags = 20, 1e-3, 1e-2, 3.5, 0.35, 1
    for k, v in kw.items():
        setattr(d, k, v)
    return d


@pytest.mark.parametrize("change,message", [
    (dict(n_steps=33), "n_steps outside"),
    (dict(n_steps=-1), "n_steps outside"),
    (dict(pos_tol=-1e-3), "tolerances"),
    (dict(rot_tol=-1e-3), "tolerances"),
    (dict(pos_tol=float("nan")), "tolerances"),
    (dict(flags=8), "unknown flags"),
])
def test_ik_refine_rejects_bad_descs(change, message):
    from cppflow_b200 import _lib

    lib = _lib.load()
    # pointers are never dereferenced: every call is rejected before a launch
    assert lib.cppflow_ik_refine(2, _desc(**change), 256, 256, 10, 10, 256, 256, 256, 256, None) == -1
    assert message.encode() in lib.cppflow_last_error()


def test_ik_calls_reject_bad_arguments():
    from cppflow_b200 import _lib, ops
    from cppflow_b200.lm_hyper_parameters import ALT_LOSS_V2_1_POSE

    lib = _lib.load()
    d = _desc()
    assert lib.cppflow_ik_refine(7, d, 256, 256, 10, 10, 256, 256, 256, 256, None) == -1
    assert b"unknown robot id" in lib.cppflow_last_error()
    assert lib.cppflow_ik_refine(2, None, 256, 256, 10, 10, 256, 256, 256, 256, None) == -1
    for args in ((None, 256, 256, 256), (256, None, 256, 256), (256, 256, None, 256), (256, 256, 256, None)):
        q, t, qo, st = args
        assert lib.cppflow_ik_refine(2, d, q, t, 10, 10, qo, st, None, None, None) == -1
        assert b"null pointer" in lib.cppflow_last_error()
    assert lib.cppflow_ik_refine(2, d, 256, 256, 10, 0, 256, 256, None, None, None) == -1
    assert lib.cppflow_ik_refine(2, d, 256, 256, 0, 10, None, None, None, None, None) == 0  # n = 0: nothing to do

    assert lib.cppflow_ik_round_inputs(256, 10, 0, 256, 0, 0, 9, 1.0, 256, 256, None) == -1
    assert b"rep must be > 0" in lib.cppflow_last_error()
    assert lib.cppflow_ik_round_inputs(256, 10, 1, 256, 0, 0, 17, 1.0, 256, 256, None) == -1
    assert lib.cppflow_ik_round_inputs(256, 10, 1, 256, 0, 0, 9, -1.0, 256, 256, None) == -1
    assert lib.cppflow_ik_round_inputs(None, 10, 1, 256, 0, 0, 9, 1.0, 256, 256, None) == -1
    assert b"null pointer" in lib.cppflow_last_error()

    sel = lambda robot=2, n=10, rep=1, q=256, cnt=256: lib.cppflow_ik_select(  # noqa: E731
        robot, q, 256, 256, n, rep, 256, 256, 256, cnt, 256, 1 << 30, None)
    assert sel(rep=0) == -1 and b"rep must be > 0" in lib.cppflow_last_error()
    assert sel(robot=3) == -1 and b"unknown robot id" in lib.cppflow_last_error()
    assert sel(n=-1) == -1 and sel(n=1 << 31) == -1
    assert sel(q=None) == -1 and b"null pointer" in lib.cppflow_last_error()
    assert sel(cnt=None) == -1
    assert lib.cppflow_ik_select_workspace_bytes(-1) == 0 and lib.cppflow_ik_select_workspace_bytes(1 << 31) == 0

    with pytest.raises(ValueError, match="at most 32"):
        ops.ik_refine_desc([1e-3] * 33, 1e-3, 1e-2, ops.make_params(ALT_LOSS_V2_1_POSE))


def _fk64(model, q):
    from oracle import kinematics as K

    return K.forward_kinematics(model, q.double())


@pytest.mark.parametrize("robot", ROBOTS)
def test_oracle_stopping_rule_is_lm_stopped_at_the_first_passing_check(robot):
    model = OR.get_model(robot)
    g = torch.Generator().manual_seed(7)
    n = 48
    q_t = _random_q(model.actuated_joints_limits, n, g, torch.float64)
    targets = _fk64(model, q_t)
    x0 = _random_q(model.actuated_joints_limits, n, g, torch.float64)
    x0[: n // 2] = q_t[: n // 2] + 0.05 * (torch.rand((n // 2, model.ndof), generator=g, dtype=torch.float64) - 0.5)
    OL.clamp_to_joint_limits(model, x0)
    pms = OL.ALT_LOSS_V2_1_POSE
    pos_tol, rot_tol, lambdas = 1e-3, 1e-2, LAMBDAS[:12]
    # every step by hand: levenberg_marquardt_only_pose + clamp_to_joint_limits
    hist = [x0.clone()]
    for lam in lambdas:
        nxt = OL.levenberg_marquardt_only_pose(model, hist[-1], targets, replace(pms, lm_lambda=lam))
        hist.append(OL.clamp_to_joint_limits(model, nxt))
    ok = torch.stack([OX.converged(model, h, targets, pos_tol, rot_tol) for h in hist])  # [steps + 1, n]

    # (torch's batched fp64 solve may round a subset of the rows differently in the last bits)
    x, status, steps = OX.refine(model, x0, targets, lambdas, pms, pos_tol, rot_tol, early_exit=False)
    torch.testing.assert_close(x, hist[-1], rtol=0, atol=1e-12)
    assert torch.equal(status, ok[-1]) and (steps == len(lambdas)).all()

    x, status, steps = OX.refine(model, x0, targets, lambdas, pms, pos_tol, rot_tol)
    first = torch.where(ok.any(dim=0), ok.to(torch.int64).argmax(dim=0), torch.full((n,), len(lambdas)))
    assert torch.equal(steps, first)
    torch.testing.assert_close(x, torch.stack(hist)[steps, torch.arange(n)], rtol=0, atol=1e-12)
    assert torch.equal(status, ok[steps, torch.arange(n)])
    assert (steps[~status] == len(lambdas)).all()
    assert 0 < int(status.sum()) < n and int((steps == 0).sum()) < n  # both outcomes occur; not every row starts done


def test_oracle_select_rule():
    status = torch.tensor([[0, 1, 1], [0, 0, 0], [1, 0, 1], [0, 0, 1]], dtype=torch.bool)
    unsolved = torch.tensor([2, 5, 6, 9], dtype=torch.int32)
    q = torch.arange(12, dtype=torch.float64)[:, None].repeat(1, 2)
    sol = torch.full((10, 2), -1.0, dtype=torch.float64)
    valid = torch.zeros(10, dtype=torch.bool)
    left = OX.select(status, unsolved, sol, valid, q)
    assert left.tolist() == [5]
    assert sol[[2, 5, 6, 9], 0].tolist() == [1.0, 3.0, 6.0, 11.0]
    assert valid.nonzero()[:, 0].tolist() == [2, 6, 9]


# ----------------------------------------------------------------------------------------------------------- GPU


def _pose_params():
    from cppflow_b200 import ops
    from cppflow_b200.lm_hyper_parameters import ALT_LOSS_V2_1_POSE

    return ops.make_params(ALT_LOSS_V2_1_POSE)


def _fp32_check(rob, q, targets, pos_tol, rot_tol):
    """The kernel's error check on the host side, in FP32: sqrt((e0*e0 + e1*e1) + e2*e2), one rounding per op."""
    from cppflow_b200 import ops

    e, _ = ops.pose_errors(rob.robot_id, rob.ndof, q, targets)
    rot = ((e[:, 0] * e[:, 0] + e[:, 1] * e[:, 1]) + e[:, 2] * e[:, 2]).sqrt()
    pos = ((e[:, 3] * e[:, 3] + e[:, 4] * e[:, 4]) + e[:, 5] * e[:, 5]).sqrt()
    return (pos < pos_tol) & (rot < rot_tol), pos, rot


def _rows(rob, n, n_targets, seed):
    """q0 [n, ndof] (half uniform in the limits, half within 0.1 rad of the target's configuration) and the targets
    [n_targets, 7] = FK of uniform in-limit configurations; row i tracks target i % n_targets."""
    from cppflow_b200 import ops

    g = torch.Generator().manual_seed(seed)
    q_t = _random_q(rob.actuated_joints_limits, n_targets, g).to(DEV)
    targets = ops.forward_kinematics(rob.robot_id, rob.ndof, q_t)
    q0 = _random_q(rob.actuated_joints_limits, n, g).to(DEV)
    near = torch.arange(n, device=DEV) % 2 == 0
    jitter = (0.2 * (torch.rand((n, rob.ndof), generator=g) - 0.5)).to(DEV)
    q0 = torch.where(near[:, None], q_t[torch.arange(n, device=DEV) % n_targets] + jitter, q0).contiguous()
    ops.clamp_to_joint_limits_(rob.robot_id, rob.ndof, q0)
    return q0, targets


@pytest.mark.gpu
@pytest.mark.parametrize("robot", ROBOTS)
def test_refine_without_early_exit_equals_lm_pose_steps(robot):
    from cppflow_b200 import ops
    from cppflow_b200.robot import get_robot

    rob = get_robot(robot)
    prm = _pose_params()
    for seed in (1, 2):
        q0, targets = _rows(rob, 100_000, 100_000, seed)
        desc = ops.ik_refine_desc(LAMBDAS, 1e-3, 1e-2, prm, early_exit=False)
        q, status, steps, err = ops.ik_refine(rob.robot_id, rob.ndof, desc, q0, targets, with_errors=True)
        ref = ops.lm_pose_steps_(rob.robot_id, rob.ndof, prm, LAMBDAS, q0.clone(), targets, True)
        assert torch.equal(q, ref)
        assert (steps == len(LAMBDAS)).all()
        ok, pos, rot = _fp32_check(rob, q, targets, 1e-3, 1e-2)
        assert torch.equal(status.bool(), ok)
        # the position error has the same bits; the rotation error goes through rotmat_to_quat and the rpy formula,
        # which the compiler may contract differently in the two kernels: last-bit differences
        assert torch.equal(err[:, 0], pos)
        torch.testing.assert_close(err[:, 1], rot, rtol=1e-5, atol=1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("robot", ROBOTS)
def test_refine_with_early_exit_equals_lm_pose_steps_per_step_count(robot):
    from cppflow_b200 import ops
    from cppflow_b200.robot import get_robot

    rob = get_robot(robot)
    prm = _pose_params()
    n, T = 100_000, 1000  # n_targets < n: row i tracks target i % T
    q0, targets = _rows(rob, n, T, 3)
    pos_tol, rot_tol = 1e-3, 1e-2
    desc = ops.ik_refine_desc(LAMBDAS, pos_tol, rot_tol, prm)
    q, status, steps = ops.ik_refine(rob.robot_id, rob.ndof, desc, q0, targets)
    # in place gives the same bits
    q_in = q0.clone()
    ops.ik_refine(rob.robot_id, rob.ndof, desc, q_in, targets, out=q_in)
    assert torch.equal(q_in, q)
    tgt = targets[torch.arange(n, device=DEV) % T].contiguous()
    counts = torch.bincount(steps.long(), minlength=len(LAMBDAS) + 1).tolist()
    print(f"{robot}: rows per step count {counts}, converged {status.float().mean().item():.3f}")
    assert counts[-1] > 0 and sum(c > 0 for c in counts[:-1]) > 5  # rows stop at many step counts, some never
    for s in range(len(LAMBDAS) + 1):
        rows = (steps == s).nonzero()[:, 0]
        if rows.numel() == 0:
            continue
        ref = q0[rows].contiguous()
        if s:
            ops.lm_pose_steps_(rob.robot_id, rob.ndof, prm, LAMBDAS[:s], ref, tgt[rows].contiguous(), True)
        assert torch.equal(q[rows], ref), s
    ok, _, _ = _fp32_check(rob, q, tgt, pos_tol, rot_tol)
    assert torch.equal(status.bool(), ok)
    assert (steps[status == 0] == len(LAMBDAS)).all()


def _oracle_check(robot, q, targets, pos_tol, rot_tol):
    model = OR.get_model(robot)
    p, r = OX.pose_error_norms(model, q.cpu().double(), targets.cpu().double())
    return p, r, model


@pytest.mark.gpu
@pytest.mark.parametrize("robot", ROBOTS)
def test_converged_rows_pass_the_fp64_check(robot):
    from oracle import geometry as G
    from cppflow_b200 import ops
    from cppflow_b200.robot import get_robot

    rob = get_robot(robot)
    prm = _pose_params()
    n = 20_000
    q0, targets = _rows(rob, n, n, 4)
    for pos_tol, rot_tol in ((1e-3, 1e-2), (1e-4, 1.745e-3)):
        desc = ops.ik_refine_desc(LAMBDAS, pos_tol, rot_tol, prm)
        q, status, _ = ops.ik_refine(rob.robot_id, rob.ndof, desc, q0, targets)
        p, r, model = _oracle_check(robot, q, targets, pos_tol, rot_tol)
        conv = status.bool().cpu()
        assert conv.sum() > n // 4
        assert (p[conv] < pos_tol + ORACLE_BAND_POS).all() and (r[conv] < rot_tol + ORACLE_BAND_ROT).all()
    # with the self-collision check: converged rows are collision-free in fp64, and a row whose pose passes but that
    # did not converge collides, each outside the band
    desc = ops.ik_refine_desc(LAMBDAS, 1e-3, 1e-2, prm, check_self_collision=True)
    q, status, _ = ops.ik_refine(rob.robot_id, rob.ndof, desc, q0, targets)
    pose_ok, _, _ = _fp32_check(rob, q, targets, 1e-3, 1e-2)
    d = G.self_collision_distances(OR.get_model(robot), q.cpu().double()).min(dim=1).values
    conv, pose_ok = status.bool().cpu(), pose_ok.cpu()
    rejected = pose_ok & ~conv
    print(f"{robot}: self-collision check: {int(conv.sum())} converged, {int(rejected.sum())} rejected at the pose")
    assert conv.sum() > n // 4
    assert (d[conv] > -SELF_BAND).all()
    assert (d[rejected] < SELF_BAND).all()
    p, r, _ = _oracle_check(robot, q, targets, 1e-3, 1e-2)
    assert (p[conv] < 1e-3 + ORACLE_BAND_POS).all() and (r[conv] < 1e-2 + ORACLE_BAND_ROT).all()


_SOLVERS = {}


def _mock(robot):
    """A random-weight flow of IKFlow's size (12 blocks, hidden 1024, 3 layers per subnet)."""
    from cppflow_b200.ikflow import IkflowSolver

    if robot.name not in _SOLVERS:
        _SOLVERS[robot.name] = IkflowSolver(robot, seed=0, device=DEV)
    return _SOLVERS[robot.name]


def _reference_rounds(solver, poses, pos_tol, rot_tol, repeat_counts, seed):
    """generate_exact_ik_solutions written with separate launches: the same latents, flow_run, one lm_pose_step launch
    per LM step with the per-row stop in torch, and torch selection."""
    from cppflow_b200 import _lib, ops

    rob, D = solver.robot, solver.robot.ndof
    prm = _pose_params()
    m = poses.shape[0]
    sol = torch.zeros((m, D), device=DEV)
    valid = torch.zeros((m,), device=DEV, dtype=torch.bool)
    unsolved = torch.arange(m, device=DEV, dtype=torch.int32)
    lists = []
    for r, rep in enumerate(repeat_counts):
        if unsolved.numel() == 0:
            break
        z, cond = ops.ik_round_inputs(unsolved, rep, poses, seed, r, solver.network_width)
        x = solver.run(z, cond, True, True)[:, :D].contiguous()
        active = torch.ones(x.shape[0], device=DEV, dtype=torch.bool)
        for lam in LAMBDAS:
            active &= ~_fp32_check(rob, x, cond, pos_tol, rot_tol)[0]
            p = _lib.LmParamsC.from_buffer_copy(prm)
            p.lm_lambda = lam
            x = torch.where(active[:, None], ops.lm_pose_step(rob.robot_id, D, p, x, cond, True), x)
        status = _fp32_check(rob, x, cond, pos_tol, rot_tol)[0]
        unsolved = OX.select(status.reshape(-1, rep), unsolved, sol, valid, x)
        lists.append(unsolved.clone())
    return sol, valid, lists


@pytest.mark.gpu
@pytest.mark.parametrize("robot", ROBOTS)
def test_exact_ik_equals_the_reference_rounds(robot):
    from cppflow_b200 import ops
    from cppflow_b200.robot import get_robot

    rob = get_robot(robot)
    solver = _mock(rob)
    m = 3000
    g = torch.Generator().manual_seed(11)
    poses = ops.forward_kinematics(rob.robot_id, rob.ndof, _random_q(rob.actuated_joints_limits, m, g).to(DEV))
    q, valid = solver.generate_exact_ik_solutions(poses, seed=5)
    ref_q, ref_valid, lists = _reference_rounds(solver, poses, 1e-3, 1e-2, (1, 3, 10), 5)
    assert torch.equal(valid, ref_valid)
    assert torch.equal(q, ref_q)
    rate = valid.float().mean().item()
    print(f"{robot}: exact-IK success {rate:.4f} after rounds leaving {[int(u.numel()) for u in lists]} unsolved")
    p, r, _ = _oracle_check(robot, q, poses, 1e-3, 1e-2)
    v = valid.cpu()
    assert (p[v] < 1e-3 + ORACLE_BAND_POS).all() and (r[v] < 1e-2 + ORACLE_BAND_ROT).all()
    assert rate >= SUCCESS_FLOOR[robot]
    # the latents of a row depend on (seed, round, target, sample) only, not on the list they were drawn for
    full, _ = ops.ik_round_inputs(torch.arange(m, device=DEV, dtype=torch.int32), 3, poses, 5, 1, 9)
    sub = torch.tensor([7, 100, 2999], device=DEV, dtype=torch.int32)
    part, cond = ops.ik_round_inputs(sub, 3, poses, 5, 1, 9)
    rows = (sub.long()[:, None] * 3 + torch.arange(3, device=DEV)).reshape(-1)
    assert torch.equal(part, full[rows]) and torch.equal(cond, poses[sub.long()].repeat_interleave(3, 0))
    assert abs(full.mean().item()) < 0.02 and abs(full.std().item() - 1.0) < 0.02


@pytest.mark.gpu
def test_exact_ik_is_deterministic_graph_capturable_and_does_not_synchronise():
    from cppflow_b200 import ops
    from cppflow_b200.ikflow import IkflowModelParameters, IkflowSolver
    from cppflow_b200.robot import get_robot

    rob = get_robot("panda")
    solver = IkflowSolver(rob, IkflowModelParameters(nb_nodes=4, coeff_fn_internal_size=256), seed=1, device=DEV)
    g = torch.Generator().manual_seed(12)
    poses = ops.forward_kinematics(rob.robot_id, rob.ndof, _random_q(rob.actuated_joints_limits, 1024, g).to(DEV))
    a = solver.generate_exact_ik_solutions(poses, seed=9, check_self_collision=True)
    b = solver.generate_exact_ik_solutions(poses, seed=9, check_self_collision=True)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])

    D, m, rep = rob.ndof, poses.shape[0], 3
    desc = ops.ik_refine_desc(LAMBDAS, 1e-3, 1e-2, _pose_params(), check_self_collision=True)
    unsolved = torch.arange(m, device=DEV, dtype=torch.int32)

    def one_round(sol, valid, out, count):
        z, cond = ops.ik_round_inputs(unsolved, rep, poses, 4, 1, solver.network_width)
        x = solver.run(z, cond, True, True)[:, :D].contiguous()
        q, status, _ = ops.ik_refine(rob.robot_id, D, desc, x, cond, out=x)
        ops.ik_select(rob.robot_id, D, q, status, unsolved, rep, sol, valid, out, count)

    def buffers():
        return (torch.zeros((m, D), device=DEV), torch.zeros((m,), device=DEV, dtype=torch.uint8),
                torch.zeros((m,), device=DEV, dtype=torch.int32), torch.zeros((1,), device=DEV, dtype=torch.int32))

    eager = buffers()
    one_round(*eager)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        again = buffers()
        one_round(*again)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    for x, y in zip(eager, again):
        assert torch.equal(x, y)

    captured = buffers()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):  # warm-up on the capture stream: its scratch buffers exist before the capture
        one_round(*captured)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    for t in captured:
        t.zero_()
    with torch.cuda.graph(graph, stream=s):
        one_round(*captured)
    for _ in range(2):
        for t in captured:
            t.zero_()
        graph.replay()
        torch.cuda.synchronize()
        n_left = int(eager[3].item())
        assert torch.equal(captured[0], eager[0]) and torch.equal(captured[1], eager[1])
        assert int(captured[3].item()) == n_left and torch.equal(captured[2][:n_left], eager[2][:n_left])
    assert 0 < n_left < m


def _refine_settings():
    from cppflow_b200.planners import IkRefineSettings

    return IkRefineSettings(LAMBDAS)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["fetch__circle", "fetch_arm__hello", "panda__1cube"])
def test_planner_refinement_reports_the_oracle_convergence(name):
    from cppflow_b200 import ops
    from cppflow_b200.data_type_utils import problem_from_filename
    from cppflow_b200.planners import IkflowCandidateGenerator

    problem = problem_from_filename(None, name, device=DEV)
    rob, T, k = problem.robot, problem.n_timesteps, 32
    plain = IkflowCandidateGenerator(_mock(rob), seed=4)(problem, k)
    none = IkflowCandidateGenerator(_mock(rob), seed=4, refine=None)
    assert torch.equal(none(problem, k), plain) and none.last_converged is None
    gen = IkflowCandidateGenerator(_mock(rob), seed=4, refine=_refine_settings())
    qs = gen(problem, k)
    conv = gen.last_converged
    assert qs.shape == (k, T, rob.ndof) and conv.shape == (k, T) and conv.dtype == torch.bool
    # the refinement is one ik_refine launch over the unrefined candidates
    desc = ops.ik_refine_desc(LAMBDAS, 1e-4, 1.745e-3, _pose_params())
    q_ref, st_ref, _ = ops.ik_refine(rob.robot_id, rob.ndof, desc, plain.reshape(k * T, -1).contiguous(),
                                     problem.target_path)
    assert torch.equal(qs.reshape(k * T, -1), q_ref) and torch.equal(conv.reshape(-1), st_ref.bool())
    # last_converged against the fp64 check, outside the rounding band of the thresholds
    p, r, _ = _oracle_check(rob.name, qs.reshape(k * T, -1), problem.target_path.repeat(k, 1), 1e-4, 1.745e-3)
    ora = (p < 1e-4) & (r < 1.745e-3)
    clear = ((p - 1e-4).abs() > ORACLE_BAND_POS) & ((r - 1.745e-3).abs() > ORACLE_BAND_ROT)
    c = conv.reshape(-1).cpu()
    print(f"{name}: {c.float().mean().item():.3f} of the waypoints converged, {int((~clear).sum())} inside the band")
    assert torch.equal(c[clear], ora[clear])
    assert (p[c] < 1e-4 + ORACLE_BAND_POS).all() and (r[c] < 1.745e-3 + ORACLE_BAND_ROT).all()


@pytest.mark.gpu
def test_planner_refinement_generate_plan_equals_plan_many():
    from cppflow_b200.data_type_utils import problem_from_filename
    from cppflow_b200.data_types import PlannerSettings
    from cppflow_b200.planners import CppFlowPlanner, IkflowCandidateGenerator, plan_many

    def planner(p):
        settings = PlannerSettings(k=32, tmax_sec=30.0, anytime_mode_enabled=False, verbosity=0)
        return CppFlowPlanner(settings, p.robot, IkflowCandidateGenerator(_mock, seed=2, refine=_refine_settings()))

    problems = [problem_from_filename(None, "fetch_arm__hello", device=DEV)]
    seq = [planner(p).generate_plan(p) for p in problems]
    con = plan_many(planner, problems)
    for a, b in zip(seq, con):
        assert a.plan.is_valid == b.plan.is_valid
        assert torch.equal(a.plan.q_path, b.plan.q_path)
