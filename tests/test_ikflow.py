"""IKFlow's GLOW network (oracle/ikflow.py) and its CUDA path (csrc/k_flow.cu, cppflow_b200/ikflow.py).

CPU: the oracle is invertible, the packed tables are laid out as include/cppflow_b200.h documents, the C ABI reports
its workspace and rejects every unsupported shape.  GPU: parity with the BF16-emulating fp64 oracle and the plain
fp32 oracle, round trip, row independence, condition broadcasting, clamp, the planner with the mock flow, and no host
synchronisation."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

from oracle import ikflow as OF

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda:0"


def _limits(name):
    from oracle import robots as R

    return R.get_model(name).actuated_joints_limits


def _params(width=9, nb=2, H=128, L=2):
    from cppflow_b200.ikflow import IkflowModelParameters

    return IkflowModelParameters(nb_nodes=nb, dim_latent_space=width, coeff_fn_config=L, coeff_fn_internal_size=H)


# ----------------------------------------------------------------------------------------------------------- CPU


@pytest.mark.parametrize("width", [7, 8, 9])
@pytest.mark.parametrize("n_layers", [1, 3])
def test_oracle_reverse_inverts_forward_fp64(width, n_layers):
    net = OF.random_glow(_limits("panda"), width, nb_nodes=4, internal=32, n_layers=n_layers, seed=width).double()
    g = torch.Generator().manual_seed(1)
    x = torch.rand((64, width), generator=g, dtype=torch.float64) * 2 - 1
    poses = torch.rand((64, 7), generator=g, dtype=torch.float64)
    z = net(x, poses)
    assert (z - x).abs().max() > 1e-2  # the network is not the identity
    back = net(z, poses, rev=True)
    assert (back - x).abs().max() < 1e-10


def test_oracle_split_and_permutation():
    assert OF.split_lengths(7) == (3, 4) and OF.split_lengths(8) == (4, 4) and OF.split_lengths(9) == (4, 5)
    np.testing.assert_array_equal(OF.permutation(3, 9), (np.random.seed(3), np.random.permutation(9))[1])


@pytest.mark.parametrize("L", [1, 3])
def test_packed_tables(L):
    from cppflow_b200.ikflow import IkflowSolver
    from cppflow_b200.robot import get_robot

    rob = get_robot("fetch")
    p = _params(width=9, nb=3, H=128, L=L)
    s = IkflowSolver(rob, p, seed=5, device="cpu")
    t = s._tables
    assert t["w_in"].shape == (3, 2, 128, 64) and t["w_in"].dtype == torch.bfloat16
    assert (t["w_hidden"] is None) if L == 1 else (t["w_hidden"].shape == (3, 2, L - 1, 128, 128)
                                                  and t["w_hidden"].dtype == torch.bfloat16)
    assert t["b_hidden"].shape == (3, 2, L, 128) and t["b_hidden"].dtype == torch.float32
    assert t["w_out"].shape == (3, 2, 16, 128) and t["w_out"].dtype == torch.float32
    assert t["b_out"].shape == (3, 2, 16) and t["scale"].shape == (9,)
    assert t["perm"].dtype == torch.int32 and t["perm_inv"].shape == (3, 9)
    ar = torch.arange(9, dtype=torch.int32)
    for b in range(3):
        assert torch.equal(t["perm"][b][t["perm_inv"][b].long()], ar) and torch.equal(t["perm_inv"][b][t["perm"][b].long()], ar)
    # zero padding: subnet1 reads len1 + 8 = 12 inputs and writes 2 * len2 = 10 outputs, subnet2 13 / 8
    assert t["w_in"][:, 0, :, 12:].abs().max() == 0 and t["w_in"][:, 0, :, :12].abs().max() > 0
    assert t["w_in"][:, 1, :, 13:].abs().max() == 0
    assert t["w_out"][:, 0, 10:].abs().max() == 0 and t["w_out"][:, 1, 8:].abs().max() == 0
    # the solver's weights are the oracle's module, name for name
    net = OF.Glow(rob.actuated_joints_limits, 9, 3, 128, L, 2.5)
    net.load_state_dict(s.state_dict)
    sd = s.state_dict
    assert torch.equal(t["w_out"][1, 1, :8], sd["module_list.4.subnet2.%d.weight" % (2 * L)])
    assert torch.equal(t["w_in"][2, 0, :, :12], sd["module_list.6.subnet1.0.weight"].to(torch.bfloat16))
    torch.testing.assert_close(t["scale"][:8].double(), torch.tensor([1 / max(abs(a), abs(b)) for a, b in
                                                                     rob.actuated_joints_limits], dtype=torch.float64))


def _desc(**kw):
    from cppflow_b200 import _lib

    d = dict(robot=0, width=9, ndof=8, dim_cond=8, nb_nodes=12, coeff_fn_config=3, coeff_fn_internal_size=1024,
             rnvp_clamp=2.5)
    d.update(kw)
    desc = _lib.FlowDescC(**d)
    for f in ("d_w_in", "d_w_hidden", "d_b_hidden", "d_w_out", "d_b_out", "d_scale", "d_perm", "d_perm_inv"):
        setattr(desc, f, 256)  # never dereferenced: every call below is rejected before a launch
    return desc


def test_workspace_bytes():
    from cppflow_b200 import _lib

    lib = _lib.load()
    a256 = lambda b: (b + 255) // 256 * 256  # noqa: E731
    n = 175 * 37
    assert lib.cppflow_flow_workspace_bytes(_desc(), n) == a256(n * 64) + a256(n * 128) + 2 * a256(n * 2048)
    assert lib.cppflow_flow_workspace_bytes(_desc(coeff_fn_config=1, coeff_fn_internal_size=256), 5) == (
        a256(5 * 64) + a256(5 * 128) + a256(5 * 512))


@pytest.mark.parametrize("change,message", [
    (dict(robot=7), "unknown robot id"),
    (dict(ndof=7), "is not the robot's"),
    (dict(width=17), "width 17 outside"),
    (dict(width=7), "width 7 outside"),
    (dict(dim_cond=6), "dim_cond 6"),
    (dict(coeff_fn_config=0), "coeff_fn_config 0"),
    (dict(coeff_fn_config=5), "coeff_fn_config 5"),
    (dict(coeff_fn_internal_size=192), "coeff_fn_internal_size 192"),
    (dict(coeff_fn_internal_size=2048), "coeff_fn_internal_size 2048"),
    (dict(nb_nodes=0), "nb_nodes 0"),
    (dict(rnvp_clamp=0.0), "rnvp_clamp"),
])
def test_unsupported_shapes_are_rejected(change, message):
    from cppflow_b200 import _lib

    lib = _lib.load()
    d = _desc(**change)
    assert lib.cppflow_flow_workspace_bytes(d, 10) == 0
    assert message.encode() in lib.cppflow_last_error()
    assert lib.cppflow_flow_run(d, 256, 256, 10, 10, 1, 256, 1 << 30, 256, None) == -1  # CPPFLOW_E_INVALID
    assert message.encode() in lib.cppflow_last_error()


def test_bad_calls_are_rejected():
    from cppflow_b200 import _lib

    lib = _lib.load()
    d = _desc()
    assert lib.cppflow_flow_run(d, 256, 256, 0, 1, 1, 256, 1 << 30, 256, None) == -1
    assert b"n = 0" in lib.cppflow_last_error()
    assert lib.cppflow_flow_run(d, 256, 256, 10, 0, 1, 256, 1 << 30, 256, None) == -1
    assert lib.cppflow_flow_run(d, 256, 256, 10, 1, 2, 256, 1 << 30, 256, None) == -1
    assert b"CPPFLOW_FLOW_CLAMP needs CPPFLOW_FLOW_REVERSE" in lib.cppflow_last_error()
    assert lib.cppflow_flow_run(d, 256, 256, 10, 1, 1, 256, 1000, 256, None) == -3  # CPPFLOW_E_WORKSPACE
    d.d_w_hidden = None
    assert lib.cppflow_flow_run(d, 256, 256, 10, 1, 1, 256, 1 << 30, 256, None) == -1


def test_flow_desc_layout_matches_the_c_header(tmp_path):
    from cppflow_b200 import _lib

    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    src = tmp_path / "flow.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "cppflow_b200.h"\nint main(void) {\n'
                   '  printf("%zu %zu %zu %zu\\n", sizeof(cppflow_flow_desc), offsetof(cppflow_flow_desc, rnvp_clamp),\n'
                   '         offsetof(cppflow_flow_desc, d_w_in), offsetof(cppflow_flow_desc, d_perm_inv));\n'
                   "  return 0;\n}\n")
    exe = tmp_path / "flow"
    subprocess.run([gcc, "-I", os.path.join(REPO, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    F = _lib.FlowDescC
    assert got == [ctypes.sizeof(F), F.rnvp_clamp.offset, F.d_w_in.offset, F.d_perm_inv.offset]


# ----------------------------------------------------------------------------------------------------------- GPU
# Tolerances (relative to max(1, |reference|)).  The CUDA path rounds to BF16 where the BF16 oracle does, so the two
# differ only where an FP32 sum (tensor-core accumulation, the last Linear, the coupling arithmetic) and its fp64
# counterpart land on different sides of a BF16 rounding boundary.  A K-term FP32 sum is within ~K * 2^-24 relative of
# the fp64 one, so about one activation in 10^3 (K = 1024) rounds the other way, by one BF16 ulp (2^-8 relative); the
# full network stores ~7 * 10^4 activations per row, i.e. tens of such flips per row, each moving the outputs by
# ~10^-4.  Against the plain fp32 oracle every stored activation carries its BF16 rounding error (2^-9 relative), the
# error of a BF16 network.  The bounds are 3-4x the worst row and 6x the mean measured on a B200 over the 6 parity
# cases (BF16 oracle: max 2.9e-3, mean 8.0e-5; fp32 oracle: max 5.0e-3, mean 4.9e-4).
PARITY_BF16 = dict(max=1e-2, mean=5e-4)
PARITY_FP32 = dict(max=2e-2, mean=3e-3)
# The reverse pass re-evaluates each subnet on an input rebuilt in FP32, not on the forward pass's bits: where the
# rebuilt value rounds to another BF16 number the subnet's s and t move by ~2^-8 relative.  Measured worst row of
# 6475: 1.4e-3 (joint units, after the 1 / M scale).
ROUND_TRIP = 5e-3


def _rel_err(got, ref):
    return ((got.double() - ref) / ref.abs().clamp(min=1.0)).abs()


def _inputs(solver, n, T, seed):
    from cppflow_b200.data_type_utils import problem_from_filename

    g = torch.Generator().manual_seed(seed)
    name = {"fetch": "fetch__circle", "fetch_arm": "fetch_arm__circle", "panda": "panda__1cube"}[solver.robot.name]
    path = problem_from_filename(None, name, device=DEV).target_path[:T].contiguous()
    z = (torch.rand((n, solver.network_width), generator=g) * 2 - 1).to(DEV)
    return z, path


def _oracle(solver):
    p = solver.params
    net = OF.Glow(solver.robot.actuated_joints_limits, p.dim_latent_space, p.nb_nodes, p.coeff_fn_internal_size,
                  p.coeff_fn_config, p.rnvp_clamp, p.softflow_enabled)
    net.load_state_dict(solver.state_dict)
    return net.to(DEV)


@pytest.mark.gpu
@pytest.mark.parametrize("robot", ["fetch", "fetch_arm", "panda"])
@pytest.mark.parametrize("size", ["small", "full"])
def test_parity_with_the_oracle(robot, size):
    from cppflow_b200.ikflow import IkflowSolver
    from cppflow_b200.robot import get_robot

    rob = get_robot(robot)
    p = _params(width=9, nb=2, H=128, L=2) if size == "small" else _params(width=9, nb=12, H=1024, L=3)
    solver = IkflowSolver(rob, p, seed=11, device=DEV)
    net = _oracle(solver).double()
    k, T = 175, 37  # n = 6475: not a multiple of any tile
    z, path = _inputs(solver, k * T, T, 0)
    cond = path.repeat(k, 1).double()
    with torch.no_grad():
        for reverse in (True, False):
            x_in = z if reverse else solver.run(z, path, True)
            got = solver.run(x_in, path, reverse)
            ref16 = net(x_in.double(), cond, rev=reverse, bf16=True)
            ref32 = net.float()(x_in, cond.float(), rev=reverse).double()
            net.double()
            e16, e32 = _rel_err(got, ref16), _rel_err(got, ref32)
            print(f"{robot} {size} reverse={reverse}: bf16 oracle max {e16.max():.2e} mean {e16.mean():.2e}; "
                  f"fp32 oracle max {e32.max():.2e} mean {e32.mean():.2e}")
            assert torch.isfinite(got).all()
            assert e16.max() < PARITY_BF16["max"] and e16.mean() < PARITY_BF16["mean"]
            assert e32.max() < PARITY_FP32["max"] and e32.mean() < PARITY_FP32["mean"]


@pytest.mark.gpu
def test_round_trip_row_independence_conditions_clamp():
    from cppflow_b200.ikflow import IkflowSolver
    from cppflow_b200.robot import get_robot

    rob = get_robot("fetch")
    solver = IkflowSolver(rob, _params(width=9, nb=12, H=1024, L=3), seed=3, device=DEV)
    k, T = 175, 37
    n = k * T
    z, path = _inputs(solver, n, T, 1)
    # round trip: the forward pass of configurations inside the limits, then the reverse pass
    lim = torch.tensor(rob.actuated_joints_limits, device=DEV)
    q = lim[:, 0] + (lim[:, 1] - lim[:, 0]) * torch.rand((n, rob.ndof), device=DEV)
    x = torch.cat([q, torch.zeros((n, 1), device=DEV)], dim=1)
    back = solver.run(solver.run(x, path, False), path, True)
    err = (back - x).abs().max().item()
    print(f"round trip max |dx| = {err:.2e}")
    assert err < ROUND_TRIP
    # rows are bit-identical whatever n and whichever rows share a tile; two runs are bit-identical
    full = solver.run(z, path, True)
    assert torch.equal(full, solver.run(z, path, True))
    cond = path.repeat(k, 1)
    for lo, hi in ((0, 1), (5, 6), (100, 229), (n - 300, n), (0, 1000)):
        part = solver.run(z[lo:hi].contiguous(), cond[lo:hi].contiguous(), True)
        assert torch.equal(part, full[lo:hi]), (lo, hi)
    # n_cond = T broadcasting == explicitly tiled conditions
    assert torch.equal(solver.run(z, cond, True), full)
    # the clamp keeps the joints inside the limits and changes nothing else
    clamped = solver.run(z, path, True, clamp=True)
    assert ((clamped[:, :8] >= lim[:, 0]) & (clamped[:, :8] <= lim[:, 1])).all()
    assert torch.equal(clamped[:, :8], torch.maximum(torch.minimum(full[:, :8], lim[:, 1]), lim[:, 0]))
    assert torch.equal(clamped[:, 8:], full[:, 8:])
    gen = solver.generate_ik_solutions(cond, z)
    assert gen.shape == (n, 8) and torch.equal(gen, clamped[:, :8])
    assert torch.equal(solver.solve_paths(path, z.reshape(k, T, 9)[:, 0]).reshape(n, 8),
                       solver.generate_ik_solutions(cond, z.reshape(k, T, 9)[:, :1].expand(k, T, 9).reshape(n, 9)))


@pytest.mark.gpu
def test_solve_paths_does_not_synchronise():
    from cppflow_b200.ikflow import IkflowSolver
    from cppflow_b200.robot import get_robot

    solver = IkflowSolver(get_robot("panda"), _params(width=9, nb=4, H=256, L=3), seed=0, device=DEV)
    z, path = _inputs(solver, 64, 50, 2)
    solver.solve_paths(path, z)  # warm-up: workspace allocation
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        q = solver.solve_paths(path, z)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert q.shape == (64, 50, 7) and torch.isfinite(q).all()


_SOLVERS = {}


def _mock(robot):
    from cppflow_b200.ikflow import IkflowSolver

    if robot.name not in _SOLVERS:
        _SOLVERS[robot.name] = IkflowSolver(robot, seed=0, device=DEV)
    return _SOLVERS[robot.name]


def _planner(robot, seed=0, k=32, **kw):
    from cppflow_b200.data_types import PlannerSettings
    from cppflow_b200.planners import CppFlowPlanner, IkflowCandidateGenerator

    settings = dict(k=k, tmax_sec=30.0, anytime_mode_enabled=False, verbosity=0)
    settings.update(kw)
    return CppFlowPlanner(PlannerSettings(**settings), robot, IkflowCandidateGenerator(_mock, seed=seed))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["fetch__circle", "panda__1cube"])
def test_planner_with_the_mock_flow(name):
    from cppflow_b200.data_type_utils import problem_from_filename
    from cppflow_b200.planners import IkflowCandidateGenerator

    problem = problem_from_filename(None, name, device=DEV)
    rob, T = problem.robot, problem.n_timesteps
    gen = IkflowCandidateGenerator(_mock(rob), seed=4)
    qs = gen(problem, 32)
    assert qs.shape == (32, T, rob.ndof) and gen.last_converged is None
    qs2 = IkflowCandidateGenerator(_mock, seed=4)(problem, 32)
    assert torch.equal(qs, qs2)
    a = _planner(rob, seed=1).generate_plan(problem)
    b = _planner(rob, seed=1).generate_plan(problem)
    assert a.plan.q_path.shape == (T, rob.ndof) and torch.isfinite(a.plan.q_path).all()
    assert torch.equal(a.plan.q_path, b.plan.q_path)
    assert a.timing.ikflow > 0


@pytest.mark.gpu
def test_planner_with_the_mock_flow_initial_configuration():
    """tests/planners_test.py:267-333 with the mock flow: the latent of the initial configuration is the centre of the
    sampled latents and path 0 keeps it, so candidate 0 starts at that configuration (within the round trip of the
    BF16 network); the search path starts exactly there (planners.py:261-265)."""
    from cppflow_b200.data_type_utils import problem_from_filename
    from cppflow_b200.data_types import Problem
    from cppflow_b200.planners import IkflowCandidateGenerator

    base = problem_from_filename(None, "panda__1cube", device=DEV)
    rob = base.robot
    lim = torch.tensor(rob.actuated_joints_limits, device=DEV)
    q0 = (lim.mean(dim=1) + 0.3 * (lim[:, 1] - lim[:, 0]) / 2)[None, :]
    problem = Problem(base.constraints, base.target_path, q0, rob, "test-problem", "test-problem", [], [], [], [])
    gen = IkflowCandidateGenerator(_mock(rob), seed=0)
    qs = gen(problem, 16)
    assert (qs[0, 0] - q0[0]).abs().max() < ROUND_TRIP
    planner = _planner(rob, seed=0, k=16)
    search_qpath, *_ = planner._run_pipeline(problem)
    assert torch.equal(search_qpath[0], q0[0])


@pytest.mark.gpu
def test_plan_many_with_the_mock_flow_equals_generate_plan():
    from cppflow_b200.data_type_utils import problem_from_filename
    from cppflow_b200.planners import plan_many

    problems = [problem_from_filename(None, name, device=DEV) for name in ("fetch__circle", "panda__1cube")]
    seq = [_planner(p.robot, seed=2).generate_plan(p) for p in problems]
    con = plan_many(lambda p: _planner(p.robot, seed=2), problems)
    for a, b in zip(seq, con):
        assert a.plan.is_valid == b.plan.is_valid
        assert torch.equal(a.plan.q_path, b.plan.q_path)
