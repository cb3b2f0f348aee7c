"""GPU parity: every C-ABI entry point (through the Python host, which only forwards pointers) against the CPU
oracle on seeded inputs, and against the golden vectors produced by the real reference code.

Tolerances (BASELINE.json north_star): FK positions 1e-5 m, rotations 1e-5 rad, LM-refined joints 1e-4 rad;
dp_search back-pointers and collision booleans bit-exact."""
import numpy as np
import pytest
import torch

from oracle import robots as R, kinematics as K, geometry as G, lm as L, search as S
from tests.helpers import OBSTACLES, cuboid_tensors, random_configs, synthetic_problem

pytestmark = pytest.mark.gpu
ROBOTS = ["fetch", "fetch_arm", "panda"]
DEV = "cuda:0"


@pytest.fixture(scope="module")
def robots():
    from cppflow_b200.robot import get_robot

    return {r: get_robot(r) for r in ROBOTS}


def quat_align(q, ref):
    s = torch.sign((q * ref).sum(dim=1, keepdim=True))
    s[s == 0] = 1
    return q * s


@pytest.mark.parametrize("r", ROBOTS)
def test_fk_and_jacobian(robots, r):
    m = R.get_model(r)
    x = random_configs(m, 20000, seed=1)
    pose = robots[r].forward_kinematics(x.to(DEV)).cpu()
    ref = K.forward_kinematics(m, x.double())
    assert (pose[:, :3].double() - ref[:, :3]).abs().max() < 1e-5
    assert (quat_align(pose[:, 3:].double(), ref[:, 3:]) - ref[:, 3:]).abs().max() < 1e-5
    J = robots[r].jacobian(x.to(DEV)).cpu()
    assert (J.double() - K.jacobian(m, x.double())).abs().max() < 1e-5


@pytest.mark.parametrize("r", ROBOTS)
def test_pose_errors(robots, r):
    from cppflow_b200.optimization_utils import get_6d_pose_errors

    m, target, x0 = synthetic_problem(r, 4, 64, seed=2)
    e, cur = get_6d_pose_errors(robots[r], x0.to(DEV), target.repeat(4, 1).to(DEV))
    e_ref, cur_ref = L.get_6d_pose_errors(m, x0.double(), target.repeat(4, 1).double())
    assert e.shape == (256, 6, 1)
    assert (e.cpu().double() - e_ref).abs().max() < 1e-5
    assert (cur.cpu()[:, :3].double() - cur_ref[:, :3]).abs().max() < 1e-5


@pytest.mark.parametrize("r", ROBOTS)
def test_collision_distances_and_jacobians(robots, r):
    m = R.get_model(r)
    x = random_configs(m, 5000, seed=3)
    d = robots[r].self_collision_distances(x.to(DEV)).cpu()
    d_ref, J_ref = G.self_collision_distances(m, x.double(), with_jacobian=True)
    assert d.shape == d_ref.shape
    assert (d.double() - d_ref).abs().max() < 1e-5
    J = robots[r].self_collision_distances_jacobian(x.to(DEV)).cpu()
    assert (J.double() - J_ref).abs().max() < 2e-4
    cuboids, Tcuboids = cuboid_tensors(OBSTACLES[r])
    for c, Tc in zip(cuboids, Tcuboids):
        d = robots[r].env_collision_distances(x.to(DEV), c.to(DEV), Tc.to(DEV)).cpu()
        d_ref, J_ref = G.env_collision_distances(m, x.double(), c, Tc, with_jacobian=True)
        assert (d.double() - d_ref).abs().max() < 1e-5
        J = robots[r].env_collision_distances_jacobian(x.to(DEV), c, Tc).cpu()
        # the gradient is discontinuous where the closest point switches feature: compare where it is well defined
        ok = (d_ref.abs() > 1e-4)
        assert ((J.double() - J_ref).abs().amax(dim=2)[ok] < 2e-3).float().mean() > 0.999


def test_rotated_cuboid(robots):
    m = R.get_model("panda")
    x = random_configs(m, 2000, seed=5)
    c = torch.tensor([-0.1, -0.2, -0.15, 0.1, 0.2, 0.15])
    Tc = torch.eye(4)
    ang = 0.7
    Tc[:3, :3] = torch.tensor([[np.cos(ang), -np.sin(ang), 0], [np.sin(ang), np.cos(ang), 0], [0, 0, 1.0]])
    Tc[:3, 3] = torch.tensor([0.3, 0.1, 0.5])
    d = robots["panda"].env_collision_distances(x.to(DEV), c, Tc).cpu()
    d_ref = G.env_collision_distances(m, x.double(), c, Tc.double())
    assert (d.double() - d_ref).abs().max() < 1e-5


@pytest.mark.parametrize("r", ROBOTS)
def test_collision_flags_bit_exact(robots, r, golden):
    from cppflow_b200.collision_detection import qpaths_batched_self_collisions, qpaths_batched_env_collisions
    from cppflow_b200.data_types import Problem, Constraints

    m = R.get_model(r)
    cuboids, Tcuboids = cuboid_tensors(OBSTACLES[r])
    k, T = 40, 128
    q = random_configs(m, k * T, seed=4).reshape(k, T, m.ndof)
    target = K.forward_kinematics(m, q[0].double()).float()
    problem = Problem(Constraints(0.01, 0.1, 7.0, 2.0), target.to(DEV), None, robots[r], "t", "t", [], Tcuboids, cuboids, [])
    s = qpaths_batched_self_collisions(problem, q.to(DEV)).cpu()
    e = qpaths_batched_env_collisions(problem, q.to(DEV)).cpu()
    assert s.dtype == torch.bool and s.shape == (k, T)
    # oracle in fp32 (the reference's dtype); booleans must agree wherever |min distance| > 1e-6 m
    q2 = q.reshape(-1, m.ndof)
    ds = G.self_collision_distances(m, q2).min(dim=1).values.reshape(k, T)
    band = ds.abs() > 1e-6
    assert torch.equal(s[band], (ds < 0)[band]) and band.float().mean() > 0.9999
    de = torch.stack([G.env_collision_distances(m, q2, c, Tc).min(dim=1).values for c, Tc in zip(cuboids, Tcuboids)]).min(dim=0).values.reshape(k, T)
    band = de.abs() > 1e-6
    assert torch.equal(e[band], (de < 0)[band]) and band.float().mean() > 0.9999
    assert s.any() and e.any() and not s.all() and not e.all()
    # golden vectors from the real reference
    gq = torch.tensor(golden[f"{r}/cd/q"])
    gc, gT = [torch.tensor(c) for c in golden[f"{r}/lm/cuboids"]], [torch.tensor(t) for t in golden[f"{r}/lm/Tcuboids"]]
    problem = Problem(Constraints(0.01, 0.1, 7.0, 2.0), target.to(DEV), None, robots[r], "t", "t", [], gT, gc, [])
    assert np.array_equal(qpaths_batched_self_collisions(problem, gq.to(DEV)).cpu().numpy(), golden[f"{r}/cd/self"])
    assert np.array_equal(qpaths_batched_env_collisions(problem, gq.to(DEV)).cpu().numpy(), golden[f"{r}/cd/env"])


@pytest.mark.parametrize("r", ROBOTS)
def test_dp_search_bit_exact(robots, r, golden):
    from cppflow_b200 import ops
    from cppflow_b200.search import dp_search, joint_limit_almost_violations_3d

    m = R.get_model(r)
    rob = robots[r]
    # golden (real reference)
    q = torch.tensor(golden[f"{r}/dp/q"])
    sv, ev = torch.tensor(golden[f"{r}/dp/self_v"]), torch.tensor(golden[f"{r}/dp/env_v"])
    best, memo, costs, chosen = ops.dp_search(rob.robot_id, rob.ndof, q.to(DEV), sv.to(DEV), ev.to(DEV))
    assert np.array_equal(memo.cpu().numpy(), golden[f"{r}/dp/memo"])
    assert np.array_equal(costs.cpu().numpy(), golden[f"{r}/dp/costs"])
    assert np.array_equal(best.cpu().numpy(), golden[f"{r}/dp/best_path"])
    assert np.array_equal(joint_limit_almost_violations_3d(rob, q.to(DEV)).cpu().numpy(), golden[f"{r}/dp/jlim"])
    # seeded random case with 2 pi wraps, ties and k not a multiple of 32
    # k <= 256 / <= 320 / <= 512 take the three register layouts of the cluster sweep, k > 512 the single-CTA sweep
    for (k, T, seed) in [(37, 50, 0), (175, 60, 1), (1, 5, 2), (33, 1, 3), (300, 40, 4), (260, 7, 5), (400, 9, 6),
                         (513, 6, 7), (5, 2, 8), (2, 300, 9)]:
        g = torch.Generator().manual_seed(seed)
        base = random_configs(m, T, seed=seed + 10)
        q = base[None] + 0.4 * torch.randn((k, T, m.ndof), generator=g)
        q[:, :, -1] += (torch.rand((k, T), generator=g) < 0.1).float() * 2 * np.pi
        if k > 4:
            q[3] = q[1]  # exact ties
        sv = torch.rand((k, T), generator=g) < 0.2
        ev = torch.rand((k, T), generator=g) < 0.2
        ref_best, ref_memo, ref_costs, ref_chosen = S.dp_search(m, q, sv, ev)
        out = dp_search(rob, q.to(DEV), sv.to(DEV), ev.to(DEV), verbosity=0)
        best, memo, costs, chosen = ops.dp_search(rob.robot_id, rob.ndof, q.to(DEV), sv.to(DEV), ev.to(DEV))
        assert torch.equal(memo.cpu(), ref_memo), (k, T)
        assert torch.equal(costs.cpu(), ref_costs)
        assert torch.equal(chosen.cpu().long(), ref_chosen)
        assert torch.equal(best.cpu(), ref_best) and torch.equal(out.cpu(), ref_best)


@pytest.mark.parametrize("r", ROBOTS)
def test_pose_step(robots, r, golden):
    from cppflow_b200 import ops
    from cppflow_b200.lm_hyper_parameters import ALT_LOSS_V2_1_POSE

    m, target, x0 = synthetic_problem(r, 16, 100, seed=6)
    rob = robots[r]
    prm = ops.make_params(ALT_LOSS_V2_1_POSE)
    xn, J, e = ops.lm_pose_step(rob.robot_id, rob.ndof, prm, x0.to(DEV), target.to(DEV), clamp=False, return_residual=True)
    x64, J64, e64 = L.levenberg_marquardt_only_pose(m, x0.double(), target.repeat(16, 1).double(), L.ALT_LOSS_V2_1_POSE, True)
    assert (J.cpu().double() - J64).abs().max() < 5e-5
    assert (e.cpu().double() - e64).abs().max() < 5e-5
    err = (xn.cpu().double() - x64).abs().max(dim=1).values
    # parity set = well-conditioned waypoints (cond(J J^T + lambda I) < 1e6): 1e-4 rad.  Near a kinematic singularity the
    # LM step itself blows up (10 rad steps that clamp_to_joint_limits then cuts): there the step must agree to 2 %.
    cond = torch.linalg.cond(J64 @ J64.transpose(1, 2) + 1e-6 * torch.eye(6, dtype=torch.float64))
    step = (x64 - x0.double()).abs().max(dim=1).values
    well = cond < 1e6
    assert well.float().mean() > 0.95
    assert err[well].max() < 1e-4, err[well].max()
    assert (err[~well] <= 2e-2 * torch.clamp(step[~well], min=1.0)).all()
    # the reference's own fp32 step is much further from exact arithmetic than the kernel is
    x32 = L.levenberg_marquardt_only_pose(m, x0, target.repeat(16, 1), L.ALT_LOSS_V2_1_POSE)
    assert err[well].max() < (x32.double() - x64).abs().max(dim=1).values[well].max()
    # golden J / e from the real reference
    gx, gt = torch.tensor(golden[f"{r}/lm/x"]), torch.tensor(golden[f"{r}/lm/target"])
    xn, J, e = ops.lm_pose_step(rob.robot_id, rob.ndof, prm, gx.to(DEV), gt.to(DEV), clamp=False, return_residual=True)
    np.testing.assert_allclose(J.cpu().numpy(), golden[f"{r}/lm/pose_step_J"], atol=2e-5)
    np.testing.assert_allclose(e.cpu().numpy(), golden[f"{r}/lm/pose_step_e"], atol=2e-5)


@pytest.mark.parametrize("r", ROBOTS)
@pytest.mark.parametrize("mode", ["diff", "all"])
def test_full_step_vs_dense_oracle(robots, r, mode):
    """Block-tridiagonal CUDA step == the reference's dense get_r_and_J + _lm_full_step (fp64 oracle).

    'diff' = ALT_LOSS_V2_1_DIFF (what run_lm_alternating_loss runs), with colliding waypoints planted so the self- and
    env-collision rows are active: 1e-4 rad.
    'all'  = pose rows switched on as well.  J^T J (entries ~10) then shares the diagonal blocks with the 4e-5-sized
    differencing / lambda terms, so ANY fp32 evaluation of the reference's normal equations is noisy in the null space
    of J: the reference's own fp32 dense step is 4e-3..4e-2 rad from exact arithmetic, and so is any other fp32
    evaluation order (per path the ratio kernel error / reference-fp32 error scatters between 0.1 and 3.5, for the
    Cholesky-based and the sweep-based block inverse alike).  Criterion over 8 paths: the MEDIAN ratio stays below 2.5
    and no path is further than 5x the reference's own fp32 distance from the fp64 result."""
    from cppflow_b200 import ops
    from cppflow_b200.lm_hyper_parameters import ALT_LOSS_V2_1_DIFF, ALT_LOSS_V2_1_POSE, OptimizationParameters

    P, T = (3, 40) if mode == "diff" else (8, 40)
    m, target, x0 = synthetic_problem(r, P, T, seed=7)
    rob = robots[r]
    cuboids, Tcuboids = cuboid_tensors(OBSTACLES[r])
    pms = OptimizationParameters(**ALT_LOSS_V2_1_DIFF.__dict__)
    ratios = []
    if mode == "diff":
        # make collisions fire: replace a few waypoints of each path by colliding configurations
        cand = random_configs(m, 6000, seed=8)
        bad_self = cand[G.self_collision_distances(m, cand).min(dim=1).values < -0.01]
        bad_env = cand[G.env_collision_distances(m, cand, cuboids[0], Tcuboids[0]).min(dim=1).values < -0.01]
        x0 = x0.reshape(P, T, -1).clone()
        x0[:, 5] = bad_self[:P]
        x0[:, 17] = bad_env[:P]
        x0[:, 18] = bad_env[P : 2 * P]
        x0 = x0.reshape(P * T, -1)
        opms = L.LmParams()
    else:
        pms.use_pose, pms.alpha_position, pms.alpha_rotation = True, ALT_LOSS_V2_1_POSE.alpha_position, ALT_LOSS_V2_1_POSE.alpha_rotation
        opms = L.LmParams(use_pose=True)
    xv = x0 + 0.01 * torch.randn(x0.shape, generator=torch.Generator().manual_seed(9))
    ob = ops.Obstacles(cuboids, Tcuboids)
    out = ops.lm_full_step(rob.robot_id, rob.ndof, ops.make_params(pms), x0.to(DEV), xv.to(DEV), target.to(DEV), P, T, ob,
                           clamp=False).cpu()
    n_active = 0
    for p in range(P):
        sl = slice(p * T, (p + 1) * T)
        xp = x0[sl].double()
        opms.virtual_configs = xv[sl].double()
        Jd, rd = L.get_r_and_J(opms, m, xp, target.double(), Tcuboids, cuboids)
        n_active += (0 if rd["self_collisions"] is None else rd["self_collisions"].shape[0])
        n_active += (0 if rd["env_collisions"] is None else rd["env_collisions"].shape[0])
        ref = L.lm_full_step(L.stack_rows(Jd), L.stack_rows(rd), xp, opms.lm_lambda)
        err = (out[sl].double() - ref).abs().max()
        if mode == "diff":
            assert err < 1e-4, (p, float(err))
        else:
            opms.virtual_configs = xv[sl]
            J32, r32 = L.get_r_and_J(opms, m, x0[sl], target, Tcuboids, cuboids)
            ref32 = L.lm_full_step(L.stack_rows(J32), L.stack_rows(r32), x0[sl], opms.lm_lambda)
            err_ref32 = (ref32.double() - ref).abs().max()
            assert err < max(5.0 * err_ref32, 1e-4), (p, float(err), float(err_ref32))
            ratios.append(float(err / err_ref32))
    if mode == "diff":
        assert n_active > 0
    else:
        assert sorted(ratios)[len(ratios) // 2] < 2.5, ratios


@pytest.mark.parametrize("P,T", [(1, 9), (5, 10), (17, 33), (2, 301)])
def test_full_step_shapes(robots, P, T):
    """Twisted block solve: odd / even / minimal T (2 * n_virtual_configs < T), path counts that do not fill a warp."""
    from cppflow_b200 import ops
    from cppflow_b200.lm_hyper_parameters import ALT_LOSS_V2_1_DIFF

    r = "fetch"
    m, target, x0 = synthetic_problem(r, P, T, seed=11)
    rob = robots[r]
    cuboids, Tcuboids = cuboid_tensors(OBSTACLES[r])
    out = ops.lm_full_step(rob.robot_id, rob.ndof, ops.make_params(ALT_LOSS_V2_1_DIFF), x0.to(DEV), None, target.to(DEV),
                           P, T, ops.Obstacles(cuboids, Tcuboids), clamp=True).cpu()
    ref = L.run_fixed_schedule(m, x0.double(), target.double(), "d", Tcuboids, cuboids)
    assert (out.double() - ref).abs().max() < 1e-4


@pytest.mark.parametrize("T", [1, 2, 3, 4])
def test_full_step_minimal_paths(robots, T):
    """Shortest paths the twisted sweep can meet (no elimination step at all for T = 1, one side only for T = 2):
    differencing + collisions without virtual configs (2 * n_virtual_configs < T cannot hold), pose rows on so that
    the T = 1 system is not singular."""
    from dataclasses import replace

    from cppflow_b200 import ops
    from cppflow_b200.lm_hyper_parameters import OptimizationParameters, all_terms_parameters

    r, P = "panda", 19
    m, target, x0 = synthetic_problem(r, P, T, seed=21)
    rob = robots[r]
    cuboids, Tcuboids = cuboid_tensors(OBSTACLES[r])
    d = dict(all_terms_parameters().__dict__)
    d.update(use_virtual_configs=False)
    out = ops.lm_full_step(rob.robot_id, rob.ndof, ops.make_params(OptimizationParameters(**d)), x0.to(DEV), None,
                           target.to(DEV), P, T, ops.Obstacles(cuboids, Tcuboids), clamp=True).cpu()
    pms = replace(L.ALL_TERMS, use_virtual_configs=False)
    ref = L.run_fixed_schedule(m, x0.double(), target.double(), "a", Tcuboids, cuboids, all_pms=pms)
    ref32 = L.run_fixed_schedule(m, x0, target, "a", Tcuboids, cuboids, all_pms=pms)
    # same fp32 noise floor as in test_full_step_vs_dense_oracle['all']: J^T J + 1e-6 I has a null-space eigenvalue of
    # 1e-6 (plus beta for T > 1), so the yardstick is the reference's own fp32 distance from the fp64 result
    err = (out.double() - ref).abs().reshape(P, T, -1).amax(dim=(1, 2))
    err32 = (ref32.double() - ref).abs().reshape(P, T, -1).amax(dim=(1, 2))
    # per path both errors are noise (the ratio scatters over two decades), so the two DISTRIBUTIONS are compared
    assert err.median() < max(2.5 * err32.median(), 1e-4) and err.max() < max(3.0 * err32.max(), 1e-4), (err, err32)


def test_full_step_rejects_bad_arguments(robots):
    from cppflow_b200 import ops, _lib
    from cppflow_b200.lm_hyper_parameters import ALT_LOSS_V2_1_DIFF

    rob = robots["fetch"]
    m, target, x0 = synthetic_problem("fetch", 1, 8, seed=1)
    with pytest.raises(_lib.CppflowError):  # 2 * n_virtual_configs (8) must be < T (optimization_utils.py:457-459)
        ops.lm_full_step(rob.robot_id, rob.ndof, ops.make_params(ALT_LOSS_V2_1_DIFF), x0.to(DEV), None, target.to(DEV), 1, 8,
                         None, clamp=True)
    with pytest.raises(RuntimeError):  # CPU tensors are refused: there is no CPU fallback
        ops.forward_kinematics(rob.robot_id, rob.ndof, x0)


def test_full_step_full_size_path_independence(robots):
    """BASELINE.json's full size (8192 paths x 300 waypoints, every term on).  Paths are independent, so the result of a
    path must not depend on how many other paths are in the launch, which solve footprint is used (deep: one CTA per SM;
    CPPFLOW_LM_OVERLAP: compact, several CTAs per SM) or how the path set is chunked over streams: all bit-identical.
    This is the regression test of a shared-memory WAR hazard (TMA refill of a ring slot against the LDS reads of its
    previous contents) that only showed with two solve CTAs on one SM, i.e. never at the sizes the oracle can check."""
    from cppflow_b200 import ops
    from cppflow_b200.lm_hyper_parameters import all_terms_parameters
    from cppflow_b200.pipeline import ResidentPipeline
    from cppflow_b200.synthetic import synthetic_problem as gpu_problem, synthetic_seeds_host

    rob = robots["fetch"]
    P, T, D = 8192, 300, rob.ndof
    problem = gpu_problem(rob, T, device=DEV)
    _, xh = synthetic_seeds_host(rob, P, T)
    x0 = xh.to(DEV)
    prm = ops.make_params(all_terms_parameters())
    ob = problem.obstacle_tables

    def step(x, n_paths, **kw):
        return ops.lm_full_step(rob.robot_id, D, prm, x, None, problem.target_path, n_paths, T, ob, True, **kw)

    ref = step(x0, P)
    for _ in range(3):  # the hazard was timing dependent: ~25 % of the paths were hit in every launch
        assert torch.equal(step(x0, P), ref)
        assert torch.equal(step(x0, P, overlap=True), ref)
    for g in (0, 7, 255, 511):  # 16-path groups on their own
        sl = slice(g * 16 * T, (g + 1) * 16 * T)
        assert torch.equal(step(x0[sl].contiguous(), 16), ref[sl])
    sl = slice(5 * T, 6 * T)  # a single path
    assert torch.equal(step(x0[sl].contiguous(), 1), ref[sl])

    seq = x0
    for it in range(3):
        seq = step(seq, P)
        if it == 1:
            seq2 = seq
    for n_chunks in (1, 3, 4):
        pipe = ResidentPipeline(problem, P, all_terms_parameters(), n_chunks=n_chunks)
        assert torch.equal(pipe.iterate(x0, 3), seq), n_chunks
    # ragged sizes: path counts that fill neither the 256-path assembly CTAs nor the 16-path solve groups
    for n_paths, n_chunks in ((1000, 3), (37, 4)):
        xs = x0[: n_paths * T].contiguous()
        one = step(step(xs, n_paths), n_paths)
        assert torch.equal(one, seq2[: n_paths * T]), (n_paths, n_chunks)
        pipe = ResidentPipeline(problem, n_paths, all_terms_parameters(), n_chunks=n_chunks)
        assert torch.equal(pipe.iterate(xs, 2), one), (n_paths, n_chunks)
    # and the full-size iterations descend: the mean over paths of the maximum position error shrinks
    m0 = ops.path_metrics(rob.robot_id, D, x0, problem.target_path, P, T, ob)
    m1 = ops.path_metrics(rob.robot_id, D, seq, problem.target_path, P, T, ob)
    assert float(m1[:, 0].mean()) < float(m0[:, 0].mean()), (m0[:, 0].mean(), m1[:, 0].mean(), m0[:, 0].max(), m1[:, 0].max())


@pytest.mark.parametrize("r", ROBOTS)
@pytest.mark.parametrize("n_steps", [1, 4, 5])
def test_pose_steps_equal_repeated_pose_step(robots, r, n_steps):
    """cppflow_lm_pose_steps (n damped pose-only steps in one call, in place) == n calls of cppflow_lm_pose_step."""
    from dataclasses import replace

    from cppflow_b200 import ops
    from cppflow_b200.lm_hyper_parameters import ALT_LOSS_V2_1_POSE

    rob = robots[r]
    m, target, x0 = synthetic_problem(r, 7, 33, seed=5, noise=0.3)
    lambdas = [1e-1, 1e-2, 1e-3, 1e-5, 1e-6][:n_steps]
    x = x0.to(DEV)
    for lam in lambdas:
        x = ops.lm_pose_step(rob.robot_id, rob.ndof, ops.make_params(replace(ALT_LOSS_V2_1_POSE, lm_lambda=lam)), x,
                             target.to(DEV), True)
    y = x0.to(DEV).clone()
    ops.lm_pose_steps_(rob.robot_id, rob.ndof, ops.make_params(ALT_LOSS_V2_1_POSE), lambdas, y, target.to(DEV), True)
    assert torch.equal(x, y)


@pytest.mark.parametrize("r", ROBOTS)
@pytest.mark.parametrize("T", [1, 2, 3, 4, 10, 33, 300])
def test_resident_solve_equals_streaming_solve(robots, r, T):
    """Up to 8 paths the block solve runs out of shared memory (lm_block_solve_resident_kernel), beyond that it streams
    the blocks with TMA: same arithmetic in the same order, so a path's result is bit-identical whichever kernel it
    went through - for the shortest paths too (no elimination step at T = 1, one side only at T = 2)."""
    from dataclasses import replace

    from cppflow_b200 import ops
    from cppflow_b200.lm_hyper_parameters import all_terms_parameters

    rob = robots[r]
    P = 24
    m, target, x0 = synthetic_problem(r, P, T, seed=31)
    cuboids, Tcuboids = cuboid_tensors(OBSTACLES[r])
    pms = all_terms_parameters() if T > 8 else replace(all_terms_parameters(), use_virtual_configs=False)
    prm, ob, x0, target = ops.make_params(pms), ops.Obstacles(cuboids, Tcuboids), x0.to(DEV), target.to(DEV)

    def step(x, n):
        return ops.lm_full_step(rob.robot_id, rob.ndof, prm, x, None, target, n, T, ob, True)

    streaming = step(x0, P)  # 24 paths: the TMA kernel
    assert torch.isfinite(streaming).all()
    for p in (0, 5, 23):
        assert torch.equal(step(x0[p * T:(p + 1) * T].contiguous(), 1), streaming[p * T:(p + 1) * T]), p
    assert torch.equal(step(x0[8 * T:16 * T].contiguous(), 8), streaming[8 * T:16 * T])
    assert torch.equal(step(x0[:3 * T].contiguous(), 3), streaming[:3 * T])


@pytest.mark.parametrize("r", ROBOTS)
def test_empty_inputs(robots, r):
    """Zero configurations / zero paths: every entry point returns an empty result of the right shape, no launch."""
    from cppflow_b200 import ops
    from cppflow_b200.lm_hyper_parameters import ALT_LOSS_V2_1_DIFF, ALT_LOSS_V2_1_POSE

    rob = robots[r]
    D = rob.ndof
    x = torch.empty((0, D), device=DEV)
    m, target, _ = synthetic_problem(r, 1, 12, seed=2)
    target = target.to(DEV)
    cuboids, Tcuboids = cuboid_tensors(OBSTACLES[r])
    ob = ops.Obstacles(cuboids, Tcuboids)
    assert rob.forward_kinematics(x).shape == (0, 7)
    assert rob.jacobian(x).shape == (0, 6, D)
    assert rob.self_collision_distances(x).shape[0] == 0
    s, e = ops.collision_flags(rob.robot_id, D, x, ob)
    assert s.numel() == 0 and e.numel() == 0
    assert ops.lm_pose_step(rob.robot_id, D, ops.make_params(ALT_LOSS_V2_1_POSE), x, target, True).shape == (0, D)
    assert ops.lm_full_step(rob.robot_id, D, ops.make_params(ALT_LOSS_V2_1_DIFF), x, None, target, 0, 12, ob, True).shape == (0, D)
    assert ops.path_metrics(rob.robot_id, D, x, target, 0, 12, ob).shape == (0, 8)


@pytest.mark.parametrize("r", ROBOTS)
def test_joint_limit_corners(robots, r):
    """FK / Jacobian / capsule distances at the corners of the joint-limit box and at the all-zero configuration
    (data_type_utils.py:68-73 relies on FK at q = 0): the extremes of every trigonometric argument the kernels see."""
    m = R.get_model(r)
    lim = torch.tensor(m.actuated_joints_limits, dtype=torch.float64)
    D = lim.shape[0]
    corners = [torch.where(torch.tensor([(i >> d) & 1 for d in range(D)], dtype=torch.bool), lim[:, 1], lim[:, 0])
               for i in range(0, 2 ** D, max(1, 2 ** D // 64))]
    x = torch.stack(corners + [torch.zeros(D, dtype=torch.float64), lim.mean(dim=1)]).float()
    pose = robots[r].forward_kinematics(x.to(DEV)).cpu().double()
    ref = K.forward_kinematics(m, x.double())
    assert (pose[:, :3] - ref[:, :3]).abs().max() < 1e-5
    assert (quat_align(pose[:, 3:], ref[:, 3:]) - ref[:, 3:]).abs().max() < 1e-5
    J = robots[r].jacobian(x.to(DEV)).cpu().double()
    assert (J - K.jacobian(m, x.double())).abs().max() < 1e-5
    d = robots[r].self_collision_distances(x.to(DEV)).cpu().double()
    assert (d - G.self_collision_distances(m, x.double())).abs().max() < 1e-5


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_random_rotated_cuboids(robots, seed):
    """Capsule-cuboid distances and flags against the oracle for random cuboid sizes, positions and rotations about
    random axes (the reference asserts zero rotation, data_type_utils.py:108; the kernels take the full 4x4 pose)."""
    from cppflow_b200 import ops

    g = torch.Generator().manual_seed(100 + seed)
    r = ROBOTS[seed % len(ROBOTS)]
    m = R.get_model(r)
    x = random_configs(m, 1500, seed=20 + seed)
    cuboids, Tcuboids = [], []
    for _ in range(3):
        half = 0.05 + 0.25 * torch.rand(3, generator=g)
        axis = torch.randn(3, generator=g)
        axis = axis / axis.norm()
        ang = float(torch.rand(1, generator=g)) * 3.0
        Kx = torch.tensor([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
        Rm = torch.eye(3) + np.sin(ang) * Kx + (1 - np.cos(ang)) * (Kx @ Kx)
        Tc = torch.eye(4)
        Tc[:3, :3] = Rm
        Tc[:3, 3] = torch.tensor([0.2, 0.0, 0.5]) + 0.5 * (torch.rand(3, generator=g) - 0.5)
        cuboids.append(torch.cat([-half, half]))
        Tcuboids.append(Tc)
    dmin = None
    for c, Tc in zip(cuboids, Tcuboids):
        d = robots[r].env_collision_distances(x.to(DEV), c, Tc).cpu().double()
        d_ref = G.env_collision_distances(m, x.double(), c.double(), Tc.double())
        assert (d - d_ref).abs().max() < 1e-5
        dmin = d_ref.min(dim=1).values if dmin is None else torch.minimum(dmin, d_ref.min(dim=1).values)
    _, e = ops.collision_flags(robots[r].robot_id, robots[r].ndof, x.to(DEV), ops.Obstacles(cuboids, Tcuboids))
    clear = dmin.abs() > 1e-6
    assert torch.equal(e.cpu().bool()[clear], (dmin < 0)[clear])
