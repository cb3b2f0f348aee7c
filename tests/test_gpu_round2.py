"""GPU parity, second set: the EXACT workload bench.py times, the reference's own alternating loop, every column of
the path metrics, the dense get_r_and_J drop-in and the standalone clamp.

  * bench workload (8192 x 300 Fetch, bench.py's generator and seeds): paths drawn from the batch are refined INSIDE
    the full-size launches and compared with the fp64 oracle - schedule `pppdd` (the steps the reference really runs,
    SURVEY config 5) at the north star's 1e-4 rad; one all-terms step `a` (the step bench.py's headline times) by the
    yardstick of test_full_step_vs_dense_oracle['all'] (the reference's own fp32 distance from the fp64 result);
  * cppflow_lm_alternating_loss against tests/golden/reference_loop_golden.npz, which holds the outputs of the
    reference's real run_lm_optimization (optimization.py:147-426) in float32 and float64;
  * cppflow_path_metrics, all seven columns, against oracle.lm.path_metrics on valid, invalid and colliding paths, for
    one path (thread-block-cluster variant) and for hundreds (one CTA per path);
  * LmResidualFns.get_r_and_J (dense) against the golden all_J / all_r of the reference's get_r_and_J;
  * cppflow_clamp_to_joint_limits against the golden clamp_in / clamp_out.
"""
import numpy as np
import pytest
import torch

from oracle import robots as R, geometry as G, lm as L
from tests.helpers import OBSTACLES, cuboid_tensors, random_configs, synthetic_problem

pytestmark = pytest.mark.gpu
ROBOTS = ["fetch", "fetch_arm", "panda"]
DEV = "cuda:0"
CONSTRAINTS = (0.01, 0.1, 7.0, 2.0)  # scripts/evaluate.py:51-56


@pytest.fixture(scope="module")
def robots():
    from cppflow_b200.robot import get_robot

    return {r: get_robot(r) for r in ROBOTS}


# ------------------------------------------------------------------------------------------------------------------
# 1a. the timed workload


@pytest.fixture(scope="module")
def bench_workload(robots):
    """bench.py's config-5 inputs, built by the same calls with the same seeds (rank 0's shard)."""
    from cppflow_b200.synthetic import synthetic_problem as gpu_problem, synthetic_seeds_host

    rob = robots["fetch"]
    P, T = 8192, 300
    problem = gpu_problem(rob, T, seed=0, device=DEV)
    _, x_host = synthetic_seeds_host(rob, P, T, seed=0, shard=0)
    return rob, problem, x_host, P, T


# spread over the batch: first / last lanes of 16-path solve groups, of 256-path assembly CTAs and of the 2048-path chunks
DRAWN = [0, 1, 15, 16, 255, 256, 1000, 2047, 2048, 4095, 4096, 5000, 6143, 6144, 8190, 8191]


def test_bench_workload_pppdd_vs_fp64_oracle(bench_workload):
    """Schedule pppdd over all 8192 x 300 waypoints in full-size launches; 16 drawn paths against the fp64 oracle
    (dense get_r_and_J + _lm_full_step per path for the differencing steps): 1e-4 rad."""
    from cppflow_b200.optimization import run_lm_fixed_schedule

    rob, problem, x_host, P, T = bench_workload
    m = R.get_model("fetch")
    cuboids, Tcuboids = cuboid_tensors(OBSTACLES["fetch"], torch.float64)
    x = run_lm_fixed_schedule(problem, x_host.to(DEV), "pppdd", parallel_count=P).cpu()
    target = problem.target_path.cpu().double()
    worst = 0.0
    for p in DRAWN:
        sl = slice(p * T, (p + 1) * T)
        ref = L.run_fixed_schedule(m, x_host[sl].double(), target, "pppdd", Tcuboids, cuboids)
        err = (x[sl].double() - ref).abs().max().item()
        worst = max(worst, err)
        assert err < 1e-4, (p, err)
    print(f"bench workload, pppdd: max |dq| vs fp64 oracle over {len(DRAWN)} drawn paths = {worst:.2e} rad")


def test_bench_workload_all_terms_step_vs_oracle(bench_workload):
    """The step bench.py's headline times (every term on, chunk-pipelined over 4 streams), 8 drawn paths.  With pose and
    differencing rows in one system any fp32 evaluation is noisy in the null space of J (DESIGN.md 4): the yardstick is
    the reference's own fp32 dense step - median ratio < 2.5, no path beyond 5x."""
    from cppflow_b200.lm_hyper_parameters import all_terms_parameters
    from cppflow_b200.pipeline import ResidentPipeline

    rob, problem, x_host, P, T = bench_workload
    m = R.get_model("fetch")
    cuboids, Tcuboids = cuboid_tensors(OBSTACLES["fetch"])
    x = ResidentPipeline(problem, P, all_terms_parameters(), n_chunks=4).iterate(x_host.to(DEV), 1).cpu()
    target = problem.target_path.cpu()
    ratios = []
    for p in DRAWN[::2]:
        sl = slice(p * T, (p + 1) * T)
        ref64 = L.run_fixed_schedule(m, x_host[sl].double(), target.double(), "a", [t.double() for t in Tcuboids],
                                     [c.double() for c in cuboids])
        ref32 = L.run_fixed_schedule(m, x_host[sl], target, "a", Tcuboids, cuboids)
        err = (x[sl].double() - ref64).abs().max().item()
        err32 = (ref32.double() - ref64).abs().max().item()
        assert err < max(5.0 * err32, 1e-4), (p, err, err32)
        ratios.append(err / max(err32, 1e-12))
    assert sorted(ratios)[len(ratios) // 2] < 2.5, ratios


# ------------------------------------------------------------------------------------------------------------------
# 1b. the reference's own loop

LOOP_PATTERNS = {  # planners.py:402-422
    "normal": dict(max_n_steps=20, return_if_valid_after_n_steps=0, convergence_threshold=1e6),
    "anytime": dict(max_n_steps=75, return_if_valid_after_n_steps=int(1e8), convergence_threshold=0.005),
}
LOOP_CASES = ["fetch_smooth", "fetch_noisy", "fetch_arm_smooth", "panda_smooth", "panda_noisy", "fetch_colliding"]


def _common_prefix(a, b):
    n = 0
    while n < min(len(a), len(b)) and a[n] == b[n]:
        n += 1
    return n


@pytest.mark.parametrize("case", LOOP_CASES)
@pytest.mark.parametrize("native", [True, False])
def test_alternating_loop_vs_reference_loop(robots, loop_golden, case, native):
    """run_lm_optimization (C++ loop and its Python twin) against the REAL reference loop's outputs.

    Where the reference's float32 and float64 runs take the same decisions (every `normal` call and the robust
    `anytime` ones) the CUDA loop must take them too - same step string, n_steps_taken, is_valid - and return the
    float64 iterate to 1e-4 rad (2e-4 after more than 20 steps).  Where the reference's own two precisions part ways
    (the convergence test |dTL| < 0.005 rad is marginal in some anytime runs) the CUDA loop must agree with them for
    as long as they agree with each other and end with the same validity."""
    from cppflow_b200.data_types import Constraints, Problem
    from cppflow_b200.optimization import run_lm_optimization

    g = loop_golden
    rname = str(g[f"{case}/robot"])
    rob = robots[rname]
    cuboids = [torch.tensor(c) for c in g[f"{case}/cuboids"]]
    Tcuboids = [torch.tensor(t) for t in g[f"{case}/Tcuboids"]]
    problem = Problem(Constraints(*CONSTRAINTS), torch.tensor(g[f"{case}/target"]).to(DEV), None, rob, "synthetic",
                      f"{rname}__synthetic", [], [t.to(DEV) for t in Tcuboids], [c.to(DEV) for c in cuboids], [])
    x_seed = torch.tensor(g[f"{case}/x_seed"]).to(DEV)
    for pat, kw in LOOP_PATTERNS.items():
        s32, s64 = str(g[f"{case}/{pat}/f32/schedule"]), str(g[f"{case}/{pat}/f64/schedule"])
        res = run_lm_optimization(problem, x_seed, tmax_sec=1e9, verbosity=0, native=native, **kw)
        assert res.is_valid == bool(g[f"{case}/{pat}/f64/is_valid"]) == bool(g[f"{case}/{pat}/f32/is_valid"]), (case, pat)
        if s32 == s64:
            assert res.schedule == s64, (case, pat, res.schedule, s64)
            assert res.n_steps_taken == int(g[f"{case}/{pat}/f64/n_steps_taken"]), (case, pat)
            err = (res.x_opt.cpu().double() - torch.tensor(g[f"{case}/{pat}/f64/x_opt"])).abs().max().item()
            assert err < (1e-4 if len(s64) <= 20 else 2e-4), (case, pat, err)
        else:
            n = _common_prefix(s32, s64)
            assert res.schedule[:n] == s64[:n], (case, pat, res.schedule, s32, s64)


# ------------------------------------------------------------------------------------------------------------------
# 1c. path metrics, every column


def _metric_paths(r, T, n_paths, seed):
    """n_paths paths of T waypoints: smooth tracking paths (valid), the same with noise (mjac / pose violations),
    with planted self-colliding and env-colliding waypoints, and with 2 pi wraps in a revolute joint."""
    m, target, x0 = synthetic_problem(r, n_paths, T, seed=seed, noise=0.0)
    cuboids, Tcuboids = cuboid_tensors(OBSTACLES[r])
    g = torch.Generator().manual_seed(seed)
    x = x0.reshape(n_paths, T, m.ndof).clone()
    cand = random_configs(m, 6000, seed=seed + 1)
    bad_self = cand[G.self_collision_distances(m, cand).min(dim=1).values < -0.01]
    bad_env = cand[G.env_collision_distances(m, cand, cuboids[0], Tcuboids[0]).min(dim=1).values < -0.01]
    for p in range(n_paths):
        kind = p % 5
        if kind == 1:
            x[p] += 0.002 * torch.randn((T, m.ndof), generator=g)  # small pose error, still smooth
        elif kind == 2:
            x[p] += 0.08 * torch.randn((T, m.ndof), generator=g)   # mjac and pose violations
        elif kind == 3:
            x[p, T // 3] = bad_self[p % bad_self.shape[0]]
            x[p, T // 2] = bad_env[p % bad_env.shape[0]]
        elif kind == 4:
            x[p, T // 2:, -1] += 2 * np.pi  # a full turn is no joint jump (angular_changes wraps) and no pose change
    return m, target, x, cuboids, Tcuboids


@pytest.mark.parametrize("r", ROBOTS)
@pytest.mark.parametrize("T", [57, 295])
def test_path_metrics_all_columns(robots, r, T):
    from cppflow_b200 import ops

    rob = robots[r]
    P = 405
    m, target, x, cuboids, Tcuboids = _metric_paths(r, T, P, seed=41)
    ob = ops.Obstacles(cuboids, Tcuboids)
    xd, td = x.reshape(P * T, -1).to(DEV), target.to(DEV)
    many = ops.path_metrics(rob.robot_id, rob.ndof, xd, td, P, T, ob).cpu()  # one CTA per path
    check = list(range(0, P, 9)) + [P - 1]
    c64 = [c.double() for c in cuboids], [t.double() for t in Tcuboids]
    n_valid = n_coll = 0
    for p in check:
        ref = L.path_metrics(m, x[p].double(), target.double(), c64[1], c64[0])
        one = ops.path_metrics(rob.robot_id, rob.ndof, x[p].contiguous().to(DEV), td, 1, T, ob).cpu()[0]  # cluster
        for got in (many[p], one):
            assert abs(got[0] - ref["max_pos_cm"]) < 2e-3, (p, "max_pos_cm", got[0], ref["max_pos_cm"])  # 2e-5 m in fp32 FK
            # fp32 geodesic distance 2 acos(min(|dot|, 1 - 1e-7)): one ulp of the dot product is 0.02 - 0.03 deg near zero
            tol_rot = 3e-2 if float(ref["max_rot_deg"]) < 1.0 else 2e-3 * float(ref["max_rot_deg"])
            assert abs(got[1] - ref["max_rot_deg"]) < tol_rot, (p, "max_rot_deg", got[1], ref["max_rot_deg"])
            assert abs(got[2] - ref["mjac_deg"]) < 1e-3, (p, "mjac_deg", got[2], ref["mjac_deg"])
            assert abs(got[3] - ref["mjac_cm"]) < 1e-4, (p, "mjac_cm", got[3], ref["mjac_cm"])
            assert abs(got[4] - ref["tl"]) < 1e-4 * max(1.0, float(ref["tl"])), (p, "tl", got[4], ref["tl"])
            # pairs are culled only against the running minimum, so the minima are exact
            for k, name in ((5, "min_self"), (6, "min_env")):
                assert abs(got[k] - ref[name]) < 1e-5, (p, name, got[k], ref[name])
        valid = (ref["max_pos_cm"] < CONSTRAINTS[0] and ref["max_rot_deg"] < CONSTRAINTS[1] and ref["mjac_deg"] < CONSTRAINTS[2]
                 and ref["mjac_cm"] < CONSTRAINTS[3] and ref["min_self"] >= 0 and ref["min_env"] >= 0)
        n_valid += bool(valid)
        n_coll += bool(ref["min_self"] < 0 or ref["min_env"] < 0)
    assert n_coll >= len(check) // 6, n_coll
    # sign-only variant (validity / cost ranking): every other column bit-identical, the two minima exact where negative
    # and non-negative where the exact minimum is
    sign = ops.path_metrics(rob.robot_id, rob.ndof, xd, td, P, T, ob, sign_only=True).cpu()
    assert torch.equal(sign[:, :5], many[:, :5])
    for k in (5, 6):
        neg = many[:, k] < 0
        assert torch.equal(sign[neg, k], many[neg, k])
        assert bool((sign[~neg, k] >= 0).all())
    assert int((many[:, 5:7] < 0).any(dim=1).sum()) >= P // 6


# ------------------------------------------------------------------------------------------------------------------
# 1d. dense get_r_and_J and the standalone clamp against the reference's golden vectors


@pytest.mark.parametrize("r", ROBOTS)
def test_dense_get_r_and_J_vs_golden(robots, golden, r):
    """cppflow_b200.optimization_utils.LmResidualFns.get_r_and_J (the dense drop-in, assembled from the CUDA kernels'
    per-term outputs) against all_J / all_r produced by the reference's LmResidualFns.get_r_and_J (all five terms,
    planted collisions, virtual configs != x): same row count and order; entries to 2e-5, collision-gradient rows to
    2e-3 (the env gradient switches feature at box edges)."""
    from cppflow_b200.lm_hyper_parameters import ALT_LOSS_V2_1_DIFF, ALT_LOSS_V2_1_POSE, OptimizationParameters
    from cppflow_b200.optimization_utils import LmResidualFns

    rob = robots[r]
    pms = OptimizationParameters(**ALT_LOSS_V2_1_DIFF.__dict__)
    pms.use_pose, pms.alpha_position, pms.alpha_rotation = True, ALT_LOSS_V2_1_POSE.alpha_position, ALT_LOSS_V2_1_POSE.alpha_rotation
    x = torch.tensor(golden[f"{r}/lm/all_x"]).to(DEV)
    pms.virtual_configs = torch.tensor(golden[f"{r}/lm/all_xv"]).to(DEV)
    cuboids = [torch.tensor(c).to(DEV) for c in golden[f"{r}/lm/cuboids"]]
    Tcuboids = [torch.tensor(t).to(DEV) for t in golden[f"{r}/lm/Tcuboids"]]
    jac, res = LmResidualFns.get_r_and_J(pms, rob, x, torch.tensor(golden[f"{r}/lm/target"]).to(DEV), Tcuboids=Tcuboids,
                                         cuboids=cuboids)
    J, rr = jac.get_J().cpu().numpy(), res.get_r().cpu().numpy()
    gJ, gr = golden[f"{r}/lm/all_J"], golden[f"{r}/lm/all_r"]
    n_self, n_env = int(golden[f"{r}/lm/all_n_self"]), int(golden[f"{r}/lm/all_n_env"])
    assert (0 if res.self_collisions is None else res.self_collisions.shape[0]) == n_self
    assert (0 if res.env_collisions is None else res.env_collisions.shape[0]) == n_env
    assert J.shape == gJ.shape and rr.shape == gr.shape
    n_coll = n_self + n_env
    n_fixed = J.shape[0] - n_coll
    np.testing.assert_allclose(rr, gr, atol=2e-5)
    np.testing.assert_allclose(J[:n_fixed], gJ[:n_fixed], atol=2e-5)
    dJ = np.abs(J[n_fixed:] - gJ[n_fixed:]).max(axis=1) / 0.01  # alpha_collision = 0.01: error of dd/dq per row
    assert (dJ < 2e-3).mean() > 0.98 and dJ.max() < 5e-2, (dJ.max(), (dJ < 2e-3).mean())
    assert n_coll > 0


@pytest.mark.parametrize("r", ROBOTS)
def test_standalone_clamp_vs_golden(robots, golden, r):
    """cppflow_clamp_to_joint_limits: in place, returns its argument (optimization_utils.py:823-833)."""
    from cppflow_b200.optimization_utils import clamp_to_joint_limits

    x = torch.tensor(golden[f"{r}/lm/clamp_in"]).to(DEV)
    y = clamp_to_joint_limits(robots[r], x)
    assert y.data_ptr() == x.data_ptr()
    assert np.array_equal(x.cpu().numpy(), golden[f"{r}/lm/clamp_out"])
    assert not np.array_equal(golden[f"{r}/lm/clamp_in"], golden[f"{r}/lm/clamp_out"])


# ------------------------------------------------------------------------------------------------------------------
# robustness items of the round-1 review


@pytest.mark.parametrize("r", ROBOTS)
def test_pose_step_at_kinematic_singularities(robots, r):
    """Fully stretched / aligned-axes configurations: J J^T + lambda I is numerically singular (pivots at the lambda
    floor).  The update must stay finite and follow the exact LM step to the tolerance used for ill-conditioned
    waypoints (2 % of the step) - never be thrown to a joint limit by a blown-up pivot."""
    from cppflow_b200 import ops
    from cppflow_b200.lm_hyper_parameters import ALT_LOSS_V2_1_POSE

    m = R.get_model(r)
    rob = robots[r]
    D = m.ndof
    lim = torch.tensor(m.actuated_joints_limits, dtype=torch.float64)
    base = torch.zeros(D, dtype=torch.float64).clamp(lim[:, 0], lim[:, 1])  # stretched arm (inside the limits)
    g = torch.Generator().manual_seed(5)
    xs = [base]
    for eps in (1e-6, 1e-4, 1e-2):
        xs += [(base + eps * torch.randn(D, generator=g, dtype=torch.float64)).clamp(lim[:, 0], lim[:, 1]) for _ in range(5)]
    x = torch.stack(xs).float()
    from oracle import kinematics as K

    target = K.forward_kinematics(m, (x.double() + 0.01 * torch.randn(x.shape, generator=g, dtype=torch.float64)).clamp(lim[:, 0], lim[:, 1])).float()
    out = ops.lm_pose_step(rob.robot_id, D, ops.make_params(ALT_LOSS_V2_1_POSE), x.to(DEV), target.to(DEV), True).cpu()
    assert torch.isfinite(out).all()
    ref = L.clamp_to_joint_limits(m, L.levenberg_marquardt_only_pose(m, x.double(), target.double(), L.ALT_LOSS_V2_1_POSE))
    step = (ref - x.double()).abs().max(dim=1).values
    err = (out.double() - ref).abs().max(dim=1).values
    assert (err <= 2e-2 * torch.clamp(step, min=1.0)).all(), (err, step)


def test_second_device(robots):
    """Tensors on cuda:1 while cuda:0 stays the current device: the shared-memory opt-in of the big kernels is per
    device and the ops make the tensor's device current for the call.  Same results as on cuda:0, bit for bit."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from cppflow_b200 import ops
    from cppflow_b200.lm_hyper_parameters import all_terms_parameters

    rob = robots["fetch"]
    P, T = 300, 64
    m, target, x0 = synthetic_problem("fetch", P, T, seed=3)
    cuboids, Tcuboids = cuboid_tensors(OBSTACLES["fetch"])
    ob = ops.Obstacles(cuboids, Tcuboids)
    prm = ops.make_params(all_terms_parameters())
    outs = []
    assert torch.cuda.current_device() == 0
    for dev in ("cuda:0", "cuda:1"):
        x, tg = x0.to(dev), target.to(dev)
        y = ops.lm_full_step(rob.robot_id, rob.ndof, prm, x, None, tg, P, T, ob, True)
        y1 = ops.lm_full_step(rob.robot_id, rob.ndof, prm, x[:T].contiguous(), None, tg, 1, T, ob, True)  # resident solve
        mt = ops.path_metrics(rob.robot_id, rob.ndof, y, tg, P, T, ob)
        outs.append((y.cpu(), y1.cpu(), mt.cpu()))
        assert torch.cuda.current_device() == 0
    for a, b in zip(*outs):
        assert torch.equal(a, b)


def test_dp_search_long_path_takes_the_single_cta_sweep(robots):
    """k <= 512 candidates but a path too long for the cluster sweep's shared-memory penalties: the search must fall
    through to the single-CTA sweep (the reference's dp_search has no limit on T), bit-exact as ever."""
    from cppflow_b200 import ops
    from oracle import search as S

    m = R.get_model("panda")
    rob = robots["panda"]
    k, T = 24, 20000  # 3 rows per CTA x 20000 x 4 B = 240 KB of penalties > 200 KB
    g = torch.Generator().manual_seed(3)
    base = random_configs(m, 1, seed=4)[0]
    q = base[None, None] + 0.05 * torch.randn((k, T, m.ndof), generator=g).cumsum(dim=1) * 0.05
    sv = torch.rand((k, T), generator=g) < 0.1
    ev = torch.rand((k, T), generator=g) < 0.1
    best, memo, costs, chosen = ops.dp_search(rob.robot_id, rob.ndof, q.to(DEV), sv.to(DEV), ev.to(DEV))
    ref_best, ref_memo, ref_costs, ref_chosen = S.dp_search(m, q, sv, ev)
    assert torch.equal(memo.cpu(), ref_memo) and torch.equal(costs.cpu(), ref_costs) and torch.equal(best.cpu(), ref_best)


@pytest.fixture(scope="module")
def rowscale_golden():
    import os

    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_rowscale_golden.npz"))


def test_row_scaling_helpers_vs_golden(robots, rowscale_golden):
    """The host mirror of the reference's row scaling / filtering helpers (device tensors, torch ops) against the
    reference's own outputs (SURVEY 8c golden items 4-6)."""
    from cppflow_b200.optimization_utils import LmResidualFns, filter_rows_from_r_J_differencing

    g = rowscale_golden
    for key in ("fetch/unit", "fetch/random", "panda/random"):
        rob = robots[str(g[f"{key}/robot"])]
        for shift in (0, 1):
            r, J = torch.tensor(g[f"{key}/diff/r_in"]).to(DEV), torch.tensor(g[f"{key}/diff/J_in"]).to(DEV)
            Jo, ro, inv = LmResidualFns._scale_down_rows_from_r_J_differencing_below_error(
                rob, r, J, mjac_threshold_m=0.25, mjac_threshold_rad=1.5, scale=0.5, shift_invalid_to_threshold=bool(shift))
            assert np.array_equal(ro.cpu().numpy(), g[f"{key}/diff/scale_shift{shift}/r"])
            assert np.array_equal(Jo.cpu().numpy(), g[f"{key}/diff/scale_shift{shift}/J"])
            assert np.array_equal(inv.cpu().numpy(), g[f"{key}/diff/scale_shift{shift}/invalid"])
            r, J = torch.tensor(g[f"{key}/diff/r_in"]).to(DEV), torch.tensor(g[f"{key}/diff/J_in"]).to(DEV)
            rf, Jf = filter_rows_from_r_J_differencing(rob, r, J, threshold_rad=1.5, threshold_m=0.25, shift_to_threshold=bool(shift))
            assert np.array_equal(rf.cpu().numpy(), g[f"{key}/diff/filter_shift{shift}/r"])
            assert np.array_equal(Jf.cpu().numpy(), g[f"{key}/diff/filter_shift{shift}/J"])
    for key in ("pose/a", "pose/b"):
        r, J = torch.tensor(g[f"{key}/r_in"]).to(DEV), torch.tensor(g[f"{key}/J_in"]).to(DEV)
        ro, Jo, inv = LmResidualFns._scale_down_rows_from_r_J_pose_below_error(r, J, error_threshold_m=0.01,
                                                                               error_threshold_rad=0.03, scale=0.25)
        assert np.array_equal(ro.cpu().numpy(), g[f"{key}/r"]) and np.array_equal(Jo.cpu().numpy(), g[f"{key}/J"])
        assert np.array_equal(inv.cpu().numpy(), g[f"{key}/invalid"])


@pytest.mark.parametrize("name", ["fetch__circle", "panda__1cube"])
def test_plan_from_qpath(name):
    """plan_from_qpath (data_type_utils.py:244-276) on the GPU: the Plan's derived metrics agree with the fast PathReport
    of the same path and with the fp64 oracle; its per-timestep collision flags are the capsule kernels'."""
    from cppflow_b200.collision_detection import qpaths_batched_collisions
    from cppflow_b200.data_type_utils import plan_from_qpath, problem_from_filename
    from cppflow_b200.data_types import PlanNp
    from cppflow_b200.planners import LatentIkCandidateGenerator, report_from_qpath

    problem = problem_from_filename(None, name, device=DEV)
    rob = problem.robot
    m = R.get_model(rob.name)
    qs = LatentIkCandidateGenerator(seed=4)(problem, 8)
    for q in (qs[0].contiguous(), qs[3].contiguous()):
        plan = plan_from_qpath(q, problem)
        rep = report_from_qpath(q, problem)
        cuboids = [c.cpu().double() for c in problem.obstacles_cuboids]
        Tcuboids = [t.cpu().double() for t in problem.obstacles_Tcuboids]
        ref = L.path_metrics(m, q.cpu().double(), problem.target_path.cpu().double(), Tcuboids, cuboids)
        assert plan.q_path.shape == (problem.n_timesteps, rob.ndof) and plan.pose_path.shape == (problem.n_timesteps, 7)
        assert abs(plan.max_positional_error_cm - float(ref["max_pos_cm"])) < 2e-3
        assert abs(plan.max_positional_error_cm - rep.max_positional_error_cm) < 1e-4
        assert abs(plan.mjac_deg - float(ref["mjac_deg"])) < 1e-3 and abs(plan.mjac_cm - float(ref["mjac_cm"])) < 1e-4
        assert abs(plan.path_length_rad - float(ref["tl"])) < 1e-4 * max(1.0, float(ref["tl"]))
        assert abs(plan.path_length_rad - rep.path_length_rad) < 1e-4 * max(1.0, rep.path_length_rad)
        sv, ev = qpaths_batched_collisions(problem, q[None].contiguous())
        assert torch.equal(plan.self_colliding_per_ts, sv[0]) and torch.equal(plan.env_colliding_per_ts, ev[0])
        assert bool(plan.env_colliding_per_ts.any()) == (float(ref["min_env"]) < 0)
        assert plan.is_valid == rep.is_valid
        assert isinstance(PlanNp(plan).q_path, np.ndarray)


# ------------------------------------------------------------------------------------------------------------------
# host-buffer pipeline: jobs in flight together give the results of the jobs run one at a time


@pytest.mark.parametrize("use_graph", [True, False])
def test_host_pipeline_async_jobs_match_single_step(robots, use_graph):
    from cppflow_b200 import ops
    from cppflow_b200.lm_hyper_parameters import all_terms_parameters
    from cppflow_b200.pipeline import HostPipeline
    from cppflow_b200.synthetic import synthetic_problem as device_problem, synthetic_seeds_host

    robot, P, T = robots["fetch"], 600, 61  # ragged: 600 paths over 7 chunks
    problem = device_problem(robot, T, seed=0, device=DEV)
    jobs = [synthetic_seeds_host(robot, P, T, seed=0, shard=k, pin=True)[1] for k in range(5)]
    outs = [torch.empty_like(j).pin_memory() for j in jobs]
    pipe = HostPipeline(problem, P, all_terms_parameters(), n_chunks=7, n_run_streams=3, use_graph=use_graph)
    prm = ops.make_params(all_terms_parameters())
    for rep in range(2):  # second round: graphs replayed, slots reused
        for o in outs:
            o.fill_(float("nan"))
        done = [pipe.refine_async(j, o) for j, o in zip(jobs, outs)]
        for ev in done:
            ev.synchronize()
        for j, o in zip(jobs, outs):
            ref = ops.lm_full_step(robot.robot_id, robot.ndof, prm, j.to(DEV), None, problem.target_path, P, T,
                                   problem.obstacle_tables, True)
            assert torch.equal(o, ref.cpu()), "a job in flight next to another must equal the job run alone, bit for bit"
    out2 = torch.empty_like(jobs[0]).pin_memory()
    pipe.refine(jobs[0], out2)
    torch.cuda.current_stream().synchronize()
    assert torch.equal(out2, outs[0])


# ------------------------------------------------------------------------------------------------------------------
# ranking key + local argmin: the library's one-launch kernel against the torch arithmetic of distributed.path_keys


@pytest.mark.parametrize("P", [1, 37, 8192, 70001])
@pytest.mark.parametrize("all_invalid", [False, True])
def test_native_key_argmin_matches_torch_keys(P, all_invalid):
    from cppflow_b200 import ops
    from cppflow_b200.data_types import DEFAULT_CONSTRAINTS as C
    from cppflow_b200.distributed import path_keys, enqueue_argmin, _INVALID_SHIFT

    g = torch.Generator().manual_seed(P)
    m = torch.zeros((P, 8))
    m[:, 0] = torch.rand(P, generator=g) * 2 * C.max_allowed_position_error_cm  # half of the paths break a threshold
    m[:, 1] = torch.rand(P, generator=g) * 1.2 * C.max_allowed_rotation_error_deg
    m[:, 2] = torch.rand(P, generator=g) * 1.1 * C.max_allowed_mjac_deg
    m[:, 3] = torch.rand(P, generator=g) * 1.1 * C.max_allowed_mjac_cm
    m[:, 4] = torch.rand(P, generator=g) * 50 + 1
    m[:, 5] = torch.rand(P, generator=g) - 0.1
    m[:, 6] = torch.where(torch.rand(P, generator=g) < 0.3, torch.full((P,), float("inf")), torch.rand(P, generator=g) - 0.1)
    if all_invalid:
        m[:, 0] = 1.0
    if P > 30:
        m[3, 4] = m[29, 4] = 0.5                       # a tie: the lowest index wins
        m[7, 4] = float("nan")                         # NaN trajectory length: invalid, sorts last
        m[11, 0] = C.max_allowed_position_error_cm     # equality with a threshold is not below it (float32 comparison)
        m[13, 5] = 0.0                                 # a distance of exactly zero is not a collision
    first = 1000
    md = m.to(DEV)
    keys = path_keys(md, C, first)
    want = [int(keys.min()), int((keys >> _INVALID_SHIFT == 0).sum()), first]
    got = ops.path_key_argmin(md, C, first).cpu().tolist()
    assert got == want
    assert tuple(enqueue_argmin(md, C, first, 1).result()) == tuple(enqueue_argmin(m, C, first, 1).result())


def test_resident_pipeline_graph_replay_equals_eager(robots):
    """ResidentPipeline.capture: the chunk-pipelined iterations replayed from a CUDA graph give the bits of the eager
    enqueue and of one single-stream step (chunks of 256 paths: register-resident solve; 300 paths: ragged)."""
    from cppflow_b200 import ops
    from cppflow_b200.lm_hyper_parameters import all_terms_parameters
    from cppflow_b200.pipeline import ResidentPipeline
    from cppflow_b200.synthetic import synthetic_problem as device_problem, synthetic_seeds_host

    robot, T = robots["fetch"], 61
    problem = device_problem(robot, T, seed=0, device=DEV)
    prm = ops.make_params(all_terms_parameters())
    for P, n_chunks in ((1024, None), (300, 3), (2048, None)):
        x = synthetic_seeds_host(robot, P, T, seed=0)[1].to(DEV)
        ref = ops.lm_full_step(robot.robot_id, robot.ndof, prm, x, None, problem.target_path, P, T, problem.obstacle_tables, True)
        pipe = ResidentPipeline(problem, P, all_terms_parameters(), n_chunks=n_chunks)
        out_e, out_g = torch.full_like(x, float("nan")), torch.full_like(x, float("nan"))
        metrics = torch.zeros((P, 8), device=DEV)

        def work(out):
            for _ in range(3):
                pipe.enqueue_step(x, out)
            pipe.enqueue_metrics(out, metrics)

        pipe.begin(); work(out_e); pipe.end()
        torch.cuda.synchronize()
        m_eager = metrics.clone()
        graph = pipe.capture(lambda: work(out_g))
        metrics.zero_()
        for _ in range(2):
            graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(out_e, ref) and torch.equal(out_g, ref)
        assert torch.equal(metrics, m_eager)


@pytest.mark.parametrize("r", ROBOTS)
def test_overlap_launch_equals_stand_alone_step(robots, r):
    """CPPFLOW_LM_OVERLAP: the solve launched to run under another chunk's assembly (the 4-slot ring, the smaller
    register-resident threshold, high priority).  Same bits as the stand-alone step, with and without clamp, for every
    path / waypoint count (one waypoint = only the middle block, even / odd T, ragged path counts, path counts on both
    sides of the solve kernels' thresholds) and parameter set."""
    from cppflow_b200 import ops
    from cppflow_b200.lm_hyper_parameters import all_terms_parameters, ALT_LOSS_V2_1_DIFF

    rob = robots[r]
    cuboids, Tcuboids = cuboid_tensors(OBSTACLES[r])
    ob = ops.Obstacles(cuboids, Tcuboids)
    for P, T in ((1, 1), (3, 2), (5, 3), (17, 4), (33, 5), (300, 9), (1000, 64), (2100, 301), (257, 295)):
        m, target, x0 = synthetic_problem(r, P, T, seed=P + T)
        x, tg = x0.to(DEV), target.to(DEV)
        for name, pm in (("all", all_terms_parameters()), ("diff", ALT_LOSS_V2_1_DIFF)):
            if pm.use_virtual_configs and 2 * pm.n_virtual_configs >= T:
                continue
            prm = ops.make_params(pm)
            xv = x.clone() if pm.use_virtual_configs else None
            for clamp in (True, False):
                ref = ops.lm_full_step(rob.robot_id, rob.ndof, prm, x, xv, tg, P, T, ob, clamp)
                got = ops.lm_full_step(rob.robot_id, rob.ndof, prm, x, xv, tg, P, T, ob, clamp, overlap=True)
                assert torch.equal(got, ref), (r, P, T, name, clamp, float((got - ref).abs().max()))


def _dense_step_fp64(lib, rob, prm, pm, x, tg, ob_args, P, T, paths):
    """fp64 solution of the normal equations the assembly kernel wrote, for a few paths: reads the packed (A_tt, b_t) blocks
    ([16-path group][t][float4 k][path in group]) back and solves the block-tridiagonal system densely."""
    from cppflow_b200 import _lib

    D = rob.ndof
    NT = D * (D + 1) // 2
    NW = (NT + D + 3) // 4 * 4
    ws = torch.zeros((lib.cppflow_lm_full_workspace_bytes(rob.robot_id, P, T),), device=DEV, dtype=torch.uint8)
    cu, tc, no = ob_args
    _lib.check(lib.cppflow_lm_full_assemble(rob.robot_id, prm, _lib.ptr(x), None, _lib.ptr(tg), P, T, cu, tc, no,
                                            _lib.ptr(ws), ws.numel(), _lib.stream_ptr(DEV)))
    torch.cuda.synchronize()
    groups = (P + 15) // 16
    blocks = ws.view(torch.float32)[: groups * T * NW * 16].cpu().numpy().reshape(groups, T, NW // 4, 16, 4)
    beta = np.array([(pm.alpha_differencing * (pm.alpha_differencing_prismatic_scaling if d in rob.prismatic_joint_idxs else 1.0)) ** 2
                     for d in range(D)]) * (1.0 if pm.use_differencing else 0.0)
    out = {}
    for p in paths:
        blk = blocks[p // 16, :, :, p % 16, :].reshape(T, NW).astype(np.float64)
        Mx = np.zeros((T * D, T * D))
        for i in range(D):
            for j in range(i + 1):
                for t in range(T):
                    Mx[t * D + i, t * D + j] = Mx[t * D + j, t * D + i] = blk[t, i * (i + 1) // 2 + j]
        for t in range(T - 1):
            for d in range(D):
                Mx[t * D + d, (t + 1) * D + d] = Mx[(t + 1) * D + d, t * D + d] = -beta[d]
        rhs = blk[:, NT:NT + D].reshape(-1)
        out[p] = (Mx, rhs, np.linalg.solve(Mx, rhs))
    return out


@pytest.mark.parametrize("r", ROBOTS)
def test_segmented_solve_equals_twisted_solve_up_to_rounding(robots, r):
    """CPPFLOW_LM_SEGMENTS (csrc/lm_segsolve.cuh): segments between separator waypoints eliminated in parallel, the
    separators' reduced system, parallel back-substitution.  Another elimination order of the same linear system.  With
    every term on the system is ill-conditioned (lambda = 1e-6: condition number ~ 3e7), so BOTH float32 solves sit
    ~1e-2 rad from the fp64 solution of the same blocks in the null-space directions; the yardsticks are therefore the
    residual of the normal equations and the distance from the fp64 solution, each against the twisted solve's own.
    For a given segment count the result of a path does NOT depend on how many paths are solved with it (bit-exact),
    and short paths fall back to the twisted solve."""
    from cppflow_b200 import ops, _lib
    from cppflow_b200.lm_hyper_parameters import all_terms_parameters, ALT_LOSS_V2_1_DIFF

    rob = robots[r]
    cuboids, Tcuboids = cuboid_tensors(OBSTACLES[r])
    ob = ops.Obstacles(cuboids, Tcuboids)
    lib = _lib.load()
    worst = {"residual": 0.0, "energy": 0.0, "distance_all": 0.0, "distance_diff": 0.0}
    for P, T in ((1, 300), (20, 301), (48, 37), (5, 9), (33, 8), (3, 7), (1100, 64)):
        m, target, x0 = synthetic_problem(r, P, T, seed=P + T)
        x, tg = x0.to(DEV), target.to(DEV)
        for name, pm in (("all", all_terms_parameters()), ("diff", ALT_LOSS_V2_1_DIFF)):
            if pm.use_virtual_configs and 2 * pm.n_virtual_configs >= T:
                continue
            prm = ops.make_params(pm)
            ref = ops.lm_full_step(rob.robot_id, rob.ndof, prm, x, None, tg, P, T, ob, False)
            paths = sorted({0, P // 2, P - 1})
            dense = _dense_step_fp64(lib, rob, prm, pm, x, tg, ops._obs(ob), P, T, paths)

            def quality(res, p):
                Mx, rhs, sol = dense[p]
                dx = (res[p * T:(p + 1) * T] - x[p * T:(p + 1) * T]).double().cpu().numpy().reshape(-1)
                e = dx - sol
                return np.linalg.norm(Mx @ dx - rhs) / np.linalg.norm(rhs), np.abs(e).max(), float(e @ Mx @ e) / float(sol @ Mx @ sol)

            for S in (2, 3, 5, 16, 200):
                got = ops.lm_full_step(rob.robot_id, rob.ndof, prm, x, None, tg, P, T, ob, False, segments=S)
                if T // 4 < 2:
                    assert torch.equal(got, ref), (r, P, T, name, S, "short path: twisted solve")
                    continue
                for p in paths:
                    (res_t, err_t, en_t), (res_s, err_s, en_s) = quality(ref, p), quality(got, p)
                    worst["residual"] = max(worst["residual"], res_s / (res_t + 1e-7))
                    worst["energy"] = max(worst["energy"], en_s / (en_t + 1e-13))
                    worst["distance_" + name] = max(worst["distance_" + name], err_s / (err_t + 2e-5))
                    assert res_s <= 3.0 * res_t + 1e-6, (r, P, T, name, S, p, "residual", res_s, res_t)
                    # error in the energy norm of the normal equations (what the LM step minimises), relative to the step
                    assert en_s <= 10.0 * en_t + 1e-12, (r, P, T, name, S, p, "energy-norm error", en_s, en_t)
                    if name == "diff":  # well-conditioned: also element-wise
                        assert err_s <= 3.0 * err_t + 2e-5, (r, P, T, name, S, p, "distance from fp64", err_s, err_t)
                # one path alone = the same path among the others
                one = ops.lm_full_step(rob.robot_id, rob.ndof, prm, x[-T:].contiguous(), None, tg, 1, T, ob, False, segments=S)
                assert torch.equal(one, got[-T:]), (r, P, T, name, S, "path count changes the result")
            clamped = ops.lm_full_step(rob.robot_id, rob.ndof, prm, x, None, tg, P, T, ob, True, segments=5)
            unclamped = ops.lm_full_step(rob.robot_id, rob.ndof, prm, x, None, tg, P, T, ob, False, segments=5)
            lim = torch.tensor(rob.actuated_joints_limits, device=DEV, dtype=torch.float32)
            assert torch.equal(clamped, torch.minimum(torch.maximum(unclamped, lim[:, 0]), lim[:, 1]))
    print("segmented / twisted, worst ratios:", r, {k: round(v, 2) for k, v in worst.items()})


def test_resident_pipeline_segmented_solve_is_chunking_independent(robots):
    """`ResidentPipeline(segments=...)`: for a given segment count the refined paths do not depend on the chunk count, on
    eager enqueue or graph replay, and equal the single-launch step with the same segment count bit for bit;
    `segments="auto"` takes 16 segments up to 2048 paths and the twisted solve above."""
    from cppflow_b200 import ops
    from cppflow_b200.lm_hyper_parameters import all_terms_parameters
    from cppflow_b200.pipeline import ResidentPipeline
    from cppflow_b200.synthetic import synthetic_problem as device_problem, synthetic_seeds_host

    robot, T = robots["fetch"], 61
    problem = device_problem(robot, T, seed=0, device=DEV)
    prm = ops.make_params(all_terms_parameters())
    P = 700  # ragged: not a multiple of 16 x chunks
    x = synthetic_seeds_host(robot, P, T, seed=0)[1].to(DEV)
    for S in (4, 15):
        ref = ops.lm_full_step(robot.robot_id, robot.ndof, prm, x, None, problem.target_path, P, T, problem.obstacle_tables,
                               True, segments=S)
        for n_chunks in (1, 2, 5):
            pipe = ResidentPipeline(problem, P, all_terms_parameters(), n_chunks=n_chunks, segments=S)
            out_e, out_g = torch.full_like(x, float("nan")), torch.full_like(x, float("nan"))
            pipe.begin(); pipe.enqueue_step(x, out_e); pipe.end()
            graph = pipe.capture(lambda: pipe.enqueue_step(x, out_g))
            graph.replay()
            torch.cuda.synchronize()
            assert torch.equal(out_e, ref), (S, n_chunks, float((out_e - ref).abs().max()))
            assert torch.equal(out_g, ref), (S, n_chunks, "graph replay")
    assert ResidentPipeline(problem, 2048, all_terms_parameters(), segments="auto").segments == 16
    assert ResidentPipeline(problem, 2049, all_terms_parameters(), segments="auto").segments == 0
    twisted = ops.lm_full_step(robot.robot_id, robot.ndof, prm, x, None, problem.target_path, P, T, problem.obstacle_tables, True)
    assert not torch.equal(twisted, ref)  # another elimination order: rounding-level differences, not the same bits
    assert float((twisted - ref).abs().max()) < 0.2


@pytest.mark.parametrize("P,T,S", [(3, 1000, 32), (2, 4000, 32), (40, 129, 255), (16, 4000, 7)])
def test_segmented_solve_long_paths(robots, P, T, S):
    """Long paths: half-segments that fit the staged pass 3's shared memory (T = 1000, 32 segments) and ones that do not
    (T = 4000: the streaming pass 3), a segment count above the cap of 32 / T / 4, few long segments.  With the
    well-conditioned differencing parameter set the segmented and the twisted step agree element-wise."""
    from cppflow_b200 import ops
    from cppflow_b200.lm_hyper_parameters import ALT_LOSS_V2_1_DIFF

    rob = robots["panda"]
    cuboids, Tcuboids = cuboid_tensors(OBSTACLES["panda"])
    ob = ops.Obstacles(cuboids, Tcuboids)
    m, target, x0 = synthetic_problem("panda", P, T, seed=P + T)
    x, tg = x0.to(DEV), target.to(DEV)
    prm = ops.make_params(ALT_LOSS_V2_1_DIFF)
    ref = ops.lm_full_step(rob.robot_id, rob.ndof, prm, x, None, tg, P, T, ob, True)
    got = ops.lm_full_step(rob.robot_id, rob.ndof, prm, x, None, tg, P, T, ob, True, segments=S)
    assert torch.isfinite(got).all()
    step = float((ref - x).abs().max())
    err = float((got - ref).abs().max())
    assert err < 1e-4 + 1e-3 * step, (P, T, S, err, step)
    assert not torch.equal(got, ref) or step == 0.0  # it IS another solve
