"""Training IKFlow on the device (csrc/k_flow_train.cu, cppflow_b200/ikflow_training.py) against the training
definition of oracle/ikflow_train.py.

CPU: the log-determinant identity of the oracle, the round trip of packed tables and GraphINN state dicts, workspace
sizes, rejected shapes and the struct layout.  GPU: forward parity (z bit-identical to cppflow_flow_run), gradient
parity with torch autograd, Adam against torch.optim.Adam, determinism, graph replay, resume, no host
synchronisation, skipped non-finite steps, a short training run that learns, and the planner on trained weights."""
import ctypes
import os
import shutil
import subprocess

import pytest
import torch

from oracle import ikflow as OF
from oracle import ikflow_train as OT

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda:0"
ROBOTS = ["fetch", "fetch_arm", "panda"]


def _model(name):
    from oracle import robots as R

    return R.get_model(name)


def _params(width=9, nb=2, H=128, L=2, softflow=True):
    from cppflow_b200.ikflow import IkflowModelParameters

    return IkflowModelParameters(nb_nodes=nb, dim_latent_space=width, coeff_fn_config=L, coeff_fn_internal_size=H,
                                 softflow_enabled=softflow)


# ----------------------------------------------------------------------------------------------------------- CPU


@pytest.mark.parametrize("robot", ROBOTS)
@pytest.mark.parametrize("extra", [0, 1, 2])
def test_log_det_is_the_jacobian_determinant(robot, extra):
    model = _model(robot)
    width = model.ndof + extra
    net = OF.random_glow(model.actuated_joints_limits, width, nb_nodes=3, internal=16, n_layers=2, seed=extra).double()
    g = torch.Generator().manual_seed(7)
    x = torch.rand((6, width), generator=g, dtype=torch.float64) * 2 - 1
    cond = torch.cat([torch.rand((6, 7), generator=g, dtype=torch.float64), torch.rand((6, 1), generator=g,
                                                                                      dtype=torch.float64)], dim=1)
    z, log_det = OT.forward_with_logdet(net, x, cond)
    # with a softflow scale of 0 it is the inference forward pass
    cond0 = cond.clone()
    cond0[:, 7] = 0
    torch.testing.assert_close(OT.forward_with_logdet(net, x, cond0)[0], net(x, cond[:, :7]), rtol=0, atol=1e-14)
    for r in range(x.shape[0]):
        jac = torch.autograd.functional.jacobian(lambda v: OT.forward_with_logdet(net, v[None], cond[r:r + 1])[0][0],
                                                 x[r])
        assert torch.allclose(log_det[r], torch.linalg.slogdet(jac)[1], rtol=0, atol=1e-10)
    assert (log_det - log_det.mean()).abs().max() > 1e-3  # depends on the row: the couplings are not volume-preserving
    torch.testing.assert_close(OT.nll(z, log_det), (0.5 * (z * z).sum(1) - log_det).mean())


def test_training_batch_definition():
    model = _model("panda")
    q, poses = OT.sample_training_data(model, 200, torch.Generator().manual_seed(0))
    assert 0 < q.shape[0] <= 200 and poses.shape == (q.shape[0], 7)
    n = 16
    idx = torch.arange(n) % q.shape[0]
    c, eps = torch.rand(n, dtype=torch.float64), torch.randn((n, 9), dtype=torch.float64)
    flip = torch.arange(n) % 2 == 1
    x, cond = OT.training_batch(q, poses, idx, c, eps, flip, 9, 8, 1e-3)
    torch.testing.assert_close(x, torch.cat([q[idx], torch.zeros((n, 2), dtype=torch.float64)], 1) + 1e-3 * c[:, None] * eps)
    assert torch.equal(cond[:, :3], poses[idx, :3]) and torch.equal(cond[:, 7], c)
    assert torch.equal(cond[flip, 3:7], -poses[idx][flip, 3:]) and torch.equal(cond[~flip, 3:7], poses[idx][~flip, 3:])
    x7, cond7 = OT.training_batch(q, poses, idx, c, eps, flip, 7, 7, 1e-3)
    assert torch.equal(x7, q[idx]) and cond7.shape == (n, 7)


@pytest.mark.parametrize("L", [1, 3])
def test_packed_tables_round_trip(L):
    from cppflow_b200.ikflow import pack_fp32, random_state_dict
    from cppflow_b200.ikflow_training import _TABLES, split_tables, unpack
    from cppflow_b200.robot import get_robot

    p = _params(width=9, nb=3, H=128, L=L)
    sd = random_state_dict(get_robot("fetch"), p, seed=4)
    packed = pack_fp32(p, sd)
    flat = torch.cat([packed[k].reshape(-1) for k in _TABLES])
    back = unpack(split_tables(flat, p), p)
    subnets = {k: v for k, v in sd.items() if ".subnet" in k}
    assert back.keys() == subnets.keys()
    for k in subnets:
        assert torch.equal(back[k], subnets[k]), k
    with pytest.raises(ValueError):
        split_tables(flat[:-1], p)


def _train_desc(**kw):
    from cppflow_b200 import _lib

    f = dict(robot=2, width=9, ndof=7, dim_cond=8, nb_nodes=12, coeff_fn_config=3, coeff_fn_internal_size=1024,
             rnvp_clamp=2.5)
    hyper = dict(lr=5e-4, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=1.8e-5, lr_decay=0.9794, lr_decay_steps=4883)
    for k in list(kw):
        if k in hyper:
            hyper[k] = kw.pop(k)
    f.update(kw)
    flow = _lib.FlowDescC(**f)
    for name in ("d_w_in", "d_w_hidden", "d_b_hidden", "d_w_out", "d_b_out", "d_scale", "d_perm", "d_perm_inv"):
        setattr(flow, name, 256)  # never dereferenced: every call below is rejected before a launch
    return _lib.FlowTrainDescC(flow, 256, 256, 256, 256, 256, 256, 256, **hyper)


def test_train_workspace_bytes():
    from cppflow_b200 import _lib

    lib = _lib.load()
    a256 = lambda b: (b + 255) // 256 * 256  # noqa: E731
    for nb, H, L, W, n in ((12, 1024, 3, 9, 512), (2, 128, 1, 7, 4096)):
        S = 2 * nb
        P = 2 * nb * (H * 64 + (L - 1) * H * H + L * H + 16 * H + 16)
        want = (2 * a256(S * n * 64) + 2 * a256(S * n * 128) + 2 * a256(S * L * n * H * 2) + 2 * a256(n * 4)
                + a256(n * W * 4) + 2 * a256(n * 64) + a256(n * 128) + a256(16 * n * 2) + a256(16 * n * 4)
                + 4 * a256(n * H * 2)
                + a256(n * 256) + a256(P * 4) + a256(1024) + a256(4))
        d = _train_desc(nb_nodes=nb, coeff_fn_internal_size=H, coeff_fn_config=L, width=W)
        assert lib.cppflow_flow_train_workspace_bytes(d, n) == want


@pytest.mark.parametrize("change,batch,message", [
    ({}, 200, "batch 200 is not a multiple of 128"),
    ({}, 0, "n = 0"),
    (dict(dim_cond=7), 512, "width 9 > ndof 7 needs softflow"),
    (dict(coeff_fn_internal_size=192), 512, "coeff_fn_internal_size 192"),
    (dict(width=17), 512, "width 17 outside"),
    (dict(beta1=1.0), 512, "hyperparameter out of range"),
    (dict(lr_decay_steps=0), 512, "hyperparameter out of range"),
])
def test_unsupported_training_shapes_are_rejected(change, batch, message):
    from cppflow_b200 import _lib

    lib = _lib.load()
    d = _train_desc(**change)
    assert lib.cppflow_flow_train_workspace_bytes(d, batch) == 0
    assert message.encode() in lib.cppflow_last_error()
    assert lib.cppflow_flow_train_step(d, 256, 256, batch, 0, 256, 1 << 40, 256, None, None) == -1
    assert message.encode() in lib.cppflow_last_error()
    assert lib.cppflow_flow_train_batch(d, 256, 256, 10, batch, 0, 1e-3, 256, 256, None, None, None) == -1


def test_bad_training_calls_are_rejected():
    from cppflow_b200 import _lib

    lib = _lib.load()
    d = _train_desc()
    assert lib.cppflow_flow_train_step(d, 256, 256, 512, 2, 256, 1 << 40, 256, None, None) == -1
    assert b"unknown flag bits" in lib.cppflow_last_error()
    assert lib.cppflow_flow_train_step(d, 256, 256, 512, 0, 256, 1 << 40, 256, None, None) == -1
    assert b"must point at their segments of d_params" in lib.cppflow_last_error()
    d.d_counters = None
    assert lib.cppflow_flow_train_step(d, 256, 256, 512, 0, 256, 1 << 40, 256, None, None) == -1
    assert b"null training table" in lib.cppflow_last_error()


def test_flow_train_desc_layout_matches_the_c_header(tmp_path):
    from cppflow_b200 import _lib

    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    fields = ["d_params", "d_w_hidden_t", "d_counters", "lr", "lr_decay", "lr_decay_steps"]
    src = tmp_path / "train.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "cppflow_b200.h"\nint main(void) {\n'
                   '  printf("%zu\\n", sizeof(cppflow_flow_train_desc));\n'
                   + "".join(f'  printf("%zu\\n", offsetof(cppflow_flow_train_desc, {f}));\n' for f in fields)
                   + "  return 0;\n}\n")
    exe = tmp_path / "train"
    subprocess.run([gcc, "-I", os.path.join(REPO, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    T = _lib.FlowTrainDescC
    assert got == [ctypes.sizeof(T)] + [getattr(T, f).offset for f in fields]


# ----------------------------------------------------------------------------------------------------------- GPU

def _trainer(robot, size="small", **kw):
    from cppflow_b200.ikflow_training import IkflowTrainer
    from cppflow_b200.robot import get_robot

    p = _params(width=9, nb=2, H=128, L=2) if size == "small" else _params(width=9, nb=12, H=1024, L=3)
    kw.setdefault("n_data", 20000)
    return IkflowTrainer(get_robot(robot), p, seed=kw.pop("seed", 3), device=DEV, **kw)


def _glow(tr, dtype=torch.float64):
    p = tr.params
    net = OF.Glow(tr.robot.actuated_joints_limits, p.dim_latent_space, p.nb_nodes, p.coeff_fn_internal_size,
                  p.coeff_fn_config, p.rnvp_clamp, p.softflow_enabled)
    net.load_state_dict(tr.state_dict())
    return net.to(DEV, dtype)


def _ws_z_logdet(tr, n):
    """z and the per-row log-det (without logDetM) of the last step, read from the workspace (layout: TrainWs in
    csrc/k_flow_train.cu)."""
    a256 = lambda b: (b + 255) // 256 * 256  # noqa: E731
    p = tr.params
    S, L, H, W = 2 * p.nb_nodes, p.coeff_fn_config, p.coeff_fn_internal_size, p.dim_latent_space
    off = 2 * a256(S * n * 64) + 2 * a256(S * n * 128) + 2 * a256(S * L * n * H * 2)
    logdet = tr.workspace[off:off + n * 4].view(torch.float32)
    off += a256(n * 4)
    z = tr.workspace[off:off + n * W * 4].view(torch.float32).view(n, W)
    return z, logdet


@pytest.mark.gpu
@pytest.mark.parametrize("robot", ROBOTS)
@pytest.mark.parametrize("size", ["small", "full"])
def test_training_forward_parity(robot, size):
    from cppflow_b200 import ops

    n = 128 * 41  # 5248 rows: a multiple of the 128-row tile, not of 256 or of the head's 32-row groups
    tr = _trainer(robot, size, batch_size=n)
    tr.draw_batch()
    x, cond = tr.x.clone(), tr.cond.clone()
    cond[:, 7] = 0  # cppflow_flow_run conditions with a softflow scale of 0
    loss, _ = tr.loss_and_grad(x, cond)
    z, ld = _ws_z_logdet(tr, n)
    # the inference forward pass on the same rows gives the same bits
    flow = tr.desc.flow
    ref_z = torch.empty_like(x)
    ws = torch.empty(ops._lib.load().cppflow_flow_workspace_bytes(ctypes.byref(flow), n), dtype=torch.uint8, device=DEV)
    ops._lib.check(ops._lib.load().cppflow_flow_run(ctypes.byref(flow), ops.ptr(x), ops.ptr(cond[:, :7].contiguous()), n, n,
                                                    0, ops.ptr(ws), ws.numel(), ops.ptr(ref_z), ops.stream_ptr()))
    assert torch.equal(z, ref_z)
    net = _glow(tr)
    with torch.no_grad():
        z64, ld64 = OT.forward_with_logdet(net, x.double(), cond.double(), bf16=True)
        z32, ld32 = OT.forward_with_logdet(_glow(tr, torch.float32), x, cond)
    ldm = float(torch.log(tr.scale.double()).sum())
    got_ld = ld.double() + ldm
    e16 = (got_ld - ld64).abs().max().item()
    e32 = (got_ld - ld32.double()).abs().max().item()
    l64 = OT.nll(z64, ld64).item()
    print(f"{robot} {size}: log_det max err vs bf16 oracle {e16:.2e}, vs fp32 oracle {e32:.2e}; loss {loss.item():.6f} "
          f"vs {l64:.6f}")
    assert torch.isfinite(z).all()
    assert e16 < 2e-2 and e32 < 5e-2
    assert abs(loss.item() - l64) < 1e-3 * max(1.0, abs(l64))


@pytest.mark.gpu
@pytest.mark.parametrize("size", ["small", "full"])
def test_gradient_parity_with_autograd(size):
    from cppflow_b200.ikflow_training import split_tables, unpack

    n = 1024
    tr = _trainer("panda", size, batch_size=n, seed=5)
    tr.draw_batch()
    x, cond = tr.x.clone(), tr.cond.clone()
    _, grad = tr.loss_and_grad(x, cond)
    got = unpack(split_tables(grad, tr.params), tr.params)

    def grads(net, xx, cc, bf16, autocast):
        net.zero_grad()
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
            OT.nll(*OT.forward_with_logdet(net, xx, cc, bf16=bf16)).backward()
        return {k: p.grad.detach().double().cpu() for k, p in net.named_parameters()}

    ref = grads(_glow(tr), x.double(), cond.double(), True, False)
    torch_bf16 = grads(_glow(tr, torch.float32), x, cond, False, True)
    worst = 0.0
    for k, r in ref.items():
        g = got[k].double()
        rel = ((g - r).norm() / r.norm()).item()
        rel_t = ((torch_bf16[k] - r).norm() / r.norm()).item()
        cos = torch.nn.functional.cosine_similarity(g.reshape(1, -1), r.reshape(1, -1)).item()
        worst = max(worst, rel / rel_t)
        print(f"{k}: rel L2 {rel:.2e} (torch bf16 autocast {rel_t:.2e}), cos {cos:.6f}")
        assert rel <= 2 * rel_t, k
        assert cos >= 0.999, k
    print(f"worst ratio to torch bf16: {worst:.2f}")


@pytest.mark.gpu
def test_adam_step_matches_torch_and_refreshes_the_tables():
    from cppflow_b200 import ops
    from cppflow_b200.ikflow import IkflowSolver

    tr = _trainer("fetch", "small", batch_size=512)
    for _ in range(2):  # second step: nonzero moments and bias corrections of t = 2
        tr.draw_batch()
        before = [t.clone() for t in (tr.params_flat, tr.adam_m, tr.adam_v)]
        _, grad = tr.loss_and_grad(tr.x, tr.cond)
        ops.flow_train_step(tr.desc, tr.x, tr.cond, tr.workspace, tr.loss)
        p = torch.nn.Parameter(before[0].clone())
        opt = torch.optim.Adam([p], lr=5e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=1.8e-5)
        if tr.counters[0].item() == 2:
            opt.state[p] = {"step": torch.tensor(1.0), "exp_avg": before[1].clone(), "exp_avg_sq": before[2].clone()}
        p.grad = grad
        opt.step()
        for name, mine, ref in (("w", tr.params_flat, p.detach()), ("m", tr.adam_m, opt.state[p]["exp_avg"]),
                                ("v", tr.adam_v, opt.state[p]["exp_avg_sq"])):
            d = (mine - ref).abs().max().item()
            print(f"step {tr.counters[0].item()}: max |{name} - torch| = {d:.3e}")
            # FP32 rounding relative to the tensor's scale: m is small where g + wd w nearly cancels
            torch.testing.assert_close(mine, ref, rtol=2e-6, atol=2e-6 * ref.abs().max().item())
    assert tr.counters.tolist() == [2, 0, 2]
    sol = IkflowSolver(tr.robot, tr.params, state_dict=tr.state_dict(), device=DEV)
    for k in ("w_in", "w_hidden"):
        assert torch.equal(tr.bf16[k], sol._tables[k]), k
    for k in ("b_hidden", "w_out", "b_out"):
        assert torch.equal(tr.tables[k], sol._tables[k]), k
    assert torch.equal(tr.bf16["w_in_t"], sol._tables["w_in"].transpose(-1, -2))
    assert torch.equal(tr.bf16["w_hidden_t"], sol._tables["w_hidden"].transpose(-1, -2))
    assert torch.equal(tr.bf16["w_out_t"][..., :16], sol._tables["w_out"].to(torch.bfloat16).transpose(-1, -2))
    assert tr.bf16["w_out_t"][..., 16:].abs().max() == 0


@pytest.mark.gpu
def test_batch_draw_matches_the_oracle_definition():
    tr = _trainer("panda", "small", batch_size=256)
    idx = torch.empty(256, dtype=torch.int64, device=DEV)
    noise = torch.empty((256, 11), device=DEV)
    tr.draw_batch(idx, noise)
    x, cond = OT.training_batch(tr.data_q, tr.data_poses, idx, noise[:, 9], noise[:, :9], noise[:, 10], 9, 8,
                                tr.softflow_noise_scale)
    assert torch.equal(tr.x, x) and torch.equal(tr.cond, cond)
    assert 0.3 < noise[:, 10].mean().item() < 0.7 and 0.3 < noise[:, 9].mean().item() < 0.7
    assert abs(noise[:, :9].std().item() - 1) < 0.1 and idx.max().item() < tr.data_q.shape[0]


@pytest.mark.gpu
def test_determinism_graph_resume_no_sync_and_skipped_steps(tmp_path):
    from cppflow_b200 import ops
    from cppflow_b200.ikflow_training import IkflowTrainer

    a, b = _trainer("panda", batch_size=512), _trainer("panda", batch_size=512)
    g = _trainer("panda", batch_size=512, use_graph=True)
    for t in (a, b, g):
        t.step(6)
    assert torch.equal(a.params_flat, b.params_flat) and torch.equal(a.adam_v, b.adam_v)
    assert torch.equal(a.params_flat, g.params_flat) and torch.equal(a.loss_history(), g.loss_history())
    # save after 6, continue to 12, against a run resumed from the file
    path = str(tmp_path / "ck.pt")
    a.save(path)
    a.step(6)
    r = IkflowTrainer.load(path, device=DEV)
    r.step(6)
    assert torch.equal(a.params_flat, r.params_flat) and torch.equal(a.adam_m, r.adam_m)
    assert torch.equal(a.loss_history(), r.loss_history()) and a.loss_history().numel() == 12
    # no host synchronisation inside a step
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        b.step(3)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    # a batch with a NaN pose: no update, the counter goes to 1
    b.draw_batch()
    b.cond[5, 4] = float("nan")
    before = (b.params_flat.clone(), b.adam_m.clone(), b.adam_v.clone(), b.bf16["w_in"].clone())
    ops.flow_train_step(b.desc, b.x, b.cond, b.workspace, b.loss)
    assert b.steps_skipped.item() == 1 and b.counters[0].item() == 9
    assert torch.equal(before[0], b.params_flat) and torch.equal(before[1], b.adam_m)
    assert torch.equal(before[2], b.adam_v) and torch.equal(before[3], b.bf16["w_in"])


@pytest.mark.gpu
def test_a_short_run_learns_and_both_quaternion_signs_work():
    import time

    from cppflow_b200.ikflow import IkflowSolver
    from cppflow_b200.ikflow_training import sample_dataset
    from cppflow_b200.robot import get_robot

    from cppflow_b200.ikflow_training import IkflowTrainer, sample_errors

    rob = get_robot("panda")
    tr = IkflowTrainer(rob, _params(width=9, nb=4, H=256, L=2), seed=1, batch_size=512, n_data=200000, use_graph=True,
                       device=DEV)
    _, held = sample_dataset(rob, 64, seed=99, device=DEV)
    pos0, _ = sample_errors(tr.solver(), held, 16, 0)
    t0 = time.time()
    tr.step(600)
    torch.cuda.synchronize()
    wall = time.time() - t0
    hist = tr.loss_history().cpu()
    sol = IkflowSolver(rob, tr.params, state_dict=tr.state_dict(), device=DEV)
    pos1, rot1 = sample_errors(sol, held, 16, 0)
    flipped = held.clone()
    flipped[:, 3:] = -flipped[:, 3:]
    pos_f, rot_f = sample_errors(sol, flipped, 16, 0)
    print(f"600 steps in {wall:.1f} s; NLL first 10 {hist[:10].mean():.3f}, last 50 {hist[-50:].mean():.3f}; median "
          f"position error {pos0.median():.4f} m -> {pos1.median():.4f} m (negated quaternions {pos_f.median():.4f} m); "
          f"median rotation error {rot1.median():.4f} rad (negated {rot_f.median():.4f})")
    assert wall < 60
    assert torch.isfinite(hist).all()
    # measured on a B200: NLL 5.7 -> -11.1, median position error 0.81 -> 0.41 m (negated quaternions 0.40 m)
    assert hist[-50:].mean() < hist[:10].mean() - 8.0
    assert pos1.median() < 0.75 * pos0.median()
    assert pos_f.median() < 1.25 * pos1.median() and rot_f.median() < 1.25 * rot1.median()


@pytest.mark.gpu
def test_planner_runs_on_trained_weights():
    """A briefly trained flow plans obstacle-free problems; its samples are still too far off for the obstacle
    problems, where the planner's "< 95 % colliding" check rejects them."""
    from cppflow_b200.data_type_utils import problem_from_filename
    from cppflow_b200.data_types import PlannerSettings
    from cppflow_b200.ikflow import IkflowSolver
    from cppflow_b200.ikflow_training import IkflowTrainer
    from cppflow_b200.planners import CppFlowPlanner, IkflowCandidateGenerator, plan_many
    from cppflow_b200.robot import get_robot

    rob = get_robot("fetch_arm")
    p = _params(width=9, nb=4, H=256, L=2)
    t = IkflowTrainer(rob, p, seed=1, batch_size=512, n_data=200000, use_graph=True, device=DEV)
    t.step(600)
    solver = IkflowSolver(rob, p, state_dict=t.state_dict(), device=DEV)
    settings = dict(k=32, tmax_sec=30.0, anytime_mode_enabled=False, verbosity=0)

    def planner(_problem):
        return CppFlowPlanner(PlannerSettings(**settings), rob, IkflowCandidateGenerator(solver, seed=0))

    problems = [problem_from_filename(None, name, device=DEV) for name in ("fetch_arm__hello", "fetch_arm__rot_yz2")]
    one = planner(problems[0]).generate_plan(problems[0])
    assert one.plan.q_path.shape == (problems[0].n_timesteps, 7) and torch.isfinite(one.plan.q_path).all()
    many = plan_many(planner, problems)
    assert len(many) == 2 and all(torch.isfinite(r.plan.q_path).all() for r in many)
    assert torch.equal(many[0].plan.q_path, one.plan.q_path)
