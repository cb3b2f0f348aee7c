"""Exact IK from IKFlow's samples (IkflowSolver.generate_exact_ik_solutions, csrc/k_ik.cu) for 10^4, 10^5 and 10^6
Panda and Fetch targets: solutions per second and success rate, against the same rounds run with one LM launch per
step.  One process: reads the card name and power limit, warms up every shape, then times.

  python tools/probe_ik_exact.py [--out profiles/r05_ik_exact_probe.json] [--sizes 10000 100000 1000000]
                                 [--checkpoint panda_sd.pt]

Targets are poses from the forward kinematics of uniform in-limit configurations (seeded).  The flow is an IKFlow-size
network (12 blocks, hidden 1024, three layers per subnet) with random weights, and with --checkpoint a trained
GraphINN state dict for the robot it was trained on.  Defaults of generate_exact_ik_solutions: 1 mm and 0.01 rad,
rounds of 1, 3 and 10 samples per unsolved target, up to 20 LM steps per sample.
  fused    - generate_exact_ik_solutions: per round ik_round_inputs, the reverse pass, ONE ik_refine launch (per-row
             early exit) and ik_select; the host reads the unsolved count once per round
  unfused  - the same latents and reverse pass, then ops.lm_pose_steps_ (cppflow_lm_pose_steps: one launch per step,
             every row takes every step), the FP32 error check and the selection in torch
Both are timed by the host clock around a call that ends in a device synchronisation.  The refinement alone is timed
with CUDA events: ik_refine with and without early exit against cppflow_lm_pose_steps over the same 20 steps, on the
reverse-pass samples of one round-0 launch."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # the probe still runs; the note says the limit is unknown
        q = f"unavailable ({e})"
    return {"name": name, "power_limit_and_max_sm_clock": q}


def wall(fn, reps):
    """Mean host time of fn() over reps calls after one warm-up call; every call ends in a device synchronisation."""
    out = fn()
    torch.cuda.synchronize()
    t = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        t.append(time.perf_counter() - t0)
    return sum(t) / len(t), out


def events(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def unfused(solver, poses, lambdas, prm, pos_tol=1e-3, rot_tol=1e-2, repeat_counts=(1, 3, 10), seed=0):
    """The rounds of generate_exact_ik_solutions with cppflow_lm_pose_steps (every row takes every step) and torch
    selection."""
    from cppflow_b200 import ops

    rob, D = solver.robot, solver.robot.ndof
    m = poses.shape[0]
    sol = torch.zeros((m, D), device=poses.device)
    valid = torch.zeros((m,), device=poses.device, dtype=torch.bool)
    unsolved = torch.arange(m, device=poses.device, dtype=torch.int32)
    for r, rep in enumerate(repeat_counts):
        if unsolved.numel() == 0:
            break
        z, cond = ops.ik_round_inputs(unsolved, rep, poses, seed, r, solver.network_width)
        x = solver.run(z, cond, True, True)[:, :D].contiguous()
        ops.lm_pose_steps_(rob.robot_id, D, prm, lambdas, x, cond, True)
        e, _ = ops.pose_errors(rob.robot_id, D, x, cond)
        ok = ((e[:, 3:].norm(dim=1) < pos_tol) & (e[:, :3].norm(dim=1) < rot_tol)).reshape(-1, rep)
        found = ok.any(dim=1)
        pick = torch.where(found, ok.to(torch.int64).argmax(dim=1), 0)
        rows = torch.arange(unsolved.numel(), device=poses.device) * rep + pick
        sol[unsolved.long()] = x[rows]
        valid[unsolved.long()] = found
        unsolved = unsolved[~found]  # the host learns the count here, as in the fused path
    return sol, valid


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
    ap.add_argument("--sizes", type=int, nargs="+", default=[10_000, 100_000, 1_000_000])
    ap.add_argument("--robots", nargs="+", default=["panda", "fetch"])
    ap.add_argument("--checkpoint", default=None, help="a trained GraphINN state dict (its robot is measured too)")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the probe measures on the GPU"
    from cppflow_b200 import ops
    from cppflow_b200.ikflow import IkflowSolver, params_from_state_dict
    from cppflow_b200.lm_hyper_parameters import ALT_LOSS_V2_1_POSE
    from cppflow_b200.planners import LmIkCandidateGenerator
    from cppflow_b200.robot import get_robot

    dev = "cuda:0"
    lambdas = LmIkCandidateGenerator.LAMBDAS
    prm = ops.make_params(ALT_LOSS_V2_1_POSE)
    res = {"card": card(), "exact_ik": [], "refine": []}
    flows = [(name, "random", IkflowSolver(get_robot(name), seed=0, device=dev)) for name in args.robots]
    if args.checkpoint:
        sd = torch.load(args.checkpoint, map_location="cpu")
        for name in ("panda", "fetch", "fetch_arm"):
            rob = get_robot(name)
            m = torch.tensor([1.0 / max(abs(lo), abs(hi)) for lo, hi in rob.actuated_joints_limits])
            diag = torch.diagonal(sd["module_list.0.M"]).float()
            if diag.numel() >= rob.ndof and torch.allclose(diag[: rob.ndof], m, rtol=1e-5):
                flows.append((name, "checkpoint", IkflowSolver(rob, params_from_state_dict(sd), state_dict=sd, device=dev)))
                break
    for name, weights, solver in flows:
        rob = solver.robot
        for m in args.sizes:
            g = torch.Generator().manual_seed(m)
            lim = torch.tensor(rob.actuated_joints_limits)
            q = (lim[:, 0] + (lim[:, 1] - lim[:, 0]) * torch.rand((m, rob.ndof), generator=g)).to(dev)
            poses = ops.forward_kinematics(rob.robot_id, rob.ndof, q)
            t_f, (_, valid_f) = wall(lambda: solver.generate_exact_ik_solutions(poses), args.reps)
            t_u, (_, valid_u) = wall(lambda: unfused(solver, poses, lambdas, prm), args.reps)
            row = {"robot": name, "weights": weights, "targets": m,
                   "fused": {"s": t_f, "success": valid_f.float().mean().item(),
                             "solutions_per_s": valid_f.sum().item() / t_f},
                   "unfused": {"s": t_u, "success": valid_u.float().mean().item(),
                               "solutions_per_s": valid_u.sum().item() / t_u},
                   "speedup": t_u / t_f}
            res["exact_ik"].append(row)
            print(json.dumps(row), flush=True)

            # the refinement alone, on the round-0 reverse-pass samples of these targets
            z, cond = ops.ik_round_inputs(torch.arange(m, device=dev, dtype=torch.int32), 1, poses, 0, 0,
                                          solver.network_width)
            x0 = solver.run(z, cond, True, True)[:, : rob.ndof].contiguous()
            x = torch.empty_like(x0)
            d_early = ops.ik_refine_desc(lambdas, 1e-3, 1e-2, prm)
            d_all = ops.ik_refine_desc(lambdas, 1e-3, 1e-2, prm, early_exit=False)
            reps = max(3, 10 * args.reps * 100_000 // m)

            def steps_():
                x.copy_(x0)
                ops.lm_pose_steps_(rob.robot_id, rob.ndof, prm, lambdas, x, cond, True)

            def copy_only():
                x.copy_(x0)

            t_copy = events(copy_only, reps)
            t_steps = events(steps_, reps) - t_copy
            t_all = events(lambda: ops.ik_refine(rob.robot_id, rob.ndof, d_all, x0, cond, out=x), reps)
            t_early = events(lambda: ops.ik_refine(rob.robot_id, rob.ndof, d_early, x0, cond, out=x), reps)
            _, st, taken = ops.ik_refine(rob.robot_id, rob.ndof, d_early, x0, cond)
            row = {"robot": name, "weights": weights, "rows": m, "steps": len(lambdas),
                   "ms": {"lm_pose_steps": t_steps, "ik_refine_no_early_exit": t_all, "ik_refine": t_early},
                   "mean_steps_taken": taken.float().mean().item(), "converged": st.float().mean().item(),
                   "speedup_no_early_exit": t_steps / t_all, "speedup": t_steps / t_early}
            res["refine"].append(row)
            print(json.dumps(row), flush=True)
            del q, poses, z, cond, x0, x
            torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
