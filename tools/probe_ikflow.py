"""IKFlow reverse pass on the CUDA path (csrc/k_flow.cu) against the same network run by torch, and a full plan with
the mock flow.  One process: reads the card name and power limit, warms up every shape, then times with CUDA events.

  python tools/probe_ikflow.py [--out profiles/r03_ikflow_probe.json] [--reps 10]

Reverse pass at N = 175 x T rows (T of fetch__circle), nb_nodes 12, hidden 1024, coeff_fn_config 1, 2, 3:
  cuda  - cppflow_flow_run (tcgen05 BF16 tensor-core layers, FP32 coupling arithmetic)
  fp32  - oracle/ikflow.py's module in fp32 (the reference's arithmetic; torch's default, TF32 off)
  bf16  - the same module converted to bfloat16
FLOPs are counted from the shapes (2 per multiply-add of every Linear); the share of peak is against the 2,250 TFLOP/s
dense BF16 data-sheet figure of one B200."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

PEAK_BF16 = 2250e12
L2_BYTES = 126e6


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # the probe still runs; the note says the limit is unknown
        q = f"unavailable ({e})"
    return {"name": name, "power_limit_and_max_sm_clock": q}


def flops_per_row(p, dim_cond):
    W, H, L = p.dim_latent_space, p.coeff_fn_internal_size, p.coeff_fn_config
    len1, len2 = W // 2, W - W // 2
    per = 0
    for c_in, c_out in ((len1 + dim_cond, 2 * len2), (len2 + dim_cond, 2 * len1)):
        per += 2 * (c_in * H + (L - 1) * H * H + H * c_out)
    return per * p.nb_nodes


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        fn()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the probe measures on the GPU"
    from cppflow_b200.data_type_utils import problem_from_filename
    from cppflow_b200.data_types import PlannerSettings
    from cppflow_b200.ikflow import IkflowModelParameters, IkflowSolver
    from cppflow_b200.planners import CppFlowPlanner, IkflowCandidateGenerator
    from oracle import ikflow as OF

    dev = "cuda:0"
    res = {"card": card(), "reverse": [], "plan": None}
    problem = problem_from_filename(None, "fetch__circle", device=dev)
    rob, T, k = problem.robot, problem.n_timesteps, 175
    n = k * T
    res["n_rows"] = n
    g = torch.Generator().manual_seed(0)
    for L in (1, 2, 3):
        p = IkflowModelParameters(nb_nodes=12, dim_latent_space=9, coeff_fn_config=L, coeff_fn_internal_size=1024)
        solver = IkflowSolver(rob, p, seed=0, device=dev)
        net = OF.Glow(rob.actuated_joints_limits, 9, 12, 1024, L, p.rnvp_clamp).to(dev)
        net.load_state_dict(solver.state_dict)
        z = (torch.rand((n, 9), generator=g) * 2 - 1).to(dev)
        cond = problem.target_path.repeat(k, 1).contiguous()
        with torch.no_grad():
            t_cuda = timed(lambda: solver.run(z, problem.target_path, True), args.reps)
            t_fp32 = timed(lambda: net(z, cond, rev=True), args.reps)
            net_bf = net.to(torch.bfloat16)
            zb, cb = z.to(torch.bfloat16), cond.to(torch.bfloat16)
            t_bf16 = timed(lambda: net_bf(zb, cb, rev=True), args.reps)
            err = (solver.run(z, problem.target_path, True).double()
                   - net.float()(z, cond, rev=True).double()).abs().max().item()
        fl = flops_per_row(p, solver.dim_cond) * n
        act = n * 1024 * 2
        row = {"coeff_fn_config": L, "gflop": fl / 1e9,
               "ms": {"cuda": t_cuda, "torch_fp32": t_fp32, "torch_bf16": t_bf16},
               "tflops": {"cuda": fl / t_cuda / 1e9, "torch_fp32": fl / t_fp32 / 1e9, "torch_bf16": fl / t_bf16 / 1e9},
               "share_of_bf16_peak": {"cuda": fl / t_cuda / 1e-3 / PEAK_BF16},
               "speedup": {"vs_torch_fp32": t_fp32 / t_cuda, "vs_torch_bf16": t_bf16 / t_cuda},
               "max_abs_diff_vs_torch_fp32": err,
               "hidden_activation_mb": act / 1e6,
               "layer_in_plus_out_fits_l2": 2 * act < L2_BYTES}
        res["reverse"].append(row)
        print(json.dumps(row), flush=True)
        del solver, net, net_bf
        torch.cuda.empty_cache()

    # full plan with the mock flow (default IkflowModelParameters: 12 x 1024 x 3, width 9)
    solver = IkflowSolver(rob, seed=0, device=dev)
    def plan():
        planner = CppFlowPlanner(PlannerSettings(k=k, tmax_sec=30.0, anytime_mode_enabled=False, verbosity=0), rob,
                                 IkflowCandidateGenerator(solver, seed=0))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = planner.generate_plan(problem)
        torch.cuda.synchronize()
        return r, time.perf_counter() - t0
    plan()
    runs = [plan() for _ in range(3)]
    res["plan"] = {"problem": "fetch__circle", "k": k, "T": T,
                   "td_ikflow_ms": [r.timing.ikflow * 1e3 for r, _ in runs],
                   "td_total_ms": [r.timing.total * 1e3 for r, _ in runs],
                   "wall_ms": [w * 1e3 for _, w in runs],
                   "is_valid": [bool(r.plan.is_valid) for r, _ in runs]}
    print(json.dumps(res["plan"]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
