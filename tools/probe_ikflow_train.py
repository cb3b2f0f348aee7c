"""Throughput of one IKFlow training step (csrc/k_flow_train.cu) against torch autograd + torch.optim.Adam on
oracle/ikflow.py's module with oracle/ikflow_train.py's loss, at IKFlow's size (width 9, 12 blocks, hidden 1024, 3
hidden layers per subnet).  One process: reads the card name and power limit, warms up every shape, then times with
CUDA events.

  python tools/probe_ikflow_train.py [--out profiles/r04_ikflow_train_probe.json] [--reps 20] [--batches 512,4096,32768]

Per batch size, samples per second of
  cuda       - IkflowTrainer.step, replayed as one CUDA graph (batch draw + forward + loss + backward + Adam)
  cuda_eager - the same two library calls launched every step
  torch_fp32 - forward_with_logdet + nll, backward, Adam (fp32, TF32 off)
  torch_bf16 - the same under torch.autocast(bfloat16)
The torch rows train on one fixed batch (their batch draw is not timed).  FLOPs are counted from the shapes: three
times the forward pass's multiply-adds (forward, input gradients, weight gradients), 2 FLOPs each."""
import argparse
import json
import os
import sys

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tools"))
from probe_ikflow import card, flops_per_row  # noqa: E402


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
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--batches", default="512,4096,32768")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the probe measures on the GPU"
    from cppflow_b200.ikflow import IkflowModelParameters
    from cppflow_b200.ikflow_training import IkflowTrainer
    from cppflow_b200.robot import get_robot
    from oracle import ikflow as OF, ikflow_train as OT

    torch.backends.cuda.matmul.allow_tf32 = False
    dev = "cuda:0"
    rob = get_robot("panda")
    p = IkflowModelParameters(nb_nodes=12, dim_latent_space=9, coeff_fn_config=3, coeff_fn_internal_size=1024)
    res = {"card": card(), "network": "width 9, nb_nodes 12, hidden 1024, coeff_fn_config 3", "rows": []}
    for B in (int(b) for b in args.batches.split(",")):
        fl = 3 * flops_per_row(p, 8) * B
        row = {"batch": B, "gflop_per_step": fl / 1e9, "ms": {}}
        for name, graph in (("cuda", True), ("cuda_eager", False)):
            tr = IkflowTrainer(rob, p, seed=0, batch_size=B, n_data=200_000, use_graph=graph, device=dev)
            tr.step(2)  # first launch, graph capture
            row["ms"][name] = timed(lambda: tr.step(1), args.reps)
            x, cond = tr.x.clone(), tr.cond.clone()
            del tr
            torch.cuda.empty_cache()
        for name, autocast in (("torch_fp32", False), ("torch_bf16", True)):
            net = OF.random_glow(rob.actuated_joints_limits, 9, 12, 1024, 3, seed=0).to(dev)
            opt = torch.optim.Adam(net.parameters(), lr=5e-4, weight_decay=1.8e-5)

            def step():
                opt.zero_grad(set_to_none=True)
                with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
                    loss = OT.nll(*OT.forward_with_logdet(net, x, cond))
                loss.backward()
                opt.step()

            row["ms"][name] = timed(step, args.reps)
            del net, opt
            torch.cuda.empty_cache()
        row["samples_per_s"] = {k: B / v * 1e3 for k, v in row["ms"].items()}
        row["tflops"] = {k: fl / v / 1e9 for k, v in row["ms"].items()}
        row["speedup_vs_torch_bf16"] = row["ms"]["torch_bf16"] / row["ms"]["cuda"]
        row["speedup_vs_torch_fp32"] = row["ms"]["torch_fp32"] / row["ms"]["cuda"]
        res["rows"].append(row)
        print(json.dumps(row), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
