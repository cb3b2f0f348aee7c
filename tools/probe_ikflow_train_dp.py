"""Data-parallel IKFlow training (IkflowTrainer with a process group) at IKFlow's size (width 9, 12 blocks, hidden
1024, 3 hidden layers per subnet, P = 52.3 M parameters): one process per GPU, NCCL over a file:// rendezvous in a
temporary directory, CUDA events on rank 0.  Reads the card name and power limit in the same run.

  python tools/probe_ikflow_train_dp.py [--gpus 1,2,4,8] [--batches 512,4096] [--reps 20] [--out profiles/r06_....json]

Per (W, per-shard batch B), with M = 1:
  samples_per_s  - W B / step time, IkflowTrainer.step replayed as one CUDA graph (collectives included)
  efficiency     - samples_per_s / (W x samples_per_s at W = 1, same B)
  parts_ms       - one eager step cut by events on rank 0: grad (draw + forward + backward), all_to_all, tree_reduce,
                   all_gather, apply (finite check, Adam, BF16 tables)
  all_reduce_ms  - for comparison only: an NCCL all_reduce (sum) of the same padded vector, whose summation order
                   is NCCL's; the difference to all_to_all + tree_reduce + all_gather is the price of the fixed order
  tree_reduce_gb_s - bytes the reduction moves (W + 1 slices of P / W floats) over its time
W values above the GPU count are skipped.  tree_reduce_kernel: cppflow_flow_grad_tree_reduce alone on cuda:0 at this
P, for the cross-rank shapes (n = W slices of P / W floats) and the local merge of two micro-batch gradients (n = 2
slices of P), in GB/s of bytes read and written, beside a device-to-device copy of P floats."""
import argparse
import datetime
import json
import os
import sys
import tempfile

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tools"))
from probe_ikflow import card  # noqa: E402


def worker(rank, W, batches, reps, rendezvous, out):
    import torch.distributed as dist

    from cppflow_b200 import ops
    from cppflow_b200.ikflow import IkflowModelParameters
    from cppflow_b200.ikflow_training import IkflowTrainer
    from cppflow_b200.robot import get_robot

    dev = f"cuda:{rank}"
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", init_method=f"file://{rendezvous}", rank=rank, world_size=W,
                            timeout=datetime.timedelta(minutes=10), device_id=torch.device(dev))
    try:
        p = IkflowModelParameters(nb_nodes=12, dim_latent_space=9, coeff_fn_config=3, coeff_fn_internal_size=1024)
        rows = []
        for B in batches:
            tr = IkflowTrainer(get_robot("panda"), p, seed=0, batch_size=B, n_data=200_000, use_graph=True, device=dev,
                               process_group=dist.group.WORLD)
            tr.step(3)  # eager step, capture, one replay
            torch.cuda.synchronize()
            dist.barrier()
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            ev[0].record()
            tr.step(reps)
            ev[1].record()
            torch.cuda.synchronize()
            step_ms = ev[0].elapsed_time(ev[1]) / reps
            # one eager step cut into its parts
            P, chunk = tr._P, tr._Ppad // W
            names = ["grad", "all_to_all", "tree_reduce", "all_gather", "apply"]
            acc = dict.fromkeys(names, 0.0)
            for _ in range(reps):
                e = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
                dist.barrier()
                e[0].record()
                tr._draw_shard(0)
                buf = tr._stack[0]
                ops.flow_train_step(tr.desc, tr.x, tr.cond, tr.workspace, buf[P:P + 1], buf[:P], update=False)
                e[1].record()
                mine = tr._G[rank * chunk:(rank + 1) * chunk]
                if W > 1:
                    dist.all_to_all_single(tr._recv.view(-1), buf, group=tr.group)
                    e[2].record()
                    ops.flow_grad_tree_reduce(tr._recv, mine, 1.0 / W)
                    e[3].record()
                    dist.all_gather_into_tensor(tr._G, mine, group=tr.group)
                else:
                    e[2].record()
                    ops.flow_grad_tree_reduce(buf.view(1, -1), tr._G, 1.0)
                    e[3].record()
                e[4].record()
                ops.flow_train_apply(tr.desc, tr._G, B, tr.workspace)
                e[5].record()
                torch.cuda.synchronize()
                for k, name in enumerate(names):
                    acc[name] += e[k].elapsed_time(e[k + 1]) / reps
            vec = torch.zeros(tr._Ppad, device=dev)
            dist.all_reduce(vec)
            torch.cuda.synchronize()
            dist.barrier()
            a = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            a[0].record()
            for _ in range(reps):
                dist.all_reduce(vec)
            a[1].record()
            torch.cuda.synchronize()
            ar_ms = a[0].elapsed_time(a[1]) / reps
            moved = (W + 1) * chunk * 4
            rows.append({"gpus": W, "batch": B, "params": P, "padded": tr._Ppad, "step_ms": step_ms,
                         "samples_per_s": W * B / step_ms * 1e3, "parts_ms": acc, "all_reduce_ms": ar_ms,
                         "tree_reduce_gb_s": moved / acc["tree_reduce"] / 1e6 if acc["tree_reduce"] > 0 else None,
                         "exchange_share": (acc["all_to_all"] + acc["tree_reduce"] + acc["all_gather"]) / sum(acc.values())})
            del tr, vec
            torch.cuda.empty_cache()
        if rank == 0:
            with open(out, "w") as f:
                json.dump(rows, f)
    finally:
        dist.destroy_process_group()


def tree_reduce_rows(P_pad, reps):
    from cppflow_b200 import ops

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        e[0].record()
        for _ in range(reps):
            fn()
        e[1].record()
        torch.cuda.synchronize()
        return e[0].elapsed_time(e[1]) / reps

    src = torch.randn(2 * P_pad, device="cuda:0")
    dst = torch.empty(P_pad, device="cuda:0")
    copy_ms = timed(lambda: dst.copy_(src[:P_pad]))
    rows = [{"what": "copy", "floats": P_pad, "ms": copy_ms, "gb_s": 2 * P_pad * 4 / copy_ms / 1e6}]
    for n, length in ((1, P_pad), (2, P_pad // 2), (4, P_pad // 4), (8, P_pad // 8), (2, P_pad)):
        slices = src[: n * length].view(n, length)
        ms = timed(lambda: ops.flow_grad_tree_reduce(slices, dst[:length], 0.5))
        rows.append({"what": "local merge" if n * length > P_pad else f"cross-rank W={n}", "n": n, "len": length,
                     "ms": ms, "gb_s": (n + 1) * length * 4 / ms / 1e6})
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--gpus", default="1,2,4,8")
    ap.add_argument("--batches", default="512,4096")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the probe measures on the GPU"
    import torch.multiprocessing as mp

    batches = [int(b) for b in args.batches.split(",")]
    res = {"card": card(), "device_count": torch.cuda.device_count(),
           "network": "width 9, nb_nodes 12, hidden 1024, coeff_fn_config 3", "micro_batches": 1, "rows": [],
           "skipped_gpus": []}
    res["tree_reduce_kernel"] = tree_reduce_rows(-(-(52_371_840 + 1) // 512) * 512, args.reps)  # P + 1 at IKFlow size, padded for W = 8
    for row in res["tree_reduce_kernel"]:
        print(json.dumps(row), flush=True)
    base = {}
    for W in (int(w) for w in args.gpus.split(",")):
        if W > torch.cuda.device_count():
            res["skipped_gpus"].append(W)
            continue
        with tempfile.TemporaryDirectory() as tmp:
            out = os.path.join(tmp, "rows.json")
            mp.spawn(worker, args=(W, batches, args.reps, os.path.join(tmp, "store"), out), nprocs=W, join=True)
            with open(out) as f:
                rows = json.load(f)
        for row in rows:
            if W == 1:
                base[row["batch"]] = row["samples_per_s"]
            if row["batch"] in base:
                row["efficiency"] = row["samples_per_s"] / (W * base[row["batch"]])
            print(json.dumps(row), flush=True)
            res["rows"].append(row)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res["card"]), "devices:", res["device_count"])


if __name__ == "__main__":
    main()
