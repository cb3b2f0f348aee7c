"""Train IKFlow for one robot on one or several GPUs (cppflow_b200/ikflow_training.py) and print one JSON line every
--every steps:
the mean NLL of those steps and the accuracy of the flow as an IK sampler at a fixed set of held-out poses (--k
reverse-pass samples with z ~ N(0, 1) per pose; mean and median position and rotation error of their forward
kinematics), and the share of those poses that IkflowSolver.generate_exact_ik_solutions solves with its defaults
(exact_ik_success: 1 mm and 0.01 rad after LM refinement, rounds of 1, 3 and 10 samples per unsolved pose).

    python tools/train_ikflow.py --robot panda --minutes 30 --out runs/panda.ckpt --state_dict runs/panda_sd.pt
    python tools/train_ikflow.py --resume runs/panda.ckpt --steps 10000 --out runs/panda.ckpt
    python tools/train_ikflow.py --gpus 8 --batch 4096 --minutes 6 --out runs/panda8.ckpt

--gpus N trains data-parallel on cuda:0 ... cuda:N-1 (N a power of two), one process per GPU joined over a file://
rendezvous in the directory of --out (of the working directory without --out); --micro_batches M (a power of two)
sums M shards per GPU and step.  A step then takes N x M shards of --batch rows (--batch stays per shard, and the
learning rate is not rescaled); the weights are those of one GPU at --micro_batches N x M, bit for bit, and a
checkpoint resumes on any N, M with the same product.  Rank 0 prints the reports and writes the files.

--out is a trainer checkpoint (weights, Adam moments, counters; --resume continues it bit for bit), written at every
report and at the end.  --state_dict is the GraphINN state dict that IkflowSolver, IkflowCandidateGenerator and
tools/evaluate.py --ikflow_checkpoint load.  Nothing else is written."""
import argparse
import datetime
import json
import os
import sys
import tempfile
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cppflow_b200.ikflow import IkflowModelParameters  # noqa: E402
from cppflow_b200.ikflow_training import IkflowTrainer, sample_accuracy, sample_dataset  # noqa: E402
from cppflow_b200.robot import get_robot  # noqa: E402


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--robot", default="panda", choices=["fetch", "fetch_arm", "panda"])
    ap.add_argument("--minutes", type=float, default=None, help="wall-time budget of the training loop")
    ap.add_argument("--steps", type=int, default=None, help="steps to take (with --minutes: whichever ends first)")
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--lr", type=float, default=5e-4)
    ap.add_argument("--nb_nodes", type=int, default=12)
    ap.add_argument("--hidden", type=int, default=1024)
    ap.add_argument("--layers", type=int, default=3)
    ap.add_argument("--width", type=int, default=9)
    ap.add_argument("--n_data", type=int, default=2_500_000)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--every", type=int, default=1000, help="steps between two reports")
    ap.add_argument("--held_out", type=int, default=256, help="held-out poses of the accuracy report")
    ap.add_argument("--k", type=int, default=16, help="samples per held-out pose")
    ap.add_argument("--no_graph", action="store_true", help="launch every step instead of replaying a CUDA graph")
    ap.add_argument("--out", default=None, help="trainer checkpoint to write")
    ap.add_argument("--state_dict", default=None, help="GraphINN state dict to write at the end")
    ap.add_argument("--resume", default=None, help="trainer checkpoint to continue")
    ap.add_argument("--device", default="cuda:0", help="the GPU of a one-GPU run")
    ap.add_argument("--gpus", type=int, default=1, help="data-parallel ranks, one per GPU (a power of two)")
    ap.add_argument("--micro_batches", type=int, default=None,
                    help="shards per GPU and step (a power of two; default 1, on --resume the checkpoint's shards / --gpus)")
    args = ap.parse_args(argv)
    if args.minutes is None and args.steps is None:
        ap.error("give --minutes or --steps")
    if args.gpus < 1 or args.gpus & (args.gpus - 1):
        ap.error(f"--gpus {args.gpus} is not a power of two")
    if args.gpus == 1:
        train(0, args, None)
        return
    import torch.multiprocessing as mp

    if torch.cuda.device_count() < args.gpus:
        ap.error(f"--gpus {args.gpus}: {torch.cuda.device_count()} GPUs present")
    where = os.path.dirname(os.path.abspath(args.out)) if args.out else os.getcwd()
    os.makedirs(where, exist_ok=True)
    with tempfile.TemporaryDirectory(dir=where, prefix=".rendezvous_") as tmp:
        mp.spawn(train, args=(args, os.path.join(tmp, "store")), nprocs=args.gpus, join=True)


def train(rank, args, rendezvous):
    """The training loop of one rank (rendezvous None: one GPU, args.device)."""
    group, device = None, args.device
    if rendezvous is not None:
        import torch.distributed as dist

        device = f"cuda:{rank}"
        torch.cuda.set_device(device)
        dist.init_process_group("nccl", init_method=f"file://{rendezvous}", rank=rank, world_size=args.gpus,
                                timeout=datetime.timedelta(minutes=10), device_id=torch.device(device))
        group = dist.group.WORLD
    try:
        loop(args, group, device, rank == 0)
    finally:
        if group is not None:
            dist.destroy_process_group()


def loop(args, group, device, main_rank):
    if args.resume:
        tr = IkflowTrainer.load(args.resume, use_graph=not args.no_graph, device=device, process_group=group,
                                micro_batches=args.micro_batches)
    else:
        p = IkflowModelParameters(nb_nodes=args.nb_nodes, dim_latent_space=args.width, coeff_fn_config=args.layers,
                                  coeff_fn_internal_size=args.hidden)
        tr = IkflowTrainer(get_robot(args.robot), p, seed=args.seed, batch_size=args.batch, lr=args.lr,
                           n_data=args.n_data, use_graph=not args.no_graph, device=device, process_group=group,
                           micro_batches=args.micro_batches or 1)
    _, held = sample_dataset(tr.robot, args.held_out, seed=1_000_003, device=tr.device)
    held = held[: args.held_out]

    def report(t_loop):
        if not main_rank:
            return
        hist = tr.loss_history()
        taken = int(tr.counters[2].item())
        solver = tr.solver()
        recent = hist[-min(args.every, hist.numel()):] if hist.numel() else hist
        line = {"step": taken, "samples": taken * tr.shards * tr.batch_size, "gpus": tr.world,
                "micro_batches": tr.micro_batches, "train_seconds": round(t_loop, 2),
                "nll": recent.mean().item() if recent.numel() else None,
                "skipped": int(tr.counters[1].item()), **sample_accuracy(solver, held, args.k),
                "exact_ik_success": solver.generate_exact_ik_solutions(held)[1].float().mean().item()}
        print(json.dumps(line), flush=True)
        if args.out:
            tr.save(args.out)

    report(0.0)
    deadline = None if args.minutes is None else args.minutes * 60
    done, t_loop = 0, 0.0
    while True:
        over = (args.steps is not None and done >= args.steps) or (deadline is not None and t_loop >= deadline)
        n = 0 if over else args.every if args.steps is None else min(args.every, args.steps - done)
        if group is not None:  # rank 0's clock decides, so that every rank takes the same steps
            import torch.distributed as dist

            go = torch.tensor([n], device=tr.device)
            dist.broadcast(go, 0, group=group)
            n = int(go.item())
        if n == 0:
            break
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        tr.step(n)
        torch.cuda.synchronize()
        t_loop += time.perf_counter() - t0
        done += n
        report(t_loop)
    if args.state_dict and main_rank:
        torch.save(tr.state_dict(), args.state_dict)


if __name__ == "__main__":
    main()
