"""Train IKFlow for one robot on one GPU (cppflow_b200/ikflow_training.py) and print one JSON line every --every steps:
the mean NLL of those steps and the accuracy of the flow as an IK sampler at a fixed set of held-out poses (--k
reverse-pass samples with z ~ N(0, 1) per pose; mean and median position and rotation error of their forward
kinematics), and the share of those poses that IkflowSolver.generate_exact_ik_solutions solves with its defaults
(exact_ik_success: 1 mm and 0.01 rad after LM refinement, rounds of 1, 3 and 10 samples per unsolved pose).

    python tools/train_ikflow.py --robot panda --minutes 30 --out runs/panda.ckpt --state_dict runs/panda_sd.pt
    python tools/train_ikflow.py --resume runs/panda.ckpt --steps 10000 --out runs/panda.ckpt

--out is a trainer checkpoint (weights, Adam moments, counters; --resume continues it bit for bit), written at every
report and at the end.  --state_dict is the GraphINN state dict that IkflowSolver, IkflowCandidateGenerator and
tools/evaluate.py --ikflow_checkpoint load.  Nothing else is written."""
import argparse
import json
import os
import sys
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
    ap.add_argument("--device", default="cuda:0")
    args = ap.parse_args(argv)
    if args.minutes is None and args.steps is None:
        ap.error("give --minutes or --steps")
    if args.resume:
        tr = IkflowTrainer.load(args.resume, use_graph=not args.no_graph, device=args.device)
    else:
        p = IkflowModelParameters(nb_nodes=args.nb_nodes, dim_latent_space=args.width, coeff_fn_config=args.layers,
                                  coeff_fn_internal_size=args.hidden)
        tr = IkflowTrainer(get_robot(args.robot), p, seed=args.seed, batch_size=args.batch, lr=args.lr,
                           n_data=args.n_data, use_graph=not args.no_graph, device=args.device)
    _, held = sample_dataset(tr.robot, args.held_out, seed=1_000_003, device=tr.device)
    held = held[: args.held_out]

    def report(t_loop):
        hist = tr.loss_history()
        taken = int(tr.counters[2].item())
        solver = tr.solver()
        recent = hist[-min(args.every, hist.numel()):] if hist.numel() else hist
        line = {"step": taken, "samples": taken * tr.batch_size, "train_seconds": round(t_loop, 2),
                "nll": recent.mean().item() if recent.numel() else None,
                "skipped": int(tr.counters[1].item()), **sample_accuracy(solver, held, args.k),
                "exact_ik_success": solver.generate_exact_ik_solutions(held)[1].float().mean().item()}
        print(json.dumps(line), flush=True)
        if args.out:
            tr.save(args.out)

    report(0.0)
    deadline = None if args.minutes is None else args.minutes * 60
    done, t_loop = 0, 0.0
    while (args.steps is None or done < args.steps) and (deadline is None or t_loop < deadline):
        n = args.every if args.steps is None else min(args.every, args.steps - done)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        tr.step(n)
        torch.cuda.synchronize()
        t_loop += time.perf_counter() - t0
        done += n
        report(t_loop)
    if args.state_dict:
        torch.save(tr.state_dict(), args.state_dict)


if __name__ == "__main__":
    main()
