"""Single-problem / all-problems CLI in the spirit of the reference's scripts/evaluate.py: run a planner on benchmark
problems and print one row per problem with the reference's column names (scripts/evaluate.py:32-50; no pandas, no
visualisation, no results directory).

    python tools/evaluate.py --planner CppFlow --problem fetch_arm__circle
    python tools/evaluate.py --planner CppFlow --all
    python tools/evaluate.py --planner PlannerSearcher --problem panda__1cube --k 64
    python tools/evaluate.py --problem_file my_problem.yaml            # a problem yaml in the reference's layout
    python tools/evaluate.py --all --ikflow_checkpoint panda_sd.pt     # candidates from a trained IKFlow

--ikflow_checkpoint takes a GraphINN state dict (tools/train_ikflow.py --state_dict, or an IKFlow checkpoint's); the
planner then draws its candidates with IkflowCandidateGenerator.  The network's shape is read from the state dict,
and problems of robots whose joint scale differs from the state dict's are skipped.

Errors come from plan_from_qpath (FK of the returned path against the target path); the validity flag is the
capsule-model one (the reference's klampt mesh check is out of scope)."""
import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cppflow_b200.data_type_utils import ALL_PROBLEM_FILENAMES, plan_from_qpath, problem_from_filename  # noqa: E402
from cppflow_b200.data_types import Constraints, PlannerSettings  # noqa: E402
from cppflow_b200.ikflow import IkflowSolver, params_from_state_dict  # noqa: E402
from cppflow_b200.planners import CppFlowPlanner, IkflowCandidateGenerator, PlannerSearcher  # noqa: E402

PLANNERS = {"CppFlow": CppFlowPlanner, "PlannerSearcher": PlannerSearcher}
COLUMNS = ["Problem", "Robot", "Planner", "Valid plan", "time, total (s)", "time, ikflow (s)", "time, coll_checking (s)",
           "time, batch_opt (s)", "time, dp_search (s)", "time, optimizer (s)", "time per opt. step (s)",
           "Max positional error (mm)", "Max rotational error (deg)", "Mean positional error (mm)",
           "Mean rotational error (deg)", "Mjac - prismatic (cm)", "Mjac - revolute (deg)"]
CONSTRAINTS = Constraints(max_allowed_position_error_cm=0.01, max_allowed_rotation_error_deg=0.1, max_allowed_mjac_deg=7.0,
                          max_allowed_mjac_cm=2.0)  # scripts/evaluate.py:51-56


def evaluate(planner_name: str, problem, settings: PlannerSettings, warmup: bool = True, generator=None):
    planner = (PLANNERS[planner_name](settings, problem.robot) if generator is None else
               PLANNERS[planner_name](settings, problem.robot, generator))
    if warmup:
        planner.generate_plan(problem)  # first call: kernel attributes, workspaces
    torch.cuda.synchronize()
    result = planner.generate_plan(problem)
    plan = plan_from_qpath(result.plan.q_path, problem)
    steps = max(1, int(result.debug_info.get("n_optimization_steps", 1)))
    t = result.timing
    r = 5
    return [problem.fancy_name, problem.robot.name, planner.name, f"`{str(bool(result.plan.is_valid)).lower()}`",
            round(t.total, 4), round(t.ikflow, 4), round(t.coll_checking, 4), round(t.batch_opt, 4), round(t.dp_search, 4),
            round(t.optimizer, 4), round(t.optimizer / steps, 5), round(plan.max_positional_error_mm, r),
            round(plan.max_rotational_error_deg, r), round(plan.mean_positional_error_mm, r),
            round(plan.mean_rotational_error_deg, r), round(plan.mjac_cm, r), round(plan.mjac_deg, r)], bool(result.plan.is_valid)


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--planner", default="CppFlow", choices=sorted(PLANNERS))
    ap.add_argument("--problem", default=None, help="one of " + ", ".join(ALL_PROBLEM_FILENAMES))
    ap.add_argument("--problem_file", default=None, help="a problem yaml in the reference's layout (problems/*.yaml)")
    ap.add_argument("--all", action="store_true", help="the 13 benchmark problems")
    ap.add_argument("--k", type=int, default=175)
    ap.add_argument("--tmax_sec", type=float, default=5.0)
    ap.add_argument("--device", default="cuda:0")
    ap.add_argument("--no_warmup", action="store_true")
    ap.add_argument("--ikflow_checkpoint", default=None, help="GraphINN state dict: plan with IkflowCandidateGenerator")
    args = ap.parse_args(argv)
    if args.ikflow_checkpoint and args.planner != "CppFlow":
        ap.error("--ikflow_checkpoint needs --planner CppFlow")
    sd = torch.load(args.ikflow_checkpoint, map_location="cpu") if args.ikflow_checkpoint else None
    if args.all:
        problems = [problem_from_filename(CONSTRAINTS, n, device=args.device) for n in ALL_PROBLEM_FILENAMES]
    elif args.problem_file:
        problems = [problem_from_filename(CONSTRAINTS, "", filepath_override=args.problem_file, device=args.device)]
    else:
        problems = [problem_from_filename(CONSTRAINTS, args.problem or "fetch_arm__circle", device=args.device)]
    settings = PlannerSettings(k=args.k, tmax_sec=args.tmax_sec, anytime_mode_enabled=False, verbosity=0,
                               do_rerun_if_large_dp_search_mjac=True, do_rerun_if_optimization_fails=True)
    rows, succeeded, failed = [], [], []
    solvers = {}
    for problem in problems:
        generator = None
        if sd is not None:
            rob = problem.robot
            m = torch.tensor([1.0 / max(abs(lo), abs(hi)) for lo, hi in rob.actuated_joints_limits])
            diag = torch.diagonal(sd["module_list.0.M"]).float()
            if diag.numel() < rob.ndof or not torch.allclose(diag[: rob.ndof], m, rtol=1e-5):
                print(f"skipping {problem.full_name}: the checkpoint is not for {rob.name}")
                continue
            if rob.name not in solvers:
                solvers[rob.name] = IkflowSolver(rob, params_from_state_dict(sd), state_dict=sd, device=args.device)
            generator = IkflowCandidateGenerator(solvers[rob.name], seed=0)
        try:
            row, ok = evaluate(args.planner, problem, settings, warmup=not args.no_warmup, generator=generator)
        except AssertionError as e:  # the reference's checks on the candidates, e.g. "too many env collisions"
            print(f"{problem.full_name}: the planner stopped: {e}")
            failed.append(problem.full_name)
            continue
        rows.append(row)
        (succeeded if ok else failed).append(problem.full_name)
    print("| " + " | ".join(COLUMNS) + " |")
    print("|" + "---|" * len(COLUMNS))
    for row in sorted(rows, key=lambda r: (r[1], r[0])):
        print("| " + " | ".join(str(v) for v in row) + " |")
    print(f"\nsucceeded: {sorted(succeeded)}\nfailed:    {sorted(failed)}")
    return rows


if __name__ == "__main__":
    main()
