"""Segmented (parallel-in-time) solve against the twisted solve: stand-alone solve time per path count and segment
count and the difference of the results.  One JSON line per path count."""
import json, os, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cppflow_b200 import ops, _lib
from cppflow_b200.robot import get_robot
from cppflow_b200.synthetic import synthetic_problem, synthetic_seeds_host
from cppflow_b200.lm_hyper_parameters import all_terms_parameters

dev = torch.device("cuda:0")
robot = get_robot("fetch"); PMAX, T, D = 8192, 300, 8
problem = synthetic_problem(robot, T, device=dev)
_, xh = synthetic_seeds_host(robot, PMAX, T)
x0 = xh.to(dev)
ob = problem.obstacle_tables
lib = _lib.load(); cu, tc, no = ops._obs(ob); st = _lib.stream_ptr(dev)
prm = ops.make_params(all_terms_parameters())
rid = robot.robot_id
SEGS = [int(s) for s in os.environ.get("SEGS", "0,2,4,8,12,16,24,32").split(",")]
PATHS = [int(s) for s in os.environ.get("PATHS", "1,16,256,1024,2048,4096,8192").split(",")]

def timeit(fn, n=30):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n

for n_paths in PATHS:
    out = {"paths": n_paths}
    ref = None
    for S in SEGS:
        flags = 1 | ops.lm_segments(S)
        ws = torch.empty((lib.cppflow_lm_full_workspace_bytes_ex(rid, n_paths, T, flags),), device=dev, dtype=torch.uint8)
        xo = torch.empty((n_paths * T, D), device=dev)
        fa = lambda: _lib.check(lib.cppflow_lm_full_assemble(rid, prm, _lib.ptr(x0), None, _lib.ptr(problem.target_path), n_paths, T, cu, tc, no, _lib.ptr(ws), ws.numel(), st))
        fs = lambda: _lib.check(lib.cppflow_lm_full_solve(rid, prm, _lib.ptr(x0), n_paths, T, flags, _lib.ptr(ws), ws.numel(), _lib.ptr(xo), st))
        def both():
            fa(); fs()
        t_a = timeit(fa); t_both = timeit(both)
        out[f"solve_ms_S{S}"] = round(t_both - t_a, 4)
        if S == 0:
            ref = xo.clone(); out["assemble_ms"] = round(t_a, 4)
        elif ref is not None:
            out[f"maxdiff_S{S}"] = float((xo - ref).abs().max())
    print(json.dumps(out), flush=True)
