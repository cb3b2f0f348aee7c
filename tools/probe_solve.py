"""Block-solve timings: stand-alone solve time at several path counts (the library picks the solve kernel by path
count), the chunk-pipelined step, and a checksum of the result (every solve kernel gives the same bits).  One JSON line."""
import hashlib, json, os, sys, time
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cppflow_b200 import ops, _lib
from cppflow_b200.robot import get_robot
from cppflow_b200.synthetic import synthetic_problem, synthetic_seeds_host
from cppflow_b200.lm_hyper_parameters import all_terms_parameters
from cppflow_b200.pipeline import ResidentPipeline

dev = torch.device("cuda:0")
robot = get_robot("fetch"); P, T, D = 8192, 300, 8
problem = synthetic_problem(robot, T, device=dev)
_, xh = synthetic_seeds_host(robot, P, T)
x0 = xh.to(dev); xo = torch.empty_like(x0)
ob = problem.obstacle_tables
lib = _lib.load(); cu, tc, no = ops._obs(ob); st = _lib.stream_ptr(dev)
prm = ops.make_params(all_terms_parameters())
rid = robot.robot_id

def timeit(fn, n=30):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n

out = {}
ws = torch.empty((lib.cppflow_lm_full_workspace_bytes(rid, P, T),), device=dev, dtype=torch.uint8)
for n_paths in (8192, 2048, 512, 16):
    fa = lambda: _lib.check(lib.cppflow_lm_full_assemble(rid, prm, _lib.ptr(x0), None, _lib.ptr(problem.target_path), n_paths, T, cu, tc, no, _lib.ptr(ws), ws.numel(), st))
    fs = lambda: _lib.check(lib.cppflow_lm_full_solve(rid, prm, _lib.ptr(x0), n_paths, T, 1, _lib.ptr(ws), ws.numel(), _lib.ptr(xo), st))
    def both():
        fa(); fs()
    t_a = timeit(fa); t_both = timeit(both)
    out[f"solve_ms_{n_paths}"] = round(t_both - t_a, 4)
    out[f"assemble_ms_{n_paths}"] = round(t_a, 4)
res = ops.lm_full_step(rid, D, prm, x0, None, problem.target_path, P, T, ob, True)
out["sha"] = hashlib.sha256(res.cpu().numpy().tobytes()).hexdigest()[:16]
for chunks in (4, 8):
    rp = ResidentPipeline(problem, P, all_terms_parameters(), n_chunks=chunks)
    def run(n):
        rp.begin()
        for _ in range(n): rp.enqueue_step(x0, xo)
        rp.end()
    run(5); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for n in (20, 100):
        e0.record(); run(n); e1.record(); torch.cuda.synchronize()
        out[f"pipe{chunks}_ms_per_step_{n}"] = round(e0.elapsed_time(e1) / n, 4)
    out[f"pipe{chunks}_sha"] = hashlib.sha256(xo.cpu().numpy().tobytes()).hexdigest()[:16]
# strong-scaling sizes
for n_paths in (1024, 2048):
    rp = ResidentPipeline(problem, n_paths, all_terms_parameters(), n_chunks=4)
    xs = x0[: n_paths * T]
    def run(n):
        rp.begin()
        for _ in range(n): rp.enqueue_step(xs, xo[: n_paths * T])
        rp.end()
    run(5); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); run(20); e1.record(); torch.cuda.synchronize()
    out[f"pipe4_P{n_paths}_ms_per_step"] = round(e0.elapsed_time(e1) / 20, 4)
print(json.dumps(out))
