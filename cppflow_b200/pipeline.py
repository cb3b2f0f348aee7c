"""Host-buffer entry point of the fused LM iteration: pinned host joint paths in, refined paths out.

The path set is cut into chunks; chunk c's host->device copy, the kernels of the chunks before it and the
device->host copy of finished chunks run concurrently (PCIe is full duplex), so the end-to-end rate approaches
max(copy in, compute, copy out) instead of their sum.  The kernels of consecutive chunks go to different streams
(round robin over `n_run_streams`): the block solve of a chunk is a latency-bound chain of T dependent steps that
fills only a few SMs, so it overlaps the assembly and the solves of its neighbours.

The whole fork / copy / launch / join pattern of one call (4 operations per chunk on 2 + n_run_streams streams) is
captured once per (slot, input buffer, output buffer) into a CUDA graph and replayed (enqueueing it from Python costs
~60 us per chunk).  Independent jobs submitted with `refine_async` go to `depth` slots of device buffers in turn and
overlap: the copy-in of one job runs under the copy-out of the job before it.

Measured at P = 8192, T = 300 (78.6 MB each way; one direction alone 1.42 ms, both directions at once 1.64 ms = the
floor): one job at a time 2.23-2.24 ms per job whatever the chunking (first copy-in, last solve and last copy-out are
exposed); two jobs deep: 16 chunks 2.00 ms, 8 chunks 1.94, 6 chunks / 3 run streams **1.75** (0.93 of the floor), 4
chunks 1.86, 3 chunks 1.88; a third slot changes nothing (1.76).  Every event between a copy and a kernel costs the
copy engines time (48.8 -> ~36 GB/s per direction with 16 chunks), so with the fill and drain hidden by the next job
fewer, larger chunks win until a chunk's own latency shows again."""
from typing import Optional

import torch

from . import ops
from .data_types import Problem
from .lm_hyper_parameters import OptimizationParameters, all_terms_parameters


class numa_local:
    """Context manager: while active, the calling thread is bound to the CPUs of the NUMA node the CUDA device hangs
    off, so that page-locked host buffers allocated inside (`tensor.pin_memory()`) come from that node's memory and the
    device's DMA does not cross the socket interconnect (matters with 8 ranks copying at once).  A no-op when the
    topology cannot be read or none of the node's CPUs is available to the process; the affinity is restored on exit."""

    def __init__(self, device):
        self.device = torch.device(device)
        self.saved = None

    def __enter__(self):
        import os

        try:
            prop = torch.cuda.get_device_properties(self.device)
            bdf = f"{prop.pci_domain_id:04x}:{prop.pci_bus_id:02x}:{prop.pci_device_id:02x}.0"
            with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
                node = int(f.read().strip())
            if node < 0:
                return self
            with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
                cpus = set()
                for part in f.read().strip().split(","):
                    lo, _, hi = part.partition("-")
                    cpus.update(range(int(lo), int(hi or lo) + 1))
            allowed = os.sched_getaffinity(0)
            local = cpus & allowed
            if local and local != allowed:
                self.saved = allowed
                os.sched_setaffinity(0, local)
        except Exception:  # noqa: BLE001 - topology files missing, no permission, ...: keep the default placement
            self.saved = None
        return self

    def __exit__(self, *exc):
        import os

        if self.saved is not None:
            try:
                os.sched_setaffinity(0, self.saved)
            except Exception:  # noqa: BLE001
                pass
        return False


class HostPipeline:
    def __init__(self, problem: Problem, n_paths: int, params: Optional[OptimizationParameters] = None,
                 n_chunks: int = 6, n_run_streams: int = 3, device=None, use_graph: bool = True, overlap: bool = True,
                 taper=None, depth: int = 2):
        """`taper`: path counts of extra small chunks at BOTH ends of the chunk list, e.g. (64, 192): the first result
        can only leave for the host one chunk latency (copy-in + assembly + the solve's ~0.25 ms chain) after the
        start, and the last chunk's latency is exposed after the last copy-in - small first and last chunks shorten both."""
        self.problem = problem
        self.robot = problem.robot
        self.T = problem.n_timesteps
        self.P = n_paths
        self.device = problem.target_path.device if device is None else torch.device(device)
        self.prm = ops.make_params(params if params is not None else all_terms_parameters())
        taper = [int(t) for t in (taper or []) if t > 0]
        if 4 * sum(taper) > n_paths:
            taper = []
        n_main = n_paths - 2 * sum(taper)
        n_chunks = max(1, min(n_chunks, n_main))
        base, rem = divmod(n_main, n_chunks)
        sizes = taper + [base + (1 if c < rem else 0) for c in range(n_chunks)] + taper[::-1]
        self.chunks = []
        start = 0
        for n in sizes:
            self.chunks.append((start, n))
            start += n
        assert start == n_paths
        D = self.robot.ndof
        # `depth` independent slots (device buffers, workspaces, events, launch stream): consecutive refine_async calls
        # alternate between them, so the copy-in of one call runs under the copy-out of the call before it
        self.depth = max(1, int(depth))
        self.x_devs = [torch.empty((n_paths * self.T, D), device=self.device, dtype=torch.float32) for _ in range(self.depth)]
        self.out_devs = [torch.empty_like(self.x_devs[0]) for _ in range(self.depth)]
        self.x_dev, self.out_dev = self.x_devs[0], self.out_devs[0]
        self.s_in, self.s_out = (torch.cuda.Stream(self.device) for _ in range(2))
        self.s_run = [torch.cuda.Stream(self.device) for _ in range(max(1, min(n_run_streams, n_chunks)))]
        self.s_launch = [torch.cuda.Stream(self.device) for _ in range(self.depth)]
        self.ev_in = [[torch.cuda.Event() for _ in self.chunks] for _ in range(self.depth)]
        self.ev_run = [[torch.cuda.Event() for _ in self.chunks] for _ in range(self.depth)]
        # one workspace per (slot, run stream) (kernels on one stream are ordered, so its workspace is reused safely)
        lib_bytes = ops._lib.load().cppflow_lm_full_workspace_bytes(self.robot.robot_id, max(n for _, n in self.chunks), self.T)
        self.wss = [[torch.empty((lib_bytes,), device=self.device, dtype=torch.uint8) for _ in self.s_run]
                    for _ in range(self.depth)]
        self.use_graph = use_graph
        self.flags = ops.LM_CLAMP | (ops.LM_OVERLAP if overlap else 0)  # overlap: the solve of a chunk runs under the
        self._graphs = {}                                              # assembly of the next (see ResidentPipeline)
        self._next = 0

    def refine(self, x_host: torch.Tensor, out_host: torch.Tensor) -> torch.Tensor:
        """One fused LM iteration (+ clamp) over all paths: x_host [P*T, D] pinned -> out_host [P*T, D] pinned.
        Asynchronous with respect to the host: the caller's current stream waits for the last copy."""
        done = self.refine_async(x_host, out_host)
        torch.cuda.current_stream(self.device).wait_event(done)
        return out_host

    def refine_async(self, x_host: torch.Tensor, out_host: torch.Tensor) -> torch.cuda.Event:
        """The same iteration, submitted without joining the caller's stream: returns the event that completes when
        out_host is filled (`event.synchronize()` before reading it on the CPU).  Calls go to `depth` slots in turn, each
        ordered after the caller's current stream at submission; calls in different slots overlap on the device (PCIe
        is full duplex: the copy-in of call i + 1 runs under the copy-out of call i), so a stream of independent
        path sets is refined at max(copy in, copy out) per set instead of their pipelined sum.  The caller keeps
        x_host unchanged and out_host unread until the event completes, and passes distinct out_host buffers to calls
        that may be in flight together."""
        assert x_host.shape == self.x_dev.shape and out_host.shape == self.x_dev.shape
        assert x_host.is_pinned() and out_host.is_pinned(), "host buffers must be pinned for asynchronous copies"
        slot = self._next
        self._next = (self._next + 1) % self.depth
        launch = self.s_launch[slot]
        launch.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(launch):
            if not self.use_graph:
                self._enqueue(x_host, out_host, slot)
            else:
                key = (slot, x_host.data_ptr(), out_host.data_ptr())
                graph = self._graphs.get(key)
                if graph is None:
                    self._enqueue(x_host, out_host, slot)  # eager once: first-call setup in the library must not be captured
                    launch.synchronize()
                    graph = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(graph):
                        self._enqueue(x_host, out_host, slot)
                    self._graphs[key] = graph
                graph.replay()
            done = torch.cuda.Event()
            done.record(launch)
        return done

    def _enqueue(self, x_host: torch.Tensor, out_host: torch.Tensor, slot: int = 0) -> torch.Tensor:
        T, D, rid = self.T, self.robot.ndof, self.robot.robot_id
        cur = torch.cuda.current_stream(self.device)
        x_dev, out_dev = self.x_devs[slot], self.out_devs[slot]
        for s in [self.s_in, self.s_out] + self.s_run:
            s.wait_stream(cur)
        lib = ops._lib.load()
        cu, tc, no = ops._obs(self.problem.obstacle_tables)
        for c, (p0, n) in enumerate(self.chunks):
            sl = slice(p0 * T, (p0 + n) * T)
            with torch.cuda.stream(self.s_in):
                x_dev[sl].copy_(x_host[sl], non_blocking=True)
                self.ev_in[slot][c].record(self.s_in)
            s_run = self.s_run[c % len(self.s_run)]
            with torch.cuda.stream(s_run):
                s_run.wait_event(self.ev_in[slot][c])
                ws = self.wss[slot][c % len(self.s_run)]
                ops.check(lib.cppflow_lm_full_step(
                    rid, self.prm, ops.ptr(x_dev[sl]), None, ops.ptr(self.problem.target_path), n, T, cu, tc, no, self.flags,
                    ops.ptr(ws), ws.numel(), ops.ptr(out_dev[sl]), ops.stream_ptr(self.device)))
                self.ev_run[slot][c].record(s_run)
            with torch.cuda.stream(self.s_out):
                self.s_out.wait_event(self.ev_run[slot][c])
                out_host[sl].copy_(out_dev[sl], non_blocking=True)
        for s in [self.s_out, self.s_in] + self.s_run:
            cur.wait_stream(s)
        return out_host


def split_paths(n_paths: int, n_chunks: int):
    """Contiguous chunks [(first path, count), ...] covering n_paths: multiples of 256 paths (the assembly CTA) when
    there are enough paths, of 16 (the solve's path group) otherwise; no empty chunks."""
    gran = 256 if n_paths >= 256 * n_chunks else 16 if n_paths >= 16 * n_chunks else 1
    units = (n_paths + gran - 1) // gran
    n_chunks = max(1, min(n_chunks, units))
    base, rem = divmod(units, n_chunks)
    chunks, start = [], 0
    for c in range(n_chunks):
        n = min((base + (1 if c < rem else 0)) * gran, n_paths - start)
        if n > 0:
            chunks.append((start, n))
        start += n
    return chunks


class ResidentPipeline:
    """LM iterations over device-resident paths with the two kernels of the step overlapped across path chunks.

    One iteration is assembly (FP32-bound, fills every SM) followed by the block solve (a latency-bound chain: 4 warps
    per 64 paths, each busy for the whole 0.25 ms however few paths there are).  Back to back they add up.  Paths are
    independent, so the path set is cut into `n_chunks` chunks, each with its own stream and workspace, and the
    iterations of a chunk are enqueued on its stream without any cross-chunk join: while chunk A is in its solve, chunk
    B is in the assembly of the same or the next iteration.  For that to happen on the SMs the solve is launched with
    CPPFLOW_LM_OVERLAP: a 105 KB shared-memory footprint that fits next to one 256-thread assembly CTA, and the highest
    launch priority so that its CTAs are dispatched before the thousands of pending assembly CTAs of the other chunks.
    Chunks are multiples of 256 paths (the assembly CTA) where P allows."""

    def __init__(self, problem: Problem, n_paths: int, params: Optional[OptimizationParameters] = None,
                 n_chunks: Optional[int] = None, device=None, overlap: bool = True, segments=0):
        """`segments`: time segments of the segmented solve (CPPFLOW_LM_SEGMENTS, csrc/lm_segsolve.cuh; 0 = the twisted
        solve).  For <= ~2000 paths per GPU the twisted solve's chain of T dependent steps is most of the iteration; the
        segmented solve's result differs by rounding and depends on `segments` only, not on the chunking.  "auto": 16
        segments up to 2048 paths (where it is faster), the twisted solve above."""
        self.problem = problem
        self.robot = problem.robot
        self.T = problem.n_timesteps
        self.P = n_paths
        self.device = problem.target_path.device if device is None else torch.device(device)
        self.prm = ops.make_params(params if params is not None else all_terms_parameters())
        self.overlap = overlap
        if segments == "auto":
            # tools/probe_segpipe.py, ms per iteration at T = 300, twisted (default chunking) against 16 segments:
            #   256 paths 0.163 / 0.077   512: 0.171 / 0.093   1024: 0.197 / 0.139   2048: 0.280 / 0.227   4096: 0.372 / 0.42
            segments = 16 if n_paths <= 2048 else 0  # at 2048 paths in two chunks: 0.228 (16 segments) / 0.237 (8)
        self.segments = segments
        if n_chunks is None and segments:
            n_chunks = 1 if n_paths <= 256 else 2  # 512: 0.098 / 0.093 (1 / 2 chunks), 1024: 0.151 / 0.139, 2048: 0.262 / 0.229
        if n_chunks is None:
            # measured at T = 300, K = 20 (tools/probe_timeline.py, ms per iteration by chunk count 1 / 2 / 3 / 4 / 6):
            #   8192 paths: - / - / - / 0.518 / 0.509      4096: 0.387 / 0.407 / 0.416 / 0.422 / 0.415
            #   2048: 0.302 / 0.282 / 0.303 / 0.310 / 0.348      1024: 0.245 / 0.231 / 0.288 / 0.194 / 0.201
            # below ~6000 paths a chunk no longer fills the SMs and the iteration is the solve's chain latency: one or two
            # chunks; at 1024 paths four chunks of 256 take the register-resident solve (ops / launch_solve)
            n_chunks = 6 if n_paths >= 6144 else 1 if n_paths >= 3072 else 2 if n_paths >= 1536 else 4
        self.chunks = split_paths(n_paths, n_chunks)
        if len(self.chunks) == 1:
            self.overlap = False  # nothing to run under: the stand-alone solve variants are faster
        self.streams = [torch.cuda.Stream(self.device) for _ in self.chunks]
        lib = ops._lib.load()
        self.ws = [torch.empty((lib.cppflow_lm_full_workspace_bytes_ex(self.robot.robot_id, n, self.T, ops.lm_segments(segments)),),
                               device=self.device, dtype=torch.uint8) for _, n in self.chunks]

    def begin(self):
        cur = torch.cuda.current_stream(self.device)
        for s in self.streams:
            s.wait_stream(cur)

    def end(self):
        cur = torch.cuda.current_stream(self.device)
        for s in self.streams:
            cur.wait_stream(s)

    def enqueue_step(self, x: torch.Tensor, out: torch.Tensor, clamp: bool = True):
        """One LM iteration x -> out ([P*T, D] device tensors) for every chunk, each on its own stream; call between
        begin() and end().  Steps enqueued back to back pipeline across chunks."""
        T, D, rid = self.T, self.robot.ndof, self.robot.robot_id
        # straight through the C ABI on each chunk's stream (the ops wrapper costs ~20 us of host time per call: with six
        # chunks that is a quarter of the step)
        lib = ops._lib.load()
        cu, tc, no = ops._obs(self.problem.obstacle_tables)
        flags = (ops.LM_CLAMP if clamp else 0) | (ops.LM_OVERLAP if self.overlap else 0) | ops.lm_segments(self.segments)
        assert x.is_cuda and out.is_cuda and x.dtype == torch.float32 and x.is_contiguous() and out.is_contiguous()
        tgt = ops.ptr(self.problem.target_path)
        with torch.cuda.device(self.device):
            for (p0, n), s, ws in zip(self.chunks, self.streams, self.ws):
                sl = slice(p0 * T, (p0 + n) * T)
                ops.check(lib.cppflow_lm_full_step(rid, self.prm, ops.ptr(x[sl]), None, tgt, n, T, cu, tc, no, flags,
                                                   ops.ptr(ws), ws.numel(), ops.ptr(out[sl]), s.cuda_stream))

    def enqueue_metrics(self, x: torch.Tensor, metrics: torch.Tensor, sign_only: bool = True):
        """Per-path validity metrics of x ([P*T, D]) into `metrics` ([P, 8]), each chunk's rows on the chunk's own stream
        right behind its last step - the metrics of a finished chunk run under the last solves of the others.  Call
        between begin() and end().  `sign_only` (default): what validity and the cost ranking need - the minimum capsule
        distances are exact only when negative (ops.path_metrics)."""
        T, D, rid = self.T, self.robot.ndof, self.robot.robot_id
        lib = ops._lib.load()
        cu, tc, no = ops._obs(self.problem.obstacle_tables)
        for (p0, n), s in zip(self.chunks, self.streams):
            ops.check(lib.cppflow_path_metrics_ex(rid, ops.ptr(x[p0 * T:(p0 + n) * T]), ops.ptr(self.problem.target_path), n, T,
                                                  cu, tc, no, ops.METRICS_SIGN_ONLY if sign_only else 0,
                                                  ops.ptr(metrics[p0:p0 + n]), s.cuda_stream))

    def capture(self, enqueue) -> torch.cuda.CUDAGraph:
        """CUDA graph of whatever `enqueue()` puts on the chunk streams between begin() and end() (steps, metrics): the
        whole fork / launch / join pattern - 2 launches per chunk and step - then costs ONE graph launch instead of one
        Python -> ctypes call per kernel, which matters when several ranks share a host's cores.  Run the same work
        eagerly once before capturing (first calls set kernel attributes)."""
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            self.begin()
            enqueue()
            self.end()
        return graph

    def iterate(self, x: torch.Tensor, n_iters: int, clamp: bool = True) -> torch.Tensor:
        """n_iters dependent LM iterations (x <- step(x)); returns the refined paths (a new tensor; x is kept)."""
        assert x.is_cuda and x.shape == (self.P * self.T, self.robot.ndof)
        bufs = [torch.empty_like(x), torch.empty_like(x)]
        src = x
        self.begin()
        for i in range(n_iters):
            dst = bufs[i % 2]
            self.enqueue_step(src, dst, clamp)
            src = dst
        self.end()
        return src if n_iters > 0 else x.clone()
