"""Builds cppflow_b200/libcppflow_b200.so (sm_100a) with nvcc.  No torch headers are involved: the library is a
plain C-ABI shared object (include/cppflow_b200.h) that the Python host binds with ctypes."""
import hashlib
import os
import shutil
import subprocess
from concurrent.futures import ThreadPoolExecutor

PKG = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libcppflow_b200.so")
OBJDIR = os.path.join(REPO, "build", "obj")

SOURCES = ["capi.cu", "k_pose.cu", "k_collision.cu", "k_lm_full.cu", "k_search.cu", "k_metrics.cu", "k_probe.cu", "lm_loop.cu", "lm_loop_batched.cu", "k_flow.cu", "k_flow_train.cu", "k_ik.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-std=c++17", "-O3", "-lineinfo", "--expt-relaxed-constexpr",
    "-Xcompiler", "-fPIC",
]


def _nvcc():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: cannot build libcppflow_b200.so")


def _digest():
    h = hashlib.sha256()
    files = sorted(os.listdir(CSRC)) + ["../../include/cppflow_b200.h"]
    for f in files:
        with open(os.path.join(CSRC, f), "rb") as fh:
            h.update(f.encode())
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def is_stale():
    stamp = LIB + ".sha256"
    if not (os.path.exists(LIB) and os.path.exists(stamp)):
        return True
    with open(stamp) as f:
        return f.read().strip() != _digest()


def build(force=False, verbose=False):
    """Compile every .cu for sm_100a and link the shared library in-tree.  Returns the library path."""
    if not force and not is_stale():
        return LIB
    nvcc = _nvcc()
    os.makedirs(OBJDIR, exist_ok=True)

    def compile_one(src):
        obj = os.path.join(OBJDIR, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        return obj, r.stderr

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 1)) as ex:
        results = list(ex.map(compile_one, SOURCES))
    if verbose:
        for _, log in results:
            print(log)
    cmd = [nvcc, "-shared", "-o", LIB] + [o for o, _ in results] + ["-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(LIB + ".sha256", "w") as f:
        f.write(_digest())
    return LIB


if __name__ == "__main__":
    import sys

    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
