"""Build libgenie_smem.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

Each source is compiled to its own object (in parallel, only when stale) and then linked, so a change
to the search kernels does not pay for the CUB-heavy index builder again."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "_obj")
LIB = os.path.join(HERE, "libgenie_smem.so")
SOURCES = ["kernels.cu", "index_device.cu", "ingest.cu", "comm.cu", "hits.cu", "chains.cu", "index_host.cpp", "ingest_host.cpp"]
HEADERS = ["fm_core.cuh", "sweep_logic.cuh", "sweep_device.cuh", "select_logic.cuh", "hits_logic.cuh", "strand_logic.cuh", "chain_logic.cuh", "host_common.hpp",
           "../../include/genie_smem.h"]
FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
         "-Xcompiler", "-fPIC,-O3,-fno-strict-aliasing", "-Xptxas", "-v"]


def _newest_header():
    return max(os.path.getmtime(os.path.join(CSRC, f)) for f in HEADERS)


def _stale(src, obj, force):
    if force or not os.path.exists(obj):
        return True
    t = os.path.getmtime(obj)
    return os.path.getmtime(src) > t or _newest_header() > t


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    os.makedirs(OBJ, exist_ok=True)
    jobs = []
    for f in SOURCES:
        src, obj = os.path.join(CSRC, f), os.path.join(OBJ, f + ".o")
        if _stale(src, obj, force):
            jobs.append((f, [nvcc] + FLAGS + ["-c", src, "-o", obj]))
    logs = {}

    def run(job):
        f, cmd = job
        r = subprocess.run(cmd, capture_output=True, text=True)
        return f, r

    with ThreadPoolExecutor(max_workers=max(1, len(jobs))) as ex:
        for f, r in ex.map(run, jobs):
            logs[f] = r.stderr
            if verbose or r.returncode != 0:
                sys.stderr.write(r.stdout + r.stderr)
            if r.returncode != 0:
                raise RuntimeError(f"nvcc failed compiling {f}")
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + \
          [os.path.join(OBJ, f + ".o") for f in SOURCES] + ["-lpthread", "-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed linking libgenie_smem.so")
    for f, text in logs.items():
        with open(os.path.join(OBJ, f"ptxas_{f.split('.')[0]}.log"), "w") as out:     # untracked; profiles/ keeps one copy per round
            out.write(text)
    return LIB


if __name__ == "__main__":
    build(force=True, verbose=True)
