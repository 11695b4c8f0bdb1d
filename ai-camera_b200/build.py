"""Build ``libaicam.so`` (the C-ABI CUDA library) in-tree with nvcc, sm_100a only.

``python -m ai_camera_b200.build`` or ``__graft_entry__.build()``.  Cross-compiles without
a GPU.  Objects are rebuilt when their source (or any header) is newer.
"""
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "_build")
LIB = os.path.join(HERE, "libaicam.so")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall",
          "--expt-relaxed-constexpr"]
# Files whose float arithmetic must match the reference bit for bit: no FMA contraction.  (counting.cu needs no entry: its
# geometry is integer-only.)
NO_FMA = {"tracker.cu", "detect_post.cu", "reid_crops.cu", "preprocess.cu"}


def nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found; the aicam library cannot be built")
    return exe


def sources():
    return sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))


def _stale(obj, src, headers):
    if not os.path.exists(obj):
        return True
    t = os.path.getmtime(obj)
    return any(os.path.getmtime(p) > t for p in [src] + headers)


def build(verbose=False, force=False):
    os.makedirs(OUT, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "aicam.h"))
    headers.append(os.path.abspath(__file__))
    jobs = []
    objs = []
    for f in sources():
        src = os.path.join(CSRC, f)
        obj = os.path.join(OUT, f[:-3] + ".o")
        objs.append(obj)
        if force or _stale(obj, src, headers):
            cmd = [nvcc()] + ARCH + COMMON + (["--fmad=false"] if f in NO_FMA else []) + \
                  (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            jobs.append((f, cmd))

    def run(job):
        f, cmd = job
        r = subprocess.run(cmd, capture_output=True, text=True)
        return f, r

    with ThreadPoolExecutor(max_workers=8) as ex:
        for f, r in ex.map(run, jobs):
            if verbose or r.returncode != 0:
                sys.stderr.write("== %s\n%s%s\n" % (f, r.stdout, r.stderr))
            if r.returncode != 0:
                raise RuntimeError("nvcc failed on %s" % f)
    if jobs or not os.path.exists(LIB):
        cmd = [nvcc()] + ARCH + ["-shared", "-o", LIB] + objs + ["-lcudart"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("linking libaicam.so failed")
    return LIB


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv, force="-f" in sys.argv))
