"""Build recipe for libslic_b200.so (the C-ABI library declared in include/slic_b200.h).

nvcc cross-compiles for sm_100a without a GPU; the .so is built in-tree (git-ignored, but shipped
to the GPU box with the snapshot).  `python -m video_similarity_search_b200.build` rebuilds it.
"""
import concurrent.futures
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
OBJ_DIR = os.path.join(CSRC, "build")
LIB_PATH = os.path.join(PKG_DIR, "libslic_b200.so")

SOURCES = ["api.cu", "primitives.cu", "prep.cu", "nn_exact.cu", "nn_screen_tc.cu", "cc.cu", "segmean.cu", "finch_small.cu",
           "masks.cu", "metrics.cu", "host_entry.cu", "finch_driver.cu", "comm.cu", "skmeans.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v"]


def _nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: the CUDA extension cannot be built")
    return exe


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile every CUDA source for sm_100a and link libslic_b200.so.  Returns the library path."""
    os.makedirs(OBJ_DIR, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(PKG_DIR), "include", "slic_b200.h"))
    nvcc = _nvcc()
    jobs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        if force or _stale(o, [s] + headers):
            jobs.append((s, o))

    def compile_one(job):
        s, o = job
        r = subprocess.run([nvcc] + NVCC_FLAGS + ["-c", s, "-o", o], capture_output=True, text=True)
        return s, r

    with concurrent.futures.ThreadPoolExecutor(max_workers=8) as ex:
        for s, r in ex.map(compile_one, jobs):
            if verbose or r.returncode != 0:
                sys.stderr.write(r.stdout + r.stderr)
            if r.returncode != 0:
                raise RuntimeError("nvcc failed on %s" % s)
    objs = [os.path.join(OBJ_DIR, s.replace(".cu", ".o")) for s in SOURCES]
    if force or jobs or _stale(LIB_PATH, objs):
        r = subprocess.run([nvcc, "-shared", "-o", LIB_PATH] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"],
                           capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("link of libslic_b200.so failed")
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
