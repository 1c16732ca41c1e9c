#!/usr/bin/env python
"""Build libhop_b200.so (sm_100a) in-tree with nvcc.  Usage: python build.py [--force]"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.environ.get("HOP_BUILD_OUT") or os.path.join(os.path.dirname(HERE), "hop", "libhop_b200.so")   # experiments: other name
SRCS = ["hop_select.cu", "hop_select_ref.cu", "hop_verify.cu", "hop_select_tpp.cu", "hop_select_epl.cu", "hop_traj.cu", "hop_ddp.cu", "hop_util.cu", "hop_cabi.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
         "-Xptxas", "-v"] + os.environ.get("HOP_EXTRA_NVCC_FLAGS", "").split()
OBJ_TAG = os.environ.get("HOP_BUILD_TAG", "")


def stale(target, deps):
    return not os.path.exists(target) or any(os.path.getmtime(d) > os.path.getmtime(target) for d in deps)


def includes_of(path, seen=None):
    """Transitive closure of the quoted #include files of `path` (the per-object dependency list)."""
    import re
    seen = set() if seen is None else seen
    if path in seen or not os.path.exists(path):
        return seen
    seen.add(path)
    with open(path) as fh:
        for inc in re.findall(r'^\s*#\s*include\s+"([^"]+)"', fh.read(), flags=re.M):
            includes_of(os.path.normpath(os.path.join(os.path.dirname(path), inc)), seen)
    return seen


def build(force=False, verbose=False):
    deps = set()
    for src in SRCS:
        includes_of(os.path.join(HERE, src), deps)
    if not (force or stale(OUT, deps)):
        return OUT

    def compile_one(src):
        obj = os.path.join(HERE, src.replace(".cu", OBJ_TAG + ".o"))
        flags_tag = obj + ".flags"
        flags_now = " ".join(FLAGS)
        same_flags = os.path.exists(flags_tag) and open(flags_tag).read() == flags_now
        if not force and same_flags and not stale(obj, sorted(includes_of(os.path.join(HERE, src)))):
            return obj                                   # object newer than its source and every header it includes
        r = subprocess.run([NVCC, *FLAGS, "-c", os.path.join(HERE, src), "-o", obj], capture_output=True, text=True)
        with open(obj + ".ptxas.log", "w") as fh:
            fh.write(r.stderr)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{r.stderr}")
        with open(flags_tag, "w") as fh:
            fh.write(flags_now)
        if verbose:
            print(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SRCS)) as ex:
        objs = list(ex.map(compile_one, SRCS))
    # static cudart (nvcc default): the library has no runtime dependency besides the driver
    subprocess.check_call([NVCC, "-shared", "-o", OUT, *objs, "-gencode", "arch=compute_100a,code=sm_100a"])
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
