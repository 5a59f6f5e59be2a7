"""Builds libsacb200.so (hand-written sm_100a CUDA + the C ABI of include/sacb200.h) in-tree with nvcc."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libsacb200.so")
SOURCES = ["sacb.cu", "program.cu", "replay.cu", "extras.cu", "dp.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O2", "--expt-relaxed-constexpr",
]


def _newer(src_paths, target):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(p) > t for p in src_paths)


def build(force=False, verbose=False):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    extra = os.environ.get("SACB_EXTRA_NVCC", "").split()       # extra nvcc flags, e.g. -DSOME_MACRO
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "sacb200.h")]
    if not force and not _newer(deps, LIB):
        return LIB
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(CSRC, src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc, *NVCC_FLAGS, *extra, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- nvcc {src}\n{out}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    subprocess.check_call([nvcc, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
