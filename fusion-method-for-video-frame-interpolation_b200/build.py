"""Build libfvfi.so (the C-ABI of include/fvfi.h) in-tree with nvcc for sm_100a.

    python fusion-method-for-video-frame-interpolation_b200/build.py [--force] [--verbose]

The .so lands in fvfi/libfvfi.so (git-ignored, but it travels to the GPU box).
"""
import glob
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
OUT = os.path.join(HERE, "fvfi", "libfvfi.so")
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-DFVFI_BUILD", "-Xcompiler", "-fPIC,-O2",
    "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(HERE, "csrc"),
]


def sources():
    return sorted(glob.glob(os.path.join(HERE, "csrc", "*.cu")))


def stale():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = sources() + glob.glob(os.path.join(HERE, "csrc", "*.cuh")) + glob.glob(os.path.join(HERE, "csrc", "*.hpp"))
    deps += glob.glob(os.path.join(ROOT, "include", "*.h"))
    deps.append(os.path.abspath(__file__))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not stale():
        return OUT
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    objs, procs = [], []
    for src in sources():
        obj = os.path.join(objdir, os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        cmd = ["nvcc"] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for cmd, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(" ".join(cmd) + "\n" + out + "\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    subprocess.check_call(["nvcc", "-shared", "-o", OUT] + objs)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
