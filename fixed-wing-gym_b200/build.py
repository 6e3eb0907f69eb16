"""Build libfwgym.so in-tree with nvcc for sm_100a (the only target)."""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "csrc", "fwgym.cu")
OUT = os.path.join(HERE, "libfwgym.so")
DEPS = [os.path.join(HERE, "csrc", f) for f in ("fwgym.cu", "dynamics.cuh", "env.cuh", "philox.cuh", "layout.h", "fwmath.cuh", "env_shapes.h",
                                                    "env_shapes_gen.h")] + [
    os.path.join(HERE, "..", "include", "fwgym.h")]


def nvcc_path():
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.isfile(p):
        raise RuntimeError("nvcc not found")
    return p


def up_to_date():
    return os.path.isfile(OUT) and all(os.path.getmtime(OUT) >= os.path.getmtime(d) for d in DEPS)


def build(force=False, verbose=False):
    if not force and up_to_date():
        return OUT
    cmd = [nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
           "--shared", "-Xcompiler", "-fPIC", "-o", OUT, SRC]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n%s\n%s" % (r.stdout, r.stderr))
    if verbose:
        print(r.stderr)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
