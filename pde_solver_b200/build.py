"""Build libpde_b200.so (hand-written CUDA for sm_100a) in-tree with nvcc.

The built library is git-ignored but travels to the GPU box with the repo snapshot."""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libpde_b200.so")
SOURCES = ["tables.cpp", "kernels.cu", "stencil3d.cu", "elast3d.cu", "heat2.cu", "solver.cu", "weighted.cu", "wmg.cu", "comm.cu", "cabi.cu"]
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"] + os.environ.get("PDE_B200_NVCC_FLAGS", "").split()


def _newest(paths):
    return max(os.path.getmtime(p) for p in paths)


def build(force: bool = False, verbose: bool = False) -> str:
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    deps = srcs + [os.path.join(CSRC, h) for h in os.listdir(CSRC) if h.endswith((".h", ".cuh"))]
    deps.append(os.path.join(HERE, "..", "include", "pde_b200.h"))
    if not force and os.path.exists(OUT) and os.path.getmtime(OUT) >= _newest(deps):
        return OUT
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    objs = []
    procs = []
    for s in srcs:
        o = os.path.join(objdir, os.path.basename(s) + ".o")
        objs.append(o)
        if not force and os.path.exists(o) and os.path.getmtime(o) >= _newest(deps):
            continue
        cmd = [nvcc] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-x", "cu", "-dc" if False else "-c", s, "-o", o]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    link = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", OUT] + objs + ["-ldl"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode:
        sys.stderr.write(r.stdout)
        raise RuntimeError("link failed")
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
