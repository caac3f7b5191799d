"""Build eirgrid_b200/libeirgrid_b200.so in-tree with nvcc for sm_100a.

    python -m eirgrid_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU. `--fmad=false` (device) and `-ffp-contract=off` (host) are part of the
numerics contract: the kernels must perform the reference's IEEE operations without FMA contraction.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, os.environ.get("EIRGRID_LIB_NAME", "libeirgrid_b200.so"))
SOURCES = ["engine.cu", "episode.cu", "site_tables.cu", "stats.cu", "update.cu", "suitability.cu", "microbench.cu", "weights.cpp", "host_tables.cpp", "report_files.cpp"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
EXTRA = os.environ.get("EIRGRID_NVCC_EXTRA", "").split()
FLAGS = EXTRA + ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "--fmad=false", "-std=c++17",
         "-Xcompiler", "-fPIC,-ffp-contract=off,-fno-fast-math,-Wall", "-Xptxas", "-v"]


def stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "eirgrid_b200.h"),
                                                                 os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not stale():
        return LIB
    objdir = os.path.join(HERE, "build", os.path.splitext(os.path.basename(LIB))[0])
    os.makedirs(objdir, exist_ok=True)
    objs = []
    log = []
    for src in SOURCES:
        obj = os.path.join(objdir, os.path.splitext(src)[0] + ".o")
        cmd = [NVCC] + FLAGS + (["-x", "cu"] if src.endswith(".cpp") else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log.append("$ " + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode != 0:
            sys.stderr.write(log[-1])
            raise RuntimeError("nvcc failed on " + src)
        objs.append(obj)
    cmd = [NVCC, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    log.append("$ " + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    if r.returncode != 0:
        sys.stderr.write(log[-1])
        raise RuntimeError("link failed")
    with open(os.path.join(objdir, "build.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
