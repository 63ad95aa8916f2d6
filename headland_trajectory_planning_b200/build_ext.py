"""Build the sm_100a shared library in-tree with nvcc (no JIT cache, so the .so
travels with the repo snapshot to the GPU box)."""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libheadland_b200.so")
SOURCES = ["hl_ctx.cu", "hl_collision.cu", "hl_rs.cu", "hl_astar.cu", "hl_grid.cu", "hl_raster.cu", "hl_bench.cu", "hl_ypark.cu", "hl_refpath.cu", "hl_dubins.cu"]


def nvcc_path():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    deps.append(os.path.join(HERE, "..", "include", "headland_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force=False, verbose=False):
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    if not force and not needs_build():
        return LIB
    objs = []
    procs = []
    for s in srcs:
        o = s[:-3] + ".o"
        cmd = [nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo",
               "-std=c++17", "-Xcompiler", "-fPIC", "--fmad=true", "-c", s, "-o", o]
        cmd[1:1] = os.environ.get("HL_NVCC_FLAGS", "").split()
        if verbose:
            cmd.insert(1, "-Xptxas")
            cmd.insert(2, "-v")
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(o)
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(out)
        if p.returncode != 0:
            failed = True
    if failed:
        raise RuntimeError("nvcc failed")
    cmd = [nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB] + objs + ["-lcudart"]
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
