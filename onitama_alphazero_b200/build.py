"""Builds libonb.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libonb.so")
SOURCES = ["onb_api.cu", "onb_env.cu", "onb_perft.cu", "onb_mcts.cu", "onb_net.cu", "onb_selfplay.cu", "onb_actor.cu", "onb_comm.cu", "onb_replay.cu", "onb_alphabeta.cu", "onb_reuse.cu", "onb_tablebase.cu"]
HEADERS = ["onb_rules.cuh", "onb_internal.h", "onb_gumbel.cuh", os.path.join("..", "..", "include", "onb.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC",
              "-Xcompiler", "-fvisibility=hidden", "--fmad=false", "-Xptxas", "-v"]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """ONB_NVCC_EXTRA (optional): extra nvcc flags for measurement builds, e.g. ONB_NVCC_EXTRA=-DONB_NET_PROFILE with force=True
    (per-phase cycle counters printed by the network kernel; rebuild without it afterwards)."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    extra = os.environ.get("ONB_NVCC_EXTRA", "").split()
    deps = [os.path.join(CSRC, h) for h in HEADERS]
    objs = []
    logs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(CSRC, src.replace(".cu", ".o"))
        if force or _stale(o, [s] + deps):
            cmd = [nvcc] + NVCC_FLAGS + extra + ["-c", s, "-o", o]
            r = subprocess.run(cmd, capture_output=True, text=True)
            logs.append(r.stderr)
            if r.returncode != 0:
                sys.stderr.write(r.stderr)
                raise RuntimeError("nvcc failed on %s" % src)
        objs.append(o)
    if force or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static", "-ldl"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stderr)
            raise RuntimeError("link failed")
    if verbose:
        sys.stderr.write("".join(logs))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
