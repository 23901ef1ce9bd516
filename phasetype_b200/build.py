"""Build libpht_b200.so in-tree with nvcc/gcc for sm_100a (no torch, no JIT cache).

Flags that matter:
  -gencode arch=compute_100a,code=sm_100a   B200 only
  -fmad=false / -ffp-contract=off            no compiler-made FMAs: device and host round alike
                                             (FMAs that are wanted are written explicitly)
  -lineinfo                                  ncu source pages map to these files
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libpht_b200.so")
CU = ["engine.cu", "k_model.cu", "k_mhrs.cu", "k_sort.cu", "k_dcs.cu", "k_ecs.cu", "k_unif.cu", "k_peak.cu"]
CC = ["gibbs_host.c", "rapi_standin.c"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-fmad=false", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=default"]
GCC_FLAGS = ["-O2", "-std=gnu11", "-fPIC", "-ffp-contract=off", "-mfma", "-Wall"]


def _newer(src_list, target):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in src_list)


def build(force=False, verbose=False, ptxas_info=False, out=None, defines=()):
    """defines/out: build an experimental variant (e.g. defines=("-DMHRS_MIN_BLOCKS=4",)) next to the default library."""
    global OUT
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if out is not None:
        OUT = os.path.join(HERE, out); force = True
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "pht_b200.h"), __file__]
    if not force and not _newer(deps, OUT):
        return OUT
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    objs = []
    for f in CU:
        o = os.path.join(objdir, f + ".o")
        cmd = [nvcc] + NVCC_FLAGS + list(defines) + (["-Xptxas", "-v"] if ptxas_info else []) + ["-c", os.path.join(CSRC, f), "-o", o]
        if verbose:
            print(" ".join(cmd))
        subprocess.run(cmd, check=True)
        objs.append(o)
    for f in CC:
        o = os.path.join(objdir, f + ".o")
        cmd = ["gcc"] + GCC_FLAGS + ["-c", os.path.join(CSRC, f), "-o", o]
        if verbose:
            print(" ".join(cmd))
        subprocess.run(cmd, check=True)
        objs.append(o)
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", OUT] + objs + ["-ldl", "-lm"]
    if verbose:
        print(" ".join(cmd))
    subprocess.run(cmd, check=True)
    return OUT


if __name__ == "__main__":
    _defs = tuple(a for a in sys.argv[1:] if a.startswith("-D"))
    _out = next((a.split("=", 1)[1] for a in sys.argv[1:] if a.startswith("--out=")), None)
    print(build(force="--force" in sys.argv, verbose=True, ptxas_info="--ptxas" in sys.argv, out=_out, defines=_defs))
