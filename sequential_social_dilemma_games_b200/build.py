"""Builds libssd_b200.so in-tree with nvcc for sm_100a (the .so is git-ignored but travels to the
GPU box with the repo snapshot).  `python -m sequential_social_dilemma_games_b200.build`."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libssd_b200.so")
SOURCES = ["ssd_step_fast.cu", "ssd_step_general.cu", "ssd_aux.cu", "ssd_capi.cu", "ssd_policy.cu", "ssd_policy_head.cu",
           "ssd_policy_pool.cu", "ssd_policy_moa.cu"]  # compiled in parallel
HEADERS = ["ssd_internal.h", "ssd_device.cuh", "ssd_phases.cuh", "ssd_umma.cuh", "ssd_policy.h", "ssd_policy_lstm.cuh", os.path.join("..", "..", "include", "ssd_b200.h")]
NVCC_FLAGS = ["-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    objs = []
    procs = []
    for s in SOURCES:
        o = os.path.join(CSRC, s.replace(".cu", ".o"))
        knobs = ["-DSSD_PROFILING_KNOBS"] if os.environ.get("SSD_PROFILING_KNOBS") else []  # profiles/skip_sweep.py only
        cmd = [_nvcc()] + NVCC_FLAGS + knobs + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, s), "-o", o]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
        objs.append(o)
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out.decode(errors="replace"))
        if p.returncode:
            raise RuntimeError("nvcc failed: %s" % " ".join(cmd))
    link = [_nvcc(), "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    subprocess.check_call(link)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
