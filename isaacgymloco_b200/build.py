"""Build libhimloco_b200.so in-tree with plain nvcc (sm_100a only; no JIT cache, no torch
extension machinery -- the library has a C ABI and is loaded with ctypes)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, os.environ.get("HL_LIB_NAME", "libhimloco_b200.so"))   # HL_LIB_NAME: experiment builds side by side
SOURCES = ["hl_env_kernels.cu", "hl_rollout_kernels.cu", "hl_amp_kernels.cu"]
HEADERS = ["hl_common.cuh", "hl_math.cuh", "hl_fused_kernel.inc", "hl_persist_kernel.inc", os.path.join("..", "..", "include", "himloco_b200.h")]
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "--shared", "-Xptxas", "-v"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    extra = os.environ.get("HL_DEFINES", "").split()          # dev experiments, e.g. HL_DEFINES=-DHL_EXP_NO_PHILOX
    cmd = [_nvcc()] + NVCC_FLAGS + extra + [os.path.join(CSRC, s) for s in SOURCES] + ["-o", LIB]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if proc.returncode != 0:
        sys.stderr.write(proc.stdout + proc.stderr)
        raise RuntimeError("nvcc failed building libhimloco_b200.so")
    if verbose:
        sys.stderr.write(proc.stderr)
    # the report of this build goes beside the library; csrc/ptxas_info.txt is the committed record and stays as it is
    with open(os.path.splitext(LIB)[0] + ".ptxas.txt", "w") as f:
        f.write(proc.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
