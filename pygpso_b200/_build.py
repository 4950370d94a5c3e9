"""
Build the C-ABI shared library ``libgpso_b200.so`` in-tree with nvcc for sm_100a.

``python -m pygpso_b200._build`` (or ``__graft_entry__.build()``) compiles ``csrc/gpso_capi.cu``; the resulting
``.so`` sits next to this file so that it travels with the source tree (it is git-ignored, not installed).
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.path.join(HERE, "libgpso_b200.so")
SOURCES = ["gpso_capi.cu"]
HEADERS = ["common.cuh", "gemm_core.cuh", "kern_cov.cuh", "kern_dense.cuh", "kern_leaves.cuh", "kern_ozaki.cuh", "kern_predict.cuh", "kern_joint.cuh", "kern_screen.cuh", "kern_probe.cuh", "kern_mean.cuh"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-shared", "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
]


def find_nvcc():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found; cannot build libgpso_b200.so")
    return nvcc


def needs_build():
    if not os.path.exists(LIB_PATH):
        return True
    built = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS]
    deps.append(os.path.join(HERE, "..", "include", "gpso_b200.h"))
    return any(os.path.getmtime(dep) > built for dep in deps)


def build_library(force=False, verbose=False):
    """Compile the library if it is missing or older than its sources.  Returns the path of the ``.so``."""
    if not force and not needs_build():
        return LIB_PATH
    cmd = [find_nvcc()] + NVCC_FLAGS + [os.path.join(CSRC, s) for s in SOURCES] + ["-o", LIB_PATH]
    # C locale: the host compiler's diagnostics (quote characters, translations) are then the same for every caller
    proc = subprocess.run(cmd, capture_output=True, text=True, env=dict(os.environ, LC_ALL="C"))
    if verbose or proc.returncode != 0:
        sys.stderr.write(proc.stdout + proc.stderr)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed building libgpso_b200.so")
    with open(os.path.join(HERE, "csrc", "ptxas_report.txt"), "w") as handle:
        # registers / spills / shared memory per kernel; the compile times, and the directory of the checkout in the
        # diagnostics, would change the file on every build
        text = (proc.stdout + proc.stderr).replace(os.path.dirname(HERE) + os.sep, "")
        handle.write("".join(line for line in text.splitlines(True) if "Compile time" not in line))
    return LIB_PATH


if __name__ == "__main__":
    print(build_library(force=True, verbose="-v" in sys.argv))
