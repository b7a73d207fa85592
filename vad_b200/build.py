"""In-tree build of the C-ABI library (nvcc, sm_100a only).  ``python -m vad_b200.build``."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libvadb200.so")
SOURCES = ["vadb200.cu", "vad_resample.cu"]
def _deps():
    """Every source the library is compiled from: csrc/*.{cu,cuh,h} and the public header."""
    names = [f for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh", ".h"))]
    return names + [os.path.join("..", "..", "include", "vadb200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "--expt-relaxed-constexpr", "-diag-suppress", "20091", "--shared", "-Xcompiler", "-fPIC"]


def is_stale():
    if not os.path.isfile(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in _deps())


LIB_DEBUG = os.path.join(HERE, "libvadb200_dbg.so")


def build(force=False, verbose=False, debug_hooks=False):
    """Compile csrc/*.cu into vad_b200/libvadb200.so (cross-compiles without a GPU).
    debug_hooks=True builds vad_b200/libvadb200_dbg.so instead: the same kernels plus the
    timing-experiment hooks (VADB200_DEBUG_SKIP phase ablation, VADB200_CTAS_PER_SM, clock64 stamps)
    used by tools/dbg_block_phase.py; select it with VADB200_LIB.  The hooks cost ~1 %, so the product
    library never contains them."""
    out = LIB_DEBUG if debug_hooks else LIB
    if not debug_hooks and not force and not is_stale():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.isfile(nvcc):
        nvcc = "nvcc"
    cmd = [nvcc] + NVCC_FLAGS + (["-DVADB_DEBUG_HOOKS"] if debug_hooks else []) + \
        (["-Xptxas", "-v"] if verbose else []) + ["-o", out] + SOURCES
    r = subprocess.run(cmd, cwd=CSRC, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or r.returncode != 0:
        sys.stderr.write(r.stdout)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed building " + os.path.basename(out))
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, debug_hooks="--debug-hooks" in sys.argv))
