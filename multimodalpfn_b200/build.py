"""Build libmmpfn_b200.so (sm_100a) in-tree with nvcc.

The library has no torch or libcuda link-time dependency (cudart is linked statically; the one
driver entry point it needs, cuTensorMapEncodeTiled, is resolved at run time), so it also loads
in a CPU-only container, where every compute entry point returns MMPFN_ENODEVICE.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")
# MMPFN_DEBUG_LIB=1 selects the tuning build (-DMMPFN_DEBUG: kernel-variant switches read from the
# environment, used by tools/ only); the product library has none of them.
DEBUG = os.environ.get("MMPFN_DEBUG_LIB", "0") == "1"
LIB = os.path.join(HERE, "libmmpfn_b200_dbg.so" if DEBUG else "libmmpfn_b200.so")
STAMP = os.path.join(HERE, ".libmmpfn_b200_dbg.stamp" if DEBUG else ".libmmpfn_b200.stamp")
SOURCES = ["api.cu", "kernels_f32.cu", "kernels_stem.cu", "kernels_tc.cu", "kernels_attn.cu", "kernels_mlp.cu", "kernels_rowgemm.cu", "kernels_featfused.cu", "kernels_tail.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "--expt-relaxed-constexpr", "-Xcompiler", "-fPIC", "-shared", "-cudart", "static",
    "-Xptxas", "-v",
] + (["-DMMPFN_DEBUG"] if DEBUG else [])
# tuning only: extra -D flags and a library name suffix for A/B builds (MMPFN_VARIANT="name:-DATTN_PIN=1 ...")
_VARIANT = os.environ.get("MMPFN_VARIANT", "")
if _VARIANT:
    _vname, _, _vflags = _VARIANT.partition(":")
    NVCC_FLAGS = NVCC_FLAGS + _vflags.split()
    LIB = os.path.join(HERE, f"libmmpfn_b200_{_vname}.so")
    STAMP = os.path.join(HERE, f".libmmpfn_b200_{_vname}.stamp")


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _digest() -> str:
    h = hashlib.sha256()
    for name in sorted(os.listdir(CSRC)) + ["../../include/mmpfn_b200.h"]:
        with open(os.path.join(CSRC, name), "rb") as f:
            h.update(name.encode())
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def is_current() -> bool:
    if not (os.path.exists(LIB) and os.path.exists(STAMP)):
        return False
    with open(STAMP) as f:
        return f.read().strip() == _digest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile if sources changed; returns the path of the shared library."""
    if not force and is_current():
        return LIB
    cmd = [_nvcc(), *NVCC_FLAGS, "-I", INCLUDE, "-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    with open(os.path.join(HERE, "build_ptxas_dbg.log" if DEBUG else "build_ptxas.log"), "w") as f:
        f.write(res.stdout + res.stderr)
    if verbose:
        print(res.stdout + res.stderr)
    with open(STAMP, "w") as f:
        f.write(_digest())
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose=True))
