"""In-tree build of the CUDA library (sm_100a only).  `python -m dart_planner_b200.build`."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
OBJDIR = os.path.join(LIBDIR, "obj")
LIB = os.path.join(LIBDIR, "libdart_se3mpc.so")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-lineinfo", "-std=c++17", "--extended-lambda", "-Xcompiler", "-fPIC"]
# per-file extra flags; the mapper needs unfused multiply/add for bit-exact voxel indices
UNITS = {
    "se3mpc_kernels.cu": [],
    "se3mpc_inst_l4.cu": [], "se3mpc_inst_l8.cu": [], "se3mpc_inst_l16.cu": [],
    "se3mpc_inst_l32.cu": [], "se3mpc_inst_l32x2.cu": [], "se3mpc_inst_l8_occ3.cu": [],
    "se3mpc_inst_l8_b64.cu": [], "se3mpc_inst_l16_occ3.cu": [], "se3mpc_inst_l32_occ3.cu": [],
    "se3mpc_inst_l6.cu": [], "se3mpc_inst_l6_occ5.cu": [], "se3mpc_vjp.cu": [],
    "mapper_kernels.cu": ["-fmad=false"],
    "probe_kernels.cu": [],
}
HEADERS = [os.path.join(CSRC, "se3mpc_core.cuh"), os.path.join(CSRC, "map_query.cuh"),
           os.path.join(CSRC, "se3mpc_kernel.cuh"),
           os.path.join(HERE, "..", "include", "dart_se3mpc.h")]


def nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: the CUDA library cannot be built")
    return exe


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _compile(unit, flags, verbose):
    src = os.path.join(CSRC, unit)
    obj = os.path.join(OBJDIR, unit.replace(".cu", ".o"))
    if not _stale(obj, [src] + HEADERS):
        return obj, ""
    cmd = [nvcc()] + ARCH + COMMON + flags + ["-Xptxas", "-v", "-c", src, "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed for {unit}:\n{r.stderr}")
    if verbose:
        print(r.stderr)
    return obj, r.stderr


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJDIR, exist_ok=True)
    if force:
        for f in os.listdir(OBJDIR):
            os.remove(os.path.join(OBJDIR, f))
    with ThreadPoolExecutor(len(UNITS)) as ex:
        res = list(ex.map(lambda kv: _compile(kv[0], kv[1], verbose), UNITS.items()))
    objs = [o for o, _ in res]
    log = "\n".join(l for _, l in res if l)
    if log:
        with open(os.path.join(LIBDIR, "ptxas.log"), "w") as fh:
            fh.write(log)
    if _stale(LIB, objs):
        cmd = [nvcc()] + ARCH + ["-shared", "-o", LIB] + objs
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stderr}")
    return LIB


# Diagnostic twin of the library for the parity A/B (tests/test_gpu_parity_sweep.py): the N <= 8
# instantiations compiled with -DDART_NO_CLOSED_FORM (the published breakpoint walk also when no
# pair is stored), everything else shared with the product build.  Never loaded by the product.
NOCF_LIB = os.path.join(LIBDIR, "libdart_se3mpc_nocf.so")
NOCF_UNITS = ["se3mpc_inst_l8.cu", "se3mpc_inst_l8_occ3.cu", "se3mpc_inst_l4.cu", "se3mpc_inst_l6.cu",
              "se3mpc_inst_l6_occ5.cu"]


def build_nocf() -> str:
    build()
    os.makedirs(OBJDIR, exist_ok=True)

    def one(unit):
        src = os.path.join(CSRC, unit)
        obj = os.path.join(OBJDIR, unit.replace(".cu", ".nocf.o"))
        if _stale(obj, [src] + HEADERS):
            r = subprocess.run([nvcc()] + ARCH + COMMON + ["-DDART_NO_CLOSED_FORM", "-c", src, "-o", obj],
                               capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError(f"nvcc failed for {unit} (nocf):\n{r.stderr}")
        return obj

    with ThreadPoolExecutor(len(NOCF_UNITS)) as ex:
        special = list(ex.map(one, NOCF_UNITS))
    objs = [os.path.join(OBJDIR, u.replace(".cu", ".o")) for u in UNITS if u not in NOCF_UNITS] + special
    if _stale(NOCF_LIB, objs):
        r = subprocess.run([nvcc()] + ARCH + ["-shared", "-o", NOCF_LIB] + objs, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed (nocf):\n{r.stderr}")
    return NOCF_LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
