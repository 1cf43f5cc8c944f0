"""Builds libmd2loss.so in-tree for sm_100a with nvcc (cross-compiles without a GPU).

    python -m monodepth2_b200.build [--force] [--verbose]
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
# development knobs: MD2_LIB_NAME / MD2_NVCC_DEFS build an experimental variant next to the product library
LIB = os.path.join(LIB_DIR, os.environ.get("MD2_LIB_NAME", "libmd2loss.so"))
EXTRA_DEFS = os.environ.get("MD2_NVCC_DEFS", "").split()
SOURCES = ["md2_kernels.cu", "md2_ops.cu", "md2_capi.cu", "md2_pyramid.cu", "md2_head.cu", "md2_monitor.cu",
           "md2_decoder.cu", "md2_depth_gt.cu", "md2_jpeg.cu", "md2_png.cu"]
HEADERS = ["md2_core.cuh", "md2_pack2.cuh", "md2_roles.cuh", "md2_plan.h", "md2_velo.h", "md2_jpeg.h", "md2_png.h",
           os.path.join("..", "..", "include", "md2_loss.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "--use_fast_math=false", "-Xcompiler", "-fPIC", "-Xptxas", "-v"]


def nvcc() -> str:
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.sep not in c or os.path.exists(c)):
            return c
    raise RuntimeError("nvcc not found")


def up_to_date() -> bool:
    if not os.path.exists(LIB):
        return False
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return all(os.path.getmtime(d) <= t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and up_to_date():
        return LIB
    os.makedirs(LIB_DIR, exist_ok=True)
    objs = []
    procs = []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        if not os.path.exists(src):
            continue
        tag = os.path.basename(LIB).replace(".so", "")
        obj = os.path.join(LIB_DIR, tag + "." + s.replace(".cu", ".o"))
        cmd = [nvcc()] + [f for f in NVCC_FLAGS if f != "--use_fast_math=false"] + EXTRA_DEFS + ["-c", src, "-o", obj]
        log = open(os.path.join(LIB_DIR, tag + "." + s + ".ptxas.log"), "w")
        procs.append((subprocess.Popen(cmd, stdout=log, stderr=subprocess.STDOUT), cmd, log))
        objs.append(obj)
    for p, cmd, log in procs:
        rc = p.wait()
        log.close()
        if rc != 0:
            sys.stderr.write(open(log.name).read())
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
        if verbose:
            sys.stdout.write(open(log.name).read())
    cmd = [nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs
    subprocess.check_call(cmd)
    return LIB


DEBUG_LIB = os.path.join(LIB_DIR, "libmd2loss_dbg.so")


def build_debug(force: bool = False) -> str:
    """libmd2loss_dbg.so: the same sources with -DMD2_DBG_DEVICE -DMD2_BOUNDS_CHECK (decision export and
    index checks inside the kernels, include/md2_debug.h).  Test infrastructure; built in a child process
    because the library name and the defines are module-level settings."""
    env = dict(os.environ, MD2_LIB_NAME="libmd2loss_dbg.so", MD2_NVCC_DEFS="-DMD2_DBG_DEVICE -DMD2_BOUNDS_CHECK")
    subprocess.check_call([sys.executable, "-m", "monodepth2_b200.build"] + (["--force"] if force else []),
                          cwd=os.path.dirname(HERE), env=env, stdout=subprocess.DEVNULL)
    return DEBUG_LIB


if __name__ == "__main__":
    if "--debug" in sys.argv:
        print(build_debug(force="--force" in sys.argv))
    else:
        print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
