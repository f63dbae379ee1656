"""Builds the CUDA extension in-tree: reflaxman_b200/libreflax_b200.so (sm_100a only, no other arch, no fallback).

nvcc cross-compiles without a GPU.  The flags matter for parity: --fmad=false (no FMA contraction in device code),
-ffp-contract=off for the host-side scene flattening, and no fast-math anywhere (IEEE div/sqrt, denormals kept).
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = [os.path.join(HERE, "csrc", f) for f in ("rfx_kernels.cu", "rfx_trace_small.cu", "rfx_trace_blob.cu", "rfx_capi.cu")]
HDR = [os.path.join(HERE, "csrc", f) for f in ("rfx_kernels.h", "rfx_types.h", "rfx_device.cuh")] + [os.path.join(HERE, "..", "include", "reflax_c.h")]
OUT = os.path.join(HERE, "libreflax_b200.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "--fmad=false", "-std=c++17",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-fvisibility=hidden,-O2",
    "-shared",
]


def stale():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(p) > t for p in SRC + HDR + [os.path.abspath(__file__)])


def build(force=False, verbose=False, defines=(), out=None):
    """defines/out: build an experimental variant (tools/variants.py) next to the product library"""
    if out is None and not force and not stale():
        return OUT
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc, *NVCC_FLAGS, *["-D" + d for d in defines], "-o", out or OUT, *SRC]
    if verbose:
        cmd += ["-Xptxas", "-v"]
        print(" ".join(cmd), file=sys.stderr)
    subprocess.run(cmd, check=True)
    return out or OUT


SHIM_HARNESS = os.path.join(HERE, "..", "build", "shim_harness")


def build_shim_harness(force=False):
    """oracle/ref_harness.cpp — the very source that drives the unmodified reference — compiled against the shim headers
    (reflaxman_b200/shim) and linked with the CUDA library instead of the reference's src/common: the drop-in proof."""
    src = os.path.join(HERE, "..", "oracle", "ref_harness.cpp")
    out = os.path.abspath(SHIM_HARNESS)
    deps = [src, OUT, os.path.join(HERE, "shim", "rfx_shim.hpp")]
    if not force and os.path.exists(out) and all(os.path.getmtime(d) <= os.path.getmtime(out) for d in deps):
        return out
    os.makedirs(os.path.dirname(out), exist_ok=True)
    subprocess.run(["g++", "-std=c++14", "-O2", "-ffp-contract=off", "-I" + os.path.join(HERE, "shim"), "-I" + os.path.join(HERE, "..", "include"),
                    "-o", out, src, "-L" + HERE, "-lreflax_b200", "-Wl,-rpath," + HERE], check=True)
    return out


SHIM_PULSE = os.path.join(HERE, "..", "build", "shim_pulse_headless")
# src/common of an upstream ReflaxMan checkout: the unmodified reference, which this repository does not contain
REFERENCE_SRC = os.environ.get("RFX_REFERENCE_SRC", "")


def build_shim_pulse(force=False):
    """The reference's UI controller — Pulse.cpp and BasePlatformInterface.cpp, compiled UNCHANGED from where they lie —
    against the shim headers, linked with the CUDA library and the headless platform stub: a front end running on the GPU
    path (SURVEY §8 f-2).  Needs the reference tree (REFERENCE_SRC).
    Returns the path, or None when neither the tree nor a prebuilt binary exists."""
    import shutil
    import tempfile
    out = os.path.abspath(SHIM_PULSE)
    drv = os.path.join(HERE, "..", "oracle", "pulse_headless.cpp")
    if not os.path.isdir(REFERENCE_SRC):
        return out if os.access(out, os.X_OK) else None
    deps = [drv, OUT, os.path.join(HERE, "shim", "rfx_shim.hpp"), os.path.join(REFERENCE_SRC, "Pulse.cpp")]
    if not force and os.path.exists(out) and all(os.path.getmtime(d) <= os.path.getmtime(out) for d in deps):
        return out
    os.makedirs(os.path.dirname(out), exist_ok=True)
    with tempfile.TemporaryDirectory() as td:
        for f in ("Pulse.h", "Pulse.cpp", "BasePlatformInterface.h", "BasePlatformInterface.cpp", "defaults.h"):
            os.symlink(os.path.join(REFERENCE_SRC, f), os.path.join(td, f))     # the reference's own files, untouched
        for f in os.listdir(os.path.join(HERE, "shim")):
            shutil.copy(os.path.join(HERE, "shim", f), td)                      # our headers stand in for Render.h, Scene.h, ...
        subprocess.run(["g++", "-std=c++14", "-O2", "-DNDEBUG", "-ffp-contract=off", "-Wno-multichar", "-I" + td, "-I" + os.path.join(HERE, "..", "include"),
                        "-o", out, drv, os.path.join(td, "Pulse.cpp"), os.path.join(td, "BasePlatformInterface.cpp"),
                        "-L" + HERE, "-lreflax_b200", "-Wl,-rpath," + HERE], check=True)
    return out


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
    build_shim_harness(force=True)
    build_shim_pulse(force=True)
