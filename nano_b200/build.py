"""In-tree build of the product libraries (nvcc cross-compiles sm_100a without a GPU).

    nano_b200/lib/libnano_b200.so        engine + C-ABI (include/nano_b200.h)        <- csrc/engine.cu, kernels.cuh
    nano_b200/lib/libnano_infer_b200.so  reference host API (infer.h symbols)        <- csrc/infer_b200.c

The outputs are git-ignored but travel to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "nano_b200", "csrc")
LIB = os.path.join(ROOT, "nano_b200", "lib")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

ENGINE_SO = os.path.join(LIB, "libnano_b200.so")
SHIM_SO = os.path.join(LIB, "libnano_infer_b200.so")


def _newer(target: str, sources) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources if os.path.exists(s))


# translation units of libnano_b200.so and what each depends on (besides itself)
UNITS = {
    "engine.cu": ["kernels.cuh", "expf_ref.cuh", "stream_args.h", "stream_host.h", "sample_host.h", "../../include/nano_b200.h"],
    "stream.cu": ["kernels.cuh", "expf_ref.cuh", "stream_args.h", "stream_host.h", "stream.cuh"],
    "sample.cu": ["kernels.cuh", "expf_ref.cuh", "sample_host.h"],
}


def build_engine(force: bool = False, verbose: bool = False) -> str:
    """One object per translation unit (compiled in parallel, only when its sources changed), then one link."""
    os.makedirs(LIB, exist_ok=True)
    base = [NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC"]
    if verbose:
        base.insert(1, "-Xptxas=-v")
    objs, procs = [], []
    for unit, deps in UNITS.items():
        obj = os.path.join(LIB, unit[:-3] + ".o")
        objs.append(obj)
        if force or _newer(obj, [os.path.join(CSRC, unit)] + [os.path.join(CSRC, d) for d in deps]):
            procs.append((unit, subprocess.Popen(base + ["-c", os.path.join(CSRC, unit), "-o", obj])))
    failed = [u for u, p in procs if p.wait() != 0]
    if failed:
        raise RuntimeError("nvcc failed for " + ", ".join(failed))
    if procs or _newer(ENGINE_SO, objs):
        subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", ENGINE_SO] + objs, check=True)
    return ENGINE_SO


TRACE_SO = os.path.join(LIB, "libnano_b200_trace.so")


def build_trace_variant() -> str:
    """Developer build of the streaming kernel with its fine cycle stamps compiled in (-DNB200_FINE_TRACE; they cost ~200
    cycles each, so the product library never carries them).  Loaded by tools/gpu_trace.py through NB200_ENGINE_SO."""
    build_engine()
    obj = os.path.join(LIB, "stream_trace.o")
    subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
                    "-DNB200_FINE_TRACE", "-c", os.path.join(CSRC, "stream.cu"), "-o", obj], check=True)
    objs = [os.path.join(LIB, u[:-3] + ".o") for u in UNITS if u != "stream.cu"] + [obj]
    subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", TRACE_SO] + objs, check=True)
    return TRACE_SO


def build_shim(force: bool = False) -> str:
    src = os.path.join(CSRC, "infer_b200.c")
    hdrs = [os.path.join(ROOT, "include", "nano_infer_abi.h"), os.path.join(ROOT, "include", "nano_b200.h")]
    if force or _newer(SHIM_SO, [src] + hdrs + [ENGINE_SO]):
        cmd = ["gcc", "-O2", "-Wall", "-fPIC", "-shared", "-I" + os.path.join(ROOT, "include"), src, "-o", SHIM_SO,
               "-L" + LIB, "-lnano_b200", "-Wl,-rpath,$ORIGIN", "-lm"]
        subprocess.run(cmd, check=True)
    return SHIM_SO


def build_all(force: bool = False, verbose: bool = False) -> None:
    build_engine(force, verbose)
    build_shim(force)


if __name__ == "__main__":
    build_all(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print("built:", ENGINE_SO, SHIM_SO)
