"""Builds liborbit_b200.so (CUDA, sm_100a only) in-tree with nvcc.  `python -m orbit_b200.build [--force]`.

The flags pin the arithmetic contract of DESIGN.md §3 a second time (the kernels already use explicit
round-to-nearest intrinsics): no fused-multiply-add contraction, IEEE division / square root, denormals kept.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "liborbit_b200.so")
SOURCES = ["api.cu", "hiz_build.cu", "entity_cull.cu", "meshlet_cull.cu", "light_cluster.cu", "scene_update.cu", "asset_bounds.cu"]
HOST_LIB_PATH = os.path.join(LIB_DIR, "liborbit_host.so")   # compiled host-side frame driver above the C ABI
HOST_SOURCES = [os.path.join(HERE, "host", "frame_driver.cpp")]
HEADERS = ["orbit_device.cuh", "scan.cuh", "params.cuh", "light_culling_kernel.cuh", "../../include/orbit_cuda.h", "../../include/orbit_layouts.h"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
    "--fmad=false", "--prec-div=true", "--prec-sqrt=true", "--ftz=false",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-fno-fast-math", "--use_fast_math=false",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def needs_build():
    if not os.path.exists(LIB_PATH) or not os.path.exists(HOST_LIB_PATH):
        return True
    t = min(os.path.getmtime(LIB_PATH), os.path.getmtime(HOST_LIB_PATH))
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + HOST_SOURCES + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, extra_flags=()):
    if not force and not needs_build():
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    flags = [f for f in NVCC_FLAGS if f != "--use_fast_math=false"] + os.environ.get("ORBIT_EXTRA_NVCC", "").split()   # development knob
    cmd = [_nvcc()] + flags + list(extra_flags) + ["-shared", "-o", os.environ.get("ORBIT_LIB_OUT", LIB_PATH)] + [os.path.join(CSRC, s) for s in SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
        print(" ".join(cmd))
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stdout + res.stderr)
    # host-side frame driver: plain C++ over the C ABI + cudart (no device code)
    cmd = [_nvcc(), "-O2", "-std=c++17", "-Xcompiler", "-fPIC", "-shared", "-I", os.path.join(HERE, "..", "include"),
           "-o", HOST_LIB_PATH] + HOST_SOURCES + ["-L", LIB_DIR, "-lorbit_b200", "-Xlinker", "-rpath=$ORIGIN"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("host driver build failed:\n" + res.stdout + res.stderr)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv or "--verbose" in sys.argv))
