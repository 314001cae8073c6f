"""Build libtcmp.so (hand-written CUDA for sm_100a + the C-ABI shim) in-tree with nvcc.

    python -m torque_constrained_motion_planning_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels with the repo snapshot to
the GPU box, where it is loaded as-is (no JIT cache, no torch extension machinery).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libtcmp.so")
SOURCES = ["rne_kernels.cu", "model_kernels.cu", "edge_kernels.cu", "ik_kernels.cu", "select_kernels.cu", "collision_kernels.cu", "dynamics_kernels.cu", "fd_kernels.cu", "rollout_kernels.cu", "track_kernels.cu", "payload_kernels.cu", "tcmp_api.cu"]
HEADERS = ["panda_model.cuh", "collision_core.cuh", "dynamics_core.cuh", "fd_core.cuh", "ik_core.cuh", "payload_core.cuh", "rollout_core.cuh", "select_core.cuh", "track_core.cuh", "sincos_table.inc", "tcmp_internal.h", os.path.join("..", "..", "include", "tcmp.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo", "--expt-relaxed-constexpr",
    "-Xcompiler", "-fPIC,-O2",
    "-Xptxas", "-v",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


# per-source flags of the product build
SOURCE_FLAGS = {}


def build(force: bool = False, verbose: bool = False, defines=(), suffix: str = "", source_flags=None) -> str:
    """defines/suffix/source_flags build an experimental variant (libtcmp<suffix>.so) next to the product library;
    source_flags = {"ik_kernels.cu": ["-fmad=false"], ...} is merged over SOURCE_FLAGS."""
    per_source = dict(SOURCE_FLAGS)
    per_source.update(source_flags or {})
    lib_path = LIB if not suffix else os.path.join(HERE, "libtcmp%s.so" % suffix)
    if not force and not suffix and not _stale():
        return LIB
    nvcc = _nvcc()
    objdir = os.path.join(HERE, "build" + suffix)
    os.makedirs(objdir, exist_ok=True)
    env = dict(os.environ)
    # the image's CC/CXX wrappers are not a supported nvcc host compiler setup; use the system g++
    ccbin = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")

    def compile_one(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc, "-ccbin", ccbin, *NVCC_FLAGS, *per_source.get(src, []), *["-D" + d for d in defines], "-c",
               os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True, env=env)
        log = r.stdout + r.stderr
        with open(os.path.join(objdir, src + ".ptxas.log"), "w") as f:
            f.write(log)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s" % (src, log))
        if verbose:
            print(log)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, "-ccbin", ccbin, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", lib_path, *objs]
    r = subprocess.run(cmd, capture_output=True, text=True, env=env)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    return lib_path


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
