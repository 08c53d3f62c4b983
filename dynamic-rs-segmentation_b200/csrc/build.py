"""Build libdrs.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python dynamic-rs-segmentation_b200/csrc/build.py [--force] [--verbose]

The shared object is written next to the package (``dynamic-rs-segmentation_b200/libdrs.so``) so that it
travels with the repo snapshot to the GPU box; it is git-ignored.  Each translation unit is compiled to an object
under ``csrc/_build/`` (cached by content digest) and the objects are linked by nvcc.
"""
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(HERE)
OUT = os.path.join(PKG, "libdrs.so")
STAMP = os.path.join(PKG, ".libdrs.stamp")
OBJ_DIR = os.path.join(HERE, "_build")
CUDA_DEPS = ["drs_api.cu", "drs_train.cuh", "drs_scene_api.cuh", "drs_common.cuh", "ptx_sm100.cuh", "conv_tc.cuh",
             "conv_simt.cuh", "ops.cuh", "scene.cuh", "wgrad_tc.cuh", "conv1_tc.cuh", "drs_comm.cuh", "variants.cuh", "pool_train.cuh", "npz_io.h", "np_softmax.h", "../../include/drs.h"]
CUDA_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC",
              "-Xcompiler", "-fvisibility=default", "--expt-relaxed-constexpr"]
# host planner: the Gaussian values must be bit-identical to NumPy's, so no fast-math and no FMA contraction
HOST_FLAGS = ["-O3", "-std=c++17", "-fPIC", "-fvisibility=default", "-ffp-contract=off", "-fno-fast-math", "-pthread"]
# (source, dependencies, compiler, flags)
UNITS = [
    ("drs_api.cu", CUDA_DEPS, "nvcc", CUDA_FLAGS),
    ("host_plan.cpp", ["host_plan.cpp", "../../include/drs.h"], "g++", HOST_FLAGS),
    ("npz_io.cpp", ["npz_io.cpp", "npz_io.h"], "g++", HOST_FLAGS),
    # the multi-scale softmax of the scene pass, for the host (drs_debug_np_softmax): same no-contraction rule as the planner
    ("np_softmax.cpp", ["np_softmax.cpp", "np_softmax.h", "../../include/drs.h"], "g++", HOST_FLAGS),
]
LINK_FLAGS = ["-shared", "-cudart", "static", "-Xcompiler", "-fPIC", "-Xlinker", "-ldl", "-Xcompiler", "-pthread"]


def _digest(deps, flags):
    h = hashlib.sha256()
    for d in deps:
        p = os.path.join(HERE, d)
        if os.path.exists(p):
            with open(p, "rb") as f:
                h.update(f.read())
    h.update(" ".join(flags).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cxx = os.environ.get("CXX", "g++")
    digs = [_digest(deps, flags) for _, deps, _, flags in UNITS]
    total = hashlib.sha256(("".join(digs) + " ".join(LINK_FLAGS)).encode()).hexdigest()
    if not force and os.path.exists(OUT) and os.path.exists(STAMP) and open(STAMP).read().strip() == total:
        return OUT
    os.makedirs(OBJ_DIR, exist_ok=True)

    def compile_unit(i):
        src, _, tool, flags = UNITS[i]
        obj = os.path.join(OBJ_DIR, os.path.splitext(src)[0] + ".o")
        stamp = obj + ".stamp"
        if not force and os.path.exists(obj) and os.path.exists(stamp) and open(stamp).read().strip() == digs[i]:
            return obj, ""
        if tool == "nvcc":
            cmd = [nvcc] + flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, os.path.join(HERE, src)]
        else:
            cmd = [cxx] + flags + ["-c", "-o", obj, os.path.join(HERE, src)]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("compiling %s failed:\n%s%s" % (src, r.stdout, r.stderr))
        with open(stamp, "w") as f:
            f.write(digs[i])
        return obj, r.stdout + r.stderr

    with ThreadPoolExecutor(max_workers=len(UNITS)) as ex:
        results = list(ex.map(compile_unit, range(len(UNITS))))
    if verbose:
        for _, log in results:
            sys.stderr.write(log)
    r = subprocess.run([nvcc] + ["-gencode", "arch=compute_100a,code=sm_100a"] + LINK_FLAGS + ["-o", OUT] + [o for o, _ in results],
                       capture_output=True, text=True)
    if verbose or r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed linking libdrs.so")
    with open(STAMP, "w") as f:
        f.write(total)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
