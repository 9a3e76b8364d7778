"""In-tree build of libpnpb200.so (hand-written CUDA for sm_100a behind the C ABI in include/pnpb200.h).

    python -m pnp_solver_test_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU.  The templated solve path (csrc/pnpb200_kernels.cu) is compiled
once per (scalar type, method group) so that the objects build in parallel; objects are cached under
csrc/_obj/ and only the stale ones are rebuilt.  The .so is git-ignored but travels with the tree.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
OBJ = os.path.join(CSRC, "_obj")
LIB_PATH = os.path.join(_HERE, "libpnpb200.so")
HEADERS = ["pnpb200_common.cuh", "pnpb200_math.cuh", "pnpb200_p3p.cuh", "pnpb200_reproject.cuh", "pnpb200_solvers.cuh", "pnpb200_tile.cuh",
           os.path.join("..", "..", "include", "pnpb200.h")]
# (object name, source, extra defines)
UNITS = [("api", "pnpb200_api.cu", []), ("aux", "pnpb200_aux.cu", []), ("robust", "pnpb200_robust.cu", []), ("ransac", "pnpb200_ransac.cu", []), ("analysis", "pnpb200_analysis.cu", []),
         ("writers", "pnpb200_writers.cpp", []), ("pack", "pnpb200_pack.cpp", [])]
UNITS += [("kernels_%s_g%d" % ("f64" if f64 else "f32", g), "pnpb200_kernels.cu", ["-DPNP_F64=%d" % f64, "-DPNP_GROUP=%d" % g])
          for f64 in (1, 0) for g in (3, 1, 0, 2)]
EXTRA = os.environ.get("PNPB200_NVCC_EXTRA", "").split()
NVCC_FLAGS = EXTRA + ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-Xcompiler", "-fPIC"]


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.sep not in c or os.path.exists(c)):
            return c
    return "nvcc"


def _ccbin():
    return ["-ccbin", "/usr/bin/g++"] if os.path.exists("/usr/bin/g++") else []


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def up_to_date():
    deps = [os.path.join(CSRC, s) for s in sorted({u[1] for u in UNITS}) + HEADERS] + [os.path.abspath(__file__)]
    return not _stale(LIB_PATH, deps)


def build(force=False, verbose=False, jobs=None):
    if not force and up_to_date():
        return LIB_PATH
    os.makedirs(OBJ, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS] + [os.path.abspath(__file__)]
    todo, objs = [], []
    for name, src, defs in UNITS:
        obj = os.path.join(OBJ, name + ".o")
        objs.append(obj)
        if force or _stale(obj, [os.path.join(CSRC, src)] + hdrs):
            todo.append([_nvcc()] + _ccbin() + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + defs + ["-c", src, "-o", obj])

    def run(cmd):
        subprocess.check_call(cmd, cwd=CSRC)

    with ThreadPoolExecutor(max_workers=jobs or min(8, os.cpu_count() or 1)) as ex:
        list(ex.map(run, todo))
    subprocess.check_call([_nvcc()] + _ccbin() + ["-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-cudart", "static", "-o", LIB_PATH] + objs, cwd=CSRC)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
