"""In-tree build of libcassie2d.so (sm_100a only): `python -m cassierl_b200.build`.

Replaces the reference's src/Makefile:1-64 (g++ -> bin/libcassie2d.so linking MuJoCo, RBDL,
qpOASES).  Translation units are compiled in parallel, objects are cached by source mtime.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "lib", "obj" + ("_" + os.environ.get("CASSIE2D_VARIANT", "") if os.environ.get("CASSIE2D_VARIANT") else ""))
# CASSIE2D_VARIANT=<name> + CASSIE2D_EXTRA_FLAGS="..." build an experimental copy lib/libcassie2d_<name>.so
# (own object cache) without touching the product library; cassierl_b200.lib loads it when CASSIE2D_LIB is set.
VARIANT = os.environ.get("CASSIE2D_VARIANT", "")
EXTRA = os.environ.get("CASSIE2D_EXTRA_FLAGS", "").split()
LIB = os.path.join(HERE, "lib", "libcassie2d%s.so" % ("_" + VARIANT if VARIANT else ""))
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
NVCC_FLAGS = ARCH + ["-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC,-O2", "--expt-relaxed-constexpr"]
UNITS = ["kernels_f32.cu", "kernels_f64.cu", "rollout_f32.cu", "rollout_f64.cu", "cassie2d_api.cu", "mjcf_flatten.cpp",
         "tree_f32.cu", "tree_f64.cu", "cassie3d_api.cu"]


def _deps(unit=None):
    """Files a translation unit is rebuilt for.  The four planar kernel units take minutes each and include neither the
    3-D tree engine (tree_*, cassie3d_*) nor the host-side flattener, so edits there do not rebuild them."""
    names = os.listdir(CSRC)
    if unit and (unit.startswith("kernels_") or unit.startswith("rollout_")):
        names = [f for f in names if f == unit or (f.endswith((".cuh", ".h")) and not f.startswith(("tree_", "cassie3d", "mjcf_flatten")))]
    elif unit and (unit.startswith("tree_") or unit.startswith("cassie3d")):
        shared = ("mjcf_flatten.h", "rollout_philox.cuh", "rollout_args.h")   # the 3-D rollout's noise and sampler launches
        names = [f for f in names if f == unit or f.startswith("tree_") and f.endswith((".cuh", ".h")) or f in shared]
    inc = ("cassie3d.h",) if unit and (unit.startswith("tree_") or unit.startswith("cassie3d")) else ("cassie2d.h",)
    return [os.path.join(CSRC, f) for f in names] + [os.path.join(HERE, "..", "include", h) for h in inc]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _compile(unit, verbose):
    src = os.path.join(CSRC, unit)
    obj = os.path.join(OBJ, unit + ".o")
    if not _stale(obj, _deps(unit)):
        return obj
    # fp32 kernels: approximate (2 ulp) single-precision division / sqrt -- removes the IEEE slow-path
    # branches from the hot instruction stream (+8..30 %, profiles/r1_variants.txt); double is unaffected
    fast = ["-prec-div=false", "-prec-sqrt=false"] if unit.endswith("_f32.cu") else []
    cmd = [NVCC] + NVCC_FLAGS + fast + EXTRA + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
    if unit.endswith(".cpp"):
        cmd = [NVCC, "-O2", "-std=c++17", "-Xcompiler", "-fPIC", "-x", "c++", "-c", src, "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed on " + unit)
    return obj


def build(verbose=False, force=False):
    """Compiles every CUDA translation unit for sm_100a and links libcassie2d.so.  Returns its path."""
    os.makedirs(OBJ, exist_ok=True)
    if force:
        for f in os.listdir(OBJ):
            os.remove(os.path.join(OBJ, f))
    with ThreadPoolExecutor(max_workers=len(UNITS)) as ex:
        objs = list(ex.map(lambda u: _compile(u, verbose), UNITS))
    if _stale(LIB, objs):
        cmd = [NVCC] + ARCH + ["-shared", "-o", LIB] + objs + ["-cudart", "static", "-ldl"]
        subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv, force="-f" in sys.argv))
