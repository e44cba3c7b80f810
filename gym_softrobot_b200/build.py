"""Build the sm_100a shared library in-tree (gym_softrobot_b200/lib/libsoftrod.so).

nvcc cross-compiles without a GPU; the built .so is git-ignored but travels to the GPU box with the gpurun
snapshot.  Every (type, CTA size, feature group) of the kernels is its own translation unit (csrc/inst_*.cu with
-D selectors), compiled in parallel into lib/obj/ and linked once.  Concurrent builders (one rank per GPU under
torchrun import the package at the same time) serialise on a file lock, and the library is moved into place
atomically, so nobody can dlopen a half-written file.
"""
import concurrent.futures
import fcntl
import os
import shutil
import subprocess
import tempfile

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_DIR = os.path.join(_HERE, "lib")
OBJ_DIR = os.path.join(LIB_DIR, "obj")
LIB_PATH = os.path.join(LIB_DIR, "libsoftrod.so")
_COMMON = ["rod_kernels.cuh", "rod_math.cuh", "launch.cuh", "util_kernels.cuh", os.path.join("..", "..", "include", "softrod.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
]
PACKED_SIZES = [(256, 2), (384, 1), (512, 1), (544, 1), (768, 1), (1024, 1)]   # (threads per CTA, CTAs per SM)
# The lean kernel's translation units: (model, layout, storage types, (threads per CTA, CTAs per SM)), by the
# enumerator names of LeanModel / LeanLayout in csrc/launch.cuh.  softrod_api.cu's lean_built() names the same sizes.
LEAN_UNITS = [
    ("PLAIN", "CTA", ("double", "float"), PACKED_SIZES),
    ("PLANE", "CTA", ("double",), PACKED_SIZES),
    ("MUSCLE", "CTA", ("double",), PACKED_SIZES),
    ("ASSEMBLY", "CTA", ("double",), PACKED_SIZES),
    # up to 768 threads: filter rods of >= 768 elements take the cluster layout
    ("FILTER", "CTA", ("double",), [s for s in PACKED_SIZES if s[0] <= 768]),
    ("SPLINE", "CTA", ("double",), PACKED_SIZES),
    # the lean kernel's CTA sizes for rods of <= 511 elements (fast-only kernel), and 768 threads: 15 rods of n = 50
    ("PLANAR", "CTA", ("double",), [s for s in PACKED_SIZES if s[0] <= 512 or s[0] == 768]),
    # a rod of exactly 512 elements in 512 threads
    ("PLAIN", "FOLD", ("double",), [(512, 1)]),
    ("PLANE", "FOLD", ("double",), [(512, 1)]),
    # rods of 512-4095 elements, one per thread-block cluster of 512-thread CTAs
    ("PLAIN", "CLUSTER", ("double",), [(512, 1)]),
    ("FILTER", "CLUSTER", ("double",), [(512, 1)]),
    ("PLANE", "CLUSTER", ("double",), [(512, 1)]),
    ("MUSCLE", "CLUSTER", ("double",), [(512, 1)]),
    ("SPLINE", "CLUSTER", ("double",), [(512, 1)]),
]


def translation_units():
    """[(object name, source, extra -D flags, header deps)]"""
    tus = [("api", "softrod_api.cu", [], _COMMON + ["copy_kernels.cuh"]), ("warp", "inst_warp.cu", [], _COMMON)]
    for model, layout, types, sizes in LEAN_UNITS:
        for t in types:
            for nt, minb in sizes:
                tus.append((f"lean_{model.lower()}_{layout.lower()}_{t}_{nt}", "inst_lean.cu",
                            [f"-DSR_TU_T={t}", f"-DSR_TU_NT={nt}", f"-DSR_TU_MINB={minb}", f"-DSR_TU_MODEL={model}",
                             f"-DSR_TU_LAYOUT={layout}"],
                            _COMMON + ["rod_kernel_lean.cuh"]))
    for nt, minb in PACKED_SIZES:
        for t in ("double", "float"):
            for grp in (1, 2, 3):    # (the lean configs of both types run rod_kernel_lean.cuh)
                tus.append((f"packed_{t}_{nt}_g{grp}", "inst_packed.cu",
                            [f"-DSR_TU_T={t}", f"-DSR_TU_F64={int(t == 'double')}", f"-DSR_TU_NT={nt}", f"-DSR_TU_MINB={minb}", f"-DSR_TU_GROUP={grp}"],
                            _COMMON + ["rod_kernel_packed.cuh"]))
    for nt, minb in ((384, 1), (1024, 1)):     # tapered rods: per-element constants in registers (168 / 64 of them)
        tus.append((f"packed_double_{nt}_g4", "inst_packed.cu",
                    ["-DSR_TU_T=double", "-DSR_TU_F64=1", f"-DSR_TU_NT={nt}", f"-DSR_TU_MINB={minb}", "-DSR_TU_GROUP=4"],
                    _COMMON + ["rod_kernel_packed.cuh"]))
    tus.append(("packed_double_384_g5", "inst_packed.cu",     # tapered assembly + COOMM muscle layers (OctoReach / OctoArmTwo)
                ["-DSR_TU_T=double", "-DSR_TU_F64=1", "-DSR_TU_NT=384", "-DSR_TU_MINB=1", "-DSR_TU_GROUP=5"],
                _COMMON + ["rod_kernel_packed.cuh"]))
    return tus


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA extension cannot be built (there is no CPU fallback)")


def _newest(paths):
    return max(os.path.getmtime(p) for p in paths)


def _tu_deps(src, deps):
    return [os.path.join(CSRC, src)] + [os.path.join(CSRC, d) for d in deps]


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(_newest(_tu_deps(src, deps)) > t for _, src, _, deps in translation_units())


def _compile(job):
    name, src, defs, obj, verbose = job
    cmd = [_nvcc()] + NVCC_FLAGS + defs + (["-Xptxas", "-v"] if verbose else []) + \
          ["-c", os.path.join(CSRC, src), "-o", obj + ".tmp"]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"nvcc failed on {name}:\n{res.stdout}")
    os.replace(obj + ".tmp", obj)
    return name, res.stdout


def build_library(force: bool = False, verbose: bool = False, only=None) -> str:
    """Compile every CUDA translation unit for sm_100a (those whose sources changed, or all with `force`)
    and link libsoftrod.so.  `only`: substring filter on the object names that get (re)compiled."""
    os.makedirs(OBJ_DIR, exist_ok=True)
    with open(os.path.join(LIB_DIR, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not is_stale():
                return LIB_PATH      # somebody else built it while we waited
            jobs, objs = [], []
            for name, src, defs, deps in translation_units():
                obj = os.path.join(OBJ_DIR, name + ".o")
                objs.append(obj)
                fresh = os.path.exists(obj) and os.path.getmtime(obj) >= _newest(_tu_deps(src, deps))
                if only is not None and only not in name and os.path.exists(obj) and \
                        os.path.getmtime(obj) >= _newest(_tu_deps(src, _COMMON)):
                    continue     # quick partial rebuild: allowed only while the shared headers (RodArgs layout!) are older
                if force or not fresh:
                    jobs.append((name, src, defs, obj, verbose))
            workers = max(1, min(len(jobs), os.cpu_count() or 1))
            if jobs:
                with concurrent.futures.ThreadPoolExecutor(max_workers=workers) as ex:
                    for name, out in ex.map(_compile, jobs):
                        if verbose and out.strip():
                            print(f"--- {name}\n{out}")
            fd, tmp = tempfile.mkstemp(suffix=".so", dir=LIB_DIR)
            os.close(fd)
            res = subprocess.run([_nvcc(), "-shared", "-o", tmp] + objs, stdout=subprocess.PIPE,
                                 stderr=subprocess.STDOUT, text=True)
            if res.returncode != 0:
                os.unlink(tmp)
                raise RuntimeError("link failed:\n" + res.stdout)
            os.chmod(tmp, 0o755)
            os.replace(tmp, LIB_PATH)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB_PATH


if __name__ == "__main__":
    import sys
    only = sys.argv[1] if len(sys.argv) > 1 else None
    print(build_library(force=only is None, verbose=True, only=only))
