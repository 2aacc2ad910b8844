"""Build recipe for the native parts of datum_b200.

    python -m datum_b200.build            # CUDA library + C++ host shim
    python -m datum_b200.build --oracle   # also the test-only oracle / oracle/_ref
    python -m datum_b200.build --ab       # also the TOOLS build with the A/B kernel variants of the
                                          # tuning history (tools/ab/libdatum_ibl_cuda_ab.so; not shipped,
                                          # loaded only when DATUM_IBL_CUDA_LIB points at it)

Everything is compiled in-tree so the built .so files travel with the source
snapshot to the GPU box.  nvcc cross-compiles sm_100a without a GPU present.
"""

import os
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "datum_b200", "csrc")
HOST = os.path.join(ROOT, "datum_b200", "host")
LIBDIR = os.path.join(ROOT, "datum_b200", "lib")

CUDA_LIB = os.path.join(LIBDIR, "libdatum_ibl_cuda.so")
HOST_LIB = os.path.join(LIBDIR, "libdatum_ibl_host.so")

CUDA_SOURCES = ["cabi.cu", "multi.cu", "prefilter_dn.cu", "prefilter_f.cu", "sh9.cu", "luts.cu", "resample.cu", "ibl_tables.cpp"]
AB_DIR = os.path.join(ROOT, "tools", "ab")
AB_LIB = os.path.join(AB_DIR, "libdatum_ibl_cuda_ab.so")
CUDA_HEADERS = ["ibl_math.cuh", "ibl_tables.h", "prefilter.h", "prefilter_f.h", "prefilter_pair.cuh", "sh9.h", "luts.h", "resample.h", "cabi_internal.h"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
    "-shared",
]


def _nvcc():
    for candidate in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if candidate and os.path.exists(candidate):
            return candidate
    raise RuntimeError("nvcc not found: the CUDA library cannot be built")


def _gxx():
    for candidate in ("/usr/bin/g++", shutil.which("g++")):
        if candidate and os.path.exists(candidate):
            return candidate
    raise RuntimeError("g++ not found")


def _stale(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.exists(s) and os.path.getmtime(s) > t for s in sources)


def _run(cmd, log_name=None):
    proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if log_name:
        with open(os.path.join(LIBDIR, log_name), "w") as f:
            f.write(" ".join(cmd) + "\n" + proc.stdout)
    if proc.returncode != 0:
        raise RuntimeError("build failed: %s\n%s" % (" ".join(cmd), proc.stdout))
    return proc.stdout


def build_cuda(force=False):
    os.makedirs(LIBDIR, exist_ok=True)
    sources = [os.path.join(CSRC, s) for s in CUDA_SOURCES if os.path.exists(os.path.join(CSRC, s))]
    deps = sources + [os.path.join(CSRC, h) for h in CUDA_HEADERS] + [os.path.join(ROOT, "include", "datum_ibl_cuda.h")]
    if force or _stale(CUDA_LIB, deps):
        _run([_nvcc()] + NVCC_FLAGS + ["-o", CUDA_LIB] + sources, "nvcc_build.log")
    return CUDA_LIB


def build_ab(force=False):
    """The same C ABI with every A/B kernel variant compiled in (-DDATUM_IBL_AB_VARIANTS) plus the
    round-1 first kernel (tools/ab/prefilter.cu).  For tools/level_times.py and friends only."""
    sources = [os.path.join(CSRC, s) for s in CUDA_SOURCES if os.path.exists(os.path.join(CSRC, s))] + [os.path.join(AB_DIR, "prefilter.cu")]
    deps = sources + [os.path.join(CSRC, h) for h in CUDA_HEADERS] + [os.path.join(ROOT, "include", "datum_ibl_cuda.h")]
    if force or _stale(AB_LIB, deps):
        _run([_nvcc()] + NVCC_FLAGS + ["-DDATUM_IBL_AB_VARIANTS", "-o", AB_LIB] + sources, "nvcc_build_ab.log")
    return AB_LIB


def build_host(force=False):
    """C++ host shim that keeps the reference's tools/ibl.h signatures."""
    sources = [os.path.join(HOST, s) for s in ("ibl.cpp", "hdr.cpp")]
    sources = [s for s in sources if os.path.exists(s)]
    if not sources:
        return None
    deps = sources + [os.path.join(HOST, h) for h in ("ibl.h", "hdr.h", "math.h")]
    if force or _stale(HOST_LIB, deps + [CUDA_LIB]):
        _run([_gxx(), "-std=c++14", "-O2", "-fPIC", "-shared", "-I", os.path.join(ROOT, "include"), "-o", HOST_LIB] + sources
             + ["-L", LIBDIR, "-ldatum_ibl_cuda", "-Wl,-rpath,$ORIGIN"], "host_build.log")
    return HOST_LIB


def build_oracle():
    """Test infrastructure only: the CPU oracle and (when /root/reference exists) oracle/_ref."""
    env = dict(os.environ)
    env.pop("CXX", None)
    proc = subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "all"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, env=env)
    if proc.returncode != 0:
        raise RuntimeError("oracle build failed:\n" + proc.stdout)
    return proc.stdout


def build_all(force=False, oracle=False, ab=False):
    build_cuda(force)
    build_host(force)
    if oracle:
        build_oracle()
    if ab:
        build_ab(force)


if __name__ == "__main__":
    build_all(force="--force" in sys.argv, oracle="--oracle" in sys.argv, ab="--ab" in sys.argv)
    print("built:", CUDA_LIB)
