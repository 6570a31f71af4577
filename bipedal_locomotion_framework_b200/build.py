"""In-tree build of the native pieces (no JIT cache: the .so files travel with the snapshot).

  lib/libblf_ccm.so        CUDA kernels + C ABI (nvcc, sm_100a only)
  lib/libblf_contact.so    C++17 host facade over the C ABI (g++)            [build_cpp]
  lib/blf_cpp_tests        the reference's Catch2 sections restated          [build_cpp]
"""
from __future__ import annotations

import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(_HERE)
LIB_DIR = os.path.join(_HERE, "lib")
CUDA_LIB = os.path.join(LIB_DIR, "libblf_ccm.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-fvisibility=hidden", "-shared",
]


def _newer(target: str, sources: list[str]) -> bool:
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(s) <= t for s in sources)


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; cannot build the sm_100a library")


def cuda_sources() -> list[str]:
    c = os.path.join(_HERE, "csrc")
    return [os.path.join(c, f) for f in sorted(os.listdir(c))] + \
        [os.path.join(ROOT, "include", "blf_ccm.h")]


def build_cuda(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(LIB_DIR, exist_ok=True)
    if not force and _newer(CUDA_LIB, cuda_sources()):
        return CUDA_LIB
    # three CUDA translation units compiled side by side (ccm_capi.cu: C ABI + contact / estimator /
    # system kernels; dyn_kernels.cu + dyn_kernels_wide.cu: the unrolled mass-matrix solves) + the host-only expansion
    # helper (plain C++, passed through to g++); one device link-free shared library
    from concurrent.futures import ThreadPoolExecutor

    obj_dir = os.path.join(LIB_DIR, "obj")
    os.makedirs(obj_dir, exist_ok=True)
    units = ["ccm_capi.cu", "dyn_kernels.cu", "dyn_kernels_wide.cu", "host_expand.cpp"]
    compile_flags = [f for f in NVCC_FLAGS if f != "-shared"]

    def compile_one(name: str) -> tuple[str, str]:
        obj = os.path.join(obj_dir, name.rsplit(".", 1)[0] + ".o")
        cmd = [_nvcc(), *compile_flags, "-c", "-o", obj, os.path.join(_HERE, "csrc", name)]
        if verbose and name.endswith(".cu"):
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed on " + name + ":\n" + r.stdout)
        return obj, r.stdout

    with ThreadPoolExecutor(max_workers=len(units)) as ex:
        results = list(ex.map(compile_one, units))
    if verbose:
        for _, out in results:
            print(out)
    cmd = [_nvcc(), *NVCC_FLAGS, "-o", CUDA_LIB, *[o for o, _ in results], "-lcudart", "-ldl", "-lpthread"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc link failed:\n" + r.stdout)
    return CUDA_LIB


CPP_DIR = os.path.join(_HERE, "cpp")
CPP_LIB = os.path.join(LIB_DIR, "libblf_contact.so")
CPP_TESTS = {
    "ContinuousContactModelUnitTests": "ContinuousContactModelTest.cpp",   # needs a GPU
    "ParametersHandlerUnitTests": "ParametersHandlerTest.cpp",             # host only
    "RecursiveLeastSquareUnitTests": "RecursiveLeastSquareTest.cpp",       # needs a GPU
    "IntegratorUnitTests": "IntegratorTest.cpp",                           # host section + GPU
    "ContactWrenchUnitTests": "ContactWrenchTest.cpp",                     # host only
    "FloatingBaseSystemDynamicsUnitTests": "FloatingBaseSystemDynamicsTest.cpp",   # needs a GPU
    "ApiConformanceUnitTests": "ApiConformanceTest.cpp",                   # compile-time signature checks
    "ContactWrenchGradientUnitTests": "ContactWrenchGradientTest.cpp",     # needs a GPU
    "RolloutGradientUnitTests": "RolloutGradientTest.cpp",                 # needs a GPU
}
CXX_FLAGS = ["-std=c++17", "-O2", "-fPIC", "-Wall", "-Wextra"]


def _cpp_sources() -> list[str]:
    out = []
    for root, _, files in os.walk(CPP_DIR):
        out += [os.path.join(root, f) for f in files if f.endswith((".h", ".cpp", ".txt"))]
    return out + [os.path.join(ROOT, "include", "blf_ccm.h")]


def build_cpp(force: bool = False) -> str:
    """C++17 host facade (libblf_contact.so, links libblf_ccm.so) and its test executables."""
    build_cuda()
    cxx = shutil.which("g++") or "g++"
    inc = ["-I", os.path.join(CPP_DIR, "include"), "-I", os.path.join(ROOT, "include")]
    srcs = sorted(os.path.join(CPP_DIR, "src", f) for f in os.listdir(os.path.join(CPP_DIR, "src"))
                  if f.endswith(".cpp"))
    deps = _cpp_sources() + [CUDA_LIB]

    def run(cmd):
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if r.returncode != 0:
            raise RuntimeError(" ".join(cmd) + "\n" + r.stdout)

    if force or not _newer(CPP_LIB, deps):
        run([cxx, *CXX_FLAGS, "-shared", "-o", CPP_LIB, *srcs, *inc, "-L", LIB_DIR, "-lblf_ccm",
             "-Wl,-rpath,$ORIGIN"])
    for exe, src in CPP_TESTS.items():
        target = os.path.join(LIB_DIR, exe)
        if force or not _newer(target, deps + [CPP_LIB]):
            run([cxx, *CXX_FLAGS, "-DCATCH_CONFIG_MAIN", "-o", target,
                 os.path.join(CPP_DIR, "tests", src), *inc, "-I", os.path.join(CPP_DIR, "tests"),
                 "-L", LIB_DIR, "-lblf_contact", "-lblf_ccm", "-Wl,-rpath,$ORIGIN"])
    # host-only test of the expansion helper and its worker pool (no CUDA, no facade library)
    target = os.path.join(LIB_DIR, "HostExpandUnitTests")
    hsrc = [os.path.join(CPP_DIR, "tests", "HostExpandTest.cpp"), os.path.join(_HERE, "csrc", "host_expand.cpp")]
    if force or not _newer(target, hsrc + [os.path.join(_HERE, "csrc", "host_expand.h")]):
        run([cxx, "-std=c++17", "-O2", "-Wall", "-Wextra", "-pthread", "-o", target, *hsrc])
    return CPP_LIB


if __name__ == "__main__":
    import sys
    print(build_cuda(force="--force" in sys.argv, verbose="-v" in sys.argv))
    print(build_cpp(force="--force" in sys.argv))
