"""Build the native code in-tree: the CUDA engine, down-converter and filter bank `pyradiotracking_b200/csrc/librtb200.so` (sm_100a only) and the CPython
helper of the host finaliser `pyradiotracking_b200/_rtfinal.so` (csrc/rt_pyfinal.c, gcc).

nvcc cross-compiles without a GPU, so this runs in the build container; the resulting
shared libraries travel to the B200 box with the source tree.
"""
import os
import shutil
import subprocess
import sys
import sysconfig

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "librtb200.so")
PYFINAL_SRC = os.path.join(CSRC, "rt_pyfinal.c")
PYFINAL = os.path.join(HERE, "_rtfinal.so")
SOURCES = ["rt_engine.cu", "rt_ddc.cu", "rt_fbank.cu", "rt_matcher.cpp"]
HEADERS = ["predicate.h", "sample_format.cuh", "fir_history.cuh", "fft_cpk.cuh", "spectro256.cuh", "spectro_tc256.cuh", "spectro_r16.cuh", os.path.join("..", "..", "include", "rt_engine.h"),
           os.path.join("..", "..", "include", "rt_matcher.h"), os.path.join("..", "..", "include", "rt_ddc.h"),
           os.path.join("..", "..", "include", "rt_fbank.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
]


def nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA engine cannot be built (there is no CPU fallback)")


def stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps)


def build_pyfinal(force: bool = False) -> str:
    """The Signal-object builder (CPython C API + datetime C API), compiled against this interpreter's headers."""
    if not force and os.path.exists(PYFINAL) and os.path.getmtime(PYFINAL) >= os.path.getmtime(PYFINAL_SRC):
        return PYFINAL
    cc = shutil.which("gcc") or shutil.which("cc")
    if not cc:
        raise RuntimeError("gcc not found: the finaliser helper cannot be built")
    cmd = [cc, "-O2", "-shared", "-fPIC", "-I" + sysconfig.get_paths()["include"], "-o", PYFINAL, PYFINAL_SRC]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("gcc failed:\n" + res.stdout + res.stderr)
    return PYFINAL


def build(force: bool = False, verbose: bool = False) -> str:
    build_pyfinal(force)
    if not force and not stale():
        return LIB
    cmd = [nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + SOURCES
    res = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        sys.stderr.write(res.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
