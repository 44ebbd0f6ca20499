"""Builds csrc/*.cu into agent0_b200/libagent0_b200.so for sm_100a with nvcc (in-tree, so the
shared object travels with the repo snapshot to the GPU box)."""
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libagent0_b200.so")
SOURCES = ["a0_replay.cu", "a0_sumtree.cu", "a0_targets.cu", "a0_ingest.cu", "a0_extend.cu", "a0_lz4enc.cu", "a0_ckpt.cu",
           "a0_weights.cu", "a0_inbox.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "--use_fast_math=false", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=default",
              "--fmad=true", "-shared", "-cudart", "static"]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [
        os.path.join(PKG, "..", "include", "agent0_b200.h"), os.path.abspath(__file__)]
    deps = [d for d in deps if not d.endswith("a0_pyingest.c")]
    return any(os.path.getmtime(d) > t for d in deps)


TRACE_LIB = os.path.join(PKG, "libagent0_b200_trace.so")


def build(force=False, verbose=False, trace=False):
    """trace=True: the same sources with -DA0_TRACE (device-side timeline records) into
    libagent0_b200_trace.so, loaded instead of the product library when A0_LIB points at it."""
    if not trace and not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + [f for f in NVCC_FLAGS if f != "--use_fast_math=false"] + (["-DA0_TRACE"] if trace else []) + \
          [os.path.join(CSRC, s) for s in SOURCES] + ["-o", TRACE_LIB if trace else LIB]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return TRACE_LIB if trace else LIB


PYINGEST_SRC = os.path.join(CSRC, "a0_pyingest.c")
PYINGEST_LIB = os.path.join(PKG, "_a0_pyingest.so")


def build_pyingest(force=False):
    """The CPython-API marshalling helper of ReplayDataset.extend (host glue, plain gcc, no CUDA)."""
    import sysconfig
    if not force and os.path.exists(PYINGEST_LIB) and os.path.getmtime(PYINGEST_LIB) >= os.path.getmtime(PYINGEST_SRC):
        return PYINGEST_LIB
    inc = sysconfig.get_paths()["include"]
    cmd = [os.environ.get("CC", "gcc"), "-O2", "-shared", "-fPIC", "-I", inc, PYINGEST_SRC, "-o", PYINGEST_LIB]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("gcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    return PYINGEST_LIB


if __name__ == "__main__":
    build_pyingest(force="--force" in sys.argv)
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, trace="--trace" in sys.argv))
