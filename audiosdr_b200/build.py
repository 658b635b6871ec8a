"""audiosdr_b200/build.py -- compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libsdr_batch.so")
SOURCES = ["sdr_kernel.cu", "sdr_pipe_t32.cu", "sdr_pipe_t16.cu", "sdr_pipe_t8.cu", "sdr_pipe_t32c.cu", "sdr_pipe_t32s.cu", "sdr_als_pass.cu", "sdr_host.cpp"]
DEPS = SOURCES + ["sdr_pipeline.cuh", "sdr_pipe_tu.cuh", "sdr_lay.h", "sdr_types.h", "sdr_kernel.h", "sdr_tables.inc", os.path.join("..", "..", "include", "sdr_batch.h")]

# -fmad=false: the reference rounds every product and every sum separately (x86-64 SSE, no FMA); contraction
# would change low bits and, through the blanker/AGC/PLL thresholds, whole decisions.  Division and square root
# stay IEEE (nvcc defaults), denormals are kept (no -ftz).
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-fmad=false", "-prec-div=true",
              "-prec-sqrt=true", "-ftz=false", "--extended-lambda", "-std=c++17", "-Xcompiler", "-fPIC", "-shared",
              "-diag-suppress", "186"]


AUX_LIB = os.path.join(HERE, "libsdr_aux.so")
AUX_DEPS = ["sdr_aux.cu", "sdr_aux_core.cuh", "aux_tables.inc", os.path.join("..", "..", "include", "sdr_aux.h")]


def _nvcc():
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in DEPS)


def build_library(force=False, verbose=False):
    """Builds audiosdr_b200/libsdr_batch.so; returns its path."""
    if not force and not needs_build():
        return LIB
    # SDR_NVCC_EXTRA: extra -D switches for A/B builds of kernel variants (tools/gpu_ab.sh); unset for the product
    cmd = [_nvcc()] + NVCC_FLAGS + ["--threads", "8"] + os.environ.get("SDR_NVCC_EXTRA", "").split() + (["-Xptxas", "-v"] if verbose else [])
    # sdr_host.cpp is plain C++ that calls the CUDA runtime: compile it as CUDA so that one nvcc call links everything
    for src in SOURCES:
        cmd += ["-x", "cu", os.path.join(CSRC, src)]
    cmd += ["-o", LIB]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stdout + r.stderr)
    return LIB


def needs_aux_build():
    return not (os.path.exists(AUX_LIB) and all(os.path.getmtime(os.path.join(CSRC, d)) <= os.path.getmtime(AUX_LIB) for d in AUX_DEPS))


def build_aux_library(force=False, verbose=False):
    """Builds audiosdr_b200/libsdr_aux.so (pre-processor + I/Q generator, include/sdr_aux.h); returns its path."""
    if not force and not needs_aux_build():
        return AUX_LIB
    cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + [os.path.join(CSRC, "sdr_aux.cu"), "-o", AUX_LIB]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stdout + r.stderr)
    return AUX_LIB


GRAPH_LIB = os.path.join(HERE, "libsdr_graph.so")
GRAPH_DEPS = ["sdr_graph.cpp"] + [os.path.join("..", "..", "include", h) for h in ("sdr_graph.h", "sdr_batch.h", "sdr_aux.h")]


def needs_graph_build():
    if not os.path.exists(GRAPH_LIB):
        return True
    t = os.path.getmtime(GRAPH_LIB)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in GRAPH_DEPS) or any(os.path.getmtime(p) > t for p in (LIB, AUX_LIB))


def build_graph_library(force=False, verbose=False):
    """Builds audiosdr_b200/libsdr_graph.so (include/sdr_graph.h) after the two libraries it links; returns its path."""
    build_library()
    build_aux_library()
    if not force and not needs_graph_build():
        return GRAPH_LIB
    # host code only (it drives the other two libraries' device entry points); $ORIGIN: they are found beside it
    cmd = [_nvcc()] + NVCC_FLAGS + [os.path.join(CSRC, "sdr_graph.cpp"), "-o", GRAPH_LIB, "-L" + HERE, "-lsdr_batch", "-lsdr_aux",
                                    "-Xlinker", "-rpath,$ORIGIN"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    return GRAPH_LIB


if __name__ == "__main__":
    import sys
    print(build_library(force="--force" in sys.argv, verbose=True))
    print(build_aux_library(force="--force" in sys.argv, verbose=True))
    print(build_graph_library(force="--force" in sys.argv))
