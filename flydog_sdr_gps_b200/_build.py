"""Build the CUDA library in-tree (flydog_sdr_gps_b200/csrc/libacq_b200.so) for sm_100a.

nvcc cross-compiles without a GPU, so this also runs in the CPU-only development container.
The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libacq_b200.so")
CU_SOURCES = ["acq_kernels.cu", "acq_api.cu", "acq_microbench.cu"]
CPP_SOURCES = ["search_dropin.cpp"]
HEADERS = ["acq_fft.cuh", "acq_geom.h", "acq_kernels.cuh", "e1b_codes.inc", os.path.join("..", "..", "include", "search_dropin.h"),
           os.path.join("..", "..", "include", "acq_b200.h")]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def _nvcc():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: cannot build libacq_b200.so")


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in CU_SOURCES + CPP_SOURCES + HEADERS]
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, defines=(), out=None):
    """Compile every CUDA/C++ source of the engine into one shared library. Returns its path.
    `defines` / `out` build an experiment variant next to the product library (A/B runs: ACQ_B200_LIB=<path>)."""
    if out is None and not force and not needs_build():
        return LIB
    lib = out or LIB
    srcs = [os.path.join(CSRC, f) for f in CU_SOURCES + CPP_SOURCES if os.path.exists(os.path.join(CSRC, f))]
    cmd = [_nvcc()] + NVCC_FLAGS + ["-D" + d for d in defines] + (["-Xptxas", "-v"] if verbose else []) + ["-o", lib + ".tmp"] + srcs
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n%s\n%s" % (" ".join(cmd), res.stderr[-4000:]))
    os.replace(lib + ".tmp", lib)
    if verbose:
        print(res.stderr)
    return lib


# Experiment variants: the reference sides of the kernel-equivalence tests, and instrumentation.  They are separate
# libraries: the product library contains none of this code and reads no environment variable.
VARIANTS = {
    "l1_multi_tw": ["ACQ_VARIANT_L1_MULTI_TW"],  # K > 1 C/A search with the twiddles (not the code run) in tensor memory
    "l1_cta": ["ACQ_FORCE_L1_CTA=1"],        # K = 1 C/A search always by k_search_l1<false> (two CTAs per SM, thread 0 stages)
    "e1b_ldg": ["ACQ_VARIANT_E1B_LDG", "ACQ_FORCE_E1B_KERNEL=1"],  # one-CTA E1B search, operands straight from L2
    "e1b_cta": ["ACQ_FORCE_E1B_KERNEL=1"],   # always the one-CTA E1B form
    "e1b_cluster": ["ACQ_FORCE_E1B_KERNEL=2"],  # always the cluster/DSMEM E1B form
    "trace": ["ACQ_TRACE"],                  # %globaltimer stamps per CTA (tools/trace_timeline.py)
    "static_tiles": ["ACQ_DYN_MIN_ROUNDS=1000000000"],  # strided search kernels always on the static stride (the product: tiles claimed from a counter from 6 rounds up)
    "dyn_tiles": ["ACQ_DYN_MIN_ROUNDS=0"],    # ... always claiming
    "argin0": ["ACQ_ARG_INPUT=0"],           # single-block captures through the staging buffer + copy node (the product: kernel argument)
}


def variant_path(name):
    return os.path.join(CSRC, "variants", "libacq_b200_%s.so" % name)


def build_variant(name, force=False):
    path = variant_path(name)
    deps = [os.path.join(CSRC, f) for f in CU_SOURCES + CPP_SOURCES + HEADERS]
    fresh = os.path.exists(path) and all(os.path.getmtime(d) <= os.path.getmtime(path) for d in deps if os.path.exists(d))
    if fresh and not force:
        return path
    os.makedirs(os.path.dirname(path), exist_ok=True)
    return build(defines=VARIANTS[name], out=path)


if __name__ == "__main__":
    print(build(force=True, verbose=True))
