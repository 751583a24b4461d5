"""Build libtrs_b200.so (sm_100a only) in-tree with nvcc.  `python -m triton_racer_sim_b200.build [--force]`."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libtrs_b200.so")
SOURCES = ["trs_api.cu", "pilot_api.cu"]
HEADERS = ["pixel_math.cuh", "preproc_kernel.cuh", "preproc_fast.cuh", "preproc_bsw.cuh", "preproc_list.h", "misc_kernels.cuh", "loc_grid.h", "loc_tracks.cuh", "jpeg_core.cuh", "jpeg_host.h", "jpeg_kernels.cuh", "jpeg_enc_core.cuh", "jpeg_enc_kernels.cuh", "pilot_kernels.cuh", "trs_internal.h", os.path.join("..", "..", "include", "trs_b200.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",   # Blackwell B200 only: no multi-arch fatbin, no PTX fallback
    "-O3", "-lineinfo", "-std=c++17",
    "-fmad=false",                                   # parity: one rounding per float op (SURVEY §7.2-6)
    "-Xcompiler", "-fPIC", "-Xcompiler", "-pthread", "-shared",
]


def nvcc_path():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    return "nvcc"


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    extra = os.environ.get("TRS_NVCC_EXTRA", "").split()          # e.g. -DTRS_PHASE_TIMERS for tools/phase_timing.py
    cmd = [nvcc_path()] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
