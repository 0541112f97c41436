"""Builds libbpe_b200.so in-tree with nvcc for sm_100a (no torch extension machinery: the library
is a plain C-ABI shared object, see include/bpe_b200.h)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libbpe_b200.so")
SOURCES = ["bpe_b200.cu", "synth.cpp"]
DEPS = ["common.cuh", "train_kernels.cuh", "encode_kernels.cuh", "encode_lanes.cuh", "mg_kernels.cuh", "round_kernels.cuh", "text_kernels.cuh", os.path.join("..", "..", "include", "bpe_b200.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17", "-shared",
    "-Xcompiler", "-fPIC,-pthread",
]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + DEPS)


def build(force: bool = False, verbose: bool = False, out: str = LIB) -> str:
    if not force and out == LIB and not needs_build():
        return LIB
    extra = ["-DBPE_FINE_PROF"] if os.environ.get("BPE_FINE_PROF") else []  # debug: sub-step timers inside phase_sites
    if os.environ.get("BPE_ML_THREADS"):
        extra.append("-DBPE_ML_THREADS=" + os.environ["BPE_ML_THREADS"])  # tuning: threads per block of the loop kernels
    if os.environ.get("BPE_TBL_STRIDE"):
        extra.append("-DBPE_TBL_STRIDE=" + os.environ["BPE_TBL_STRIDE"])  # tuning: 8 = one 32-byte entry per pair-table slot
    for knob in ("BPE_R_SMALL_LOG", "BPE_R_BATCH_LOG", "BPE_K1B_CHUNK_LOG", "BPE_STAGE_T"):  # tuning: size limits of a round's batch, staged neighbours (round_kernels.cuh)
        if os.environ.get(knob):
            extra.append("-D%s=%s" % (knob, os.environ[knob]))
    if os.environ.get("BPE_RD_THREADS"):
        extra.append("-DBPE_RD_THREADS=" + os.environ["BPE_RD_THREADS"])  # tuning: threads per block of k_merge_rounds
    cmd = [nvcc_path()] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-o", out] + [os.path.join(CSRC, f) for f in SOURCES]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed (%d)" % r.returncode)
    return out


SYNTH_LIB = os.path.join(HERE, "libbpe_synth.so")


def build_synth(force: bool = False) -> str:
    """The corpus generator alone (csrc/synth.cpp, host only, plain g++): bench.py's reference arm and the tests
    generate the synthetic text through this library so that they never map the CUDA product library."""
    src = os.path.join(CSRC, "synth.cpp")
    if not force and os.path.exists(SYNTH_LIB) and os.path.getmtime(SYNTH_LIB) >= os.path.getmtime(src):
        return SYNTH_LIB
    cxx = os.environ.get("CXX") or shutil.which("g++") or "g++"
    r = subprocess.run([cxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-pthread", "-o", SYNTH_LIB, src], capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("g++ failed on synth.cpp (%d)" % r.returncode)
    return SYNTH_LIB


if __name__ == "__main__":
    build_synth(force="--force" in sys.argv)
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
