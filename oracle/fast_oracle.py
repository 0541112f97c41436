"""TEST INFRASTRUCTURE ONLY -- ctypes binding of ``fast_oracle.cpp``, the incremental CPU oracle for mergeUntil
(core.ts:365-383) that reaches BASELINE config 3 at full size.  Pinned against the literal oracles by
``tests/test_oracle_golden.py``; used by ``tests/golden/check_cfg3_full.py`` to check the GPU's full cfg3 merge log."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libbpe_fast_oracle.so")
_lib = None


def build_fast_oracle(force: bool = False) -> str:
    src = os.path.join(_HERE, "fast_oracle.cpp")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s", "-B", "libbpe_fast_oracle.so"])
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build_fast_oracle()
        L = C.CDLL(_LIB_PATH)
        i32p, i64p = C.POINTER(C.c_int32), C.POINTER(C.c_int64)
        L.fast_create.restype = C.c_void_p
        L.fast_destroy.argtypes = [C.c_void_p]
        L.fast_set_len16.argtypes = [C.c_void_p, i32p, C.c_int32]
        L.fast_add_documents.argtypes = [C.c_void_p, i32p, i64p, C.c_int64]
        L.fast_total_tokens.argtypes = [C.c_void_p]
        L.fast_total_tokens.restype = C.c_int64
        L.fast_get_corpus.argtypes = [C.c_void_p, i32p]
        L.fast_num_documents.argtypes = [C.c_void_p]
        L.fast_num_documents.restype = C.c_int64
        L.fast_document_lengths.argtypes = [C.c_void_p, i64p]
        L.fast_merge_until.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_int32, i32p, i32p, i64p, C.c_int64]
        L.fast_merge_until.restype = C.c_int64
        _lib = L
    return _lib


def _p32(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


def _p64(a):
    return a.ctypes.data_as(C.POINTER(C.c_int64))


class FastOracle:
    """Same call shape as oracle.int_oracle.IntOracle for the training path."""

    def __init__(self):
        self.L = lib()
        self.h = C.c_void_p(self.L.fast_create())

    def __del__(self):
        if getattr(self, "h", None):
            self.L.fast_destroy(self.h)
            self.h = None

    def set_len16(self, len16) -> None:
        a = np.ascontiguousarray(len16, dtype=np.int32)
        self.L.fast_set_len16(self.h, _p32(a), a.size)

    def add_documents(self, ids, offsets) -> None:
        a = np.ascontiguousarray(ids, dtype=np.int32)
        o = np.ascontiguousarray(offsets, dtype=np.int64)
        if self.L.fast_add_documents(self.h, _p32(a), _p64(o), o.size - 1) != 0:
            raise ValueError("corpus too large for the fast oracle")

    def merge_until(self, min_weight: int, max_length: int, max_iterations: int, first_new_index: int, cap: int):
        la, lb, lw = np.zeros(cap, dtype=np.int32), np.zeros(cap, dtype=np.int32), np.zeros(cap, dtype=np.int64)
        n = self.L.fast_merge_until(self.h, min_weight, max_length, max_iterations, first_new_index, _p32(la), _p32(lb), _p64(lw), cap)
        return la[:n], lb[:n], lw[:n]

    def corpus(self) -> np.ndarray:
        out = np.zeros(max(self.L.fast_total_tokens(self.h), 1), dtype=np.int32)
        self.L.fast_get_corpus(self.h, _p32(out))
        return out[: self.L.fast_total_tokens(self.h)]

    def document_lengths(self) -> np.ndarray:
        """Current number of tokens of every document, empty documents included (corpus() holds them back to back)."""
        out = np.zeros(self.L.fast_num_documents(self.h), dtype=np.int64)
        if out.size:
            self.L.fast_document_lengths(self.h, _p64(out))
        return out
