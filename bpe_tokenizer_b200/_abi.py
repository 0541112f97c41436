"""ctypes binding of include/bpe_b200.h.  There is no CPU fallback: if the CUDA library is missing
or no device is usable, construction fails loudly."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libbpe_b200.so")

BPE_OK, BPE_E_INVALID, BPE_E_CUDA, BPE_E_CAPACITY, BPE_E_DOMAIN, BPE_E_NOMEM, BPE_E_INTERNAL = 0, -1, -2, -3, -4, -5, -6
BPE_MAX_TOKENS = 56319
MG_MAX_WORLD = 8
_CODE_NAMES = {-1: "BPE_E_INVALID", -2: "BPE_E_CUDA", -3: "BPE_E_CAPACITY", -4: "BPE_E_DOMAIN", -5: "BPE_E_NOMEM", -6: "BPE_E_INTERNAL"}


class BpeError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"{_CODE_NAMES.get(code, code)}: {message}")
        self.code = code
        self.message = message


class bpe_merge(C.Structure):
    _fields_ = [("a", C.c_int32), ("b", C.c_int32), ("c", C.c_int32), ("reserved", C.c_int32), ("weight", C.c_int64)]


class bpe_stats(C.Structure):
    _fields_ = [(n, C.c_int64) for n in (
        "kernel_launches", "merges_applied", "index_builds", "hot_rebuilds", "tie_breaks", "sites_merged",
        "corpus_positions", "corpus_tokens", "distinct_pairs", "pool_used")] + [(n, C.c_double) for n in (
        "ms_index_build", "ms_argmax", "ms_apply", "ms_encode", "ms_last_merge_until")] + [("ms_loop_phase", C.c_double * 8)] + [(n, C.c_int64) for n in (
        "loop_rounds", "loop_round_merges", "loop_round_tried", "loop_rounds_cut", "encode_path")]


MERGE_DTYPE = np.dtype([("a", "<i4"), ("b", "<i4"), ("c", "<i4"), ("reserved", "<i4"), ("weight", "<i8")])
assert MERGE_DTYPE.itemsize == C.sizeof(bpe_merge)

i32p, i64p, u8p, vp = C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_uint8), C.c_void_p

# every symbol include/bpe_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "bpe_abi_version": (C.c_int, []),
    "bpe_create": (C.c_int, [C.c_int, C.POINTER(vp)]),
    "bpe_create_group": (C.c_int, [C.POINTER(C.c_int), C.c_int, C.POINTER(vp)]),
    "bpe_destroy": (None, [vp]),
    "bpe_last_error": (C.c_char_p, [vp]),
    "bpe_set_stream": (C.c_int, [vp, vp]),
    "bpe_synchronize": (C.c_int, [vp]),
    "bpe_get_stats": (C.c_int, [vp, C.POINTER(bpe_stats)]),
    "bpe_set_profiling": (C.c_int, [vp, C.c_int]),
    "bpe_set_tokens": (C.c_int, [vp, i32p, C.c_int32]),
    "bpe_num_tokens": (C.c_int, [vp, i32p]),
    "bpe_load_merges": (C.c_int, [vp, i32p, C.c_int64]),
    "bpe_add_documents": (C.c_int, [vp, i32p, i64p, C.c_int64]),
    "bpe_add_documents_dev": (C.c_int, [vp, vp, i64p, C.c_int64]),
    "bpe_restore_documents": (C.c_int, [vp, i32p, i64p, C.c_int64]),
    "bpe_clear_corpus": (C.c_int, [vp]),
    "bpe_corpus_size": (C.c_int, [vp, i64p, i64p]),
    "bpe_get_corpus": (C.c_int, [vp, C.c_int64, C.c_int64, i32p, C.c_int64, i64p, i64p]),
    "bpe_find_next_merge": (C.c_int, [vp, C.c_int64, C.c_int32, C.POINTER(bpe_merge), C.POINTER(C.c_int)]),
    "bpe_apply_merge": (C.c_int, [vp, C.c_int32, C.c_int32, C.c_int32, i64p]),
    "bpe_apply_merges": (C.c_int, [vp, i32p, C.c_int64, i64p]),
    "bpe_merge_until": (C.c_int, [vp, C.c_int64, C.c_int32, C.c_int64, vp, C.c_int64, i64p]),
    "bpe_pair_counts": (C.c_int, [vp, i32p, i32p, i64p, C.c_int64, i64p]),
    "bpe_encode_batch": (C.c_int, [vp, i32p, i64p, C.c_int64, i32p, C.c_int32, i32p, C.c_int64, i64p, i64p, i64p]),
    "bpe_encode_batch_dev": (C.c_int, [vp, vp, vp, C.c_int64, C.c_int64, C.c_int64, vp, C.c_int32, vp, vp, vp, i64p]),
    "bpe_decode_batch": (C.c_int, [vp, i32p, i64p, C.c_int64, i32p, C.c_int32, u8p, i64p, C.c_int32, u8p, C.c_int64, i64p, i64p, i64p]),
    "bpe_set_chars": (C.c_int, [vp, i32p, i32p, C.c_int32]),
    "bpe_add_text": (C.c_int, [vp, u8p, i64p, C.c_int64, i32p, C.c_int32, i32p, i64p, C.c_int64]),
    "bpe_add_text_stage": (C.c_int, [vp, u8p, i64p, C.c_int64, i32p, i64p, C.c_int32, i32p]),
    "bpe_add_text_commit": (C.c_int, [vp, i32p, C.c_int32, i64p, C.c_int64]),
    "bpe_debug_lane_table": (C.c_int, [i32p, C.c_int64, C.c_int32, i32p, i32p, i32p, i32p, i32p, i32p, C.c_int64, i64p]),
    "bpe_debug_plan_chunks": (C.c_int, [i64p, C.c_int64, C.c_int64, i64p, C.c_int64, i64p, i64p]),
    "bpe_encode_text_batch": (C.c_int, [vp, u8p, i64p, C.c_int64, i32p, C.c_int32, i32p, C.c_int64, i64p, i64p, i64p, i64p, i32p]),
    "bpe_encode_text_batch_dev": (C.c_int, [vp, vp, C.c_int64, vp, C.c_int64, vp, C.c_int32, vp, vp, vp, i64p, i64p, i32p]),
    "bpe_pad_batch_dev": (C.c_int, [vp, vp, vp, C.c_int64, C.c_int64, C.c_int32, vp, vp]),
    "bpe_mg_init": (C.c_int, [vp, C.c_int, C.c_int, vp]),
    "bpe_mg_connect": (C.c_int, [vp, C.c_char_p]),
    "bpe_mg_state": (C.c_int, [vp, C.POINTER(C.c_int)]),
    "bpe_mg_export_counts": (C.c_int, [vp, vp, vp, C.c_int64, i64p]),
    "bpe_mg_import_counts": (C.c_int, [vp, vp, vp, C.c_int64, C.c_int]),
    "bpe_synth_corpus": (C.c_int, [C.c_int64, C.c_uint64, C.c_int32, C.c_uint64, u8p, C.c_int64, i64p, C.c_int64, i64p, i64p]),
}

_lib = None


def load_library(build_if_missing: bool = True) -> C.CDLL:
    """Load libbpe_b200.so (building it in-tree with nvcc when absent) and bind every symbol."""
    global _lib
    if _lib is not None:
        return _lib
    if build_if_missing:
        from . import build as _build

        if _build.needs_build():
            _build.build()
    path = os.environ.get("BPE_LIB") or LIB_PATH  # BPE_LIB: a differently tuned build of the same library (A/B timing)
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing: build it with `python -m bpe_tokenizer_b200.build` (no CPU fallback exists)")
    lib = C.CDLL(path)
    for name, (restype, argtypes) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError here = header and library disagree
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def p32(a: np.ndarray):
    return a.ctypes.data_as(i32p)


def p64(a: np.ndarray):
    return a.ctypes.data_as(i64p)
