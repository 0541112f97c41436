"""Host side of the drop-in: a mirror of the reference's ``class BPETokenizer``
(/root/reference/core.ts:77-495) with the same member names, argument meaning and error
messages.  Dictionary / Token / JSON work stays here (as it would stay in TypeScript);
everything that touches the corpus -- pair counting, arg-max, in-place merging, encoding --
runs on the B200 through the C ABI of ``include/bpe_b200.h``.  There is no CPU path:
constructing a tokenizer without the CUDA library and a device raises.

Node is not available in this image, so this Python class is the host the tests drive; the
TypeScript host + N-API shim a maintainer would use is shown in INTEGRATION.md.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np

from . import _abi
from ._abi import BpeError, MERGE_DTYPE, bpe_merge, bpe_stats, p32, p64

# core.ts:36-45
FS = chr(28)
EOF = chr(4)
LF = "\n"
CR = "\r"

_CUDA_STREAM_LEGACY = 1  # cudaStreamLegacy: the legacy default stream, which torch's default stream is (handle 0)

_JS_WS = (
    "\t\n\x0b\x0c\r \xa0\u1680\u2000\u2001\u2002\u2003\u2004\u2005\u2006\u2007\u2008\u2009\u200a"
    "\u2028\u2029\u202f\u205f\u3000\ufeff"
)


def fileContentToCorpus(content) -> str:  # core.ts:55-58
    text = content.decode("utf-8") if isinstance(content, (bytes, bytearray)) else str(content)
    return FS + text + EOF


def linesToCorpus(text: str) -> List[str]:  # core.ts:61-64
    return ["\r" + line.strip(_JS_WS) + "\n" for line in text.split("\n")]


def linesTrimmedToCorpus(text: str) -> List[str]:  # core.ts:67-75
    out = []
    for line in text.split("\n"):
        if line.endswith("\r"):
            line = line[:-1]
        out.append("\r" + line + "\n")
    return out


def _utf16_len(s: str) -> int:
    return len(s) + sum(1 for ch in s if ord(ch) > 0xFFFF)


def _js_stringify(s: str) -> str:
    short = {'"': '\\"', "\\": "\\\\", "\b": "\\b", "\f": "\\f", "\n": "\\n", "\r": "\\r", "\t": "\\t"}
    out = ['"']
    for ch in s:
        o = ord(ch)
        if ch in short:
            out.append(short[ch])
        elif o < 0x20 or 0xD800 <= o <= 0xDFFF:
            out.append("\\u%04x" % o)
        else:
            out.append(ch)
    out.append('"')
    return "".join(out)


class Token:
    """core.ts:1-10"""

    __slots__ = ("chars", "weight", "original_weight", "code", "index")

    def __init__(self, chars: str, weight: int, original_weight: int, code: str, index: int):
        self.chars = chars
        self.weight = weight
        self.original_weight = original_weight
        self.code = code
        self.index = index

    def _row(self):
        return (self.chars, self.weight, self.original_weight, self.code, self.index)

    def __eq__(self, other):
        return isinstance(other, Token) and self._row() == other._row()

    def __hash__(self):
        return id(self)

    def __repr__(self):
        return "Token(chars=%r, weight=%d, original_weight=%d, code=%r, index=%d)" % self._row()


MergeToken = Tuple[Token, Token, Token]


def compactMerge(merge: MergeToken):  # core.ts:500-503
    a, b, c = merge
    return [a.code, b.code, c.weight]


def _options(options, kw) -> dict:
    o = dict(options or {})
    o.update(kw)
    return o


def _min_weight(o) -> int:
    mw = o.get("min_weight") or 2  # core.ts:256
    return max(1, int(math.ceil(mw)))


class BPETokenizer:
    def __init__(self, device: int = 0, devices: Optional[Sequence[int]] = None):
        """One engine on `device`, or, with `devices`, one engine over those GPUs of this process (bpe_create_group): the corpus is
        sharded by document across them and every method keeps the single-engine results."""
        self._lib = _abi.load_library()
        h = C.c_void_p()
        if devices is None:
            rc = self._lib.bpe_create(device, C.byref(h))
        else:
            devices = [int(d) for d in devices]
            rc = self._lib.bpe_create_group((C.c_int * max(len(devices), 1))(*devices), len(devices), C.byref(h))
            if rc == _abi.BPE_E_INVALID:
                raise BpeError(rc, "devices must list 1 to %d distinct GPUs, got %r" % (_abi.MG_MAX_WORLD, devices))
            device = devices[0]
        if rc != _abi.BPE_OK:
            raise BpeError(rc, "cannot create the CUDA engine (no usable device, or GPUs without peer access? there is no CPU fallback)")
        self._h = h
        self._device = device
        self._stream = 0  # the stream set_stream gave the engine (0: its own); the C ABI has no getter
        self._reset_host()

    # ---- plumbing -------------------------------------------------------------------------
    def _reset_host(self) -> None:
        self.char_to_token: Dict[str, Token] = {}  # core.ts:79
        self.code_to_token: Dict[str, Token] = {}  # core.ts:82
        self.token_table: List[Token] = []  # core.ts:85
        self.merge_tokens: List[MergeToken] = []  # core.ts:88
        self.merge_codes: List[Tuple[str, str]] = []  # core.ts:91
        self.to_vector_index: Optional[Dict[int, int]] = None  # core.ts:97 (sparse array)
        self.from_vector_index: Optional[Dict[int, int]] = None  # core.ts:103
        self._pending: List[np.ndarray] = []  # documents added on the host, not yet uploaded
        self._tvi_dev: Optional[np.ndarray] = None
        self._tvi_cuda = None  # _tvi_dev as a CUDA tensor on the engine's device (encodeTextTensor)
        self._chars_synced = -1  # entries of char_to_token the engine's character table holds (-1: never pushed)

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self._lib.bpe_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def close(self) -> None:
        self.__del__()

    def _check(self, rc: int) -> None:
        if rc != _abi.BPE_OK:
            raise BpeError(rc, (self._lib.bpe_last_error(self._h) or b"").decode("utf-8", "replace"))

    @staticmethod
    def _check_offsets(doc_offsets: np.ndarray, n_units: int) -> None:
        """The C ABI carries no length for `ids` / `utf8`: the offsets are the only bound, so they must stay inside the
        array the caller handed over (and be non-decreasing) before a pointer to it crosses the boundary."""
        if doc_offsets.ndim != 1 or doc_offsets.size < 1:
            raise BpeError(_abi.BPE_E_INVALID, "doc_offsets must hold n_docs + 1 entries")
        if int(doc_offsets[0]) < 0 or int(doc_offsets[-1]) > n_units or (doc_offsets.size > 1 and bool(np.any(np.diff(doc_offsets) < 0))):
            raise BpeError(_abi.BPE_E_INVALID, "document offsets must be non-decreasing and lie inside the ids / bytes array (0 .. %d)" % n_units)

    def _dev_num_tokens(self) -> int:
        n = C.c_int32()
        self._check(self._lib.bpe_num_tokens(self._h, C.byref(n)))
        return n.value

    def _sync_tokens(self) -> None:
        if self._dev_num_tokens() != len(self.token_table):
            lens = np.fromiter((_utf16_len(t.chars) for t in self.token_table), dtype=np.int32, count=len(self.token_table))
            self._check(self._lib.bpe_set_tokens(self._h, p32(lens), len(lens)))

    def _flush(self) -> None:
        self._sync_tokens()
        if not self._pending:
            return
        docs, self._pending = self._pending, []
        offsets = np.zeros(len(docs) + 1, dtype=np.int64)
        np.cumsum([d.size for d in docs], out=offsets[1:])
        ids = np.concatenate(docs) if offsets[-1] else np.zeros(0, dtype=np.int32)
        self._check(self._lib.bpe_add_documents(self._h, p32(np.ascontiguousarray(ids, dtype=np.int32)), p64(offsets), len(docs)))

    def set_stream(self, cuda_stream: int) -> None:
        """Run the engine on an existing CUDA stream (e.g. ``torch.cuda.current_stream().cuda_stream``)."""
        self._check(self._lib.bpe_set_stream(self._h, C.c_void_p(cuda_stream)))
        self._stream = cuda_stream or 0

    def stats(self) -> dict:
        s = bpe_stats()
        self._check(self._lib.bpe_get_stats(self._h, C.byref(s)))
        return {n: (list(getattr(s, n)) if n == "ms_loop_phase" else getattr(s, n)) for n, _ in bpe_stats._fields_}

    # ---- snapshot (core.ts:112-171) ---------------------------------------------------------
    def toJSON(self) -> dict:
        return {
            "version": 2,
            "char_count": len(self.char_to_token),
            "token_table": [[t.chars, t.weight, t.original_weight] for t in self.token_table],
            "merge_codes": [[a.code, b.code, c.code] for a, b, c in self.merge_tokens],
        }

    def fromJSON(self, json: dict) -> None:
        if (
            not isinstance(json, dict)
            or json.get("version") != 2
            or not isinstance(json.get("token_table"), list)
            or not isinstance(json.get("merge_codes"), list)
        ):
            raise ValueError("invalid format")  # core.ts:136
        char_count = json.get("char_count")
        self._reset_host()  # core.ts:138-146: every field, corpus included, is replaced
        self._check(self._lib.bpe_clear_corpus(self._h))
        for chars, weight, original_weight in json["token_table"]:
            index = len(self.token_table)
            code = chr(index + 1)
            token = Token(chars, weight, original_weight, code, index)
            if char_count is not None and index < char_count:
                self.char_to_token[chars] = token
            self.code_to_token[code] = token
            self.token_table.append(token)
        if len(self.token_table) > _abi.BPE_MAX_TOKENS:
            raise BpeError(_abi.BPE_E_DOMAIN, "token table exceeds %d entries" % _abi.BPE_MAX_TOKENS)
        for a_code, b_code, c_code in json["merge_codes"]:
            a, b, c = self.code_to_token[a_code], self.code_to_token[b_code], self.code_to_token[c_code]
            self.merge_tokens.append((a, b, c))
            self.merge_codes.append((a.code + b.code, c.code))
        lens = np.fromiter((_utf16_len(t.chars) for t in self.token_table), dtype=np.int32, count=len(self.token_table))
        self._check(self._lib.bpe_set_tokens(self._h, p32(lens), len(lens)))
        abc = np.array([[a.index, b.index, c.index] for a, b, c in self.merge_tokens], dtype=np.int32).reshape(-1)
        self._check(self._lib.bpe_load_merges(self._h, p32(abc), len(self.merge_tokens)))
        self.compactVectorIndex()  # core.ts:170

    def _invalidateVectorIndex(self) -> None:  # core.ts:173-176
        self.to_vector_index = None
        self.from_vector_index = None
        self._tvi_dev = None
        self._tvi_cuda = None

    # ---- corpus -----------------------------------------------------------------------------
    def _char_ids(self, content: str, create: bool) -> np.ndarray:
        """core.ts:185-204 / :396-402: code-point iteration, first-appearance index assignment."""
        table, c2t = self.token_table, self.char_to_token
        ids = np.empty(len(content), dtype=np.int32)
        for i, char in enumerate(content):
            token = c2t.get(char)
            if token is None:
                if not create:
                    raise ValueError("unknown token, char: " + _js_stringify(char))  # core.ts:399
                index = len(table)
                if index >= _abi.BPE_MAX_TOKENS:
                    raise BpeError(_abi.BPE_E_DOMAIN, "token table exceeds %d entries" % _abi.BPE_MAX_TOKENS)
                code = chr(index + 1)
                token = Token(char, 1, 1, code, index)
                c2t[char] = token
                self.code_to_token[code] = token
                table.append(token)
            elif create:
                token.weight += 1
                token.original_weight += 1
            ids[i] = token.index
        return ids

    def addToCorpus(self, content: str) -> None:  # core.ts:182-207
        self._pending.append(self._char_ids(content, create=True))

    def addDocuments(self, ids: np.ndarray, doc_offsets: np.ndarray) -> None:
        """Bulk addToCorpus for documents already mapped to single-character token indices
        (every index must exist in token_table).  Weights are bumped as core.ts:201-202 does."""
        self._flush()
        ids = np.ascontiguousarray(ids, dtype=np.int32)
        doc_offsets = np.ascontiguousarray(doc_offsets, dtype=np.int64)
        self._check_offsets(doc_offsets, ids.size)
        counts = np.bincount(ids[doc_offsets[0]:doc_offsets[-1]], minlength=len(self.token_table))
        if counts.size > len(self.token_table):
            raise ValueError("document holds an index outside token_table")
        for i in np.nonzero(counts)[0]:
            t = self.token_table[i]
            t.weight += int(counts[i])
            t.original_weight += int(counts[i])
        self._check(self._lib.bpe_add_documents(self._h, p32(ids), p64(doc_offsets), len(doc_offsets) - 1))

    # ---- text front end on the device (csrc/text_kernels.cuh) -----------------------------------------
    def _sync_chars(self) -> None:
        if self._chars_synced == len(self.char_to_token):
            return
        # only one-code-point keys can match a character of a text; after `addToCorpus` following merges, fromJSON files
        # multi-character tokens under char_to_token (core.ts:157-159 takes the first char_count entries) -- they are inert
        items = [(ord(ch), t.index) for ch, t in self.char_to_token.items() if len(ch) == 1]
        cps = np.array([c for c, _ in items], dtype=np.int32)
        idx = np.array([i for _, i in items], dtype=np.int32)
        self._check(self._lib.bpe_set_chars(self._h, p32(cps), p32(idx), len(cps)))
        self._chars_synced = len(self.char_to_token)

    def _add_text_tokens(self, new_code_points: Sequence[int], counts: np.ndarray) -> None:
        """Host half of a text ingest: the tokens the engine just appended for the new characters, in its order
        (core.ts:188-199), then the batch's occurrence counts of every token (core.ts:201-202)."""
        for cp in new_code_points:
            index = len(self.token_table)
            token = Token(chr(cp), 0, 0, chr(index + 1), index)
            self.char_to_token[token.chars] = token
            self.code_to_token[token.code] = token
            self.token_table.append(token)
        self._chars_synced = len(self.char_to_token)
        for i in np.nonzero(counts[: len(self.token_table)])[0]:
            t = self.token_table[i]
            t.weight += int(counts[i])
            t.original_weight += int(counts[i])

    def addTextBatch(self, utf8: bytes, doc_byte_offsets: np.ndarray) -> None:
        """addToCorpus (core.ts:182-207) for many documents given as UTF-8 bytes, with the code-point loop, the
        first-appearance token creation and the weight counts done on the device.  Equivalent to calling
        ``addToCorpus(doc)`` for every document in order."""
        self._flush()
        self._sync_chars()
        doc_byte_offsets = np.ascontiguousarray(doc_byte_offsets, dtype=np.int64)
        self._check_offsets(doc_byte_offsets, len(utf8))
        buf = np.frombuffer(utf8 or b"\0", dtype=np.uint8)
        new_cps = np.empty(1 << 16, dtype=np.int32)
        counts = np.zeros(len(self.token_table) + (1 << 16), dtype=np.int64)
        n_new = C.c_int32()
        self._check(self._lib.bpe_add_text(self._h, buf.ctypes.data_as(_abi.u8p), p64(doc_byte_offsets), len(doc_byte_offsets) - 1,
                                           p32(new_cps), new_cps.size, C.byref(n_new), p64(counts), counts.size))
        self._add_text_tokens(new_cps[: n_new.value].tolist(), counts)
        # like addToCorpus (core.ts:182-207) this does NOT invalidate the vector index: a following encodeToVector with a
        # stale index throws `unknown token index` for the new characters, exactly as the reference does

    def encodeTextBatch(self, utf8: bytes, doc_byte_offsets: np.ndarray, vector: bool = True):
        """encodeBatch with the char -> index step on the device: -> (values, out_offsets, first_bad)."""
        self._flush()
        self._sync_chars()
        doc_byte_offsets = np.ascontiguousarray(doc_byte_offsets, dtype=np.int64)
        self._check_offsets(doc_byte_offsets, len(utf8))
        n_docs = len(doc_byte_offsets) - 1
        buf = np.frombuffer(utf8 or b"\0", dtype=np.uint8)
        total = int(doc_byte_offsets[-1] - doc_byte_offsets[0]) if n_docs else 0
        out = np.empty(max(total, 1), dtype=np.int32)
        out_off = np.zeros(n_docs + 1, dtype=np.int64)
        bad = np.full(max(n_docs, 1), -1, dtype=np.int64)
        n, upos, ucp = C.c_int64(), C.c_int64(-1), C.c_int32()
        tvi = None
        if vector:
            if self.to_vector_index is None:
                self.compactVectorIndex()
            tvi = self._tvi_array()
        rc = self._lib.bpe_encode_text_batch(self._h, buf.ctypes.data_as(_abi.u8p), p64(doc_byte_offsets), n_docs,
                                             p32(tvi) if tvi is not None else None, len(tvi) if tvi is not None else 0, p32(out), out.size,
                                             p64(out_off), p64(bad), C.byref(n), C.byref(upos), C.byref(ucp))
        if rc == _abi.BPE_E_INVALID and upos.value >= 0:
            raise ValueError("unknown token, char: " + _js_stringify(chr(ucp.value)))  # core.ts:399
        self._check(rc)
        return out[: n.value], out_off, bad[:n_docs]

    def encodeTextTensor(self, texts, doc_byte_offsets=None, *, vector: bool = True, pad_to=None, pad_value: int = -1):
        """encodeTextBatch into CUDA tensors on the engine's device, for a model that consumes the vectors there.
        `texts`: a sequence of str (UTF-8 with lone surrogates as 'surrogatepass' writes them), bytes with host offsets, or a
        torch.uint8 CUDA tensor with an int64 CUDA offsets tensor (both on the engine's device; they are read in place).
        -> (values int32[N], offsets int64[B+1]) when pad_to is None, else (ids int32[B, L], lengths int64[B]) with
        L = pad_to, or the longest document for pad_to="longest"; longer documents are cut on the right and the rest of a
        row holds pad_value.  Raises as encodeTextBatch (unknown character) and, with vector=True, as encodeToVector at the
        first hole in document order.  The work runs on torch.cuda.current_stream() of the engine's device and is complete
        when the call returns; the engine's own stream setting is restored afterwards."""
        import torch

        self._flush()
        self._sync_chars()
        dev = torch.device("cuda", self._device)
        if pad_to is not None and not (isinstance(pad_to, str) and pad_to == "longest"):
            if isinstance(pad_to, (bool, str, float)) or not hasattr(pad_to, "__index__") or pad_to.__index__() < 0:
                raise ValueError('pad_to must be None, "longest" or an int >= 0, got %r' % (pad_to,))
            pad_to = pad_to.__index__()
        if isinstance(texts, str):
            raise ValueError("texts must be a sequence of str (one per document), not one str")
        if isinstance(texts, torch.Tensor):
            if not isinstance(doc_byte_offsets, torch.Tensor):
                raise ValueError("a text tensor takes its document offsets as an int64 tensor on the same device")
            if texts.device != dev or doc_byte_offsets.device != dev:
                raise ValueError("text and offsets must be on %s, the engine's device (got %s and %s)" % (dev, texts.device, doc_byte_offsets.device))
            if texts.dtype != torch.uint8 or texts.dim() != 1 or doc_byte_offsets.dtype != torch.int64 or doc_byte_offsets.dim() != 1:
                raise ValueError("text must be a 1-D uint8 tensor and offsets a 1-D int64 tensor")
            text_d, off_d = texts.contiguous(), doc_byte_offsets.contiguous()
        else:
            if isinstance(texts, (bytes, bytearray, memoryview)):
                if doc_byte_offsets is None:
                    raise ValueError("bytes need doc_byte_offsets")
                data, off = bytes(texts), np.ascontiguousarray(doc_byte_offsets, dtype=np.int64)
            else:
                if doc_byte_offsets is not None:
                    raise ValueError("a sequence of str carries its own document boundaries")
                chunks = [s.encode("utf-8", "surrogatepass") for s in texts]
                off = np.zeros(len(chunks) + 1, dtype=np.int64)
                np.cumsum([len(c) for c in chunks], out=off[1:])
                data = b"".join(chunks)
            with torch.cuda.device(dev):  # the copies go out on the current stream of the engine's device
                if data:
                    import warnings

                    with warnings.catch_warnings():  # (the tensor only reads the bytes: that they are immutable does not matter)
                        warnings.simplefilter("ignore", UserWarning)
                        text_d = torch.frombuffer(data, dtype=torch.uint8).to(dev)
                else:
                    text_d = torch.empty(0, dtype=torch.uint8, device=dev)
                off_d = torch.from_numpy(off).to(dev)
        if off_d.numel() < 1:
            raise BpeError(_abi.BPE_E_INVALID, "doc_byte_offsets must hold n_docs + 1 entries")
        n_docs, n_bytes = off_d.numel() - 1, text_d.numel()
        tvi = None
        if vector:
            if self.to_vector_index is None:
                self.compactVectorIndex()
            if self._tvi_cuda is None:
                self._tvi_cuda = torch.from_numpy(self._tvi_array()).to(dev)
            tvi = self._tvi_cuda
        out = torch.empty(max(n_bytes, 1), dtype=torch.int32, device=dev)
        out_off = torch.empty(n_docs + 1, dtype=torch.int64, device=dev)
        bad = torch.empty(max(n_docs, 1), dtype=torch.int64, device=dev) if vector else None
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731
        n, upos, ucp = C.c_int64(), C.c_int64(-1), C.c_int32()
        # torch's default stream has the handle 0, which bpe_set_stream reads as the engine's own (non-blocking) stream: that
        # stream is not ordered after the work torch queued on the legacy default stream, so name that stream explicitly
        self._check(self._lib.bpe_set_stream(self._h, C.c_void_p(torch.cuda.current_stream(dev).cuda_stream or _CUDA_STREAM_LEGACY)))
        try:
            rc = self._lib.bpe_encode_text_batch_dev(self._h, ptr(text_d), n_bytes, ptr(off_d), n_docs, ptr(tvi), tvi.numel() if vector else 0,
                                                     ptr(out), ptr(out_off), ptr(bad), C.byref(n), C.byref(upos), C.byref(ucp))
            if rc == _abi.BPE_E_INVALID and upos.value >= 0:
                raise ValueError("unknown token, char: " + _js_stringify(chr(ucp.value)))  # core.ts:399
            self._check(rc)
            values = out[: n.value]
            if vector:
                holes = torch.nonzero(bad[:n_docs] >= 0)
                if holes.numel():  # encodeToVector throws at its document's first hole (core.ts:437-441)
                    d = int(holes[0, 0])
                    raise ValueError("unknown token index: %d" % (-int(values[int(out_off[d]) + int(bad[d])]) - 1))
            if pad_to is None:  # (a copy of the N values: `out` holds 4 B per byte of input, a multiple of what they need)
                return values.clone(), out_off
            width = pad_to if pad_to != "longest" else (int((out_off[1:] - out_off[:-1]).max()) if n_docs else 0)
            ids = torch.empty((n_docs, width), dtype=torch.int32, device=dev)
            lengths = torch.empty(n_docs, dtype=torch.int64, device=dev)
            self._check(self._lib.bpe_pad_batch_dev(self._h, ptr(out), ptr(out_off), n_docs, width, int(pad_value), ptr(ids), ptr(lengths)))
            return ids, lengths
        finally:
            # bpe_set_stream waits for the stream it leaves: the pad kernel is done when this returns
            self._check(self._lib.bpe_set_stream(self._h, C.c_void_p(self._stream)))

    def restoreToCorpus(self, content: str) -> None:  # core.ts:213-216
        ids = self._char_ids(content, create=False)
        self._flush()
        off = np.array([0, ids.size], dtype=np.int64)
        self._check(self._lib.bpe_restore_documents(self._h, p32(ids), p64(off), 1))

    def restoreDocuments(self, ids: np.ndarray, doc_offsets: np.ndarray) -> None:
        """Bulk restoreToCorpus (documents as single-character token indices)."""
        self._flush()
        ids = np.ascontiguousarray(ids, dtype=np.int32)
        doc_offsets = np.ascontiguousarray(doc_offsets, dtype=np.int64)
        self._check_offsets(doc_offsets, ids.size)
        self._check(self._lib.bpe_restore_documents(self._h, p32(ids), p64(doc_offsets), len(doc_offsets) - 1))

    def corpusIds(self) -> Tuple[np.ndarray, np.ndarray]:
        """Current token indices of every document: (ids, doc_offsets)."""
        self._flush()
        nd, nt = C.c_int64(), C.c_int64()
        self._check(self._lib.bpe_corpus_size(self._h, C.byref(nd), C.byref(nt)))
        out = np.empty(max(nt.value, 1), dtype=np.int32)
        offs = np.zeros(nd.value + 1, dtype=np.int64)
        n = C.c_int64()
        self._check(self._lib.bpe_get_corpus(self._h, 0, nd.value, p32(out), out.size, p64(offs), C.byref(n)))
        return out[: n.value], offs

    @property
    def corpus_in_code(self) -> List[str]:  # core.ts:106 -- materialised from the device on demand
        ids, offs = self.corpusIds()
        codes = (ids.astype(np.uint32) + 1).tolist()
        return ["".join(map(chr, codes[offs[d]:offs[d + 1]])) for d in range(len(offs) - 1)]

    @corpus_in_code.setter
    def corpus_in_code(self, value: Sequence[str]) -> None:  # example/import-merge-log-to-ram.ts:22
        self._pending = []
        self._check(self._lib.bpe_clear_corpus(self._h))
        self._sync_tokens()
        docs = [np.fromiter((ord(ch) - 1 for ch in s), dtype=np.int32, count=len(s)) for s in value]
        if docs:
            offsets = np.zeros(len(docs) + 1, dtype=np.int64)
            np.cumsum([d.size for d in docs], out=offsets[1:])
            ids = np.concatenate(docs) if offsets[-1] else np.zeros(0, dtype=np.int32)
            self._check(self._lib.bpe_add_documents(self._h, p32(np.ascontiguousarray(ids)), p64(offsets), len(docs)))

    # ---- vector index (core.ts:222-241) -------------------------------------------------------
    def compactVectorIndex(self) -> None:
        if len(self.token_table) == 0:
            raise ValueError("token table is empty, have you called tokenizer.addToCorpus()?")
        to_vi: Dict[int, int] = {}
        from_vi: Dict[int, int] = {}
        vector_index = 0
        for index, token in enumerate(self.token_table):
            if token.weight > 0:
                to_vi[index] = vector_index
                from_vi[vector_index] = index
                vector_index += 1
        self.to_vector_index, self.from_vector_index = to_vi, from_vi
        self._tvi_dev = None
        self._tvi_cuda = None

    def _tvi_array(self) -> np.ndarray:
        if self._tvi_dev is None:
            arr = np.full(len(self.token_table), -1, dtype=np.int32)
            if self.to_vector_index:
                idx = np.fromiter(self.to_vector_index.keys(), dtype=np.int64, count=len(self.to_vector_index))
                val = np.fromiter(self.to_vector_index.values(), dtype=np.int32, count=len(self.to_vector_index))
                arr[idx] = val
            self._tvi_dev = arr
        return self._tvi_dev

    # ---- training -----------------------------------------------------------------------------
    def findNextMerge(self, options: Optional[dict] = None, **kw) -> Optional[MergeToken]:  # core.ts:247-326
        o = _options(options, kw)
        max_length = o.get("max_length")
        self._flush()
        if max_length and max_length < 2:
            return None  # no pair of non-empty tokens is that short (core.ts:272)
        m, found = bpe_merge(), C.c_int()
        self._check(self._lib.bpe_find_next_merge(self._h, _min_weight(o), int(max_length or 0), C.byref(m), C.byref(found)))
        if not found.value:
            return None
        a, b = self.token_table[m.a], self.token_table[m.b]
        new_index = len(self.token_table)
        return (a, b, Token(a.chars + b.chars, m.weight, m.weight, chr(new_index + 1), new_index))

    def _record_merge(self, a: Token, b: Token, c: Token) -> None:  # core.ts:345-354
        a.weight -= c.weight
        b.weight -= c.weight
        self.code_to_token[c.code] = c
        self.token_table.append(c)
        self.merge_tokens.append((a, b, c))
        self.merge_codes.append((a.code + b.code, c.code))

    def applyMerge(self, merge: MergeToken) -> None:  # core.ts:332-360
        a, b, c = merge
        self._flush()
        if c.index != len(self.token_table):
            raise ValueError("merge is stale: its token index %d is not the next free index %d" % (c.index, len(self.token_table)))
        self._check(self._lib.bpe_apply_merge(self._h, a.index, b.index, c.index, None))
        self._record_merge(a, b, c)
        self._invalidateVectorIndex()

    def mergeUntil(self, options: Optional[dict] = None, **kw) -> int:  # core.ts:365-383
        o = _options(options, kw)
        max_length = o.get("max_length")
        max_iterations = o.get("max_iterations")
        self._flush()
        if max_length and max_length < 2:
            return 0
        if max_iterations and max_iterations < 1:
            return 0  # `iteration <= max_iterations` fails at once (core.ts:376)
        room = _abi.BPE_MAX_TOKENS - len(self.token_table)
        cap = min(room, int(max_iterations)) if max_iterations else room
        if cap <= 0:
            if room <= 0:
                raise BpeError(_abi.BPE_E_DOMAIN, "token table exceeds %d entries" % _abi.BPE_MAX_TOKENS)
            return 0
        log = np.zeros(cap, dtype=MERGE_DTYPE)
        n = C.c_int64()
        rc = self._lib.bpe_merge_until(self._h, _min_weight(o), int(max_length or 0), int(max_iterations or 0),
                                       log.ctypes.data_as(C.c_void_p), cap, C.byref(n))
        table = self.token_table
        for a_i, b_i, _c, _r, w in log[: n.value].tolist():  # replay on the host exactly as core.ts:315-325,345-354
            a, b = table[a_i], table[b_i]
            index = len(table)
            self._record_merge(a, b, Token(a.chars + b.chars, w, w, chr(index + 1), index))
        if n.value:
            self._invalidateVectorIndex()
        self._check(rc)
        return n.value

    def restoreMerge(self, compact) -> None:  # core.ts:477-494
        a_code, b_code, c_weight = compact
        a = self.code_to_token.get(a_code)
        if a is None:
            raise ValueError("unknown token, a_code: " + _js_stringify(a_code))
        b = self.code_to_token.get(b_code)
        if b is None:
            raise ValueError("unknown token, b_code: " + _js_stringify(b_code))
        index = len(self.token_table)
        self.applyMerge((a, b, Token(a.chars + b.chars, c_weight, c_weight, chr(index + 1), index)))

    def restoreMerges(self, compacts: Sequence) -> None:
        """Replay a whole merge log -- lines ``[a_code, b_code, c_weight]`` as written by ``compactMerge``
        (core.ts:500-503; example/scan-to-merge-log.ts:38-40) -- in ONE device call.  Equivalent to calling
        ``restoreMerge`` per line (core.ts:477-494; example/import-merge-log-to-ram.ts:24-31), including its throws."""
        self._flush()
        base = len(self.token_table)
        pending: List[Tuple[Token, Token, Token]] = []
        code_to_new: Dict[str, Token] = {}
        ab = np.empty((len(compacts), 2), dtype=np.int32)
        for i, (a_code, b_code, c_weight) in enumerate(compacts):
            a = self.code_to_token.get(a_code) or code_to_new.get(a_code)
            if a is None:
                raise ValueError("unknown token, a_code: " + _js_stringify(a_code))  # core.ts:481
            b = self.code_to_token.get(b_code) or code_to_new.get(b_code)
            if b is None:
                raise ValueError("unknown token, b_code: " + _js_stringify(b_code))  # core.ts:483
            index = base + i
            c = Token(a.chars + b.chars, c_weight, c_weight, chr(index + 1), index)
            code_to_new[c.code] = c
            pending.append((a, b, c))
            ab[i] = (a.index, b.index)
        if not pending:
            return
        self._check(self._lib.bpe_apply_merges(self._h, p32(ab.reshape(-1)), len(pending), None))
        for a, b, c in pending:
            self._record_merge(a, b, c)
        self._invalidateVectorIndex()

    # ---- encode / decode ------------------------------------------------------------------------
    def encodeBatch(self, ids: np.ndarray, doc_offsets: np.ndarray, vector: bool = True):
        """Encode many documents (single-character token indices) in one device call.
        -> (values int32, out_offsets int64[n_docs+1], first_bad int64[n_docs]); with ``vector=True`` values are
        vector indices and first_bad[d] >= 0 marks documents the reference would throw on (core.ts:437-441)."""
        self._flush()
        ids = np.ascontiguousarray(ids, dtype=np.int32)
        doc_offsets = np.ascontiguousarray(doc_offsets, dtype=np.int64)
        self._check_offsets(doc_offsets, ids.size)
        n_docs = len(doc_offsets) - 1
        total = int(doc_offsets[-1] - doc_offsets[0]) if n_docs else 0
        out = np.empty(max(total, 1), dtype=np.int32)
        out_off = np.zeros(n_docs + 1, dtype=np.int64)
        bad = np.full(max(n_docs, 1), -1, dtype=np.int64)
        n = C.c_int64()
        tvi = None
        if vector:
            if self.to_vector_index is None:
                self.compactVectorIndex()
            tvi = self._tvi_array()
        self._check(self._lib.bpe_encode_batch(self._h, p32(ids), p64(doc_offsets), n_docs,
                                               p32(tvi) if tvi is not None else None, len(tvi) if tvi is not None else 0,
                                               p32(out), out.size, p64(out_off), p64(bad), C.byref(n)))
        return out[: n.value], out_off, bad[:n_docs]

    def _encode_ids(self, content: str) -> np.ndarray:
        ids = self._char_ids(content, create=False)  # core.ts:396-402
        out, _, _ = self.encodeBatch(ids, np.array([0, ids.size], dtype=np.int64), vector=False)
        return out

    def encodeToCode(self, content: str) -> str:  # core.ts:392-409
        return "".join(map(chr, (self._encode_ids(content).astype(np.uint32) + 1).tolist()))

    def encodeToTokens(self, content: str) -> List[Token]:  # core.ts:411-422
        table = self.token_table
        return [table[i] for i in self._encode_ids(content).tolist()]

    def encodeToVector(self, content: str) -> List[int]:  # core.ts:424-445
        if self.to_vector_index is None:
            self.compactVectorIndex()
        ids = self._char_ids(content, create=False)
        out, _, bad = self.encodeBatch(ids, np.array([0, ids.size], dtype=np.int64), vector=True)
        if bad[0] >= 0:
            raise ValueError("unknown token index: %d" % (-int(out[bad[0]]) - 1))  # core.ts:440
        return out.tolist()

    def decodeBatch(self, values: np.ndarray, doc_offsets: np.ndarray, vector: bool = True):
        """decodeVector / decodeTokens (core.ts:447-471) for many documents in one device call.
        -> (utf8 bytes, out_offsets int64[n_docs+1], first_bad int64[n_docs]); first_bad[d] >= 0 is the position of the
        first value of document d the reference would throw `unknown vector index` on."""
        self._flush()
        values = np.ascontiguousarray(values, dtype=np.int32)
        doc_offsets = np.ascontiguousarray(doc_offsets, dtype=np.int64)
        self._check_offsets(doc_offsets, values.size)
        n_docs = len(doc_offsets) - 1
        fvi = None
        if vector:
            if self.from_vector_index is None:
                self.compactVectorIndex()
            n = (max(self.from_vector_index) + 1) if self.from_vector_index else 0
            fvi = np.full(max(n, 1), -1, dtype=np.int32)
            for k, v in self.from_vector_index.items():
                fvi[k] = v
        chunks = [t.chars.encode("utf-8", "surrogatepass") for t in self.token_table]
        tok_off = np.zeros(len(chunks) + 1, dtype=np.int64)
        np.cumsum([len(c) for c in chunks], out=tok_off[1:])
        arena = np.frombuffer(b"".join(chunks) or b"\0", dtype=np.uint8)
        total = int(doc_offsets[-1] - doc_offsets[0]) if n_docs else 0
        longest = max((len(c) for c in chunks), default=0)
        out = np.empty(max(total * longest, 1), dtype=np.uint8)
        out_off = np.zeros(n_docs + 1, dtype=np.int64)
        bad = np.full(max(n_docs, 1), -1, dtype=np.int64)
        n = C.c_int64()
        self._check(self._lib.bpe_decode_batch(self._h, p32(values), p64(doc_offsets), n_docs, p32(fvi) if fvi is not None else None,
                                               len(fvi) if fvi is not None else 0, arena.ctypes.data_as(_abi.u8p), p64(tok_off), len(chunks),
                                               out.ctypes.data_as(_abi.u8p), out.size, p64(out_off), p64(bad), C.byref(n)))
        return out[: n.value].tobytes(), out_off, bad[:n_docs]

    def decodeTensor(self, values, offsets=None, *, lengths=None, vector: bool = True) -> List[str]:
        """decodeVector (core.ts:455-471) per document for vectors held in tensors, e.g. a model's output on the GPU: ragged
        (values, offsets) or dense (ids[B, L], lengths=[B]) as encodeTextTensor returns them.  The values come to the host once
        and are decoded in one bpe_decode_batch call.  With vector=False they are raw token indices."""
        if values.dim() == 2:
            if lengths is None or offsets is not None:
                raise ValueError("dense ids take their row lengths as lengths=, and no offsets")
            ids, lens = values.cpu().numpy(), lengths.cpu().numpy().astype(np.int64)
            if lens.shape != (ids.shape[0],) or bool(np.any(lens < 0)) or bool(np.any(lens > ids.shape[1])):
                raise ValueError("lengths must hold one value in [0, %d] per row" % ids.shape[1])
            vals = ids[np.arange(ids.shape[1])[None, :] < lens[:, None]]
            off = np.zeros(len(lens) + 1, dtype=np.int64)
            np.cumsum(lens, out=off[1:])
        elif values.dim() == 1:
            if offsets is None or lengths is not None:
                raise ValueError("ragged values take their document offsets, and no lengths")
            vals = values.cpu().numpy()
            off = np.ascontiguousarray(offsets.cpu().numpy() if hasattr(offsets, "cpu") else offsets, dtype=np.int64)
        else:
            raise ValueError("values must be 1-D (with offsets) or 2-D (with lengths)")
        utf8, out_off, bad = self.decodeBatch(vals, off, vector=vector)
        holes = np.flatnonzero(bad >= 0)
        if holes.size:
            d = int(holes[0])
            v = int(vals[int(off[d]) + int(bad[d])])
            raise ValueError(("unknown vector index: %s" if vector else "unknown token index: %s") % (v,))  # core.ts:467
        return [utf8[out_off[d]:out_off[d + 1]].decode("utf-8", "surrogatepass") for d in range(len(off) - 1)]

    def decodeTokens(self, tokens: Iterable[Token]) -> str:  # core.ts:447-453
        return "".join(t.chars for t in tokens)

    def decodeVector(self, vector: Iterable[int]) -> str:  # core.ts:455-471
        if self.from_vector_index is None:
            self.compactVectorIndex()
        from_vi, table = self.from_vector_index, self.token_table
        out = []
        for vector_index in vector:
            index = from_vi.get(vector_index)
            if index is None:
                raise ValueError("unknown vector index: %s" % (vector_index,))  # core.ts:467
            out.append(table[index].chars)
        return "".join(out)
