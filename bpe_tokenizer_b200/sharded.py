"""BPETokenizer over a corpus sharded by document across the GPUs of one node (one process per GPU).

The reference has a single in-memory corpus (core.ts:106) and no notion of devices; this class keeps its API and
results bit-exact while each rank holds only a contiguous range of the documents.  SPMD contract: every rank
constructs the tokenizer on its own device and calls the same methods in the same order.

* ``addToCorpus(text)`` is called with EVERY document on EVERY rank: the host-side dictionary work (first-appearance
  indices, character weights, core.ts:185-203) is then identical everywhere without communication; at upload time a
  rank keeps only its shard (contiguous in ``addToCorpus`` order, balanced by token count), so global scan order is
  (rank, local position) -- what the reference's position tie-break needs (core.ts:294-305).
* ``addDocuments(ids, offsets, local_shard=True)`` is the bulk form for corpora too large to replicate: each rank
  passes only its own documents (rank order = document order); character weights are summed over the group.
* ``addTextBatch(utf8, offsets, local_shard=True)`` is the same from raw UTF-8 text: each rank decodes its shard on its
  device (bpe_add_text_stage), the ranks exchange their new characters with their first positions and order them by
  (rank, position), and every rank appends its shard with that one global order (bpe_add_text_commit).
* ``mergeUntil`` first sums the pair histograms of all shards (one all-gather of (pair, count) lists over NCCL), then
  runs the persistent sharded kernel (csrc/mg_kernels.cuh): count deltas travel GPU to GPU over NVLink inside the
  kernel, the arg-max is replicated, every rank returns the same merge log and replays it on its host table.
* ``encode*`` / ``decode*`` need no communication (each rank encodes what it is given).
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np

from . import _abi
from .tokenizer import BPETokenizer, BpeError, p32, p64


def shard_bounds(sizes: Sequence[int], world: int) -> List[int]:
    """Document boundaries of a contiguous, token-balanced partition: rank r owns documents [b[r], b[r+1]).
    A document belongs to the rank whose token range [r*T/world, (r+1)*T/world) contains its first token
    (empty trailing documents go to the last rank)."""
    starts = np.zeros(len(sizes) + 1, dtype=np.int64)
    np.cumsum(np.asarray(sizes, dtype=np.int64), out=starts[1:])
    total = int(starts[-1])
    bounds = [0]
    for r in range(1, world):
        cut = (total * r + world - 1) // world  # ceil
        bounds.append(int(np.searchsorted(starts[:-1], cut, side="left")))
    bounds.append(len(sizes))
    for r in range(1, len(bounds)):
        bounds[r] = max(bounds[r], bounds[r - 1])
    return bounds


def exchange_pair_counts(lib, handle, rank: int, world: int, device, group=None) -> None:
    """Sum the K1 pair histograms of all shards into every rank's table (once per index build): each rank exports
    (pair, count) device arrays, one NCCL all-gather moves them, every rank imports its peers' lists."""
    import torch
    import torch.distributed as dist

    def check(rc):
        if rc != _abi.BPE_OK:
            raise BpeError(rc, (lib.bpe_last_error(handle) or b"").decode("utf-8", "replace"))

    if world == 1:
        return
    state = C.c_int()
    check(lib.bpe_mg_state(handle, C.byref(state)))
    n = C.c_int64()
    if not state.value:
        check(lib.bpe_mg_export_counts(handle, None, None, 0, C.byref(n)))
    meta = torch.tensor([int(state.value), int(n.value)], dtype=torch.int64, device=device)
    metas = [torch.empty_like(meta) for _ in range(world)]
    dist.all_gather(metas, meta, group=group)
    metas = [m.tolist() for m in metas]
    flags = [m[0] for m in metas]
    if all(flags):
        return
    if any(flags):
        raise BpeError(_abi.BPE_E_INTERNAL, "ranks disagree on whether the pair counts were exchanged: %r" % (flags,))
    cap = max(max(m[1] for m in metas), 1)
    mine = torch.zeros((2, cap), dtype=torch.int32, device=device)
    check(lib.bpe_mg_export_counts(handle, C.c_void_p(mine[0].data_ptr()), C.c_void_p(mine[1].data_ptr()), cap, C.byref(n)))
    cnt = torch.tensor([int(n.value)], dtype=torch.int64, device=device)
    cnts = [torch.empty_like(cnt) for _ in range(world)]
    dist.all_gather(cnts, cnt, group=group)
    gathered = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(gathered, mine, group=group)
    sizes = [int(c.item()) for c in cnts]
    torch.cuda.synchronize(device)
    peers = [q for q in range(world) if q != rank]
    for q in peers:
        g = gathered[q]
        check(lib.bpe_mg_import_counts(handle, C.c_void_p(g[0].data_ptr()), C.c_void_p(g[1].data_ptr()), sizes[q], int(q == peers[-1])))


def order_new_chars(per_rank: Sequence[Tuple[Sequence[int], Sequence[int]]]) -> List[int]:
    """The new characters of a sharded text batch in the global first-appearance order of core.ts:186-199.
    per_rank[r] = (code_points, first_pos) as rank r's engine reported them, positions local to its shard.  Ranks hold
    contiguous document ranges in rank order, so the order key is (rank, first_pos) and a character that several ranks
    report belongs to the first of them, whatever its local positions."""
    seen, out = set(), []
    for cps, pos in per_rank:
        cps = np.asarray(cps, dtype=np.int64).reshape(-1)
        pos = np.asarray(pos, dtype=np.int64).reshape(-1)
        for k in np.argsort(pos, kind="stable").tolist():
            cp = int(cps[k])
            if cp not in seen:
                seen.add(cp)
                out.append(cp)
    return out


def _error_of(ex: Exception) -> Tuple[int, str]:
    if isinstance(ex, BpeError):
        return ex.code, ex.message
    return _abi.BPE_E_INTERNAL, repr(ex)


def text_ingest_collective(stage: Callable[[], Tuple[Sequence[int], Sequence[int]]], commit: Callable[[List[int]], np.ndarray],
                           n_tokens: int, world: int, group=None, device=None) -> Tuple[List[int], np.ndarray]:
    """The rank-side protocol of a sharded text ingest.  stage() decodes this rank's shard and returns its new
    characters with their local first positions; commit(code_points) appends the shard with the agreed characters and
    returns its counts (int64, n_tokens + len(code_points)).  -> (new characters in global order, counts summed over
    the ranks).  Two collectives on success: a gather of every rank's status and list, an all-reduce of the counts.
    A failure on any rank raises the same BpeError on every rank, and no rank is left waiting in a collective: a stage
    failure travels with the lists, a commit failure as a flag after the counts (then one more gather names it)."""
    import torch
    import torch.distributed as dist

    err: Optional[Tuple[int, str]] = None
    cps: Sequence[int] = []
    pos: Sequence[int] = []
    try:
        cps, pos = stage()
    except Exception as ex:  # (every rank must reach the gather below)
        err = _error_of(ex)
    mine = (err, [int(c) for c in cps], [int(p) for p in pos])
    parts = [mine]
    if world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, mine, group=group)
    for e in parts:
        if e[0] is not None:
            raise BpeError(*e[0])  # the first failing rank's error, on every rank
    new = order_new_chars([(p[1], p[2]) for p in parts])
    if n_tokens + len(new) > _abi.BPE_MAX_TOKENS:  # judged on the global count, identically everywhere
        raise BpeError(_abi.BPE_E_DOMAIN, "token table would exceed %d entries (%d new characters over %d ranks)" % (_abi.BPE_MAX_TOKENS, len(new), world))
    counts = np.zeros(n_tokens + len(new) + 1, dtype=np.int64)  # [-1]: ranks whose commit failed
    try:
        counts[:-1] = np.asarray(commit(new), dtype=np.int64)[: n_tokens + len(new)]
    except Exception as ex:
        err = _error_of(ex)
        counts[:] = 0
        counts[-1] = 1
    if world > 1:
        nccl = dist.get_backend(group) == "nccl"
        t = torch.from_numpy(counts).to(device if nccl else "cpu")
        dist.all_reduce(t, group=group)
        counts = t.cpu().numpy()
    if counts[-1]:
        errs = [err]
        if world > 1:
            errs = [None] * world
            dist.all_gather_object(errs, err, group=group)
        raise BpeError(*next(e for e in errs if e is not None))
    return new, counts[:-1]


class ShardedBPETokenizer(BPETokenizer):
    def __init__(self, device: Optional[int] = None, group=None):
        import torch
        import torch.distributed as dist

        if not dist.is_initialized():
            raise RuntimeError("ShardedBPETokenizer needs an initialised torch.distributed process group")
        self._dist = dist
        self._group = group
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)
        if device is None:
            device = torch.cuda.current_device()
        super().__init__(device)
        self._torch_device = torch.device("cuda", device)
        if self.world > _abi.MG_MAX_WORLD:
            raise BpeError(_abi.BPE_E_INVALID, "at most %d ranks (one NVLink domain)" % _abi.MG_MAX_WORLD)
        if self.world > 1:
            handle = C.create_string_buffer(64)
            self._check(self._lib.bpe_mg_init(self._h, self.rank, self.world, handle))
            handles: List[bytes] = [b""] * self.world
            dist.all_gather_object(handles, bytes(handle.raw), group=group)
            self._check(self._lib.bpe_mg_connect(self._h, b"".join(handles)))
            dist.barrier(group=group)

    # ---- corpus: keep only this rank's shard ------------------------------------------------------
    _ONCE = ("sharded corpus: add every document before the first merge/encode of the corpus "
             "(a later batch would break the global document order); clear the corpus first")

    def _reset_host(self) -> None:
        super()._reset_host()
        self._pending_restore: List[np.ndarray] = []  # restoreToCorpus documents (raw character ids), not yet uploaded
        self._uploaded = False  # fromJSON drops the corpus (core.ts:138-146)

    def _upload_shard(self, docs: List[np.ndarray], restore: bool) -> None:
        """Every rank holds ALL `docs` (SPMD); it uploads the contiguous, token-balanced range it owns."""
        if self._uploaded:
            raise BpeError(_abi.BPE_E_INVALID, self._ONCE)
        b = shard_bounds([d.size for d in docs], self.world)
        mine = docs[b[self.rank]:b[self.rank + 1]]
        offsets = np.zeros(len(mine) + 1, dtype=np.int64)
        np.cumsum([d.size for d in mine], out=offsets[1:])
        ids = np.concatenate(mine) if offsets[-1] else np.zeros(0, dtype=np.int32)
        fn = self._lib.bpe_restore_documents if restore else self._lib.bpe_add_documents
        self._check(fn(self._h, p32(np.ascontiguousarray(ids, dtype=np.int32)), p64(offsets), len(mine)))
        self._uploaded = True

    def _flush(self) -> None:
        self._sync_tokens()
        if self._pending and self._pending_restore:
            raise BpeError(_abi.BPE_E_INVALID, "sharded corpus: addToCorpus and restoreToCorpus documents cannot be mixed in one upload")
        if self._pending:
            docs, self._pending = self._pending, []
            self._upload_shard(docs, restore=False)
        elif self._pending_restore:
            docs, self._pending_restore = self._pending_restore, []
            self._upload_shard(docs, restore=True)

    def restoreToCorpus(self, content: str) -> None:  # core.ts:213-216, called with EVERY document on EVERY rank
        self._pending_restore.append(self._char_ids(content, create=False))

    def restoreDocuments(self, ids: np.ndarray, doc_offsets: np.ndarray, local_shard: bool = False) -> None:
        """Bulk restoreToCorpus.  local_shard=False: every rank passes ALL documents and keeps its shard;
        local_shard=True: the arrays hold only this rank's documents (ranks in document order)."""
        self._flush()
        if self._uploaded:
            raise BpeError(_abi.BPE_E_INVALID, self._ONCE)
        ids = np.ascontiguousarray(ids, dtype=np.int32)
        doc_offsets = np.ascontiguousarray(doc_offsets, dtype=np.int64)
        self._check_offsets(doc_offsets, ids.size)
        lo, hi = 0, len(doc_offsets) - 1
        if not local_shard:
            b = shard_bounds(np.diff(doc_offsets), self.world)
            lo, hi = b[self.rank], b[self.rank + 1]
        off = np.ascontiguousarray(doc_offsets[lo:hi + 1])
        self._check(self._lib.bpe_restore_documents(self._h, p32(ids), p64(off), hi - lo))
        self._uploaded = True

    def addTextBatch(self, utf8: bytes, doc_byte_offsets: np.ndarray, local_shard: bool = False) -> None:
        """Bulk addToCorpus from UTF-8 text (core.ts:182-207), bit-exact with one engine holding the whole batch.
        local_shard=False: every rank passes ALL documents and keeps a contiguous range balanced by bytes;
        local_shard=True: the arguments hold only this rank's documents (ranks in document order).  Each rank decodes
        its own shard on its device; the ranks then agree on the new characters' global first-appearance order (a list
        of at most 65 536 entries per rank, whatever the corpus size) and each appends its shard with it."""
        def stage():
            self._flush()
            if self._uploaded:
                raise BpeError(_abi.BPE_E_INVALID, self._ONCE)
            self._sync_chars()
            off = np.ascontiguousarray(doc_byte_offsets, dtype=np.int64)
            self._check_offsets(off, len(utf8))
            lo, hi = 0, len(off) - 1
            if not local_shard:
                b = shard_bounds(np.diff(off), self.world)
                lo, hi = b[self.rank], b[self.rank + 1]
            mine = np.ascontiguousarray(off[lo:hi + 1])
            buf = np.frombuffer(utf8, dtype=np.uint8) if len(utf8) else np.zeros(1, dtype=np.uint8)
            cps = np.empty(1 << 16, dtype=np.int32)
            pos = np.empty(1 << 16, dtype=np.int64)
            n = C.c_int32()
            self._check(self._lib.bpe_add_text_stage(self._h, buf.ctypes.data_as(_abi.u8p), p64(mine), hi - lo, p32(cps), p64(pos), cps.size, C.byref(n)))
            return cps[: n.value], pos[: n.value]

        def commit(new: List[int]) -> np.ndarray:
            cps = np.asarray(new, dtype=np.int32)
            counts = np.zeros(len(self.token_table) + cps.size, dtype=np.int64)
            self._check(self._lib.bpe_add_text_commit(self._h, p32(cps), cps.size, p64(counts), counts.size))
            return counts

        new, counts = text_ingest_collective(stage, commit, len(self.token_table), self.world, self._group, self._torch_device)
        self._uploaded = True
        self._add_text_tokens(new, counts)

    @property
    def corpus_in_code(self) -> List[str]:  # this rank's shard (corpusIdsAllRanks gathers every shard)
        return BPETokenizer.corpus_in_code.fget(self)

    @corpus_in_code.setter
    def corpus_in_code(self, value: Sequence[str]) -> None:  # every rank passes ALL documents, `[]` clears
        self.clearCorpus()
        self._sync_tokens()
        docs = [np.fromiter((ord(ch) - 1 for ch in s), dtype=np.int32, count=len(s)) for s in value]
        if docs:
            self._upload_shard(docs, restore=False)

    def addDocuments(self, ids: np.ndarray, doc_offsets: np.ndarray, local_shard: bool = False) -> None:
        """Bulk addToCorpus.  local_shard=False: every rank passes ALL documents and keeps its shard;
        local_shard=True: the arrays hold only this rank's documents (ranks in document order)."""
        import torch

        self._flush()
        if self._uploaded:
            raise BpeError(_abi.BPE_E_INVALID, "sharded corpus: documents were already uploaded; clear the corpus first")
        ids = np.ascontiguousarray(ids, dtype=np.int32)
        doc_offsets = np.ascontiguousarray(doc_offsets, dtype=np.int64)
        self._check_offsets(doc_offsets, ids.size)
        n_docs = len(doc_offsets) - 1
        counts = np.bincount(ids[doc_offsets[0]:doc_offsets[-1]], minlength=len(self.token_table)).astype(np.int64)
        if counts.size > len(self.token_table):
            raise ValueError("document holds an index outside token_table")
        if local_shard:
            if self.world > 1:
                backend = self._dist.get_backend(self._group)
                t = torch.from_numpy(counts).to(self._torch_device if backend == "nccl" else "cpu")
                self._dist.all_reduce(t, group=self._group)
                counts = t.cpu().numpy()
            lo, hi = 0, n_docs
        else:
            b = shard_bounds(np.diff(doc_offsets), self.world)
            lo, hi = b[self.rank], b[self.rank + 1]
        for i in np.nonzero(counts)[0]:
            t_ = self.token_table[i]
            t_.weight += int(counts[i])
            t_.original_weight += int(counts[i])
        off = np.ascontiguousarray(doc_offsets[lo:hi + 1])
        self._check(self._lib.bpe_add_documents(self._h, p32(ids), p64(off), hi - lo))
        self._uploaded = True

    def addDocumentsDevice(self, dev_ids_ptr: int, doc_offsets: np.ndarray, char_counts: np.ndarray) -> None:
        """local_shard bulk form with the ids already on this rank's device (bench path): `char_counts` = this shard's
        per-character counts, summed over the group here."""
        import torch

        self._flush()
        if self._uploaded:
            raise BpeError(_abi.BPE_E_INVALID, self._ONCE)
        counts = np.asarray(char_counts, dtype=np.int64)
        if self.world > 1:
            t = torch.from_numpy(counts.copy()).to(self._torch_device)
            self._dist.all_reduce(t, group=self._group)
            counts = t.cpu().numpy()
        for i in np.nonzero(counts)[0]:
            t_ = self.token_table[i]
            t_.weight += int(counts[i])
            t_.original_weight += int(counts[i])
        doc_offsets = np.ascontiguousarray(doc_offsets, dtype=np.int64)
        self._check(self._lib.bpe_add_documents_dev(self._h, C.c_void_p(dev_ids_ptr), p64(doc_offsets), len(doc_offsets) - 1))
        self._uploaded = True

    def clearCorpus(self) -> None:
        self._pending = []
        self._pending_restore = []
        self._check(self._lib.bpe_clear_corpus(self._h))
        self._uploaded = False

    def corpusIdsAllRanks(self) -> Tuple[np.ndarray, np.ndarray]:
        """The whole corpus in document order, gathered from every rank (tests / small corpora)."""
        ids, off = self.corpusIds()
        parts: List[Optional[tuple]] = [None] * self.world
        self._dist.all_gather_object(parts, (ids, off), group=self._group)
        all_ids = np.concatenate([p[0] for p in parts]) if parts else ids
        offs = [np.zeros(1, dtype=np.int64)]
        base = 0
        for p in parts:
            offs.append(p[1][1:] + base)
            base += int(p[1][-1])
        return all_ids, np.concatenate(offs)

    # ---- training -------------------------------------------------------------------------------------
    def _exchange_counts(self) -> None:
        exchange_pair_counts(self._lib, self._h, self.rank, self.world, self._torch_device, self._group)

    def mergeUntil(self, options: Optional[dict] = None, **kw) -> int:  # core.ts:365-383, on the sharded corpus
        self._flush()
        self._exchange_counts()
        return super().mergeUntil(options, **kw)

    def findNextMerge(self, options: Optional[dict] = None, **kw):
        raise BpeError(_abi.BPE_E_INVALID, "single-step findNextMerge/applyMerge are not available on a sharded corpus; use mergeUntil(max_iterations=1)")

    def applyMerge(self, merge) -> None:
        raise BpeError(_abi.BPE_E_INVALID, "single-step findNextMerge/applyMerge are not available on a sharded corpus; use mergeUntil(max_iterations=1)")
