"""GPU: bpe_add_text_stage / bpe_add_text_commit, the two halves of the text ingest a sharded corpus runs on every rank.
Several engines in one process act as ranks: each stages its shard, order_new_chars orders the reported lists, each
commits that order.  The new characters, the summed counts and the concatenated corpus must equal what one engine
running bpe_add_text on the whole batch produces.  Also: every rejection of a commit leaves the engine unchanged."""
import ctypes as C
import random

import numpy as np
import pytest

from bpe_tokenizer_b200 import _abi
from bpe_tokenizer_b200._abi import p32, p64
from bpe_tokenizer_b200.sharded import order_new_chars

pytestmark = pytest.mark.gpu

CAP = 1 << 16


@pytest.fixture(scope="module")
def lib():
    return _abi.load_library()


class Engine:
    def __init__(self, lib, table=(), merged=()):
        """table: the characters the table already knows (indices 0..), then `merged` multi-character tokens."""
        self.lib = lib
        self.h = C.c_void_p()
        assert lib.bpe_create(0, C.byref(self.h)) == 0
        toks = list(table) + list(merged)
        lens = np.array([len(t.encode("utf-16-le", "surrogatepass")) // 2 for t in toks], dtype=np.int32)
        self.ok(lib.bpe_set_tokens(self.h, p32(lens), len(lens)))
        cps = np.array([ord(c) for c in table], dtype=np.int32)
        self.ok(lib.bpe_set_chars(self.h, p32(cps), p32(np.arange(len(cps), dtype=np.int32)), len(cps)))

    def ok(self, rc):
        assert rc == 0, (rc, self.lib.bpe_last_error(self.h))

    def close(self):
        self.lib.bpe_destroy(self.h)

    def n_tokens(self):
        n = C.c_int32()
        self.ok(self.lib.bpe_num_tokens(self.h, C.byref(n)))
        return n.value

    def corpus(self):
        nd, nt = C.c_int64(), C.c_int64()
        self.ok(self.lib.bpe_corpus_size(self.h, C.byref(nd), C.byref(nt)))
        out = np.empty(max(nt.value, 1), dtype=np.int32)
        offs = np.zeros(nd.value + 1, dtype=np.int64)
        n = C.c_int64()
        self.ok(self.lib.bpe_get_corpus(self.h, 0, nd.value, p32(out), out.size, p64(offs), C.byref(n)))
        return out[: n.value], offs

    def add_text(self, docs):
        buf, off = _utf8(docs)
        cps = np.zeros(CAP, dtype=np.int32)
        n = C.c_int32()
        counts = np.zeros(self.n_tokens() + CAP, dtype=np.int64)
        self.ok(self.lib.bpe_add_text(self.h, buf.ctypes.data_as(_abi.u8p), p64(off), len(off) - 1, p32(cps), CAP, C.byref(n), p64(counts), counts.size))
        return cps[: n.value].tolist(), counts[: self.n_tokens()]

    def stage(self, docs):
        buf, off = _utf8(docs)
        cps = np.zeros(CAP, dtype=np.int32)
        pos = np.zeros(CAP, dtype=np.int64)
        n = C.c_int32()
        self.ok(self.lib.bpe_add_text_stage(self.h, buf.ctypes.data_as(_abi.u8p), p64(off), len(off) - 1, p32(cps), p64(pos), CAP, C.byref(n)))
        return cps[: n.value].tolist(), pos[: n.value].tolist()

    def commit(self, new):
        cps = np.array(new, dtype=np.int32)
        counts = np.zeros(self.n_tokens() + len(new), dtype=np.int64)
        rc = self.lib.bpe_add_text_commit(self.h, p32(cps), len(new), p64(counts), counts.size)
        return rc, counts


def _utf8(docs):
    parts = [d.encode("utf-8", "surrogatepass") for d in docs]
    off = np.zeros(len(parts) + 1, dtype=np.int64)
    np.cumsum([len(p) for p in parts], out=off[1:])
    buf = np.frombuffer(b"".join(parts) or b"\0", dtype=np.uint8)
    return buf, off


def _check_split(lib, docs, bounds, table=(), merged=()):
    """bounds: document ranges of the ranks, contiguous in rank order (empty ranges allowed)."""
    one = Engine(lib, table, merged)
    want_new, want_counts = one.add_text(docs)
    want_ids, want_off = one.corpus()
    ranks = [Engine(lib, table, merged) for _ in range(len(bounds) - 1)]
    reports = [r.stage(docs[bounds[q]:bounds[q + 1]]) for q, r in enumerate(ranks)]
    new = order_new_chars(reports)
    assert new == want_new
    counts = np.zeros(len(want_counts), dtype=np.int64)
    for r in ranks:
        rc, c = r.commit(new)
        assert rc == 0, r.lib.bpe_last_error(r.h)
        counts += c
        assert r.n_tokens() == one.n_tokens()
    assert counts.tolist() == want_counts.tolist()
    ids, offs, base = [], [np.zeros(1, dtype=np.int64)], 0
    for r in ranks:
        i, o = r.corpus()
        ids.append(i)
        offs.append(o[1:] + base)
        base += int(o[-1])
    assert np.array_equal(np.concatenate(ids), want_ids)
    assert np.array_equal(np.concatenate(offs), want_off)
    for e in ranks + [one]:
        e.close()
    return new


def test_stage_commit_over_ranks_equals_one_engine(lib):
    docs = ["héllo wörld", "", "中文字", "emoji \U0001F600\U0001F600 end", "lone \ud800 and \udfff",
            "max \U0010FFFF!", "a", "é中\U0001F600a", "\x00\x7f\x80߿ࠀ￿\U00010000"]
    for bounds in ([0, 9], [0, 4, 9], [0, 0, 5, 9], [0, 3, 3, 7, 9], [0, 9, 9], [0, 1, 2, 3, 9]):
        _check_split(lib, docs, bounds)
    # a character whose local first position on a later rank is smaller than on the earlier one
    new = _check_split(lib, ["xxxxxxxxxxé", "é\U0001F600"], [0, 1, 2])
    assert new == [ord("x"), 0xE9, 0x1F600]


def test_stage_commit_after_merged_tokens_and_without_new_characters(lib):
    # the table holds characters and merged tokens: new characters take the indices after all of them
    docs = ["abab é", "ba\U0001F600", "", "zz\ud800"]
    new = _check_split(lib, docs, [0, 2, 2, 4], table="ab ", merged=["ab", "ab ", "bab"])
    assert new == [0xE9, 0x1F600, ord("z"), 0xD800]
    # nothing new: every character is known
    assert _check_split(lib, ["abba", "", "b a"], [0, 1, 3], table="ab ", merged=["ab"]) == []
    # no documents at all, on every rank
    assert _check_split(lib, [], [0, 0, 0]) == []


def test_stage_commit_on_zipf_text(lib):
    from bpe_tokenizer_b200.synth import synth_corpus

    text, off = synth_corpus(300_000, seed=47)
    docs = [bytes(text[off[d]:off[d + 1]]).decode() for d in range(len(off) - 1)]
    rng = random.Random(3)
    for d in rng.sample(range(len(docs)), 20):  # scatter a few non-ASCII characters over the documents
        docs[d] = docs[d] + rng.choice(["é", "中", "\U0001F600", "\ud800", "\U0010FFFF"])
    n = len(docs)
    _check_split(lib, docs, [0, n // 5, n // 2, n // 2, n])


def _unchanged(e, before):
    assert e.n_tokens() == before[0]
    ids, off = e.corpus()
    assert np.array_equal(ids, before[1]) and np.array_equal(off, before[2])


def test_commit_rejections_change_nothing(lib):
    e = Engine(lib, "ab")
    assert e.add_text(["ab"])[0] == []
    state = lambda: (e.n_tokens(),) + e.corpus()  # noqa: E731
    before = state()
    # nothing staged
    rc, _ = e.commit([])
    assert rc == _abi.BPE_E_INVALID
    _unchanged(e, before)
    new, _ = e.stage(["bé中 a"])
    assert new == [0xE9, 0x4E2D, ord(" ")]
    for bad in ([0xE9, 0x4E2D],                      # misses a staged code point
                [0xE9, 0x4E2D, ord(" "), 0xE9],      # repeats one
                [0xE9, 0x4E2D, ord(" "), ord("a")],  # names one the table knows
                [0xE9, 0x4E2D, ord(" "), 0x110000],  # not a code point
                [0xE9, 0x4E2D, ord(" "), -5]):
        rc, _ = e.commit(bad)
        assert rc == _abi.BPE_E_INVALID, bad
        _unchanged(e, before)
    # a rejected commit leaves the batch staged: the right list (with a character only another rank saw) goes through
    rc, counts = e.commit([0x1F600, 0xE9, 0x4E2D, ord(" ")])
    assert rc == 0
    assert e.n_tokens() == 6 and counts.tolist() == [1, 1, 0, 1, 1, 1]
    ids, off = e.corpus()
    assert ids.tolist() == [0, 1, 1, 3, 4, 5, 0] and off.tolist() == [0, 2, 7]
    before = state()
    rc, _ = e.commit([0xE9, 0x4E2D, ord(" ")])  # committed once: nothing staged any more
    assert rc == _abi.BPE_E_INVALID
    _unchanged(e, before)
    # any call that reuses the staging buffers or replaces the character table discards the staged batch
    for other in ("encode_text", "encode_ids", "set_chars"):
        e.stage(["àb"])
        if other == "encode_text":
            buf, off = _utf8(["ab"])
            out, ooff, n = np.zeros(8, dtype=np.int32), np.zeros(2, dtype=np.int64), C.c_int64()
            e.ok(e.lib.bpe_encode_text_batch(e.h, buf.ctypes.data_as(_abi.u8p), p64(off), 1, None, 0, p32(out), out.size, p64(ooff), None, C.byref(n), None, None))
        elif other == "encode_ids":
            ids_in, off_in = np.array([0, 1], dtype=np.int32), np.array([0, 2], dtype=np.int64)
            out, ooff, n = np.zeros(8, dtype=np.int32), np.zeros(2, dtype=np.int64), C.c_int64()
            e.ok(e.lib.bpe_encode_batch(e.h, p32(ids_in), p64(off_in), 1, None, 0, p32(out), out.size, p64(ooff), None, C.byref(n)))
        else:
            cps = np.array([ord("a"), ord("b"), 0xE9, 0x4E2D, ord(" "), 0x1F600], dtype=np.int32)
            e.ok(e.lib.bpe_set_chars(e.h, p32(cps), p32(np.array([0, 1, 3, 4, 5, 2], dtype=np.int32)), len(cps)))
        rc, _ = e.commit([0xE0])
        assert rc == _abi.BPE_E_INVALID, other
        _unchanged(e, before)
    e.close()


def test_commit_domain_limit(lib):
    e = Engine(lib, "")
    lens = np.ones(_abi.BPE_MAX_TOKENS - 1, dtype=np.int32)
    e.ok(e.lib.bpe_set_tokens(e.h, p32(lens), len(lens)))
    e.ok(e.lib.bpe_set_chars(e.h, p32(np.array([ord("a")], dtype=np.int32)), p32(np.array([0], dtype=np.int32)), 1))
    assert e.stage(["ab"])[0] == [ord("b")]
    rc, _ = e.commit([ord("b"), ord("c")])  # the union of the ranks' characters no longer fits
    assert rc == _abi.BPE_E_DOMAIN
    assert e.n_tokens() == _abi.BPE_MAX_TOKENS - 1 and e.corpus()[0].size == 0
    rc, _ = e.commit([ord("b")])  # the last free index
    assert rc == 0 and e.n_tokens() == _abi.BPE_MAX_TOKENS
    assert e.corpus()[0].tolist() == [0, _abi.BPE_MAX_TOKENS - 1]
    e.close()

