"""One engine over several GPUs of one process (bpe_create_group, BPETokenizer(devices=[...])): the corpus is sharded by
document across the members, and every result equals the CPU oracle's and a single engine's.  The GPU tests run at 2 members
and at min(device_count, 4) on distinct GPUs; on a host with one GPU they skip, or, with BPE_GROUP_SHARE_DEVICE=1, run 2 and 4
members that share it."""
import ctypes as C
import random

import numpy as np
import pytest

from bpe_tokenizer_b200 import _abi

SIZES = pytest.mark.parametrize("members", ["2", "up to 4"])
# every size with the default loop, and again with BPE_LOOP_ROUNDS=0: then the sharded k_merge_loop runs every merge, where by default
# it only takes those above 2^20 global sites, which these corpora never reach
_LOOPS = [("2", None), ("up to 4", None), ("2", "0"), ("up to 4", "0")]
SIZES_LOOPS = pytest.mark.parametrize("members,loop_rounds", _LOOPS, ids=[m if r is None else m + "-rounds0" for m, r in _LOOPS])


def _set_loop(monkeypatch, loop_rounds):
    if loop_rounds is None:
        monkeypatch.delenv("BPE_LOOP_ROUNDS", raising=False)
    else:
        monkeypatch.setenv("BPE_LOOP_ROUNDS", loop_rounds)


def _devices(members):
    """Distinct GPUs; on a host with one GPU, members that share it when BPE_GROUP_SHARE_DEVICE=1 (each with its share of the SMs)."""
    import os

    import torch

    n = torch.cuda.device_count()
    if n < 2:
        if n == 1 and os.environ.get("BPE_GROUP_SHARE_DEVICE") == "1":
            return [0] * (2 if members == "2" else 4)
        pytest.skip("needs 2 GPUs (or BPE_GROUP_SHARE_DEVICE=1)")
    devs = list(range(2 if members == "2" else min(n, 4)))
    if not all(torch.cuda.can_device_access_peer(a, b) for a in devs for b in devs if a != b):
        pytest.skip("needs GPUs with peer access")
    return devs


def _merges(t):
    return [[a.index, b.index, c.weight] for a, b, c in t.merge_tokens]


def _offsets(lengths):
    off = np.zeros(len(lengths) + 1, dtype=np.int64)
    np.cumsum(lengths, out=off[1:])
    return off


def _utf8_batch(docs):
    chunks = [d.encode("utf-8", "surrogatepass") for d in docs]
    return b"".join(chunks), _offsets([len(c) for c in chunks])


def test_create_group_without_a_device_is_a_cuda_error():
    import torch

    if torch.cuda.is_available():
        pytest.skip("checks the answer without a device")
    from bpe_tokenizer_b200 import BPETokenizer, BpeError

    lib = _abi.load_library()
    h = C.c_void_p()
    assert lib.bpe_create_group((C.c_int * 2)(0, 1), 2, C.byref(h)) == _abi.BPE_E_CUDA
    assert lib.bpe_create_group((C.c_int * 1)(0), 1, C.byref(h)) == _abi.BPE_E_CUDA
    # the argument checks come first
    assert lib.bpe_create_group((C.c_int * 2)(1, 1), 2, C.byref(h)) == _abi.BPE_E_INVALID
    assert lib.bpe_create_group((C.c_int * 9)(*range(9)), 9, C.byref(h)) == _abi.BPE_E_INVALID
    assert lib.bpe_create_group((C.c_int * 1)(0), 0, C.byref(h)) == _abi.BPE_E_INVALID
    with pytest.raises(BpeError) as ex:
        BPETokenizer(devices=[0, 1])
    assert ex.value.code == _abi.BPE_E_CUDA


@pytest.mark.gpu
@SIZES_LOOPS
def test_fuzz_against_literal(members, loop_rounds, monkeypatch):
    """Small alphabets, runs, empty documents, option mixes; every other case adds documents after a mergeUntil (they go to the
    last member) and merges again.  The small alphabets make position tie-breaks, which each loop kernel must settle."""
    devs = _devices(members)
    _set_loop(monkeypatch, loop_rounds)
    from bpe_tokenizer_b200 import BPETokenizer
    from oracle import LiteralTokenizer

    def docs_of(rng, alphabet):
        return ["".join(rng.choice(alphabet) for _ in range(rng.randint(0, rng.choice([0, 20, 100, 400])))) for _ in range(rng.randint(1, 12))]

    tie_breaks = 0
    for case in range(10):
        rng = random.Random(7100 + case)
        alphabet = "ab" if case % 3 == 0 else "abcde "
        opts = [{"min_weight": rng.choice([None, 2, 4]), "max_length": rng.choice([None, 5, 9]), "max_iterations": rng.choice([None, None, 7])}
                for _ in range(2)]
        lit, grp = LiteralTokenizer(), BPETokenizer(devices=devs)
        docs = docs_of(rng, alphabet)
        for d in docs:
            lit.addToCorpus(d)
            grp.addToCorpus(d)
        assert grp.mergeUntil(opts[0]) == lit.mergeUntil(opts[0])
        assert _merges(grp) == _merges(lit), case
        if case % 2:
            more = docs_of(rng, alphabet + "xy")
            docs += more
            for d in more:
                lit.addToCorpus(d)
                grp.addToCorpus(d)
            assert grp.mergeUntil(opts[1]) == lit.mergeUntil(opts[1])
            assert _merges(grp) == _merges(lit), case
        assert grp.toJSON() == lit.toJSON(), case
        assert grp.corpus_in_code == lit.corpus_in_code, case
        for d in docs[:4]:
            try:
                want = lit.encodeToVector(d)
            except ValueError as ex:
                with pytest.raises(ValueError) as got:
                    grp.encodeToVector(d)
                assert str(got.value) == str(ex)
                continue
            assert grp.encodeToVector(d) == want
            assert grp.decodeVector(want) == lit.decodeVector(want)
        tie_breaks += grp.stats()["tie_breaks"]
        grp.close()
    assert tie_breaks > 0


def _zipf_tokenizers(devs, n_bytes):
    from bpe_tokenizer_b200 import BPETokenizer
    from bpe_tokenizer_b200.synth import first_appearance_ids, synth_corpus
    from oracle.int_oracle import IntOracleTokenizer

    text, off = synth_corpus(n_bytes, seed=43)
    ids, alphabet = first_appearance_ids(text)
    grp, one, orc = BPETokenizer(devices=devs), BPETokenizer(devs[0]), IntOracleTokenizer()
    for t in (grp, one, orc):
        t.addToCorpus("".join(chr(c) for c in alphabet))
        if hasattr(t, "_pending"):
            t._pending = []
        else:
            t._o.clear_corpus()
        for tk in t.token_table:
            tk.weight = 0
            tk.original_weight = 0
    grp.addDocuments(ids, off)
    one.addDocuments(ids, off)
    orc.add_ids(ids, off)
    return grp, one, orc


@pytest.mark.gpu
@SIZES_LOOPS
def test_zipf_1mb_500_merges(members, loop_rounds, monkeypatch):
    devs = _devices(members)
    _set_loop(monkeypatch, loop_rounds)
    grp, one, orc = _zipf_tokenizers(devs, 1_000_000)
    assert [t.mergeUntil({"max_iterations": 500}) for t in (grp, one, orc)] == [500] * 3
    assert _merges(grp) == _merges(orc) == _merges(one)
    assert grp.toJSON() == orc.toJSON()
    got, got_off = grp.corpusIds()
    want, want_off = one.corpusIds()
    assert np.array_equal(got, want) and np.array_equal(got_off, want_off)
    assert np.array_equal(got, np.concatenate([orc._o.document(d) for d in range(orc._o.num_documents())]))
    s = grp.stats()
    assert s["corpus_positions"] == one.stats()["corpus_positions"]
    assert s["corpus_tokens"] == got.size
    assert s["sites_merged"] == one.stats()["sites_merged"]
    grp.close()
    one.close()


# characters of 1 to 4 UTF-8 bytes whose first appearances fall into documents far apart in the batch, so on different members
_SPECIALS = ["é", "€", "\U0001d11e", "ж", "中", "\U0001f600", "ß", "\U00010348", "\x7f"]


def _text_docs(seed, n_docs, specials):
    rng = random.Random(seed)
    docs = []
    for i in range(n_docs):
        body = "".join(rng.choice("ab ") for _ in range(rng.randint(40, 80)))
        for s in specials[(i * 5) % len(specials):][: (i % 3)]:
            p = rng.randint(0, len(body))
            body = body[:p] + s + body[p:]
        docs.append(body if i % 7 != 5 else "")
    return docs


def _text_arrays(t):
    return t.toJSON()["token_table"], _merges(t)


@pytest.mark.gpu
@SIZES
def test_text_ingest_equals_one_engine(members):
    devs = _devices(members)
    from bpe_tokenizer_b200 import BPETokenizer
    from bpe_tokenizer_b200.tokenizer import _js_stringify

    grp, one = BPETokenizer(devices=devs), BPETokenizer(devs[0])
    first = _text_docs(11, 40, _SPECIALS)
    later = _text_docs(12, 9, _SPECIALS[::-1] + ["Ω", "\U0001f680"])  # a later batch goes to the last member
    for batch in (first, later):
        utf8, off = _utf8_batch(batch)
        for t in (grp, one):
            t.addTextBatch(utf8, off)
        assert _text_arrays(grp) == _text_arrays(one)
        assert grp.mergeUntil({"max_iterations": 60}) == one.mergeUntil({"max_iterations": 60})
        assert _text_arrays(grp) == _text_arrays(one)
        assert grp.corpus_in_code == one.corpus_in_code
    # unknown characters in two members: the first in batch order (document 15: member 0 of 2, member 1 of 4) wins over the one of
    # the last member (document 35)
    docs = _text_docs(13, 40, ["a"])
    docs[15] = docs[15][:9] + "☃" + docs[15][9:]
    docs[35] = "☄" + docs[35]
    utf8, off = _utf8_batch(docs)
    for t in (grp, one):
        with pytest.raises(ValueError) as ex:
            t.encodeTextBatch(utf8, off)
        assert str(ex.value) == "unknown token, char: " + _js_stringify("☃")
    answers = []
    for t in (grp, one):
        out = np.empty(len(utf8), dtype=np.int32)
        oo, bad = np.zeros(len(docs) + 1, dtype=np.int64), np.full(len(docs), -1, dtype=np.int64)
        n, upos, ucp = C.c_int64(), C.c_int64(-1), C.c_int32()
        rc = t._lib.bpe_encode_text_batch(t._h, np.frombuffer(utf8, dtype=np.uint8).ctypes.data_as(_abi.u8p), _abi.p64(off), len(docs), None, 0,
                                          _abi.p32(out), out.size, _abi.p64(oo), _abi.p64(bad), C.byref(n), C.byref(upos), C.byref(ucp))
        answers.append((rc, upos.value, ucp.value))
    assert answers[0] == answers[1] and answers[0][0] == _abi.BPE_E_INVALID and answers[0][2] == 0x2603
    grp.close()
    one.close()


def _trained_pair(devs):
    """A group and a single engine trained on the same documents; x occurs only before y, so merging (x, y) leaves x with
    weight 0 (a hole of the vector index)."""
    from bpe_tokenizer_b200 import BPETokenizer

    rng = random.Random(21)
    docs = ["".join(rng.choice("abcd e") for _ in range(rng.randint(0, 300))) for _ in range(60)] + ["xy" * 200 + " ab"] * 3
    grp, one = BPETokenizer(devices=devs), BPETokenizer(devs[0])
    for t in (grp, one):
        for d in docs:
            t.addToCorpus(d)
        t.mergeUntil({"max_iterations": 80})
        t.compactVectorIndex()
    assert _merges(grp) == _merges(one)
    assert grp.to_vector_index == one.to_vector_index and len(grp.to_vector_index) < len(grp.token_table)
    return grp, one, docs


def _raw_encode(t, ids, off, out_cap, vector=True):
    out = np.empty(max(out_cap, 1), dtype=np.int32)
    oo, bad = np.zeros(len(off), dtype=np.int64), np.full(max(len(off) - 1, 1), -1, dtype=np.int64)
    n = C.c_int64()
    tvi = t._tvi_array() if vector else None
    rc = t._lib.bpe_encode_batch(t._h, _abi.p32(ids), _abi.p64(off), len(off) - 1, _abi.p32(tvi) if tvi is not None else None,
                                 len(tvi) if tvi is not None else 0, _abi.p32(out) if out_cap else None, out_cap, _abi.p64(oo), _abi.p64(bad), C.byref(n))
    return rc, n.value, out[: n.value].copy() if rc == 0 else None, oo, bad


@pytest.mark.gpu
@SIZES
def test_encode_decode_equal_one_engine(members):
    devs = _devices(members)
    grp, one, docs = _trained_pair(devs)
    batch = docs[:50] + ["x", "", "xy", "yx" * 7] + docs[50:]
    ids = np.concatenate([one._char_ids(d, create=False) for d in batch]).astype(np.int32)
    off = _offsets([len(d) for d in batch])
    for vector in (True, False):
        a, b = grp.encodeBatch(ids, off, vector=vector), one.encodeBatch(ids, off, vector=vector)
        for x, y in zip(a, b):
            assert np.array_equal(x, y)
    vals, voff, bad = one.encodeBatch(ids, off)
    assert (bad >= 0).any()
    utf8, boff = _utf8_batch(batch)
    for x, y, z in zip(grp.encodeTextBatch(utf8, boff), one.encodeTextBatch(utf8, boff), (vals, voff, bad)):
        assert np.array_equal(x, y) and np.array_equal(x, z)
    # decode, with a value no vector index has
    dvals = vals.copy()
    dvals[voff[int(np.nonzero(np.diff(voff))[0][0])]] = 10 ** 6
    ga, oa = grp.decodeBatch(dvals, voff), one.decodeBatch(dvals, voff)
    assert ga[0] == oa[0] and np.array_equal(ga[1], oa[1]) and np.array_equal(ga[2], oa[2]) and (ga[2] >= 0).any()
    # out_cap: too small by one, exactly the output (less than the input: the members write past it), a size query
    need = vals.size
    assert need < ids.size
    for cap in (need - 1, need, 0):
        rg, ro = _raw_encode(grp, ids, off, cap), _raw_encode(one, ids, off, cap)
        assert rg[0] == ro[0] == (_abi.BPE_OK if cap == need else _abi.BPE_E_CAPACITY)
        assert rg[1] == ro[1] == need
        assert np.array_equal(rg[3], ro[3]) and np.array_equal(rg[4], ro[4])
        if cap == need:
            assert np.array_equal(rg[2], ro[2]) and np.array_equal(rg[2], vals)
    grp.close()
    one.close()


@pytest.mark.gpu
@SIZES
def test_resume_equals_uninterrupted_run(members):
    """toJSON -> fromJSON on a group -> restoreToCorpus of every document -> mergeUntil (and restoreMerge on an emptied corpus)."""
    devs = _devices(members)
    from bpe_tokenizer_b200 import BPETokenizer, compactMerge
    from bpe_tokenizer_b200.synth import synth_corpus

    text, off = synth_corpus(120_000, seed=47)
    docs = [bytes(text[off[d]:off[d + 1]]).decode() for d in range(len(off) - 1)]
    full, part = BPETokenizer(devices=devs), BPETokenizer(devices=devs)
    for t in (full, part):
        for d in docs:
            t.addToCorpus(d)
    full.mergeUntil({"max_iterations": 300})
    part.mergeUntil({"max_iterations": 120})
    snap = part.toJSON()
    part.close()
    resumed = BPETokenizer(devices=devs)
    resumed.fromJSON(snap)
    for d in docs:
        resumed.restoreToCorpus(d)
    resumed.mergeUntil({"max_iterations": 180})
    assert resumed.toJSON() == full.toJSON()
    assert resumed.corpus_in_code == full.corpus_in_code
    # the merge-log route (example/import-merge-log-to-ram.ts): characters, an emptied corpus, one restoreMerge per line
    replay = BPETokenizer(devices=devs)
    for d in docs:
        replay.addToCorpus(d)
    replay.corpus_in_code = []
    for m in full.merge_tokens[:40]:
        replay.restoreMerge(compactMerge(m))
    assert replay.toJSON()["merge_codes"] == full.toJSON()["merge_codes"][:40]
    full.close()
    resumed.close()
    replay.close()


@pytest.mark.gpu
def test_refusals(monkeypatch):
    import os

    devs = _devices("up to 4")
    share = os.environ.pop("BPE_GROUP_SHARE_DEVICE", None)  # (repeated devices are refused by default)
    from bpe_tokenizer_b200 import BPETokenizer, BpeError
    from bpe_tokenizer_b200.tokenizer import Token
    from oracle import LiteralTokenizer

    lib = _abi.load_library()
    h = C.c_void_p()
    for bad in ([0, 1, 0], list(range(9))):
        assert lib.bpe_create_group((C.c_int * len(bad))(*bad), len(bad), C.byref(h)) == _abi.BPE_E_INVALID
        with pytest.raises(BpeError) as ex:
            BPETokenizer(devices=bad)
        assert ex.value.code == _abi.BPE_E_INVALID
    if share is not None:
        monkeypatch.setenv("BPE_GROUP_SHARE_DEVICE", share)
    docs = ["abababcab", "", "cabcab ab", "abc" * 20]
    grp, lit = BPETokenizer(devices=devs), LiteralTokenizer()
    # a refused upload adds nothing on any member (here the last document names a token that does not exist)
    lens = np.ones(3, dtype=np.int32)
    assert grp._lib.bpe_set_tokens(grp._h, _abi.p32(lens), 3) == 0
    bad_ids = np.array([0, 1, 0, 1, 2, 0, 1, 2, 0, 1, 7], dtype=np.int32)
    bad_off = np.array([0, 3, 6, 9, 11], dtype=np.int64)
    assert grp._lib.bpe_add_documents(grp._h, _abi.p32(bad_ids), _abi.p64(bad_off), 4) == _abi.BPE_E_INVALID
    nd, nt = C.c_int64(), C.c_int64()
    assert grp._lib.bpe_corpus_size(grp._h, C.byref(nd), C.byref(nt)) == 0 and nd.value == nt.value == 0
    # an id outside the token table in encode: its position within the batch, as one engine reports it
    out, oo, n = np.empty(11, dtype=np.int32), np.zeros(5, dtype=np.int64), C.c_int64()
    assert grp._lib.bpe_encode_batch(grp._h, _abi.p32(bad_ids), _abi.p64(bad_off), 4, None, 0, _abi.p32(out), 11, _abi.p64(oo), None, C.byref(n)) == _abi.BPE_E_INVALID
    assert b"id 7 at 10 outside the token table" in grp._lib.bpe_last_error(grp._h)
    assert grp._lib.bpe_set_tokens(grp._h, None, 0) == 0
    for t in (grp, lit):
        for d in docs:
            t.addToCorpus(d)
    before = grp.toJSON()
    with pytest.raises(BpeError) as ex:
        grp.findNextMerge()
    assert ex.value.code == _abi.BPE_E_INVALID
    m, found = _abi.bpe_merge(), C.c_int()
    assert grp._lib.bpe_find_next_merge(grp._h, 2, 0, C.byref(m), C.byref(found)) == _abi.BPE_E_INVALID
    a, b = grp.token_table[0], grp.token_table[1]
    n = len(grp.token_table)
    with pytest.raises(BpeError) as ex:
        grp.applyMerge((a, b, Token(a.chars + b.chars, 1, 1, chr(n + 1), n)))
    assert ex.value.code == _abi.BPE_E_INVALID
    with pytest.raises(BpeError) as ex:
        grp.restoreMerges([[a.code, b.code, 1]])
    assert ex.value.code == _abi.BPE_E_INVALID
    assert grp._lib.bpe_apply_merge(grp._h, a.index, b.index, n, None) == _abi.BPE_E_INVALID
    assert grp._lib.bpe_set_stream(grp._h, None) == _abi.BPE_E_INVALID
    with pytest.raises(BpeError) as ex:
        grp.set_stream(0)
    assert ex.value.code == _abi.BPE_E_INVALID
    assert grp.toJSON() == before  # nothing on the host moved
    # the group still trains exactly
    assert grp.mergeUntil() == lit.mergeUntil()
    assert grp.toJSON() == lit.toJSON() and grp.corpus_in_code == lit.corpus_in_code
    grp.close()
