"""GPU: the CUDA path (through the C ABI) against the CPU oracle -- the reference's known answers,
the committed golden fixtures, seeded fuzzing step by step, and MB-scale Zipf corpora."""
import json
import os
import random

import numpy as np
import pytest

import kat_suite
from oracle import LiteralTokenizer, compact_merge
from oracle.int_oracle import IntOracleTokenizer
from pair_counts import device_counts, loop_counts, recount

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "literal_cases.json")


def make():
    from bpe_tokenizer_b200 import BPETokenizer

    return BPETokenizer()


def rows(t):
    return [(x.chars, x.weight, x.original_weight, x.code, x.index) for x in t.token_table]


@pytest.mark.parametrize("kat", kat_suite.ALL, ids=lambda f: f.__name__)
def test_reference_known_answers(kat):
    kat(make)


def test_reference_merge_log_resume():
    from bpe_tokenizer_b200 import compactMerge

    kat_suite.kat_merge_log_resume(make, compactMerge)


def test_committed_golden_fixtures():
    with open(GOLDEN, encoding="utf-8") as f:
        cases = json.load(f)
    for case in cases:
        t = make()
        for d in case["docs"]:
            t.addToCorpus(d)
        t.mergeUntil(case["options"])
        assert [[a.index, b.index, c.weight] for a, b, c in t.merge_tokens] == case["merges"], case["name"]
        assert t.toJSON() == case["json"], case["name"]
        for text, want in case["encode"]:
            try:
                got = list(t.encodeToVector(text))
            except ValueError as e:
                got = "throws: " + str(e)
            assert got == want, (case["name"], text)


def _random_docs(rng, alphabet, n_docs, max_len):
    return ["".join(rng.choice(alphabet) for _ in range(rng.randint(0, max_len))) for _ in range(n_docs)]


@pytest.mark.parametrize("scan_mode", [0, 1])
@pytest.mark.parametrize("seed", range(24))
def test_fuzz_step_by_step_against_literal(seed, scan_mode):
    """findNextMerge / applyMerge one at a time: same winner (tie-breaks included), same corpus,
    same pair histogram after every merge.  scan_mode=1 discovers sites by a full scan instead of the
    occurrence lists; both must agree with the literal restatement."""
    rng = random.Random(1000 + seed)
    alphabet = "abc"[: 1 + seed % 3] if seed % 2 else "abcdefgh"[: 2 + seed % 7]
    docs = _random_docs(rng, alphabet, rng.randint(1, 5), rng.choice([8, 30, 120]))
    max_length = rng.choice([None, None, 3, 4, 8])
    min_weight = rng.choice([None, 2, 3])
    lit, gpu = LiteralTokenizer(), make()
    gpu._lib.bpe_set_profiling(gpu._h, 2 if scan_mode else 0)
    for d in docs:
        lit.addToCorpus(d)
        gpu.addToCorpus(d)
    assert gpu.corpus_in_code == lit.corpus_in_code
    opts = {"min_weight": min_weight, "max_length": max_length}
    for step in range(300):
        m1 = lit.findNextMerge(opts)
        m2 = gpu.findNextMerge(opts)
        if m1 is None:
            assert m2 is None
            break
        assert (m2[0].index, m2[1].index, m2[2].weight, m2[2].chars) == (m1[0].index, m1[1].index, m1[2].weight, m1[2].chars), step
        lit.applyMerge(m1)
        gpu.applyMerge(m2)
        assert gpu.corpus_in_code == lit.corpus_in_code, step
        toks = [[ord(ch) - 1 for ch in doc] for doc in lit.corpus_in_code]
        assert device_counts(gpu) == recount([x for d in toks for x in d], [len(d) for d in toks]), step
    assert gpu.toJSON() == lit.toJSON()
    for d in docs + _random_docs(rng, alphabet, 3, 60):
        try:
            want = lit.encodeToCode(d)
        except ValueError as e:
            with pytest.raises(ValueError) as ei:
                gpu.encodeToCode(d)
            assert str(ei.value) == str(e)
            continue
        assert gpu.encodeToCode(d) == want


@pytest.mark.parametrize("mode", [0, 2])  # 0: persistent kernel, 2: persistent + full-scan sites
@pytest.mark.parametrize("seed", range(18))
def test_fuzz_merge_until_against_literal(seed, mode):
    rng = random.Random(2000 + seed)
    alphabet = "ab" if seed % 3 == 0 else "abcde "
    docs = _random_docs(rng, alphabet, rng.randint(1, 8), rng.choice([20, 100, 400]))
    opts = {"min_weight": rng.choice([None, 2, 4]), "max_length": rng.choice([None, 5, 9]), "max_iterations": rng.choice([None, None, 7])}
    lit, gpu = LiteralTokenizer(), make()
    gpu._lib.bpe_set_profiling(gpu._h, mode)
    for d in docs:
        lit.addToCorpus(d)
        gpu.addToCorpus(d)
    lit.mergeUntil(opts)
    gpu.mergeUntil(opts)
    assert [[a.index, b.index, c.weight] for a, b, c in gpu.merge_tokens] == [[a.index, b.index, c.weight] for a, b, c in lit.merge_tokens]
    assert gpu.toJSON() == lit.toJSON()
    assert gpu.corpus_in_code == lit.corpus_in_code
    for d in docs:
        try:
            want = lit.encodeToVector(d)
        except ValueError as e:
            with pytest.raises(ValueError, match=str(e)):
                gpu.encodeToVector(d)
            continue
        assert gpu.encodeToVector(d) == want
        assert gpu.decodeVector(want) == d


def test_long_runs_and_chains():
    for text in ["x" * 1000, "ab" * 700, "aab" * 300 + "a" * 77, "x" * 33 + "y" + "x" * 64]:
        lit, gpu = LiteralTokenizer(), make()
        lit.addToCorpus(text)
        gpu.addToCorpus(text)
        lit.mergeUntil({})
        gpu.mergeUntil({})
        assert gpu.toJSON() == lit.toJSON(), text[:10]
        assert gpu.corpus_in_code == lit.corpus_in_code
        assert gpu.encodeToVector(text) == lit.encodeToVector(text)


def test_pair_histogram_matches_oracle_counts():
    import ctypes as C
    from bpe_tokenizer_b200 import _abi
    from bpe_tokenizer_b200.synth import synth_corpus

    text, off = synth_corpus(300000)
    docs = [bytes(text[off[d]:off[d + 1]]).decode() for d in range(len(off) - 1)]
    lit, gpu = LiteralTokenizer(), make()
    for d in docs:
        lit.addToCorpus(d)
        gpu.addToCorpus(d)
    gpu._flush()
    cap = 1 << 16
    a = np.zeros(cap, dtype=np.int32)
    b = np.zeros(cap, dtype=np.int32)
    c = np.zeros(cap, dtype=np.int64)
    n = C.c_int64()
    gpu._check(gpu._lib.bpe_pair_counts(gpu._h, _abi.p32(a), _abi.p32(b), _abi.p64(c), cap, C.byref(n)))
    got = {(int(a[i]), int(b[i])): int(c[i]) for i in range(n.value)}
    assert got == loop_counts([[ord(ch) - 1 for ch in doc] for doc in lit.corpus_in_code])


def _zipf_pair(n_bytes, seed=43):
    from bpe_tokenizer_b200.synth import synth_corpus, first_appearance_ids

    text, off = synth_corpus(n_bytes, seed=seed)
    ids, alphabet = first_appearance_ids(text)
    return text, off, ids, alphabet


def _seed_tables(tok_gpu, tok_orc, alphabet):
    # register the single-character tokens in first-appearance order (what addToCorpus would do)
    for t in (tok_gpu, tok_orc):
        t.addToCorpus("".join(chr(c) for c in alphabet))
        if hasattr(t, "_pending"):
            t._pending = []
        else:
            t._o.clear_corpus()
        for tk in t.token_table:
            tk.weight = 0
            tk.original_weight = 0


def test_zipf_1mb_500_merges_bit_exact():
    text, off, ids, alphabet = _zipf_pair(1_000_000)
    gpu, orc = make(), IntOracleTokenizer()
    _seed_tables(gpu, orc, alphabet)
    gpu.addDocuments(ids, off)
    orc.add_ids(ids, off)
    assert rows(gpu) == rows(orc)
    n1 = gpu.mergeUntil({"max_iterations": 500})
    n2 = orc.mergeUntil({"max_iterations": 500})
    assert n1 == n2 == 500
    assert [[a.index, b.index, c.weight] for a, b, c in gpu.merge_tokens] == [[a.index, b.index, c.weight] for a, b, c in orc.merge_tokens]
    assert gpu.toJSON() == orc.toJSON()
    got_ids, got_off = gpu.corpusIds()
    want = np.concatenate([orc._o.document(d) for d in range(orc._o.num_documents())])
    assert np.array_equal(got_ids, want)
    # token.weight == live occurrences of the token in the corpus (core.ts:201,345-346 bookkeeping)
    assert np.array_equal(np.bincount(got_ids, minlength=len(gpu.token_table)), np.array([t.weight for t in gpu.token_table]))
    # encode unseen text (seed 44): vectors or the same throw
    text2, off2, _, _ = _zipf_pair(60_000, seed=44)
    lut = np.full(256, -1, dtype=np.int32)
    lut[alphabet] = np.arange(len(alphabet))
    ids2 = lut[text2]
    vals, ooff, bad = gpu.encodeBatch(ids2, off2, vector=True)
    raw, roff, _ = gpu.encodeBatch(ids2, off2, vector=False)
    orc.compactVectorIndex()
    for d in range(len(off2) - 1):
        want_raw = orc.encode_ids(ids2[off2[d]:off2[d + 1]])
        assert np.array_equal(raw[roff[d]:roff[d + 1]], want_raw), d
        holes = [i for i, x in enumerate(want_raw.tolist()) if x not in orc.to_vector_index]
        assert bad[d] == (holes[0] if holes else -1)
        if not holes:
            assert vals[ooff[d]:ooff[d + 1]].tolist() == [orc.to_vector_index[x] for x in want_raw.tolist()]


@pytest.mark.parametrize("opts", [{}, {"max_length": 6}, {"min_weight": 150}], ids=["plain", "max_length6", "min_weight150"])
@pytest.mark.parametrize("k", ["16", "4", "1", "off"])
def test_merge_rounds_equal_the_oracle(k, opts, monkeypatch):
    """mergeUntil commits several merges per barrier round (csrc/round_kernels.cuh): whatever the batch size (BPE_LOOP_K;
    "off" = the one-merge-per-iteration kernel), the merge log, weights and corpus must equal the incremental CPU oracle's
    (core.ts:365-383 semantics, pinned to the literal restatement by tests/test_oracle_golden.py)."""
    from oracle.fast_oracle import FastOracle

    if k == "off":
        monkeypatch.setenv("BPE_LOOP_ROUNDS", "0")
    else:
        monkeypatch.setenv("BPE_LOOP_K", k)
    text, off, ids, alphabet = _zipf_pair(6_000_000)
    merges = 3000
    gpu = make()
    gpu.addToCorpus("".join(chr(c) for c in alphabet))
    gpu.corpus_in_code = []
    for tk in gpu.token_table:
        tk.weight = tk.original_weight = 0
    gpu.addDocuments(ids, off)
    n = gpu.mergeUntil(dict(opts, max_iterations=merges))
    o = FastOracle()
    o.set_len16(np.ones(len(alphabet), dtype=np.int32))
    o.add_documents(ids, off)
    la, lb, lw = o.merge_until(int(opts.get("min_weight", 2)), int(opts.get("max_length", 0)), merges, len(alphabet), merges)
    got = [[a.index, b.index, c.original_weight] for a, b, c in gpu.merge_tokens]
    want = [[int(a), int(b), int(w)] for a, b, w in zip(la, lb, lw)]
    first_bad = next((i for i, (g, w) in enumerate(zip(got, want)) if g != w), None)
    assert first_bad is None, (first_bad, got[first_bad], want[first_bad])
    assert n == len(want)
    got_ids, _ = gpu.corpusIds()
    assert np.array_equal(got_ids, o.corpus())
    st = gpu.stats()
    if k not in ("off", "1") and not opts:
        assert st["loop_rounds"] > 0 and st["loop_round_merges"] == n
        assert st["loop_round_merges"] > 1.5 * st["loop_rounds"], st  # the batches really are batches


def test_cfg2_full_size_merge_log_matches_the_oracle():
    """BASELINE config 2 at FULL size (10 MB seeded Zipf corpus, 4 000 merges, SURVEY.md section 8(d) "cfg2: full bit-exact"): the
    product's merge log -- pairs, new indices and weights, in the byte layout bench.py hashes -- equals the one the CPU restatement
    of core.ts produced offline (tests/golden/make_cfg2_golden.py, minutes of CPU; the fixture keeps its SHA-1 and both ends)."""
    import hashlib

    from bpe_tokenizer_b200._abi import MERGE_DTYPE
    from bpe_tokenizer_b200.synth import first_appearance_ids, synth_corpus

    with open(os.path.join(os.path.dirname(__file__), "golden", "cfg2_merge_log.json")) as f:
        golden = json.load(f)
    text, off = synth_corpus(10_000_000, seed=43)
    ids, alphabet = first_appearance_ids(text)
    assert len(alphabet) == golden["alphabet"] and "%d B" % text.size in golden["workload"] and "%d docs" % (len(off) - 1) in golden["workload"]
    gpu = make()
    gpu.addToCorpus("".join(chr(c) for c in alphabet))  # the single-character tokens in first-appearance order
    gpu._pending = []
    for tk in gpu.token_table:
        tk.weight = tk.original_weight = 0
    gpu.addDocuments(ids, off)
    assert gpu.mergeUntil({"max_iterations": golden["merges"]}) == golden["merges"]
    log = np.zeros(golden["merges"], dtype=MERGE_DTYPE)
    log["a"] = [a.index for a, _, _ in gpu.merge_tokens]
    log["b"] = [b.index for _, b, _ in gpu.merge_tokens]
    log["c"] = [c.index for _, _, c in gpu.merge_tokens]
    log["weight"] = [c.original_weight for _, _, c in gpu.merge_tokens]
    assert [[int(r["a"]), int(r["b"]), int(r["weight"])] for r in log[:8]] == golden["first"]
    assert [[int(r["a"]), int(r["b"]), int(r["weight"])] for r in log[-4:]] == golden["last"]
    assert hashlib.sha1(log["weight"].astype(np.int64).tobytes()).hexdigest() == golden["weights_sha1"]
    assert hashlib.sha1(log.tobytes()).hexdigest() == golden["sha1"]


def test_resume_routes_equal_uninterrupted_run():
    """cfg5 shape at test size: max_length=8, split run resumed (a) via toJSON -> fromJSON -> restoreToCorpus
    (core.ts:213-216) and (b) via addToCorpus + restoreMerge(compactMerge(...)) (core.ts:477-494); both must equal the
    uninterrupted run -- and every stage must equal the ORACLE doing the same thing (the compiled restatement for the
    mergeUntil stages, the literal one for restoreToCorpus / restoreMerge on a sample)."""
    from bpe_tokenizer_b200.synth import synth_corpus

    text, off = synth_corpus(200_000)
    docs = [bytes(text[off[d]:off[d + 1]]).decode() for d in range(len(off) - 1)]
    opts = {"max_length": 8, "max_iterations": 60}

    def run(factory, n):
        t = factory()
        for d in docs:
            t.addToCorpus(d)
        t.mergeUntil({"max_length": 8, "max_iterations": n})
        return t

    full, o_full = run(make, 120), run(IntOracleTokenizer, 120)
    assert full.toJSON() == o_full.toJSON()
    assert full.corpus_in_code == o_full.corpus_in_code
    first, o_first = run(make, 60), run(IntOracleTokenizer, 60)
    assert first.toJSON() == o_first.toJSON()
    assert first.corpus_in_code == o_first.corpus_in_code
    snap = json.loads(json.dumps(first.toJSON()))
    # the reference logs compactMerge(merge) at findNextMerge time, when c.weight is still its original weight
    log = [[a.code, b.code, c.original_weight] for a, b, c in first.merge_tokens]
    assert log == [[a.code, b.code, c.original_weight] for a, b, c in o_first.merge_tokens]
    # route (a): the GPU and the oracle both restore every document from the same snapshot
    a, o_a = make(), IntOracleTokenizer()
    for t in (a, o_a):
        t.fromJSON(json.loads(json.dumps(snap)))
        for d in docs:
            t.restoreToCorpus(d)
    assert a.corpus_in_code == o_a.corpus_in_code == first.corpus_in_code
    assert a.toJSON() == o_a.toJSON()
    lit = LiteralTokenizer()  # the string-level restatement's restoreToCorpus on a sample of the documents (it is slow)
    lit.fromJSON(json.loads(json.dumps(snap)))
    for d in docs[:40]:
        lit.restoreToCorpus(d)
    assert lit.corpus_in_code == a.corpus_in_code[:40]
    a.mergeUntil(opts)
    o_a.mergeUntil(opts)
    assert a.toJSON() == o_a.toJSON() == full.toJSON()
    assert a.corpus_in_code == o_a.corpus_in_code == full.corpus_in_code
    # route (b): replay the merge log line by line
    b, o_b = make(), IntOracleTokenizer()
    for t in (b, o_b):
        for d in docs:
            t.addToCorpus(d)
        for m in log:
            t.restoreMerge(list(m))
    assert b.toJSON() == o_b.toJSON() == first.toJSON()
    assert b.corpus_in_code == o_b.corpus_in_code
    b.mergeUntil(opts)
    o_b.mergeUntil(opts)
    assert b.toJSON() == o_b.toJSON() == full.toJSON()
    assert b.corpus_in_code == o_b.corpus_in_code
    # merge log replay with the corpus emptied (example/import-merge-log-to-ram.ts:22-31)
    c, o_c = make(), LiteralTokenizer()
    for t in (c, o_c):
        for d in docs[:50]:
            t.addToCorpus(d)
        t.corpus_in_code = []
        for m in log:
            t.restoreMerge(list(m))
    assert c.toJSON() == o_c.toJSON()
    assert [t.chars for t in c.token_table] == [t.chars for t in first.token_table]


def test_encode_edge_cases():
    t, lit = make(), LiteralTokenizer()
    docs = ["", "a", "ab" * 10, "hello world " * 200, "", "zzz"]
    for d in docs:
        t.addToCorpus(d)
        lit.addToCorpus(d)
    t.mergeUntil({})
    lit.mergeUntil({})
    assert t.toJSON() == lit.toJSON()
    assert t.corpus_in_code == lit.corpus_in_code  # empty documents are kept (core.ts:206)
    long_text = "hello world " * 500  # > 1024 tokens: the global-scratch encode path
    assert t.encodeToCode(long_text) == lit.encodeToCode(long_text)
    assert t.encodeToCode("") == ""
    assert t.encodeToVector("") == []
    with pytest.raises(ValueError, match="unknown token, char"):
        t.encodeToVector("hello?")
    for text in ["world hello", "hello world ", "zzz", "a"]:
        try:
            want = lit.encodeToVector(text)
        except ValueError as e:
            with pytest.raises(ValueError) as ei:
                t.encodeToVector(text)
            assert str(ei.value) == str(e)
            continue
        assert t.encodeToVector(text) == want
        assert t.decodeVector(want) == text


def test_add_to_corpus_after_merges_appends_raw_ids():
    t, lit = make(), LiteralTokenizer()
    for x in (t, lit):
        x.addToCorpus("abababab")
        x.mergeUntil({})
        x.addToCorpus("ababcab")  # core.ts:204 appends raw single-character codes; 'c' is a new token after the merges
        x.mergeUntil({})
    assert t.toJSON() == lit.toJSON()
    assert t.corpus_in_code == lit.corpus_in_code


@pytest.mark.parametrize("lmax", ["auto", "48", "32", "24", "20", "16"])
@pytest.mark.parametrize("seed", range(6))
def test_encode_batch_lane_path_fuzz(seed, lmax, monkeypatch):
    """K4: the lane path (encode_lanes.cuh, the default; "auto": the geometry the batch's longest document selects, else one
    forced geometry per value) on batches of ragged documents -- empty, single-token, runs, documents longer than one lane
    batch (per-document fallback) -- against the sequential replaceAll of core.ts:404-406, with the per-document kernel as
    the cross-check."""
    if lmax == "auto":
        monkeypatch.delenv("BPE_ENC_LMAX", raising=False)
    else:
        monkeypatch.setenv("BPE_ENC_LMAX", lmax)
    rng = random.Random(7000 + seed)
    alphabet = ["ab", "abc", "abcdef ", "ab", "abcdefghijklmnopqrstuvwxyz ", "xy "][seed]
    train = _random_docs(rng, alphabet, rng.randint(2, 10), rng.choice([50, 300, 2000]))
    lit, gpu = LiteralTokenizer(), make()
    for d in train:
        lit.addToCorpus(d)
        gpu.addToCorpus(d)
    opts = {"max_length": rng.choice([None, 6]), "max_iterations": rng.choice([None, 3, 40])}
    lit.mergeUntil(opts)
    gpu.mergeUntil(opts)
    assert gpu.toJSON() == lit.toJSON()
    known = [ch for ch in alphabet if ch in lit.char_to_token]
    docs = []
    for _ in range(rng.randint(40, 400)):
        kind = rng.random()
        if kind < 0.08:
            docs.append("")
        elif kind < 0.16:
            docs.append(rng.choice(known) * rng.randint(1, 130))
        elif kind < 0.20:
            docs.append("".join(rng.choice(known) for _ in range(rng.randint(1400, 4000))))
        elif kind < 0.5:
            docs.append("".join(rng.choice(known) for _ in range(rng.randint(1, 12))))
        else:
            docs.append("".join(rng.choice(known) for _ in range(rng.randint(1, 700))))
    ids = np.array([lit.char_to_token[ch].index for d in docs for ch in d], dtype=np.int32)
    off = np.zeros(len(docs) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(d) for d in docs])
    raw, roff, _ = gpu.encodeBatch(ids, off, vector=False)
    assert roff[0] == 0 and roff[-1] == raw.size
    for d, text in enumerate(docs):
        want = [ord(ch) - 1 for ch in lit.encodeToCode(text)]
        assert raw[roff[d]:roff[d + 1]].tolist() == want, (d, len(text))
    assert gpu.stats()["encode_path"] == 2, "the lane path was expected to take this batch"
    # the per-document kernel must agree with the lane path on every document
    monkeypatch.setenv("BPE_ENC_OLD", "1")
    old = make()
    old.fromJSON(gpu.toJSON())
    raw2, roff2, _ = old.encodeBatch(ids, off, vector=False)
    assert np.array_equal(raw, raw2) and np.array_equal(roff, roff2)


@pytest.mark.parametrize("chunk", ["1", "97", "1000", "5000"])
def test_host_buffer_encode_pipeline_chunks(chunk, monkeypatch):
    """bpe_encode_batch / bpe_encode_text_batch run as a three-stream pipeline over chunks of whole documents
    (copy in | encode | copy out, bpe_b200.cu encode_pipeline).  Forced to tiny chunks, the vectors, offsets and
    first-offender reports must equal the one-chunk call and the sequential replaceAll of core.ts:404-406; errors keep
    their batch-relative positions when they occur in a late chunk."""
    import ctypes as C

    from bpe_tokenizer_b200 import _abi
    from bpe_tokenizer_b200.tokenizer import BpeError

    rng = random.Random(4242)
    alphabet = "abcdé中 \n"
    train = _random_docs(rng, alphabet, 8, 400)
    lit, one = LiteralTokenizer(), make()
    for d in train:
        lit.addToCorpus(d)
        one.addToCorpus(d)
    lit.mergeUntil({"max_iterations": 60})
    one.mergeUntil({"max_iterations": 60})
    assert one.toJSON() == lit.toJSON()
    known = [ch for ch in alphabet if ch in lit.char_to_token]
    docs = []
    for _ in range(300):
        kind = rng.random()
        n = 0 if kind < 0.1 else rng.randint(1, 12) if kind < 0.4 else rng.randint(1, 300) if kind < 0.95 else rng.randint(1100, 2600)
        docs.append("".join(rng.choice(known) for _ in range(n)))
    docs += ["", ""]  # the batch ends with empty documents
    ids = np.array([lit.char_to_token[ch].index for d in docs for ch in d], dtype=np.int32)
    off = np.zeros(len(docs) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(d) for d in docs])
    text, boff = _utf8_batch(docs)
    want = [one.encodeBatch(ids, off, vector=v) for v in (False, True)] + [one.encodeTextBatch(text, boff, vector=v) for v in (False, True)]
    for d, doc in enumerate(docs[:40]):
        raw, roff, _ = want[0]
        assert raw[roff[d]:roff[d + 1]].tolist() == [ord(ch) - 1 for ch in lit.encodeToCode(doc)], d
    assert all(np.array_equal(a, b) for a, b in zip(want[0], want[2])) and all(np.array_equal(a, b) for a, b in zip(want[1], want[3]))

    monkeypatch.setenv("BPE_ENC_CHUNK", chunk)
    t = make()
    t.fromJSON(one.toJSON())
    got = [t.encodeBatch(ids, off, vector=v) for v in (False, True)] + [t.encodeTextBatch(text, boff, vector=v) for v in (False, True)]
    for g, w in zip(got, want):
        assert all(np.array_equal(a, b) for a, b in zip(g, w))
    # a window of the batch (offsets that do not start at zero)
    lo, hi = 17, 203
    raw, roff, _ = t.encodeBatch(ids, off[lo:hi + 1], vector=False)
    w_raw, w_off, _ = want[0]
    assert np.array_equal(raw, w_raw[w_off[lo]:w_off[hi]]) and np.array_equal(roff, w_off[lo:hi + 1] - w_off[lo])
    # an id outside the table / an unknown character in a late chunk: position relative to the batch
    bad_at = int(off[250]) + 1
    assert off[251] > bad_at
    ids_bad = ids.copy()
    ids_bad[bad_at] = 60000
    with pytest.raises(BpeError, match="id 60000 at %d outside" % bad_at):
        t.encodeBatch(ids_bad, off, vector=False)
    docs_bad = list(docs)
    docs_bad[250] = docs_bad[250][:1] + "☃" + docs_bad[250][1:]
    with pytest.raises(ValueError, match="unknown token, char"):
        t.encodeTextBatch(*_utf8_batch(docs_bad), vector=False)
    tb, ob = _utf8_batch(docs_bad)
    buf = np.frombuffer(tb, dtype=np.uint8)
    out = np.empty(len(tb), dtype=np.int32)
    ooff = np.zeros(len(docs) + 1, dtype=np.int64)
    n, upos, ucp = C.c_int64(), C.c_int64(-1), C.c_int32()
    rc = t._lib.bpe_encode_text_batch(t._h, buf.ctypes.data_as(_abi.u8p), _abi.p64(ob), len(docs), None, 0, _abi.p32(out), out.size, _abi.p64(ooff),
                                      None, C.byref(n), C.byref(upos), C.byref(ucp))
    assert rc == _abi.BPE_E_INVALID and upos.value == bad_at and ucp.value == ord("☃")
    # an output buffer that is too small: BPE_E_CAPACITY and the size that is needed
    small = np.empty(10, dtype=np.int32)
    rc = t._lib.bpe_encode_batch(t._h, _abi.p32(ids), _abi.p64(off), len(docs), None, 0, _abi.p32(small), small.size, _abi.p64(ooff), None, C.byref(n))
    assert rc == _abi.BPE_E_CAPACITY and n.value == want[0][0].size and np.array_equal(ooff, want[0][1])
    # offsets that go backwards are refused before anything is read through them
    off_bad = off.copy()
    off_bad[260] = off_bad[259] - 1
    with pytest.raises(BpeError, match="non-decreasing"):
        t.encodeBatch(ids, off_bad, vector=False)
    # the engine still works after the failed calls
    assert all(np.array_equal(a, b) for a, b in zip(t.encodeBatch(ids, off, vector=True), want[1]))


def test_decode_batch_matches_host_decode():
    """Device decodeVector (core.ts:455-471): bytes equal the concatenated token chars; the first unknown vector index
    of a document is reported where the reference throws."""
    rng = random.Random(31)
    t, lit = make(), LiteralTokenizer()
    docs = ["the cat sat on the mat\n" * 30, "café \U0001F600 naïve 中文 " * 20, "", "zzz", "ab" * 100]
    for d in docs:
        t.addToCorpus(d)
        lit.addToCorpus(d)
    t.mergeUntil({"max_iterations": 60})
    lit.mergeUntil({"max_iterations": 60})
    lit.compactVectorIndex()
    vecs = []
    for d in docs + ["the mat sat", "", "中文café"]:
        try:
            vecs.append(lit.encodeToVector(d))
        except ValueError:
            vecs.append([])
    values = np.array([v for vec in vecs for v in vec], dtype=np.int32)
    off = np.zeros(len(vecs) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(v) for v in vecs])
    raw, boff, bad = t.decodeBatch(values, off, vector=True)
    assert (bad == -1).all()
    for d, vec in enumerate(vecs):
        assert raw[boff[d]:boff[d + 1]].decode("utf-8") == lit.decodeVector(vec)
    # raw token indices (decodeTokens semantics)
    idx = np.array([rng.randrange(len(t.token_table)) for _ in range(500)], dtype=np.int32)
    raw2, boff2, _ = t.decodeBatch(idx, np.array([0, 200, 200, 500], dtype=np.int64), vector=False)
    want = ["".join(t.token_table[i].chars for i in idx[a:b]) for a, b in ((0, 200), (200, 200), (200, 500))]
    assert [raw2[boff2[d]:boff2[d + 1]].decode("utf-8") for d in range(3)] == want
    # unknown vector indices: first offender per document
    n_vec = len(lit.from_vector_index)
    vals = np.array([0, 1, n_vec + 5, 2, -3, 1, 0], dtype=np.int32)
    _, _, bad3 = t.decodeBatch(vals, np.array([0, 4, 4, 7], dtype=np.int64), vector=True)
    assert bad3.tolist() == [2, -1, 0]
    with pytest.raises(ValueError, match="unknown vector index: %d" % (n_vec + 5)):
        lit.decodeVector(vals[:4].tolist())


@pytest.mark.parametrize("seed", range(4))
def test_batched_merge_log_replay_equals_line_by_line(seed):
    """restoreMerges (one device call, replay mode of the loop kernel) == restoreMerge per line (core.ts:477-494) ==
    the run that produced the log; pairs that no longer occur, unknown codes and an emptied corpus included."""
    from bpe_tokenizer_b200 import compactMerge

    rng = random.Random(500 + seed)
    alphabet = "ab" if seed == 0 else "abcdef "
    docs = _random_docs(rng, alphabet, rng.randint(2, 9), rng.choice([40, 300]))
    first = make()
    for d in docs:
        first.addToCorpus(d)
    first.mergeUntil({"max_length": rng.choice([None, 6])})
    # compactMerge is taken when the merge is found (core.spec.ts:176-183): c.weight == c.original_weight at that moment
    log = [[a.code, b.code, c.original_weight] for a, b, c in first.merge_tokens]
    assert compactMerge((first.merge_tokens[0][0], first.merge_tokens[0][1], first.merge_tokens[0][2]))[:2] == log[0][:2]
    one, batch, lit = make(), make(), LiteralTokenizer()
    for d in docs:
        one.addToCorpus(d)
        batch.addToCorpus(d)
        lit.addToCorpus(d)
    for line in log:
        one.restoreMerge(line)
        lit.restoreMerge(line)
    cut = len(log) // 2
    batch.restoreMerges(log[:cut])  # two calls: the second continues on the rewritten corpus
    batch.restoreMerges(log[cut:])
    assert batch.toJSON() == one.toJSON() == lit.toJSON() == first.toJSON()
    assert batch.corpus_in_code == one.corpus_in_code == lit.corpus_in_code == first.corpus_in_code
    # the resumed tokenizer keeps merging like the uninterrupted one (the index is rebuilt after a replay)
    more = docs[0] + docs[-1]
    for x in (batch, first):
        x.addToCorpus(more)
        x.mergeUntil({"max_iterations": 5})
    assert batch.toJSON() == first.toJSON()
    # corpus emptied before the replay (example/import-merge-log-to-ram.ts:22): only tables grow
    empty = make()
    for d in docs:
        empty.addToCorpus(d)
    empty.corpus_in_code = []
    empty.restoreMerges(log)
    assert [t.chars for t in empty.token_table] == [t.chars for t in first.token_table][: len(empty.token_table)]
    assert empty.encodeToCode(docs[0]) == lit.encodeToCode(docs[0])
    with pytest.raises(ValueError, match="unknown token, a_code"):
        batch.restoreMerges([["￿", "a", 3]])


def _utf8_batch(docs):
    chunks = [d.encode("utf-8", "surrogatepass") for d in docs]
    off = np.zeros(len(chunks) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(c) for c in chunks])
    return b"".join(chunks), off


def test_device_text_front_end_equals_add_to_corpus():
    """addTextBatch / encodeTextBatch (UTF-8 decode, first-appearance token creation and weights on the device,
    csrc/text_kernels.cuh) against addToCorpus / encodeToVector (core.ts:182-207, :392-445): 1- to 4-byte characters,
    empty documents, characters first seen late, a second batch that adds more characters after merges."""
    rng = random.Random(77)
    pool = "abc déf ÿ中文字 \U0001F600\U0001F389\n\r\t" + "".join(chr(c) for c in (0x7F, 0x80, 0x7FF, 0x800, 0xFFFF, 0x10000, 0x10FFFF))
    docs = ["".join(rng.choice(pool) for _ in range(rng.randint(0, 300))) for _ in range(60)] + ["", "a" * 5000, "ÿ" * 4100]
    dev, host, lit = make(), make(), LiteralTokenizer()
    text, off = _utf8_batch(docs)
    dev.addTextBatch(text, off)
    for d in docs:
        host.addToCorpus(d)
        lit.addToCorpus(d)
    assert rows(dev) == rows(host) == rows(lit)
    assert dev.corpus_in_code == host.corpus_in_code == lit.corpus_in_code
    for x in (dev, host, lit):
        x.mergeUntil({"max_iterations": 40})
    assert dev.toJSON() == host.toJSON() == lit.toJSON()
    # second batch after merges: new characters get indices after the merged tokens (core.ts:188-199, :204)
    more = ["xyz" + d for d in docs[:10]] + ["§§§ new § chars ¶"]
    text2, off2 = _utf8_batch(more)
    dev.addTextBatch(text2, off2)
    for d in more:
        host.addToCorpus(d)
        lit.addToCorpus(d)
    assert rows(dev) == rows(host) == rows(lit)
    for x in (dev, host, lit):
        x.mergeUntil({"max_iterations": 20})
    assert dev.toJSON() == lit.toJSON()
    assert dev.corpus_in_code == lit.corpus_in_code
    # encode from text
    probe = [d for d in docs[:20]] + ["abc", ""]
    ptext, poff = _utf8_batch(probe)
    raw, roff, _ = dev.encodeTextBatch(ptext, poff, vector=False)
    for d, textd in enumerate(probe):
        assert raw[roff[d]:roff[d + 1]].tolist() == [ord(ch) - 1 for ch in lit.encodeToCode(textd)], d
    vals, voff, bad = dev.encodeTextBatch(ptext, poff, vector=True)
    lit.compactVectorIndex()
    for d, textd in enumerate(probe):
        try:
            want = lit.encodeToVector(textd)
        except ValueError:
            assert bad[d] >= 0
            continue
        assert bad[d] == -1 and vals[voff[d]:voff[d + 1]].tolist() == want
    with pytest.raises(ValueError) as ei:
        dev.encodeTextBatch(*_utf8_batch(["abc", "ab☃c"]))
    with pytest.raises(ValueError) as ej:
        lit.encodeToVector("ab☃c")
    assert str(ei.value) == str(ej.value)
    # a snapshot restored into a fresh engine knows the characters again
    back = make()
    back.fromJSON(dev.toJSON())
    raw2, roff2, _ = back.encodeTextBatch(ptext, poff, vector=False)
    assert np.array_equal(raw, raw2) and np.array_equal(roff, roff2)


def test_scale_properties_64mb():
    """Size-independent properties at a size the oracle cannot reach in test time (64 MB, 2000 merges): weights equal the
    live occurrences of every token, token count conservation, encode -> decode round trip of unseen text (byte exact),
    idempotence of encode on its own decoded output, monotone offsets; plus an oracle check of a slice."""
    import ctypes as C

    from bpe_tokenizer_b200 import _abi
    from oracle.int_oracle import IntOracle

    lib = _abi.load_library()

    def synth(target, seed):
        nb, nd = C.c_int64(), C.c_int64()
        assert lib.bpe_synth_corpus(target, seed, 50000, 42, None, 0, None, 0, C.byref(nb), C.byref(nd)) == 0
        text = np.empty(nb.value, dtype=np.uint8)
        off = np.empty(nd.value + 1, dtype=np.int64)
        assert lib.bpe_synth_corpus(target, seed, 50000, 42, text.ctypes.data_as(_abi.u8p), text.size, _abi.p64(off), off.size, C.byref(nb), C.byref(nd)) == 0
        return text, off

    text, off = synth(64_000_000, 43)
    t = make()
    t.addTextBatch(text.tobytes(), off)  # device text front end: characters, indices and weights
    n0 = int(text.size)
    assert sum(tk.weight for tk in t.token_table) == n0 and len(t.token_table) == 29
    done = t.mergeUntil({"max_iterations": 2000})
    assert done == 2000
    ids, offs = t.corpusIds()
    weights = np.array([tk.weight for tk in t.token_table])
    assert np.array_equal(np.bincount(ids, minlength=len(t.token_table)), weights)           # core.ts:201,345-346 bookkeeping
    assert ids.size == n0 - sum(c.original_weight for _, _, c in t.merge_tokens)              # every replacement removes one token
    assert np.all(np.diff(offs) >= 0) and offs[-1] == ids.size
    w = [c.original_weight for _, _, c in t.merge_tokens]
    assert all(w[i] >= w[i + 1] for i in range(len(w) - 1))                                   # counts never grow: weights are sorted
    # unseen text: encode -> decode is the identity, encode is idempotent on its own output
    text2, off2 = synth(32_000_000, 44)
    raw, roff, _ = t.encodeTextBatch(text2.tobytes(), off2, vector=False)
    assert np.all(np.diff(roff) >= 0) and roff[-1] == raw.size
    back, boff, bad = t.decodeBatch(raw, roff, vector=False)
    assert (bad == -1).all() and back == text2.tobytes() and np.array_equal(boff, off2)
    raw2, roff2, _ = t.encodeTextBatch(back, boff, vector=False)
    assert np.array_equal(raw, raw2) and np.array_equal(roff, roff2)
    # a slice against the compiled oracle (sequential replaceAll per merge, core.ts:404-406)
    o = IntOracle()
    o.set_len16(np.ones(len(t.token_table), dtype=np.int32))
    o.load_merges(np.array([[a.index, b.index, c.index] for a, b, c in t.merge_tokens], dtype=np.int32))
    lut = np.full(256, -1, dtype=np.int32)
    for ch, tk in t.char_to_token.items():
        lut[ord(ch)] = tk.index
    for d in list(range(0, 40)) + list(range(len(off2) - 41, len(off2) - 1)):
        assert np.array_equal(raw[roff[d]:roff[d + 1]], o.encode(lut[text2[off2[d]:off2[d + 1]]], fast=True)), d
