"""CPU: pin the oracle against the reference's own known-answer tests
(core.spec.ts) and cross-check its two forms (string-level literal vs compiled
int-level) by seeded fuzzing, including the closed-form tie-break of
SURVEY.md Appendix A.2."""
import json
import os
import random

import numpy as np
import pytest

import kat_suite
from oracle import LiteralTokenizer, compact_merge, utf16_len
from oracle.int_oracle import IntOracleTokenizer

IMPLS = {"literal": LiteralTokenizer, "int": IntOracleTokenizer}


@pytest.mark.parametrize("impl", sorted(IMPLS))
@pytest.mark.parametrize("kat", kat_suite.ALL, ids=lambda f: f.__name__)
def test_reference_known_answers(impl, kat):
    kat(IMPLS[impl])


@pytest.mark.parametrize("impl", sorted(IMPLS))
def test_reference_merge_log_resume(impl):
    kat_suite.kat_merge_log_resume(IMPLS[impl], compact_merge)


def _random_docs(rng, alphabet, n_docs, max_len):
    return ["".join(rng.choice(alphabet) for _ in range(rng.randint(0, max_len))) for _ in range(n_docs)]


def _closed_form_next_merge(t: LiteralTokenizer, min_weight, max_length):
    """SURVEY.md A.1/A.2: count with run parity, then
    argmax (weight desc, a.index+b.index asc, position of last counted occurrence asc)."""
    count, last = {}, {}
    pos = 0
    for doc in t.corpus_in_code:
        toks = [t.code_to_token[c].index for c in doc]
        run = 0  # number of pairs (x,x) seen so far in the current run of identical tokens
        for i in range(1, len(toks)):
            a, b = toks[i - 1], toks[i]
            if a == b:
                run = run + 1 if (i >= 2 and toks[i - 2] == a) else 1
                counted = run % 2 == 1
            else:
                run = 0
                counted = True
            if max_length and utf16_len(t.token_table[a].chars) + utf16_len(t.token_table[b].chars) > max_length:
                counted = False
            if counted:
                count[(a, b)] = count.get((a, b), 0) + 1
                last[(a, b)] = pos + i
        pos += len(toks) + 1
    if not count:
        return None
    w = max(count.values())
    if w < (min_weight or 2):
        return None
    a, b = min((k for k, v in count.items() if v == w), key=lambda k: (k[0] + k[1], last[k]))
    return a, b, w


@pytest.mark.parametrize("seed", range(40))
def test_literal_vs_int_vs_closed_form(seed):
    rng = random.Random(seed)
    alphabet = "abc"[: rng.randint(1, 3)] if seed % 2 else "abcdefg"[: rng.randint(2, 7)]
    docs = _random_docs(rng, alphabet, rng.randint(1, 4), rng.choice([6, 20, 60]))
    max_length = rng.choice([None, None, 3, 4, 8])
    min_weight = rng.choice([None, 2, 3])
    lit, fast = LiteralTokenizer(), IntOracleTokenizer()
    for d in docs:
        lit.addToCorpus(d)
        fast.addToCorpus(d)
    for _ in range(200):
        want = _closed_form_next_merge(lit, min_weight, max_length)
        m1 = lit.find_next_merge(min_weight, max_length)
        m2 = fast.find_next_merge(min_weight, max_length)
        if m1 is None:
            assert m2 is None and want is None
            break
        assert (m1[0].index, m1[1].index, m1[2].weight) == (m2[0].index, m2[1].index, m2[2].weight) == want
        lit.apply_merge(m1)
        fast.apply_merge(m2)
        assert lit.corpus_in_code == fast.corpus_in_code
    assert lit.to_json() == fast.to_json()
    for d in docs + _random_docs(rng, alphabet, 3, 40):
        try:
            want_code = lit.encode_to_code(d)
        except ValueError as e:
            with pytest.raises(ValueError, match="unknown token, char"):
                fast.encode_to_code(d)
            continue
        assert fast.encode_to_code(d) == want_code
        ids = [lit.char_to_token[ch].index for ch in d]
        assert "".join(chr(int(i) + 1) for i in fast.encode_ids(ids, fast=True)) == want_code


def test_int_merge_until_matches_literal_loop():
    rng = random.Random(7)
    docs = _random_docs(rng, "abcd ", 6, 200)
    lit, fast = LiteralTokenizer(), IntOracleTokenizer()
    for d in docs:
        lit.addToCorpus(d)
        fast.addToCorpus(d)
    n1 = lit.merge_until(min_weight=2, max_length=6)
    n2 = fast.merge_until(min_weight=2, max_length=6)
    assert n1 == n2 and n1 > 10
    assert lit.to_json() == fast.to_json()
    assert lit.corpus_in_code == fast.corpus_in_code


def test_astral_characters_count_two_utf16_units():
    # core.ts:272 uses chars.length (UTF-16); one astral char is one token (core.ts:185) of length 2
    t = LiteralTokenizer()
    t.addToCorpus("\U0001F600\U0001F600\U0001F600\U0001F600ab" * 3)
    assert t.find_next_merge(max_length=3) is not None  # 'ab' (1+1) still allowed
    m = t.find_next_merge(max_length=4)
    assert m[2].chars in ("\U0001F600\U0001F600",)
    u = IntOracleTokenizer()
    u.addToCorpus("\U0001F600\U0001F600\U0001F600\U0001F600ab" * 3)
    m2 = u.find_next_merge(max_length=3)
    assert m2[2].chars == t.find_next_merge(max_length=3)[2].chars


GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "literal_cases.json")


def test_committed_golden_fixtures_still_match_literal_oracle():
    with open(GOLDEN, encoding="utf-8") as f:
        cases = json.load(f)
    assert len(cases) >= 8
    for case in cases:
        for cls in (LiteralTokenizer, IntOracleTokenizer):
            t = cls()
            for d in case["docs"]:
                t.addToCorpus(d)
            t.mergeUntil(case["options"])
            assert t.toJSON() == case["json"], case["name"]
            assert [[a.index, b.index, c.weight] for a, b, c in t.merge_tokens] == case["merges"], case["name"]
            for text, want in case["encode"]:
                try:
                    got = list(t.encodeToVector(text))
                except ValueError as e:
                    got = "throws: " + str(e)
                assert got == want, (case["name"], text)


def test_cfg3_gpu_merge_table_starts_like_the_oracle_on_the_full_corpus():
    """SURVEY.md section 8(d), parity at scale (1): the first merges of BASELINE config 3 -- pairs, new indices AND weights on the full
    1 GB corpus -- as the CPU restatement computes them (tests/golden/make_cfg3_prefix_golden.py, ~8 s per merge, run offline) equal
    the head of the merge log the GPU run produced (tools/data/merges_cfg3_abc.npy + merges_cfg3_weights.npy, written from
    tools/dump_merges.py's output).  That log is the one every cfg3 bench line reports: its SHA-1 is profiles/*bench*.json's."""
    import hashlib
    import json

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    from bpe_tokenizer_b200._abi import MERGE_DTYPE

    abc = np.load(os.path.join(root, "tools", "data", "merges_cfg3_abc.npy"))
    weights = np.load(os.path.join(root, "tools", "data", "merges_cfg3_weights.npy"))
    alphabet = np.load(os.path.join(root, "tools", "data", "alphabet_cfg3.npy"))
    log = np.zeros(len(abc), dtype=MERGE_DTYPE)
    log["a"], log["b"], log["c"], log["weight"] = abc[:, 0], abc[:, 1], abc[:, 2], weights
    sha = hashlib.sha1(log.tobytes()).hexdigest()
    with open(os.path.join(root, "profiles", "r01_bench_n1.json")) as f:
        assert json.load(f)["config"]["merge_log_sha1"] == sha == "add92aa1a96c276f03b63e3a952370ef04cb60f0"
    with open(os.path.join(root, "tests", "golden", "cfg3_prefix.json")) as f:
        golden = json.load(f)
    assert golden["alphabet"] == alphabet.tolist()
    n = len(golden["merges"])
    assert n >= 8
    assert [[int(r["a"]), int(r["b"]), int(r["c"]), int(r["weight"])] for r in log[:n]] == golden["merges"]
    # weights never increase from one merge to the next (a born pair occurs at most as often as the pair that bore it)
    assert np.all(np.diff(weights.astype(np.int64)) <= 0)


# ---- the incremental oracle (oracle/fast_oracle.cpp) is pinned to the literal restatement ------------------------------------
def _int_vs_fast(docs, nsym, mw, ml, mi, len16_chars=None, cap=400):
    from oracle.fast_oracle import FastOracle
    from oracle.int_oracle import IntOracle

    ids = np.array([t for d in docs for t in d], dtype=np.int32)
    off = np.zeros(len(docs) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(d) for d in docs])
    len16 = np.ones(nsym + cap + 1, dtype=np.int32)
    if len16_chars is not None:
        len16[:nsym] = len16_chars
    lit, fast = IntOracle(), FastOracle()
    lit.set_len16(len16)
    lit.add_documents(ids, off)
    fast.set_len16(len16[:nsym])
    fast.add_documents(ids, off)
    want, got = lit.merge_until(mw, ml, mi, nsym, cap), fast.merge_until(mw, ml, mi, nsym, cap)
    assert all(np.array_equal(x, y) for x, y in zip(want, got)), ([x[:12].tolist() for x in want], [x[:12].tolist() for x in got])
    corpus = np.concatenate([lit.document(d) for d in range(lit.num_documents())]) if lit.num_documents() else np.zeros(0, np.int32)
    assert np.array_equal(corpus, fast.corpus())
    return len(want[0])


@pytest.mark.parametrize("chunk", range(8))
def test_fast_oracle_equals_literal_oracle_fuzz(chunk):
    """tiny alphabets (ties on weight and index sum, runs like 'aaa', chains like 'abab'), empty and one-token documents, every
    option: same merges, same weights, same final corpus as the literal restatement"""
    total = 0
    for seed in range(chunk * 120, (chunk + 1) * 120):
        rng = random.Random(40000 + seed)
        nsym = rng.choice([1, 2, 2, 3, 3, 5, 8])
        docs = [[rng.randrange(nsym) for _ in range(rng.choice([0, 1, 2, 5, 20, 60, 200]))] for _ in range(rng.randint(1, 6))]
        chars = [rng.choice([1, 2]) for _ in range(nsym)] if rng.random() < 0.3 else None
        total += _int_vs_fast(docs, nsym, rng.choice([1, 2, 2, 3, 5]), rng.choice([0, 0, 3, 4, 8]), rng.choice([0, 0, 1, 5, 40]), chars)
    assert total > 300  # the cases do merge


def test_fast_oracle_equals_literal_oracle_on_zipf_text():
    from bpe_tokenizer_b200.synth import first_appearance_ids, synth_corpus

    text, off = synth_corpus(200_000, seed=43)
    ids, alphabet = first_appearance_ids(text)
    docs = [ids[off[d]:off[d + 1]].tolist() for d in range(len(off) - 1)]
    assert _int_vs_fast(docs, len(alphabet), 2, 0, 300, cap=300) == 300
    assert _int_vs_fast(docs, len(alphabet), 2, 6, 200, cap=200) == 200


def _int_vs_fast_calls(docs, nsym, calls):
    """One corpus trained through a sequence of merge_until calls (min_weight, max_length, max_iterations) on both oracles: the
    logs of every call, the corpus and the document lengths after every call must be equal.  -> merges done"""
    from oracle.fast_oracle import FastOracle
    from oracle.int_oracle import IntOracle

    ids = np.array([t for d in docs for t in d], dtype=np.int32)
    off = np.zeros(len(docs) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(d) for d in docs])
    lit, fast = IntOracle(), FastOracle()
    for o in (lit, fast):
        o.set_len16(np.ones(nsym, dtype=np.int32))
        o.add_documents(ids, off)
    done = 0
    for i, (mw, ml, mi) in enumerate(calls):
        cap = mi if mi > 0 else 1000
        want, got = lit.merge_until(mw, ml, mi, nsym + done, cap), fast.merge_until(mw, ml, mi, nsym + done, cap)
        assert all(np.array_equal(x, y) for x, y in zip(want, got)), (i, [x[:12].tolist() for x in want], [x[:12].tolist() for x in got])
        done += len(want[0])
        assert np.array_equal(fast.document_lengths(), [lit.document(d).size for d in range(lit.num_documents())]), i
        corpus = np.concatenate([lit.document(d) for d in range(lit.num_documents())]) if docs else np.zeros(0, np.int32)
        assert np.array_equal(corpus, fast.corpus()), i
    return done


def test_fast_oracle_keeps_pairs_a_max_length_excluded():
    """(3, 2) -- the token of the first merge, then 2 -- is too long under max_length 2 and is the next merge once the limit is gone:
    a call that skips a pair for its length must leave it to later calls."""
    docs = [[0, 1, 2]] * 10 + [[0, 1]] * 2 + [[2, 2]] * 3
    assert _int_vs_fast_calls(docs, 3, [(2, 2, 5), (2, 0, 5)]) == 3
    assert _int_vs_fast_calls(docs + [[]], 3, [(2, 2, 1), (2, 2, 1), (2, 0, 1), (2, 2, 1), (2, 0, 5)]) == 3


@pytest.mark.parametrize("chunk", range(4))
def test_fast_oracle_equals_literal_oracle_across_calls(chunk):
    """sequences of calls whose max_length and min_weight change between calls, and cuts at max_iterations, on the corpora of
    the fuzz test above: empty and one-token documents, runs, ties"""
    total = 0
    for seed in range(chunk * 60, (chunk + 1) * 60):
        rng = random.Random(50000 + seed)
        nsym = rng.choice([1, 2, 3, 3, 5, 8])
        docs = [[rng.randrange(nsym) for _ in range(rng.choice([0, 1, 2, 5, 20, 60, 200]))] for _ in range(rng.randint(1, 6))]
        calls = [(rng.choice([1, 2, 2, 3, 5]), rng.choice([0, 0, 2, 3, 4, 8]), rng.choice([1, 2, 3, 5, 40])) for _ in range(rng.randint(2, 6))]
        total += _int_vs_fast_calls(docs, nsym, calls)
    assert total > 300


def test_fast_oracle_equals_literal_oracle_across_calls_on_zipf_text():
    """the option sequences the GPU state tests train through (tests/test_gpu_merge_state.py), at 100 kB"""
    from bpe_tokenizer_b200.synth import first_appearance_ids, synth_corpus

    text, off = synth_corpus(100_000, seed=43)
    ids, alphabet = first_appearance_ids(text)
    docs = [ids[off[d]:off[d + 1]].tolist() for d in range(len(off) - 1)]
    for calls in ([(2, 4, 40), (2, 0, 40), (2, 6, 40)], [(150, 0, 60), (2, 0, 40)], [(3, 9, 60), (2, 0, 40)]):
        assert _int_vs_fast_calls(docs, len(alphabet), calls) > 60


def test_fast_oracle_reproduces_the_cfg2_golden_log():
    """10 MB, 4 000 merges: the incremental oracle (seconds) gives the SHA-1 the literal restatement needed 34 minutes for
    (tests/golden/cfg2_merge_log.json) -- and the GPU gives (test_gpu_parity.py)"""
    import hashlib
    import json

    from bpe_tokenizer_b200._abi import MERGE_DTYPE
    from bpe_tokenizer_b200.synth import first_appearance_ids, synth_corpus
    from oracle.fast_oracle import FastOracle

    with open(os.path.join(os.path.dirname(__file__), "golden", "cfg2_merge_log.json")) as f:
        golden = json.load(f)
    text, off = synth_corpus(10_000_000, seed=43)
    ids, alphabet = first_appearance_ids(text)
    o = FastOracle()
    o.set_len16(np.ones(len(alphabet), dtype=np.int32))
    o.add_documents(ids, off)
    la, lb, lw = o.merge_until(2, 0, golden["merges"], len(alphabet), golden["merges"])
    log = np.zeros(len(la), dtype=MERGE_DTYPE)
    log["a"], log["b"], log["weight"] = la, lb, lw
    log["c"] = len(alphabet) + np.arange(len(la))
    assert hashlib.sha1(log.tobytes()).hexdigest() == golden["sha1"]


def test_cfg3_full_run_was_checked_against_the_incremental_oracle():
    """BASELINE config 3 at FULL size: tests/golden/check_cfg3_full.py ran oracle/fast_oracle.cpp over the 1 GB corpus (14 minutes of CPU,
    ~40 GB of RAM -- too heavy for this suite) and found all 32 000 merges and weights of the GPU's log equal; the fixture records
    that run.  Here: the fixture belongs to the committed GPU table and to the SHA-1 the cfg3 bench lines report."""
    import hashlib
    import json

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    from bpe_tokenizer_b200._abi import MERGE_DTYPE

    with open(os.path.join(root, "tests", "golden", "cfg3_full_check.json")) as f:
        check = json.load(f)
    assert check["equals_gpu_merge_log"] is True and check["merges"] == 32000 and "first_difference" not in check
    abc = np.load(os.path.join(root, "tools", "data", "merges_cfg3_abc.npy"))
    log = np.zeros(len(abc), dtype=MERGE_DTYPE)
    log["a"], log["b"], log["c"] = abc[:, 0], abc[:, 1], abc[:, 2]
    log["weight"] = np.load(os.path.join(root, "tools", "data", "merges_cfg3_weights.npy"))
    assert hashlib.sha1(log.tobytes()).hexdigest() == check["sha1"]
    with open(os.path.join(root, "profiles", "r01_bench_n1.json")) as f:
        bench_line = json.load(f)
    assert bench_line["config"]["merge_log_sha1"] == check["sha1"]
    # token conservation: every merge removes exactly `weight` tokens
    n0 = int(check["workload"].split(" B ")[0])
    assert n0 - int(log["weight"].sum()) == check["tokens_left"]


def test_cfg4_full_encode_token_count_equals_the_cpu_golden():
    """BASELINE config 4 at FULL size: the literal encodeToCode restatement, one call per document over the whole 1 GB seed-44 text
    (tests/golden/make_cfg4_encode_golden.py, ~4 core-hours), produced exactly as many tokens as the GPU reports for the same text
    and merge table in its bench line; bench.py compares the token stream itself by SHA-1 (encode.cpu_baseline.full_output)."""
    import json

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "tests", "golden", "cfg4_encode.json")) as f:
        golden = json.load(f)
    with open(os.path.join(root, "profiles", "r01_bench_n1.json")) as f:
        line = json.load(f)
    assert line["config"]["merges_done"] == 32000 and line["config"]["merge_log_sha1"] == "add92aa1a96c276f03b63e3a952370ef04cb60f0"
    assert ("%d B" % line["encode"]["chars"]) in golden["workload"] and ("%d docs" % line["encode"]["docs"]) in golden["workload"]
    assert golden["tokens_out"] == line["encode"]["tokens_out"] == 176384677
