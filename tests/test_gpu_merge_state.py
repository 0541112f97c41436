"""GPU: what every exit of mergeUntil leaves behind for the next caller.  DESIGN §3: a launch leaves every occurrence list complete
and every delta cell zero, and the incremental pair table holds the counts of the corpus.  Each case trains through a sequence of
calls -- mergeUntil cut at max_iterations, single findNextMerge / applyMerge steps, options that change between calls, a replayed
merge log -- on one engine that keeps its index, and after every call takes a checkpoint:

  * the merge log so far, (a, b, weight), equals the CPU oracle's;
  * the corpus equals the oracle's corpus;
  * the device's pair table (bpe_pair_counts, read without rebuilding the index: stats()["index_builds"] stays put) equals
    recount(), the literal counting rule (core.ts:265-310) applied to the ORACLE's corpus and document lengths, so that the check
    shares nothing with the device;
  * stats()["corpus_tokens"] equals the corpus size.

A pair whose count a round gets wrong shows here even if it never wins.  The oracle is oracle/fast_oracle.py (the incremental
one, pinned to the literal restatement across calls with changing options by tests/test_oracle_golden.py), or IntOracle (the
literal recount per merge) on small corpora.

On a device group bpe_pair_counts reads member 0's table only, and no ABI reads the others.  A count that drifts on another
member is likely, but not certain, to surface as a different decision or as ERR_ROUND_MISMATCH when a run goes on to exhaustion
(test_run_to_exhaustion).

Every case asserts, in the stats or on the corpus, that it reached what it is named after; test_exit_statuses_are_reached runs
one engine's cases with BPE_TRACE=1 and asserts that the launches ended in every status the host driver continues from."""
import functools
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from pair_counts import device_counts, loop_counts, recount
from test_gpu_block_cells import STAGE, _alphabet, _mixed
from test_gpu_fresh_token_rounds import N_ALPHA, _remerging
from test_gpu_group_edges import _devices, _engine, _log, _set, _upload
from test_gpu_loop_stage import _giant_corpus

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAX_TOKENS = 56319  # BPE_MAX_TOKENS
CUTS = [1, 2, 3, 5, 8, 13, 16, 17, 31, 64, 100]  # merges per mergeUntil call, then the rest in one call
RB = 16  # merges one round of k_merge_rounds commits at most (round_kernels.cuh)
KNOBS = ("BPE_LOOP_K", "BPE_LOOP_ROUNDS", "BPE_BLOCK_CELLS_MIN_SITES", "BPE_LOOP_BLOCKS")
TALLY = {"checkpoints": 0, "max_pairs": 0}


# ---- the oracle, driven call by call ----
class Ref:
    """The CPU oracle on the same ids, trained through the same calls; `log` holds (a, b, weight) of every merge so far."""

    def __init__(self, ids, off, n_alpha, literal=False):
        from oracle.fast_oracle import FastOracle
        from oracle.int_oracle import IntOracle

        self.o = IntOracle() if literal else FastOracle()
        self.literal = literal
        self.n_alpha = n_alpha
        self.o.set_len16(np.ones(n_alpha, dtype=np.int32))
        self.o.add_documents(ids, off)
        self.log = []

    def merge_until(self, opts):
        mi = opts.get("max_iterations") or 0
        room = MAX_TOKENS - self.n_alpha - len(self.log)
        la, lb, lw = self.o.merge_until(opts.get("min_weight") or 2, opts.get("max_length") or 0, mi, self.n_alpha + len(self.log),
                                        min(mi, room) if mi else room)
        got = [(int(a), int(b), int(w)) for a, b, w in zip(la, lb, lw)]
        self.log += got
        return got

    def corpus(self):
        """(ids, document lengths)"""
        if not self.literal:
            return self.o.corpus(), self.o.document_lengths()
        docs = [self.o.document(d) for d in range(self.o.num_documents())]
        return (np.concatenate(docs) if docs else np.zeros(0, np.int32)), np.array([d.size for d in docs], dtype=np.int64)


def checkpoint(t, ref, what=""):
    got = [tuple(x) for x in _log(t)]
    bad = next((i for i, (g, w) in enumerate(zip(got, ref.log)) if g != w), None)
    assert bad is None and len(got) == len(ref.log), (what, bad, got[bad] if bad is not None else len(got), ref.log[bad] if bad is not None else len(ref.log))
    ids, lengths = ref.corpus()
    got_ids, got_off = t.corpusIds()
    assert np.array_equal(got_ids, ids), what
    assert np.array_equal(np.diff(got_off), lengths), what
    want = recount(ids, lengths)
    dev = device_counts(t)
    if dev != want:
        wrong = sorted(k for k in set(dev) | set(want) if dev.get(k) != want.get(k))
        raise AssertionError("%s: %d pairs differ from the recount, e.g. %s" % (what, len(wrong), [(k, dev.get(k), want.get(k)) for k in wrong[:8]]))
    assert t.stats()["corpus_tokens"] == ids.size, what
    TALLY["checkpoints"] += 1
    TALLY["max_pairs"] = max(TALLY["max_pairs"], len(want))


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    sys.stderr.write("\n[test_gpu_merge_state] checkpoints %d, most distinct pairs compared at one checkpoint %d\n"
                     % (TALLY["checkpoints"], TALLY["max_pairs"]))


# ---- corpora ----
@functools.lru_cache(maxsize=None)
def _corpus(name):
    """(ids, offsets, alphabet size, merges of the cut runs)"""
    if name == "mixed":
        return _mixed(1, 2_000_000) + (600, 1500)
    if name == "remerging":
        return _remerging(1, 1_000_000) + (N_ALPHA, 1500)
    if name == "giant":
        return _giant_corpus(7, 1_100_000) + (600, 300)
    if name == "many_pairs":  # uniform ids over 3000 tokens: pairs enough to grow the table during the run (test_gpu_k1_lists)
        rng = np.random.default_rng(7)
        head = rng.integers(0, 3000, size=200_000).astype(np.int32)
        tail, toff = _mixed(4, 300_000)
        return np.concatenate([head, tail]), np.concatenate([[0, 100_000], toff + head.size]).astype(np.int64), 3000, 400
    if name == "tie":  # test_gpu_loop_stage's tie corpus with 4 000 each of (5, 10) and (6, 9): the tie comes after other merges
        rng = np.random.default_rng(11)
        pairs = np.array([[5, 10], [6, 9]], dtype=np.int32)[rng.permutation(np.repeat([0, 1], 4_000))]
        tail, toff = _mixed(6, 500_000)
        ids = np.concatenate([pairs.ravel(), tail])
        return ids, np.concatenate([np.arange(0, 2 * len(pairs), 2, dtype=np.int64), toff + 2 * len(pairs)]), 600, 600
    if name == "small_mixed":
        return _mixed(2, 100_000) + (600, 0)
    if name == "small_remerging":
        return _remerging(2, 100_000) + (N_ALPHA, 0)
    raise KeyError(name)


def _start(name, devs=None, layout="split", literal=False):
    ids, off, n_alpha, _ = _corpus(name)
    t = _engine(devs, _alphabet(n_alpha))
    _upload(t, ids, off, layout)
    return t, Ref(ids, off, n_alpha, literal)


def _call(t, ref, opts):
    """one mergeUntil on the engine and the oracle -> merges done"""
    n = t.mergeUntil(dict(opts))
    assert n == len(ref.merge_until(opts)), opts
    return n


def _cut_run(t, ref, merges, steps=None):
    """mergeUntil in calls of CUTS merges, then the rest, a checkpoint after each; steps(t, ref, i) runs after checkpoint i."""
    done = 0
    for i, k in enumerate(CUTS + [None]):
        k = merges - done if k is None else min(k, merges - done)
        if k <= 0:
            break
        assert _call(t, ref, {"max_iterations": k}) == k
        done = len(ref.log)
        checkpoint(t, ref, "after call %d" % i)
        if steps:
            steps(t, ref, i)
            done = len(ref.log)
    assert done >= merges


# ---- cut batches ----
ONE = {
    "rounds": {},
    "rounds_k4": {"BPE_LOOP_K": "4"},
    "rounds_k1": {"BPE_LOOP_K": "1"},
    "loop": {"BPE_LOOP_ROUNDS": "0"},
    # staged / unstaged: BPE_BLOCK_CELLS_MIN_SITES forces the count deltas of every merge through the blocks' shared-memory cells, or
    # of none (as test_gpu_block_cells); no stat shows which way a merge went
    "rounds_staged": {"BPE_BLOCK_CELLS_MIN_SITES": STAGE["on"]},
    "rounds_unstaged": {"BPE_BLOCK_CELLS_MIN_SITES": STAGE["off"]},
    "loop_staged": {"BPE_LOOP_ROUNDS": "0", "BPE_BLOCK_CELLS_MIN_SITES": STAGE["on"]},
}
# "last": every document but the first on the last member, whose pair table is then sized for the corpus while the others' tables are
# small; only some members grow their tables during the run, and every member must rebuild its hot list after a growth, or the
# members' hot-list thresholds differ and they leave the kernel at different merges (a peer timeout in the exchange)
GROUPS = [pytest.param(m, r, lay, id="%d-%s-%s" % (m, "loop" if r else "rounds", lay)) for m in (2, 4) for r in (None, "0") for lay in ("split", "last")]


def _knobs(monkeypatch, env):
    _set(monkeypatch, **{k: env.get(k) for k in KNOBS})


@pytest.mark.gpu
@pytest.mark.parametrize("loop", sorted(ONE))
def test_cut_batches_one_engine(loop, monkeypatch):
    _knobs(monkeypatch, ONE[loop])
    t, ref = _start("mixed")
    _cut_run(t, ref, _corpus("mixed")[3])
    st = t.stats()
    if loop == "rounds_k1":
        assert st["loop_rounds"] > 0 and st["loop_round_merges"] == st["loop_rounds"], st  # one merge per round
    elif loop.startswith("rounds"):
        assert st["loop_rounds"] > 0 and st["loop_round_merges"] > 1.5 * st["loop_rounds"], st  # the cuts fall inside batches
    if loop.startswith("loop"):
        assert st["loop_rounds"] == 0, st
    t.close()


@pytest.mark.gpu
@pytest.mark.parametrize("members,loop_rounds,layout", GROUPS)
def test_cut_batches_group(members, loop_rounds, layout, monkeypatch):
    devs = _devices(members, monkeypatch)
    _knobs(monkeypatch, {"BPE_LOOP_ROUNDS": loop_rounds})
    t, ref = _start("mixed", devs, layout)
    _cut_run(t, ref, _corpus("mixed")[3])
    st = t.stats()
    assert (st["loop_round_merges"] > 1.5 * st["loop_rounds"]) if loop_rounds is None else st["loop_rounds"] == 0, st
    t.close()


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["rounds", "rounds_k4", "loop", "group2"])
def test_cut_batches_fresh_tokens(where, monkeypatch):
    """_remerging makes the tokens of one round merge again in the next.  Some cuts fall between a merge and a merge of its new token
    at most RB merges later (a round's batch at most): the next call's first round takes that pair from the occurrence lists the
    cut launch left."""
    devs = _devices(2, monkeypatch) if where == "group2" else None
    _knobs(monkeypatch, ONE.get(where, {}))
    t, ref = _start("remerging", devs)
    _cut_run(t, ref, _corpus("remerging")[3])
    cuts = np.cumsum(CUTS)
    fresh = [int(p) for p in cuts if max(ref.log[p][:2]) >= N_ALPHA + p - RB]  # the first merge after the cut takes a token made by
    assert len(fresh) >= 2, fresh                                            # one of the last RB merges before it
    if where != "loop":
        st = t.stats()
        assert st["loop_round_merges"] > 1.5 * st["loop_rounds"], st
    t.close()


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["one", "group2"])
def test_cut_batches_giant_merge(where, monkeypatch):
    """The first call is max_iterations=1: the giant (0, 1), above R_HUGE, runs in k_merge_loop and the checkpoint follows that
    hand-off; the rounds take the merges of the later calls."""
    devs = _devices(2, monkeypatch) if where == "group2" else None
    _knobs(monkeypatch, {})
    t, ref = _start("giant", devs)
    _cut_run(t, ref, _corpus("giant")[3])
    assert ref.log[0][:2] == (0, 1) and ref.log[0][2] > 1 << 20, ref.log[0]
    st = t.stats()
    assert 0 < st["loop_round_merges"] < len(ref.log), st
    t.close()


# ---- single steps continuing a launch ----
def _single_steps(rounds_of, group=False):
    """steps(t, ref, i): 1..5 findNextMerge + applyMerge after checkpoint i (on a group: mergeUntil(max_iterations=1)), each winner
    and the corpus compared with the oracle's next merge"""

    def steps(t, ref, i):
        for s in range(rounds_of(i)):
            want = ref.merge_until({"max_iterations": 1})
            if group:
                t.mergeUntil({"max_iterations": 1})
            else:
                m = t.findNextMerge()
                assert (m is None) == (not want)
                if m is None:
                    return
                assert (m[0].index, m[1].index, m[2].weight) == want[0], (i, s)
                t.applyMerge(m)
            checkpoint(t, ref, "after step %d of call %d" % (s, i))

    return steps


@pytest.mark.gpu
@pytest.mark.parametrize("scan", [0, 2], ids=["lists", "full_scan"])
@pytest.mark.parametrize("name", ["mixed", "remerging"])
def test_single_steps_continue_a_launch(name, scan, monkeypatch):
    """Profiling bit 1 (scan=2) finds the steps' sites by a full scan of the corpus instead of the occurrence lists the rounds
    filled: both must leave the same corpus and counts."""
    _knobs(monkeypatch, {})
    t, ref = _start(name)
    t._lib.bpe_set_profiling(t._h, scan)
    _cut_run(t, ref, _corpus(name)[3] // 2, _single_steps(lambda i: 1 + i % 5))
    assert t.stats()["loop_rounds"] > 0
    t.close()


@pytest.mark.gpu
@pytest.mark.parametrize("scan", [0, 2], ids=["lists", "full_scan"])
def test_single_step_tie_break_after_a_launch(scan, monkeypatch):
    """The run stops on the merge just before (5, 10) / (6, 9) -- same weight, same a + b: findNextMerge then breaks the tie on the
    last counted positions, read from the occurrence lists that the rounds wrote."""
    _knobs(monkeypatch, {})
    t, ref = _start("tie")
    t._lib.bpe_set_profiling(t._h, scan)
    full = Ref(*_corpus("tie")[:3])
    full.merge_until({"max_iterations": _corpus("tie")[3]})
    k = next(i for i, (a, b, _) in enumerate(full.log) if (a, b) in ((5, 10), (6, 9)))
    assert k >= 5 and full.log[k + 1][:2] in ((5, 10), (6, 9)) and full.log[k][2] == full.log[k + 1][2], (k, full.log[k:k + 2])
    assert _call(t, ref, {"max_iterations": k}) == k
    checkpoint(t, ref, "before the tie")
    before = t.stats()["tie_breaks"]
    _single_steps(lambda i: 2)(t, ref, 0)
    assert t.stats()["tie_breaks"] > before
    _call(t, ref, {"max_iterations": 200})
    checkpoint(t, ref, "after the tie")
    t.close()


@pytest.mark.gpu
def test_single_steps_on_a_group(monkeypatch):
    devs = _devices(2, monkeypatch)
    _knobs(monkeypatch, {})
    t, ref = _start("remerging", devs)
    _cut_run(t, ref, 600, _single_steps(lambda i: 1 + i % 5, group=True))
    t.close()


# ---- options that change between calls ----
SEQUENCES = {
    "max_length_4_none_6": [{"max_length": 4, "max_iterations": 120}, {"max_iterations": 120}, {"max_length": 6, "max_iterations": 120}],
    "min_weight_150_default": [{"min_weight": 150}, {"max_iterations": 200}],
    "max_length_9_min_weight_3_none": [{"max_length": 9, "min_weight": 3, "max_iterations": 150}, {"max_iterations": 150}],
}


def _zipf(n_bytes):
    from bpe_tokenizer_b200.synth import first_appearance_ids, synth_corpus

    text, off = synth_corpus(n_bytes, seed=43)
    ids, alphabet = first_appearance_ids(text)
    return ids, off, len(alphabet)


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["one", "group2"])
@pytest.mark.parametrize("size", ["small", "mb"])
@pytest.mark.parametrize("seq", sorted(SEQUENCES))
def test_options_change_between_calls(seq, size, where, monkeypatch):
    """small: 100 kB against IntOracle (the literal recount per merge); mb: 3 MB against the incremental oracle."""
    devs = _devices(2, monkeypatch) if where == "group2" else None
    _knobs(monkeypatch, {})
    ids, off, n_alpha = _zipf(100_000 if size == "small" else 3_000_000)
    t = _engine(devs, _alphabet(n_alpha))
    _upload(t, ids, off, "split")
    ref = Ref(ids, off, n_alpha, literal=size == "small")
    calls = []
    for i, opts in enumerate(SEQUENCES[seq]):
        assert _call(t, ref, opts) > 0, (i, opts)
        calls.append(len(ref.log))
        checkpoint(t, ref, "after call %d %s" % (i, opts))
    assert _options_acted(ref, n_alpha, SEQUENCES[seq], calls)
    t.close()


def _options_acted(ref, n_alpha, seq, ends):
    """Every call keeps to its options, and a later call merges a pair that an earlier call's options excluded."""
    lens = np.ones(n_alpha + len(ref.log), dtype=np.int64)
    for j, (a, b, _) in enumerate(ref.log):
        lens[n_alpha + j] = lens[a] + lens[b]

    def allowed(j, opts):
        return lens[n_alpha + j] <= (opts.get("max_length") or 1 << 30) and ref.log[j][2] >= (opts.get("min_weight") or 2)

    begins = [0] + ends[:-1]
    assert all(allowed(j, o) for o, b, e in zip(seq, begins, ends) for j in range(b, e))
    return any(not allowed(j, seq[i]) for i in range(len(seq)) for j in range(ends[i], len(ref.log)))


# ---- replay, then training ----
@pytest.mark.gpu
def test_replay_then_training(monkeypatch):
    """restoreMerges of the first half of a log (k_merge_loop's replay mode) updates the same table that mergeUntil goes on with."""
    _knobs(monkeypatch, {})
    t, ref = _start("mixed")
    full = Ref(*_corpus("mixed")[:3])
    full.merge_until({"max_iterations": 1000})
    assert ref.merge_until({"max_iterations": 500}) == full.log[:500]
    t.restoreMerges([[chr(a + 1), chr(b + 1), w] for a, b, w in full.log[:500]])
    checkpoint(t, ref, "after the replay")
    assert _call(t, ref, {"max_iterations": 500}) == 500
    checkpoint(t, ref, "after training on")
    assert ref.log == full.log
    t.close()


@pytest.mark.gpu
def test_apply_merges_after_a_partial_merge_until(monkeypatch):
    """bpe_apply_merges continues a mergeUntil cut at 300 merges with the oracle's next 300; every replayed merge replaces as many
    occurrences as the oracle's weight; then mergeUntil trains on."""
    from bpe_tokenizer_b200._abi import p32, p64
    from bpe_tokenizer_b200.tokenizer import Token

    _knobs(monkeypatch, {})
    t, ref = _start("remerging")
    assert _call(t, ref, {"max_iterations": 300}) == 300
    checkpoint(t, ref, "after mergeUntil")
    nxt = ref.merge_until({"max_iterations": 300})
    ab = np.array([[a, b] for a, b, _ in nxt], dtype=np.int32).reshape(-1)
    n_replaced = np.zeros(len(nxt), dtype=np.int64)
    t._check(t._lib.bpe_apply_merges(t._h, p32(ab), len(nxt), p64(n_replaced)))
    assert n_replaced.tolist() == [w for _, _, w in nxt]
    for a, b, w in nxt:  # (the host table, as restoreMerges keeps it)
        ta, tb, i = t.token_table[a], t.token_table[b], len(t.token_table)
        t._record_merge(ta, tb, Token(ta.chars + tb.chars, w, w, chr(i + 1), i))
    checkpoint(t, ref, "after bpe_apply_merges")
    assert _call(t, ref, {"max_iterations": 300}) == 300
    checkpoint(t, ref, "after training on")
    t.close()


# ---- run to exhaustion ----
def _tie_quarters():
    from test_gpu_group_edges import _tie_corpus

    (ids, off), _ = _tie_corpus()
    return ids, off, 64


@pytest.mark.gpu
@pytest.mark.parametrize("members", [None, 2, 4], ids=["one", "group2", "group4"])
@pytest.mark.parametrize("name", ["small_mixed", "small_remerging", "tie_quarters"])
def test_run_to_exhaustion(name, members, monkeypatch):
    """No limit: the run ends when no pair reaches min_weight; the last histogram is the recount's, and every count in it is 1."""
    devs = _devices(members, monkeypatch) if members else None
    _knobs(monkeypatch, {})
    ids, off, n_alpha = _tie_quarters() if name == "tie_quarters" else _corpus(name)[:3]
    t = _engine(devs, _alphabet(n_alpha))
    _upload(t, ids, off, "split")
    ref = Ref(ids, off, n_alpha)
    assert _call(t, ref, {}) > 5
    checkpoint(t, ref, "exhausted")
    assert max(recount(*ref.corpus()).values()) == 1
    assert t.mergeUntil({}) == 0
    if name == "tie_quarters":
        assert t.stats()["tie_breaks"] > 0
    t.close()


# ---- which exits were reached ----
def _trace_cases():
    """One engine's cases, run by test_exit_statuses_are_reached in a child process with BPE_TRACE=1."""
    for name in ("mixed", "giant", "many_pairs"):
        t, ref = _start(name)
        _cut_run(t, ref, _corpus(name)[3])
        t.close()
    t, ref = _start("many_pairs")  # to exhaustion: its count-1 pairs keep the hot list's threshold above 1 until the end
    _call(t, ref, {})
    checkpoint(t, ref, "exhausted")
    t.close()


@pytest.mark.gpu
def test_exit_statuses_are_reached():
    """The trace flag is latched at a process's first mergeUntil, hence the child process.  The launches of the cases end in
    statuses 2 (hot-list rebuild), 3 (table or pool growth), 6 (max_iterations reached) and 7 (a winner above R_HUGE)."""
    env = dict(os.environ, BPE_TRACE="1")
    for k in KNOBS:
        env.pop(k, None)
    code = "import sys; sys.path[:0] = [%r, %r]; import test_gpu_merge_state as t; t._trace_cases()" % (ROOT, os.path.join(ROOT, "tests"))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr[-3000:]
    seen = sorted({int(s) for s in re.findall(r"\[bpe\] k_merge_loop: \d+ merges in [\d.]+ ms, status (\d+)", r.stderr)})
    sys.stderr.write("\n[test_gpu_merge_state] exit statuses seen: %s\n" % seen)
    assert {2, 3, 6, 7} <= set(seen), seen


# ---- CPU: the recount is the literal rule ----
def _fuzz_docs(rng, alphabet, n_docs, max_len):
    return ["".join(rng.choice(alphabet) for _ in range(rng.randint(0, max_len))) for _ in range(n_docs)]


def _ids_and_lengths(docs):
    lengths = np.array([len(d) for d in docs], dtype=np.int64)
    return np.array([x for d in docs for x in d], dtype=np.int64), lengths


@pytest.mark.parametrize("seed", range(30))
def test_recount_equals_the_per_pair_loop(seed):
    """Corpora of the fuzz generators, before and after LiteralTokenizer merges: empty and one-token documents, runs that start
    and end at document edges."""
    import random

    from oracle import LiteralTokenizer

    rng = random.Random(3000 + seed)
    alphabet = "ab" if seed % 3 == 0 else "abc" if seed % 3 == 1 else "abcdefg "
    docs = _fuzz_docs(rng, alphabet, rng.randint(1, 8), rng.choice([1, 8, 40, 200]))
    docs += ["", alphabet[0], alphabet[0] * rng.randint(2, 9), "", alphabet[-1] * rng.randint(1, 7) + alphabet[0] * rng.randint(1, 7)]
    rng.shuffle(docs)
    lit = LiteralTokenizer()
    for d in docs:
        lit.addToCorpus(d)
    for _ in range(4):
        toks = [[ord(ch) - 1 for ch in d] for d in lit.corpus_in_code]
        assert recount(*_ids_and_lengths(toks)) == loop_counts(toks)
        lit.mergeUntil({"max_iterations": rng.choice([1, 3, 10])})


def test_recount_edges():
    assert recount([], []) == {} and recount([4], [1]) == {}
    assert recount([0, 0, 0, 0, 0], [5]) == {(0, 0): 2}
    assert recount([0, 0, 0, 0, 0], [2, 3]) == {(0, 0): 2}  # runs end at the document edge
    assert recount([1, 0, 0, 0, 1], [0, 2, 0, 3, 0]) == {(1, 0): 1, (0, 1): 1, (0, 0): 1}
    assert recount([0, 1, 0, 1], [1, 1, 1, 1]) == {}
    ids = np.random.default_rng(1).integers(0, 3, size=5000)
    lengths = np.random.default_rng(2).multinomial(5000, np.ones(700) / 700)
    docs = np.split(ids, np.cumsum(lengths)[:-1])
    assert recount(ids, lengths) == loop_counts([d.tolist() for d in docs])
