"""GPU: the site passes of k_merge_loop stage the count deltas of frequent neighbours per block as k_merge_rounds does
(csrc/train_kernels.cuh: agg_new_dense, agg_dec2, loop_flush_stage).  The corpora of test_gpu_block_cells run through
k_merge_loop alone (BPE_LOOP_ROUNDS=0) with staging forced on and off; a pair above R_HUGE sends its merge from the rounds to
k_merge_loop under default knobs; a replayed merge log (restoreMerges, replay mode of k_merge_loop) runs staged.  Merge log,
weights and corpus must equal the incremental CPU oracle's (oracle/fast_oracle.py) or the uninterrupted run's.  The list
filling of a staged merge (phase_fill with `stage`) runs in the whole-block fills: next to a big merge's site pass, before a
tie-break, before a winner born by the previous merge, and on exit."""
import numpy as np
import pytest

from test_gpu_block_cells import EDGE, STAGE, _alphabet, _check, _mixed

pytestmark = pytest.mark.gpu


def _loop_only(monkeypatch, stage):
    monkeypatch.setenv("BPE_LOOP_ROUNDS", "0")
    monkeypatch.setenv("BPE_BLOCK_CELLS_MIN_SITES", STAGE[stage])


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("stage", ["on", "off"])
def test_loop_staged_deltas_equal_the_oracle(stage, seed, monkeypatch):
    _loop_only(monkeypatch, stage)
    ids, off = _mixed(seed, 3_000_000)
    _check(ids, off, 600, 1500)


@pytest.mark.parametrize("stage", ["on", "off"])
def test_loop_staged_deltas_one_block(stage, monkeypatch):
    """One block: its staged rows hold the whole grid's deltas of the frequent neighbours."""
    _loop_only(monkeypatch, stage)
    monkeypatch.setenv("BPE_LOOP_BLOCKS", "1")
    ids, off = _mixed(1, 3_000_000)
    _check(ids, off, 600, 600)


@pytest.mark.parametrize("stage", ["on", "off"])
def test_loop_staged_deltas_many_distinct_neighbours(stage, monkeypatch):
    """test_gpu_block_cells' corpus whose first merge has 17 000 sites, each with a different neighbour on either side (ids
    2 .. 17 001, below and above R_STAGE_T), on one block."""
    _loop_only(monkeypatch, stage)
    monkeypatch.setenv("BPE_LOOP_BLOCKS", "1")
    n = 17_000
    x = np.arange(2, 2 + n, dtype=np.int32)
    head = np.stack([x, np.zeros(n, np.int32), np.ones(n, np.int32), x[::-1]], axis=1).ravel()
    tail, toff = _mixed(3, 40_000)
    ids = np.concatenate([head, tail])
    off = np.concatenate([np.arange(0, 4 * n, 4, dtype=np.int64), toff + 4 * n])
    _check(ids, off, 2 + n, 300)


@pytest.mark.parametrize("stage", ["on", "off"])
def test_loop_staged_fill_before_a_tie_break(stage, monkeypatch):
    """(5, 10) and (6, 9) -- same weight, same a + b -- in 40 000 two-token documents each: their merge is a tie broken by the
    last counted position, which reads occurrence lists, so the previous merge's lists are filled first (staged when on)."""
    _loop_only(monkeypatch, stage)
    rng = np.random.default_rng(11)
    pairs = np.array([[5, 10], [6, 9]], dtype=np.int32)[rng.permutation(np.repeat([0, 1], 40_000))]
    tail, toff = _mixed(6, 500_000)
    ids = np.concatenate([pairs.ravel(), tail])
    off = np.concatenate([np.arange(0, 2 * len(pairs), 2, dtype=np.int64), toff + 2 * len(pairs)])
    st = _check(ids, off, 600, 600)
    assert st["tie_breaks"] > 0, st


def _giant_corpus(seed, groups):
    """`groups` times [x, 0, 1] with Zipf-weighted x over the EDGE ids and a few others (documents of whole groups), then
    test_gpu_block_cells' mixed text: the pair (0, 1) has more than `groups` sites."""
    rng = np.random.default_rng(seed)
    vocab = np.array(EDGE + [2, 3, 4, 5, 300, 400], dtype=np.int32)
    p = 1.0 / np.arange(1, len(vocab) + 1)
    rng.shuffle(p)
    x = rng.choice(vocab, size=groups, p=p / p.sum()).astype(np.int32)
    head = np.stack([x, np.zeros(groups, np.int32), np.ones(groups, np.int32)], axis=1).ravel()
    cuts = np.cumsum(3 * rng.integers(1, 33, size=groups // 8))
    tail, toff = _mixed(seed, 200_000)
    ids = np.concatenate([head, tail])
    off = np.concatenate([[0], cuts[cuts < 3 * groups], toff + 3 * groups]).astype(np.int64)
    return ids, off


def test_giant_merge_leaves_the_rounds_staged_and_returns(monkeypatch):
    """Default knobs: the first pair has 1.1 M sites, above R_HUGE = 2^20, so the rounds hand it to k_merge_loop
    (LOOP_NEED_LEGACY), whose site pass stages (1.1 M list entries > BPE_BLOCK_CELLS_MIN_SITES), and the rounds take the
    merges after it."""
    for k in ("BPE_BLOCK_CELLS_MIN_SITES", "BPE_LOOP_ROUNDS", "BPE_LOOP_BLOCKS"):
        monkeypatch.delenv(k, raising=False)
    ids, off = _giant_corpus(7, 1_100_000)
    # the 1.1 M groups alone hold (0, 1) inside their documents, one site each: above R_HUGE, which the rounds cannot take
    assert np.count_nonzero((ids[:-1] == 0) & (ids[1:] == 1)) > 1 << 20
    st = _check(ids, off, 600, 300)
    assert st["loop_round_merges"] > 0, st


def _engine(ids, off, n_alpha):
    from bpe_tokenizer_b200 import BPETokenizer

    t = BPETokenizer()
    t.addToCorpus("".join(chr(c) for c in _alphabet(n_alpha)))
    t.corpus_in_code = []
    for tk in t.token_table:
        tk.weight = tk.original_weight = 0
    t.addDocuments(ids, off)
    return t


def test_replay_staged_equals_the_uninterrupted_run(monkeypatch):
    """restoreMerges with staging forced on leaves the corpus of the run that wrote the log, and every replayed merge
    replaces exactly as many occurrences as that merge's weight (k_merge_loop logs its site count as the weight)."""
    from bpe_tokenizer_b200._abi import p32, p64

    ids, off = _mixed(5, 2_000_000)
    first = _engine(ids, off, 600)
    first.mergeUntil({"max_iterations": 500})
    log = [[a.code, b.code, c.original_weight] for a, b, c in first.merge_tokens]
    monkeypatch.setenv("BPE_BLOCK_CELLS_MIN_SITES", STAGE["on"])
    again = _engine(ids, off, 600)
    again.restoreMerges(log)
    assert np.array_equal(again.corpusIds()[0], first.corpusIds()[0])
    assert [t.chars for t in again.token_table] == [t.chars for t in first.token_table]
    raw = _engine(ids, off, 600)
    raw._flush()
    ab = np.array([[a.index, b.index] for a, b, _ in first.merge_tokens], dtype=np.int32).reshape(-1)
    n_replaced = np.zeros(len(log), dtype=np.int64)
    assert raw._lib.bpe_apply_merges(raw._h, p32(ab), len(log), p64(n_replaced)) == 0
    assert n_replaced.tolist() == [w for _, _, w in log]
