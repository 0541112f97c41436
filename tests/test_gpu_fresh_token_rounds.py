"""GPU: a pair that contains a token the previous round of k_merge_rounds created joins the next round's batch, and its site
pass walks that round's site records instead of its occurrence list, which the helper warps are still writing
(csrc/round_kernels.cuh: RoundSm::src).  The corpora below make new tokens merge again at once -- back-to-back pairs
(x y x y ..), runs (x x x ..), chains (x y z x y z .. w), text over a Zipf-weighted lexicon of words -- so that batches hold
pairs (c, y), (x, c), (c, c) and pairs of two new tokens of the previous round, winners included.  The merge log (a, b, weight) and the corpus must
equal the incremental CPU oracle's (oracle/fast_oracle.py), on one engine and on a two-member device group (the sharded
rounds).  A site pass that finds another number of sites than the pair's count sets ERR_ROUND_MISMATCH, which mergeUntil
reports as an error."""
import numpy as np
import pytest

from test_gpu_group_edges import _devices, _engine

pytestmark = pytest.mark.gpu

N_ALPHA = 64


def _remerging(seed, n_tokens):
    """Pieces over a Zipf-weighted alphabet of N_ALPHA ids, 1..8 pieces per document: x y repeated, x repeated, x y z repeated
    with a w after it, or (five pieces in eight) 1..23 words of a Zipf-weighted lexicon of 400 words of 2..8 ids -- whose merges
    build the frequent words one new token after the other."""
    rng = np.random.default_rng(seed)
    p = 1.0 / np.arange(1, N_ALPHA + 1)
    p /= p.sum()
    lex = [rng.choice(N_ALPHA, size=int(rng.integers(2, 9)), p=p).astype(np.int32) for _ in range(400)]
    lw = 1.0 / np.arange(1, len(lex) + 1)
    lw /= lw.sum()
    pieces, ends, total = [], [], 0
    while total < n_tokens:
        x, y, z, w = rng.choice(N_ALPHA, 4, p=p)
        h = int(rng.integers(1, 24))
        kind = int(rng.integers(0, 8))
        if kind == 0:
            piece = np.tile([x, y], h)
        elif kind == 1:
            piece = np.full(h, x)
        elif kind == 2:
            piece = np.concatenate([np.tile([x, y, z], h), [w]])
        else:
            piece = np.concatenate([lex[i] for i in rng.choice(len(lex), size=h, p=lw)])
        pieces.append(piece.astype(np.int32))
        total += len(piece)
        ends.append(total)
    ids = np.concatenate(pieces)
    cuts = np.array(ends, dtype=np.int64)[:: int(rng.integers(1, 9))]
    off = np.unique(np.concatenate([[0], cuts, [len(ids)]])).astype(np.int64)
    return ids, off


def _oracle(ids, off, merges, max_length):
    from oracle.fast_oracle import FastOracle

    o = FastOracle()
    o.set_len16(np.ones(N_ALPHA, dtype=np.int32))
    o.add_documents(ids, off)
    la, lb, lw = o.merge_until(2, max_length, merges, N_ALPHA, merges)
    return [[int(a), int(b), int(w)] for a, b, w in zip(la, lb, lw)], o.corpus()


def _run(devs, ids, off, merges, max_length):
    gpu = _engine(devs, [0x4E00 + i for i in range(N_ALPHA)])
    gpu.addDocuments(ids, off)
    opts = {"max_iterations": merges}
    if max_length:
        opts["max_length"] = max_length
    n = gpu.mergeUntil(opts)
    want, corpus = _oracle(ids, off, merges, max_length)
    got = [[a.index, b.index, c.original_weight] for a, b, c in gpu.merge_tokens]
    first_bad = next((i for i, (g, w) in enumerate(zip(got, want)) if g != w), None)
    assert first_bad is None, (first_bad, got[first_bad], want[first_bad])
    assert n == len(want)
    got_ids, _ = gpu.corpusIds()
    assert np.array_equal(got_ids, corpus)
    return gpu.stats()


@pytest.mark.parametrize("max_length", [0, 4, 9], ids=["plain", "max_length4", "max_length9"])
@pytest.mark.parametrize("seed", [1, 2])
def test_fresh_tokens_join_the_batch(seed, max_length):
    ids, off = _remerging(seed, 3_000_000)
    st = _run(None, ids, off, 1500, max_length)
    assert st["loop_rounds"] > 0 and st["loop_round_merges"] > 1.5 * st["loop_rounds"], st


def test_fresh_tokens_join_the_batch_sharded(monkeypatch):
    """The same on two members: each rank walks its own records of the previous round."""
    devs = _devices(2, monkeypatch)
    ids, off = _remerging(3, 3_000_000)
    _run(devs, ids, off, 1500, 0)
