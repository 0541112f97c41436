"""GPU: the site passes of k_merge_rounds stage the count deltas of frequent neighbours (token ids below the build's R_STAGE_T)
in per-block shared-memory cells and add them to the global cells once per block (csrc/round_kernels.cuh).  With staging
forced on for every merge and forced off (BPE_BLOCK_CELLS_MIN_SITES), the merge log -- pairs and weights -- and the corpus must
equal the incremental CPU oracle's (oracle/fast_oracle.py, pinned to the literal restatement by tests/test_oracle_golden.py)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

STAGE = {"on": "0", "off": "4294967295"}  # list entries above which a merge stages: every merge / none
# neighbour ids on both sides of each threshold a build may stage below (BPE_STAGE_T = 128, 256 or 512)
EDGE = [t + d for t in (128, 256, 512) for d in (-1, 0, 1)]


def _alphabet(n):
    return [0x4E00 + i for i in range(n)]  # n distinct single-character tokens (CJK ideographs: no surrogates, no controls)


def _mixed(seed, n_tokens):
    """Zipf-weighted text over the EDGE ids and a few others, with back-to-back pairs (a b a b ..), runs (a a a ..) pasted in
    and documents of 1..64 tokens, so that the big merges have neighbours on both sides of the staging threshold, merges with
    a == b occur, sites sit at document boundaries, and the merges of one round share their frequent neighbours."""
    rng = np.random.default_rng(seed)
    vocab = np.array(EDGE + [0, 1, 2, 3, 300, 400], dtype=np.int32)
    p = 1.0 / np.arange(1, len(vocab) + 1)
    rng.shuffle(p)
    ids = rng.choice(vocab, size=n_tokens, p=p / p.sum()).astype(np.int32)
    for _ in range(n_tokens // 300):
        at = int(rng.integers(0, n_tokens - 64))
        a, b = rng.choice(vocab, 2)
        half = int(rng.integers(2, 16))
        ids[at:at + 2 * half] = np.tile(np.array([a, b], dtype=np.int32), half)
        at = int(rng.integers(0, n_tokens - 64))
        ids[at:at + int(rng.integers(3, 33))] = rng.choice(vocab)
    cuts = np.cumsum(rng.integers(1, 65, size=n_tokens // 16))
    off = np.concatenate([[0], cuts[cuts < n_tokens], [n_tokens]]).astype(np.int64)
    return ids, off


def _check(ids, off, n_alpha, merges):
    from bpe_tokenizer_b200 import BPETokenizer
    from oracle.fast_oracle import FastOracle

    gpu = BPETokenizer()
    gpu.addToCorpus("".join(chr(c) for c in _alphabet(n_alpha)))
    gpu.corpus_in_code = []
    for tk in gpu.token_table:
        tk.weight = tk.original_weight = 0
    gpu.addDocuments(ids, off)
    n = gpu.mergeUntil({"max_iterations": merges})
    o = FastOracle()
    o.set_len16(np.ones(n_alpha, dtype=np.int32))
    o.add_documents(ids, off)
    la, lb, lw = o.merge_until(2, 0, merges, n_alpha, merges)
    got = [[a.index, b.index, c.original_weight] for a, b, c in gpu.merge_tokens]
    want = [[int(a), int(b), int(w)] for a, b, w in zip(la, lb, lw)]
    first_bad = next((i for i, (g, w) in enumerate(zip(got, want)) if g != w), None)
    assert first_bad is None, (first_bad, got[first_bad], want[first_bad])
    assert n == len(want)
    got_ids, _ = gpu.corpusIds()
    assert np.array_equal(got_ids, o.corpus())
    return gpu.stats()


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("stage", ["on", "off"])
def test_staged_cells_equal_the_oracle(stage, seed, monkeypatch):
    monkeypatch.setenv("BPE_BLOCK_CELLS_MIN_SITES", STAGE[stage])
    ids, off = _mixed(seed, 3_000_000)
    st = _check(ids, off, 600, 1500)
    assert st["loop_round_merges"] > 1.5 * st["loop_rounds"], st  # rounds of several merges that share neighbours


@pytest.mark.parametrize("stage", ["on", "off"])
def test_staged_cells_with_a_full_cell_list(stage, monkeypatch):
    """One block, and a first merge (a, b) whose 17 000 sites each have a different neighbour on either side (ids 2 .. 17 001,
    below and above the threshold): 34 000 touched cells overflow the block's list (R_LISTCAP = 32 768), so the round clears and
    visits the cells by scanning the rows.  Zipf text after it gives the following rounds their merges."""
    monkeypatch.setenv("BPE_BLOCK_CELLS_MIN_SITES", STAGE[stage])
    monkeypatch.setenv("BPE_LOOP_BLOCKS", "1")
    n = 17_000
    x = np.arange(2, 2 + n, dtype=np.int32)
    head = np.stack([x, np.zeros(n, np.int32), np.ones(n, np.int32), x[::-1]], axis=1).ravel()
    tail, toff = _mixed(3, 40_000)
    ids = np.concatenate([head, tail])
    off = np.concatenate([np.arange(0, 4 * n, 4, dtype=np.int64), toff + 4 * n])
    _check(ids, off, 2 + n, 300)
