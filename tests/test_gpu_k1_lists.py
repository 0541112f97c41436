"""GPU: K1b (`k_scatter`, csrc/train_kernels.cuh) stages each chunk's occurrence lists in shared memory and copies them out as
contiguous runs; pairs that find no room in the block's shared table go straight to the pool.  On corpora built to hit the
edges of that scheme, the merge log -- pairs and weights -- and the final corpus must equal the incremental CPU oracle's
(oracle/fast_oracle.py), with the product library (chunks of 2^15 positions) and with a build of 2^10-position chunks, which
puts many chunk boundaries inside documents and runs.  Each case runs in its own process, because a process binds one library."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL_CHUNK_LOG = 10
BIG = 1 << 15  # the product library's chunk (BPE_K1B_CHUNK_LOG in csrc/train_kernels.cuh)


def _mixed(rng, n_tokens, n_alpha):
    """Zipf-weighted ids with runs (a a a ..) of odd and even length pasted in, in documents of 1..300 tokens."""
    p = 1.0 / np.arange(1, n_alpha + 1)
    ids = rng.choice(n_alpha, size=n_tokens, p=p / p.sum()).astype(np.int32)
    for _ in range(n_tokens // 500):
        at = int(rng.integers(0, n_tokens - 40))
        ids[at:at + int(rng.integers(2, 40))] = rng.integers(0, 4)
    cuts = np.cumsum(rng.integers(1, 301, size=n_tokens // 100 + 1))
    return ids, np.concatenate([[0], cuts[cuts < n_tokens], [n_tokens]]).astype(np.int64)


def _case(name):
    """(ids, doc offsets, alphabet size, merges) of one corpus."""
    rng = np.random.default_rng(7)
    if name == "straddle_odd_length":
        # 3 big chunks + 7 positions: not a multiple of 4 or of any chunk; documents and runs cross every chunk boundary
        n = 3 * BIG + 7
        ids, off = _mixed(rng, n, 40)
        for b in range(1 << SMALL_CHUNK_LOG, n, 1 << SMALL_CHUNK_LOG):
            if rng.integers(0, 4) == 0:
                ids[b - 5:b + 6] = 2  # a run of 11 across the boundary
        off = np.union1d(off, [0, n])
        off = off[(off % BIG != 0) | (off == 0) | (off == n)]  # no document starts on a big chunk's first position
        return ids, off.astype(np.int64), 40, 400
    if name == "many_pairs":
        # uniform ids over 3000 tokens: ~30 000 distinct pairs per big chunk, far more than the 2048 slots of the shared
        # table, so most adjacencies take the global path; Zipf text after it gives the merges something to do
        head = rng.integers(0, 3000, size=2 * BIG + 1001).astype(np.int32)
        tail, toff = _mixed(rng, BIG, 40)
        ids = np.concatenate([head, tail])
        off = np.concatenate([[0, 40_000], toff + head.size]).astype(np.int64)
        return ids, off, 3000, 300
    if name == "one_char_documents":
        # every other document is a single character (no adjacency); the others are short
        lens = np.where(np.arange(60_000) % 2 == 0, 1, rng.integers(2, 9, size=60_000))
        ids = rng.integers(0, 30, size=int(lens.sum())).astype(np.int32)
        return ids, np.concatenate([[0], np.cumsum(lens)]).astype(np.int64), 30, 200
    if name == "runs":
        # runs a a a .. of every length 1..600 in one document each and back to back inside long documents, so that the
        # counted-occurrence parity (floor(len/2) per run) is tested on runs that cross chunk boundaries
        parts = [np.full(k, k % 5, dtype=np.int32) for k in range(1, 601)]
        ids = np.concatenate(parts + parts)
        lens = [len(q) for q in parts] + [sum(len(q) for q in parts[i:i + 50]) for i in range(0, 600, 50)]
        return ids, np.concatenate([[0], np.cumsum(lens)]).astype(np.int64), 5, 300
    if name == "single_chunk":
        ids, off = _mixed(rng, 1000, 12)
        return ids, off, 12, 100
    if name == "one_pair_fills_a_chunk":
        # one document of BIG + 1 copies of one token: the first big chunk (and every small one it covers) holds BIG
        # adjacencies of (0, 0), a single run as long as the chunk; then a b a b .. over a whole big chunk.  (The oracle's
        # time grows with the square of a run's length, so the run is not longer.)
        ids = np.concatenate([np.zeros(BIG + 1, np.int32), np.tile(np.array([1, 2], np.int32), BIG // 2)])
        return ids, np.array([0, BIG + 1, ids.size], np.int64), 3, 40
    raise KeyError(name)


CASES = ["straddle_odd_length", "many_pairs", "one_char_documents", "runs", "single_chunk", "one_pair_fills_a_chunk"]


def _check(ids, off, n_alpha, merges):
    """Run in the child process: the GPU engine of whichever library BPE_LIB names against the CPU oracle."""
    from bpe_tokenizer_b200 import BPETokenizer
    from oracle.fast_oracle import FastOracle

    gpu = BPETokenizer()
    gpu.addToCorpus("".join(chr(0x4E00 + i) for i in range(n_alpha)))  # n_alpha single-character tokens
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
    assert n == len(want) > 0
    got_ids, _ = gpu.corpusIds()
    assert np.array_equal(got_ids, o.corpus())


@pytest.fixture(scope="module")
def small_chunk_lib(tmp_path_factory):
    from bpe_tokenizer_b200 import build

    out = str(tmp_path_factory.mktemp("k1b") / ("libbpe_b200_chunk%d.so" % SMALL_CHUNK_LOG))
    old = os.environ.get("BPE_K1B_CHUNK_LOG")
    os.environ["BPE_K1B_CHUNK_LOG"] = str(SMALL_CHUNK_LOG)
    try:
        return build.build(force=True, out=out)
    finally:
        if old is None:
            del os.environ["BPE_K1B_CHUNK_LOG"]
        else:
            os.environ["BPE_K1B_CHUNK_LOG"] = old


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("chunk", ["product", "small"])
def test_lists_equal_the_oracle(chunk, case, request):
    env = dict(os.environ)
    env.pop("BPE_LIB", None)
    if chunk == "small":
        env["BPE_LIB"] = request.getfixturevalue("small_chunk_lib")
    code = "import sys; sys.path[:0] = [%r, %r]; import test_gpu_k1_lists as t; t._check(*t._case(%r))" % (ROOT, os.path.join(ROOT, "tests"), case)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr[-3000:]


def test_cases_hit_the_edges():
    """CPU: the corpora have the shapes the GPU test relies on."""
    ids, off, _, _ = _case("straddle_odd_length")
    assert ids.size % 4 and ids.size % BIG and off[-1] == ids.size
    starts = set(off[:-1].tolist())
    assert not any(b in starts for b in range(BIG, ids.size, BIG))  # the big chunks' boundaries fall inside documents
    ids, off, _, _ = _case("many_pairs")
    chunk = ids[BIG:2 * BIG].astype(np.int64)
    assert np.unique(chunk[:-1] * 3000 + chunk[1:]).size > 20_000
    ids, off, _, _ = _case("one_char_documents")
    assert np.sum(np.diff(off) == 1) >= 30_000
    ids, off, _, _ = _case("single_chunk")
    assert ids.size < 1 << SMALL_CHUNK_LOG
    ids, off, _, _ = _case("one_pair_fills_a_chunk")
    assert off[1] == BIG + 1 and not ids[:off[1]].any()
