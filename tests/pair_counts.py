"""The reference pair histogram of the state tests (test_gpu_merge_state.py, test_gpu_parity.py): the literal counting rule over
a corpus, and the engine's incremental pair table read through the C ABI."""
import ctypes as C

import numpy as np


def recount(ids, lengths):
    """{(a, b): count > 0} of the literal counting rule (core.ts:265-310) over documents of `lengths` tokens laid back to back in
    `ids`: adjacent pairs inside a document, never across a boundary; inside a run of L equal tokens x, the pairs at even offsets
    from the run's start, floor(L / 2) of them."""
    ids = np.asarray(ids, dtype=np.int64)
    n = ids.size
    if n < 2:
        return {}
    starts = np.concatenate([[0], np.cumsum(np.asarray(lengths, dtype=np.int64))[:-1]])
    first = np.zeros(n, dtype=bool)
    first[starts[starts < n]] = True
    a, b = ids[:-1], ids[1:]
    inside = ~first[1:]
    run_start = first.copy()
    run_start[1:] |= a != b
    run_first = np.maximum.accumulate(np.where(run_start, np.arange(n), 0))
    counted = inside & ((a != b) | ((np.arange(n - 1) - run_first[:-1]) % 2 == 0))
    keys, cnt = np.unique((a[counted] << 32) | b[counted], return_counts=True)
    return {(int(k >> 32), int(k & 0xFFFFFFFF)): int(c) for k, c in zip(keys, cnt)}


def loop_counts(docs):
    """The per-pair loop of test_gpu_parity.py::test_pair_histogram_matches_oracle_counts, over documents given as lists of ids."""
    want = {}
    for toks in docs:
        run = 0
        for i in range(1, len(toks)):
            x, y = toks[i - 1], toks[i]
            if x == y:
                run = run + 1 if (i >= 2 and toks[i - 2] == x) else 1
                if run % 2 == 0:
                    continue
            else:
                run = 0
            want[(x, y)] = want.get((x, y), 0) + 1
    return want


def device_counts(t):
    """The engine's incremental pair table, {(a, b): count > 0}; the dump must not rebuild the index (a fresh build would be
    compared instead of the table the merges updated)."""
    from bpe_tokenizer_b200 import _abi

    before = t.stats()["index_builds"]
    cap = 1 << 16
    for attempt in range(2):
        a, b, c = np.zeros(cap, np.int32), np.zeros(cap, np.int32), np.zeros(cap, np.int64)
        n = C.c_int64()
        rc = t._lib.bpe_pair_counts(t._h, _abi.p32(a), _abi.p32(b), _abi.p64(c), cap, C.byref(n))
        if rc == _abi.BPE_E_CAPACITY and attempt == 0:
            cap = n.value
            continue
        t._check(rc)
        break
    assert t.stats()["index_builds"] == before, "bpe_pair_counts rebuilt the index"
    k = n.value
    return dict(zip(zip(a[:k].tolist(), b[:k].tolist()), c[:k].tolist()))
