"""CPU: the host side of the sharded text ingest (ShardedBPETokenizer.addTextBatch) -- the global first-appearance order
of the new characters, and the collective protocol around stage and commit on gloo, with stub steps in place of the
engines: every rank gets the same result, and a failure on one rank raises the same error on every rank."""
import datetime
import os
import random

import numpy as np
import pytest

from bpe_tokenizer_b200 import BpeError, _abi
from bpe_tokenizer_b200.sharded import order_new_chars, text_ingest_collective


def _local_report(piece, known, rng):
    """What a rank's stage reports for its piece: each code point the table does not know, with its first local
    position, in an arbitrary order."""
    first = {}
    for i, cp in enumerate(piece):
        if cp not in known and cp not in first:
            first[cp] = i
    items = list(first.items())
    rng.shuffle(items)
    return [cp for cp, _ in items], [p for _, p in items]


def _first_appearance(seq, known):
    out, seen = [], set(known)
    for cp in seq:
        if cp not in seen:
            seen.add(cp)
            out.append(cp)
    return out


def test_order_new_chars_matches_a_scan_of_the_concatenation():
    rng = random.Random(11)
    for case in range(400):
        world = rng.randint(1, 8)
        alphabet = rng.sample([0x41, 0x61, 0xE9, 0x3B1, 0x4E2D, 0xD800, 0xDFFF, 0x1F600, 0x10FFFF, 0x0, 0x7F, 0x80, 0x7FF, 0x800, 0xFFFF, 0x10000],
                              rng.randint(1, 16))
        seq = [rng.choice(alphabet) for _ in range(rng.randint(0, 200))]
        cuts = sorted(rng.randint(0, len(seq)) for _ in range(world - 1))
        pieces = [seq[a:b] for a, b in zip([0] + cuts, cuts + [len(seq)])]
        known = set(rng.sample(alphabet, rng.randint(0, len(alphabet) // 2)))
        per_rank = [_local_report(p, known, rng) for p in pieces]
        assert order_new_chars(per_rank) == _first_appearance(seq, known), case


def test_order_new_chars_rank_before_position():
    # rank 1 sees 'b' at local position 0, rank 0 at 10^6: it is rank 0's character
    assert order_new_chars([([ord("a"), ord("b")], [0, 10**6]), ([ord("b"), ord("c")], [0, 1])]) == [ord("a"), ord("b"), ord("c")]
    # characters only a later rank sees, behind empty ranks
    assert order_new_chars([([], []), ([0x10FFFF, 0xD800], [7, 3]), ([], []), ([0xD800, 0x41], [0, 5])]) == [0xD800, 0x10FFFF, 0x41]
    assert order_new_chars([]) == []
    assert order_new_chars([(np.array([5, 4], dtype=np.int32), np.array([1, 0], dtype=np.int64))]) == [4, 5]


def test_protocol_single_rank_needs_no_process_group():
    new, counts = text_ingest_collective(lambda: ([9, 7], [3, 1]), lambda cps: np.arange(2 + len(cps), dtype=np.int64), 2, 1)
    assert new == [7, 9] and counts.tolist() == [0, 1, 2, 3]


def _raised(fn):
    try:
        fn()
    except BpeError as ex:
        return (ex.code, ex.message)
    return None


def _gloo_protocol_worker(rank, world, port):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    # a regression that leaves one rank waiting must fail the test, not hang it
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=datetime.timedelta(seconds=60))
    try:
        n_tokens = 3
        lists = {0: ([ord("x"), ord("y")], [4, 0]), 1: ([ord("z"), ord("x")], [0, 2])}

        def stage_ok():
            return lists[rank]

        def commit_ok(cps):
            assert cps == [ord("y"), ord("x"), ord("z")]
            return np.arange(n_tokens + len(cps), dtype=np.int64) * (rank + 1)

        def stage_fails_on_1():
            if rank == 1:
                raise BpeError(_abi.BPE_E_INVALID, "document offsets must be non-decreasing (rank 1)")
            return lists[rank]

        def stage_raises_other_on_0():
            if rank == 0:
                raise ValueError("not a BpeError")
            return lists[rank]

        def commit_fails_on_0(cps):
            if rank == 0:
                raise BpeError(_abi.BPE_E_CUDA, "commit failed on rank 0")
            return np.zeros(n_tokens + len(cps), dtype=np.int64)

        committed = []

        def commit_recorded(cps):
            committed.append(cps)
            return np.zeros(n_tokens + len(cps), dtype=np.int64)

        results = {}
        new, counts = text_ingest_collective(stage_ok, commit_ok, n_tokens, world)
        results["ok"] = (new, counts.tolist())
        assert new == [ord("y"), ord("x"), ord("z")]
        assert counts.tolist() == [3 * i for i in range(6)]  # summed over both ranks
        results["stage"] = _raised(lambda: text_ingest_collective(stage_fails_on_1, commit_recorded, n_tokens, world))
        results["other"] = _raised(lambda: text_ingest_collective(stage_raises_other_on_0, commit_recorded, n_tokens, world))
        assert committed == []  # no rank commits after a failed stage
        results["commit"] = _raised(lambda: text_ingest_collective(stage_ok, commit_fails_on_0, n_tokens, world))
        # each rank's list alone fits, the union does not: every rank raises, none commits
        full = _abi.BPE_MAX_TOKENS - 2
        results["domain"] = _raised(lambda: text_ingest_collective(stage_ok, commit_recorded, full, world))
        assert committed == []
        # the protocol still works after the failures (no collective was left half done)
        results["again"] = text_ingest_collective(stage_ok, commit_ok, n_tokens, world)[0]
        assert results["stage"] == (_abi.BPE_E_INVALID, "document offsets must be non-decreasing (rank 1)")
        assert results["other"][0] == _abi.BPE_E_INTERNAL and "not a BpeError" in results["other"][1]
        assert results["commit"] == (_abi.BPE_E_CUDA, "commit failed on rank 0")
        assert results["domain"][0] == _abi.BPE_E_DOMAIN
        everyone = [None] * world
        dist.all_gather_object(everyone, results)
        assert all(r == everyone[0] for r in everyone), everyone
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(180)
def test_protocol_failures_reach_every_rank_world2_gloo():
    import torch.multiprocessing as mp

    mp.spawn(_gloo_protocol_worker, args=(2, 29547), nprocs=2, join=True)
