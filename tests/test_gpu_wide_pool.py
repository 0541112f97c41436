"""GPU: the occurrence pool's cell indices are 64-bit, so one engine trains on corpora whose pool passes 2^32 cells.  BPE_POOL_BASE
starts the pool's cursor just below 2^32 (memory is reserved below it), so that the lists of MB-sized corpora sit on both sides of
cell 2^32 and straddle it; the merge logs and corpora must stay those of the CPU oracles.  Every test checks that the pool really
passed 2^32 cells."""
import json
import os
import random

import numpy as np
import pytest

from oracle import LiteralTokenizer

pytestmark = pytest.mark.gpu

TOP = 1 << 32
BASE_MB = str(TOP - (1 << 20))  # MB corpora: K1 alone writes several million cells, most of them above 2^32
BASE_SMALL = str(TOP - 64)      # fuzz corpora of a few hundred positions


def _fresh(alphabet):
    from bpe_tokenizer_b200 import BPETokenizer

    gpu = BPETokenizer()
    gpu.addToCorpus("".join(chr(c) for c in alphabet))  # the single-character tokens in first-appearance order
    gpu.corpus_in_code = []
    for tk in gpu.token_table:
        tk.weight = tk.original_weight = 0
    return gpu


def _crossed(gpu):
    assert gpu.stats()["pool_used"] > TOP


def test_cfg2_golden_with_a_straddling_pool(monkeypatch):
    """cfg2 (10 MB, 4 000 merges) against the literal restatement's fixture: SHA-1 of the log, its first and last entries."""
    import hashlib

    from bpe_tokenizer_b200._abi import MERGE_DTYPE
    from bpe_tokenizer_b200.synth import first_appearance_ids, synth_corpus

    monkeypatch.setenv("BPE_POOL_BASE", BASE_MB)
    with open(os.path.join(os.path.dirname(__file__), "golden", "cfg2_merge_log.json")) as f:
        golden = json.load(f)
    text, off = synth_corpus(10_000_000, seed=43)
    ids, alphabet = first_appearance_ids(text)
    gpu = _fresh(alphabet)
    gpu.addDocuments(ids, off)
    assert gpu.mergeUntil({"max_iterations": golden["merges"]}) == golden["merges"]
    log = np.zeros(golden["merges"], dtype=MERGE_DTYPE)
    log["a"] = [a.index for a, _, _ in gpu.merge_tokens]
    log["b"] = [b.index for _, b, _ in gpu.merge_tokens]
    log["c"] = [c.index for _, _, c in gpu.merge_tokens]
    log["weight"] = [c.original_weight for _, _, c in gpu.merge_tokens]
    assert [[int(r["a"]), int(r["b"]), int(r["weight"])] for r in log[:8]] == golden["first"]
    assert [[int(r["a"]), int(r["b"]), int(r["weight"])] for r in log[-4:]] == golden["last"]
    assert hashlib.sha1(log.tobytes()).hexdigest() == golden["sha1"]
    _crossed(gpu)
    gpu.close()


# rounds (k_merge_rounds, 16 merges per batch), the one-merge kernel (k_merge_loop), and both with every merge staging its
# neighbours' deltas and list cells per block (BPE_BLOCK_CELLS_MIN_SITES=0: the staged list fill of the giant merges)
LOOPS = {"rounds16": {"BPE_LOOP_K": "16"}, "one_merge": {"BPE_LOOP_ROUNDS": "0"},
         "rounds16_staged": {"BPE_LOOP_K": "16", "BPE_BLOCK_CELLS_MIN_SITES": "0"},
         "one_merge_staged": {"BPE_LOOP_ROUNDS": "0", "BPE_BLOCK_CELLS_MIN_SITES": "0"}}


@pytest.mark.parametrize("loop", list(LOOPS))
def test_merge_loops_with_a_straddling_pool_equal_the_oracle(loop, monkeypatch):
    from bpe_tokenizer_b200.synth import first_appearance_ids, synth_corpus
    from oracle.fast_oracle import FastOracle

    monkeypatch.setenv("BPE_POOL_BASE", BASE_MB)
    for k, v in LOOPS[loop].items():
        monkeypatch.setenv(k, v)
    text, off = synth_corpus(6_000_000, seed=43)
    ids, alphabet = first_appearance_ids(text)
    merges = 3000
    gpu = _fresh(alphabet)
    gpu.addDocuments(ids, off)
    n = gpu.mergeUntil({"max_iterations": merges})
    o = FastOracle()
    o.set_len16(np.ones(len(alphabet), dtype=np.int32))
    o.add_documents(ids, off)
    la, lb, lw = o.merge_until(2, 0, merges, len(alphabet), merges)
    got = [[a.index, b.index, c.original_weight] for a, b, c in gpu.merge_tokens]
    want = [[int(a), int(b), int(w)] for a, b, w in zip(la, lb, lw)]
    first_bad = next((i for i, (g, w) in enumerate(zip(got, want)) if g != w), None)
    assert first_bad is None, (first_bad, got[first_bad], want[first_bad])
    assert n == len(want)
    got_ids, _ = gpu.corpusIds()
    assert np.array_equal(got_ids, o.corpus())
    _crossed(gpu)
    gpu.close()


def _docs(seed):
    rng = random.Random(7000 + seed)
    alphabet = "ab" if seed % 2 == 0 else "abcdef "
    return [("".join(rng.choice(alphabet) for _ in range(rng.randint(40, 160)))) for _ in range(rng.randint(3, 8))]


@pytest.mark.parametrize("seed", range(3))
def test_single_steps_and_batched_replay_with_a_straddling_pool(seed, monkeypatch):
    """findNextMerge / applyMerge one at a time (K1's lists and the stand-alone apply kernels), then restoreMerges in one device
    call (the replay mode of the loop kernel), against the literal restatement of core.ts."""
    monkeypatch.setenv("BPE_POOL_BASE", BASE_SMALL)
    from bpe_tokenizer_b200 import BPETokenizer

    docs = _docs(seed)
    lit, gpu = LiteralTokenizer(), BPETokenizer()
    for d in docs:
        lit.addToCorpus(d)
        gpu.addToCorpus(d)
    for step in range(400):
        m1 = lit.findNextMerge({})
        m2 = gpu.findNextMerge({})
        if m1 is None:
            assert m2 is None
            break
        assert (m2[0].index, m2[1].index, m2[2].weight) == (m1[0].index, m1[1].index, m1[2].weight), step
        lit.applyMerge(m1)
        gpu.applyMerge(m2)
        assert gpu.corpus_in_code == lit.corpus_in_code, step
    assert gpu.toJSON() == lit.toJSON()
    _crossed(gpu)
    log = [[a.code, b.code, c.original_weight] for a, b, c in lit.merge_tokens]
    batch, lit2 = BPETokenizer(), LiteralTokenizer()
    for d in docs:
        batch.addToCorpus(d)
        lit2.addToCorpus(d)
    batch.findNextMerge({})  # builds the index: the replay starts on a pool that straddles 2^32
    batch.restoreMerges(log)
    for line in log:
        lit2.restoreMerge(line)
    assert batch.toJSON() == lit2.toJSON() == lit.toJSON()
    assert batch.corpus_in_code == lit2.corpus_in_code
    _crossed(batch)
    for x in (gpu, batch):
        x.close()


def test_count_import_past_32_bits_is_a_domain_error(monkeypatch):
    """The sharded count import adds every rank's counts with 32-bit atomics: a sum past 2^32 - 1 must not wrap silently."""
    import ctypes as C

    import torch

    from bpe_tokenizer_b200 import BPETokenizer, _abi
    from bpe_tokenizer_b200.tokenizer import BpeError

    monkeypatch.setenv("BPE_POOL_BASE", BASE_SMALL)
    gpu = BPETokenizer()
    gpu.addToCorpus("ab" * 200)
    gpu.findNextMerge({})  # uploads the corpus and builds the index (no merge is applied)
    index = {t.chars: t.index for t in gpu.token_table}
    a, b = index["a"], index["b"]
    keys = torch.tensor([(a << 16) | b], dtype=torch.int32, device="cuda")
    cnts = torch.tensor([-1], dtype=torch.int32, device="cuda")  # 2^32 - 1 as u32, on top of the pair's own count
    rc = gpu._lib.bpe_mg_import_counts(gpu._h, C.c_void_p(keys.data_ptr()), C.c_void_p(cnts.data_ptr()), 1, 1)
    assert rc == _abi.BPE_E_DOMAIN, (rc, gpu._lib.bpe_last_error(gpu._h))
    assert b"2^32" in gpu._lib.bpe_last_error(gpu._h)
    with pytest.raises(BpeError):
        gpu._check(rc)
    _crossed(gpu)
    gpu.close()


def _sharded_cfg2(rank, world, port, base):
    import hashlib

    import torch
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    assert os.environ.get("BPE_POOL_BASE") == base
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from bpe_tokenizer_b200._abi import MERGE_DTYPE
        from bpe_tokenizer_b200.sharded import ShardedBPETokenizer, shard_bounds
        from bpe_tokenizer_b200.synth import first_appearance_ids, synth_corpus

        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cfg2_merge_log.json")) as f:
            golden = json.load(f)
        text, off = synth_corpus(10_000_000, seed=43)
        ids, alphabet = first_appearance_ids(text)
        gpu = ShardedBPETokenizer(rank)
        gpu.addToCorpus("".join(chr(c) for c in alphabet))
        gpu._pending = []
        for tk in gpu.token_table:
            tk.weight = tk.original_weight = 0
        b = shard_bounds(np.diff(off), world)
        lo, hi = b[rank], b[rank + 1]
        gpu.addDocuments(ids[off[lo]:off[hi]], off[lo:hi + 1] - off[lo], local_shard=True)
        assert gpu.mergeUntil({"max_iterations": golden["merges"]}) == golden["merges"]
        log = np.zeros(golden["merges"], dtype=MERGE_DTYPE)
        log["a"] = [a.index for a, _, _ in gpu.merge_tokens]
        log["b"] = [b_.index for _, b_, _ in gpu.merge_tokens]
        log["c"] = [c.index for _, _, c in gpu.merge_tokens]
        log["weight"] = [c.original_weight for _, _, c in gpu.merge_tokens]
        assert hashlib.sha1(log.tobytes()).hexdigest() == golden["sha1"], rank
        assert gpu.stats()["pool_used"] > TOP, rank
        gpu.close()
    finally:
        dist.destroy_process_group()


def test_sharded_cfg2_with_a_straddling_pool_world2(monkeypatch):
    import torch
    import torch.multiprocessing as mp

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    monkeypatch.setenv("BPE_POOL_BASE", BASE_MB)  # (set before the spawn: the workers inherit it)
    mp.spawn(_sharded_cfg2, args=(2, 29541, BASE_MB), nprocs=2, join=True)


def _sharded_large(rank, world, port, n_bytes, merges, out_path):
    """rank r of the 4 GB corpus sharded over `world` GPUs (bench.py's strong construction): writes rank 0's merge log."""
    import torch
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        import ctypes as C

        import sys

        sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
        from bench import alphabet_lut, synth
        from bpe_tokenizer_b200 import _abi
        from bpe_tokenizer_b200._abi import MERGE_DTYPE, p32, p64
        from bpe_tokenizer_b200.sharded import exchange_pair_counts, shard_bounds

        text, off = synth(None, n_bytes, 43)
        lut, alphabet = alphabet_lut(text)
        b = shard_bounds(np.diff(off), world)
        lo, hi = b[rank], b[rank + 1]
        ids = torch.from_numpy(lut[text[off[lo]:off[hi]]]).cuda()
        my_off = np.ascontiguousarray(off[lo:hi + 1] - off[lo])
        del text
        lib = _abi.load_library()
        h = C.c_void_p()
        assert lib.bpe_create(rank, C.byref(h)) == 0
        handle = C.create_string_buffer(64)
        assert lib.bpe_mg_init(h, rank, world, handle) == 0
        handles = [b""] * world
        dist.all_gather_object(handles, bytes(handle.raw))
        assert lib.bpe_mg_connect(h, b"".join(handles)) == 0
        dist.barrier()
        len16 = np.ones(len(alphabet), dtype=np.int32)
        assert lib.bpe_set_tokens(h, p32(len16), len(len16)) == 0
        assert lib.bpe_add_documents_dev(h, C.c_void_p(ids.data_ptr()), p64(my_off), len(my_off) - 1) == 0
        exchange_pair_counts(lib, h, rank, world, torch.device("cuda", rank))
        log = np.zeros(merges, dtype=MERGE_DTYPE)
        done = C.c_int64()
        rc = lib.bpe_merge_until(h, 2, 0, merges, log.ctypes.data_as(C.c_void_p), merges, C.byref(done))
        assert rc == 0, lib.bpe_last_error(h)
        if rank == 0:
            np.save(out_path, log[:done.value])
        lib.bpe_destroy(h)
    finally:
        dist.destroy_process_group()


def test_4gb_on_one_gpu_equals_the_same_corpus_on_four(tmp_path):
    """4.0 G characters (seed 43), 32 000 merges on ONE engine, whose pool passes 2^32 cells without any test hook, against the
    same corpus sharded over four ranks (1 GB shards, each rank's pool below 2^32 cells)."""
    import torch
    import torch.multiprocessing as mp

    if torch.cuda.device_count() < 4:
        pytest.skip("needs 4 GPUs")
    import sys

    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import large_corpus

    n_bytes, merges = 4_000_000_000, 32000
    res, log1 = large_corpus.run(n_bytes, merges)
    assert res["rc"] == 0 and res["merges_done"] == merges, res
    assert res["pool_used"] > TOP, res
    out = str(tmp_path / "log4.npy")
    mp.spawn(_sharded_large, args=(4, 29547, n_bytes, merges, out), nprocs=4, join=True)
    log4 = np.load(out)
    assert log4.shape == log1.shape and np.array_equal(log4, log1)
