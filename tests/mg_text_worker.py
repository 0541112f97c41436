"""Multi-GPU worker (one process per GPU): ShardedBPETokenizer.addTextBatch, in both sharding modes, then mergeUntil,
against the CPU oracles fed the same documents one addToCorpus call at a time.  Run by tests/test_multi_gpu_text.py
(torch.multiprocessing spawn) or directly:
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29512 tests/mg_text_worker.py"""
import os
import random
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def _merges(t):
    return [[a.index, b.index, c.weight] for a, b, c in t.merge_tokens]


def _rows(t):
    return [(tk.chars, tk.weight, tk.original_weight) for tk in t.token_table]


def _utf8(docs):
    parts = [d.encode("utf-8", "surrogatepass") for d in docs]
    off = np.zeros(len(parts) + 1, dtype=np.int64)
    np.cumsum([len(p) for p in parts], out=off[1:])
    return b"".join(parts), off


def _ingest(gpu, docs, rank, world, local_bounds):
    """local_bounds None: every rank passes every document; else rank r passes docs[local_bounds[r]:local_bounds[r + 1]]."""
    if local_bounds is None:
        gpu.addTextBatch(*_utf8(docs))
    else:
        gpu.addTextBatch(*_utf8(docs[local_bounds[rank]:local_bounds[rank + 1]]), local_shard=True)


def _compare(gpu, ref, docs, n_encode, tag):
    assert _rows(gpu) == _rows(ref), tag
    assert _merges(gpu) == _merges(ref), tag
    assert gpu.toJSON() == ref.toJSON(), tag
    ids, off = gpu.corpusIdsAllRanks()
    codes = (ids.astype(np.uint32) + 1).tolist()
    assert ["".join(map(chr, codes[off[d]:off[d + 1]])) for d in range(len(off) - 1)] == ref.corpus_in_code, tag
    sample = docs[:n_encode]
    out, out_off, _ = gpu.encodeTextBatch(*_utf8(sample), vector=False)
    got = [out[out_off[d]:out_off[d + 1]].tolist() for d in range(len(sample))]
    assert got == [[ord(c) - 1 for c in ref.encodeToCode(d)] for d in sample], tag


def run_checks(rank: int, world: int, fuzz_cases: int = 8, zipf_bytes: int = 300_000, zipf_merges: int = 300) -> None:
    import torch

    from bpe_tokenizer_b200.sharded import ShardedBPETokenizer
    from oracle import LiteralTokenizer
    from oracle.int_oracle import IntOracleTokenizer

    dev = torch.cuda.current_device()
    # ---- fuzz: small alphabets with 2- to 4-byte characters, lone surrogates, U+10FFFF, empty documents and shards ----
    alphabets = ["ab", "abé ", "a中\U0001F600 b", "xy\ud800\U0010FFFFé", "é", "abcde "]
    for case in range(fuzz_cases):
        rng = random.Random(7100 + case)
        alphabet = alphabets[case % len(alphabets)]
        n_docs = 1 if case == 1 else rng.randint(2, 9)  # case 1: one document, so one rank's shard is empty
        docs = ["".join(rng.choice(alphabet) for _ in range(rng.randint(0, rng.choice([20, 100, 400])))) for _ in range(n_docs)]
        if case == 2 and len(docs) > 1:
            docs[-1] = "Ω" + docs[-1]  # a character only the last rank sees, at its local position 0
        opts = {"min_weight": rng.choice([None, 2, 3]), "max_length": rng.choice([None, 5, 9]), "max_iterations": rng.choice([None, 40, 7])}
        cut = rng.randint(0, n_docs)  # local mode: an arbitrary split, empty ranges included
        for local_bounds in (None, [0] + [cut] * (world - 1) + [n_docs]):
            lit, gpu = LiteralTokenizer(), ShardedBPETokenizer(dev)
            for d in docs:
                lit.addToCorpus(d)
            _ingest(gpu, docs, rank, world, local_bounds)
            assert _rows(gpu) == _rows(lit), (case, rank, local_bounds)
            lit.mergeUntil(opts)
            gpu.mergeUntil(opts)
            _compare(gpu, lit, docs, 4, (case, rank, local_bounds))
            gpu.close()
    # ---- Zipf text with a few non-ASCII characters: merge log against the compiled oracle ----
    if zipf_bytes:
        from bpe_tokenizer_b200.sharded import shard_bounds
        from bpe_tokenizer_b200.synth import synth_corpus

        text, off = synth_corpus(zipf_bytes, seed=43)
        docs = [bytes(text[off[d]:off[d + 1]]).decode() for d in range(len(off) - 1)]
        rng = random.Random(5)
        for d in rng.sample(range(len(docs)), 30):
            docs[d] = docs[d] + rng.choice(["é", "中", "\U0001F600", "\ud800", "\U0010FFFF"])
        orc = IntOracleTokenizer()
        for d in docs:
            orc.addToCorpus(d)
        orc.mergeUntil({"max_iterations": zipf_merges})
        by_docs = shard_bounds([1] * len(docs), world)  # local mode: balanced by document count, not by bytes
        for local_bounds in (None, by_docs):
            gpu = ShardedBPETokenizer(dev)
            _ingest(gpu, docs, rank, world, local_bounds)
            n = gpu.mergeUntil({"max_iterations": zipf_merges})
            assert n == zipf_merges, n
            _compare(gpu, orc, docs, 200, ("zipf", rank, local_bounds))
            if rank == 0:
                print("mg text parity ok: world %d, %d merges on %d B, local_shard=%s" % (world, n, zipf_bytes, local_bounds is not None), flush=True)
            gpu.close()


def _spawn_entry(rank: int, world: int, port: int, kwargs: dict) -> None:
    import torch
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        run_checks(rank, world, **kwargs)
    finally:
        dist.destroy_process_group()


if __name__ == "__main__":
    import torch
    import torch.distributed as dist

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    run_checks(rank, world)
    dist.destroy_process_group()
