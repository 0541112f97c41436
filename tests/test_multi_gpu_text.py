"""GPU, >= 2 devices: ShardedBPETokenizer.addTextBatch (each rank decodes its shard, the ranks agree on one global
first-appearance order of the new characters) followed by mergeUntil, against the CPU oracles.  Skipped on
single-GPU boxes."""
import pytest

pytestmark = pytest.mark.gpu


def test_sharded_text_ingest_matches_oracle_world2():
    import torch
    import torch.multiprocessing as mp

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import mg_text_worker

    mp.spawn(mg_text_worker._spawn_entry, args=(2, 29535, {"fuzz_cases": 8, "zipf_bytes": 300_000, "zipf_merges": 300}), nprocs=2, join=True)
