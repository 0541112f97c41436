"""Sharded training from raw UTF-8 text against the same training from host ids, in one run:
    python -m torch.distributed.run --nproc-per-node N tools/mg_text_bench.py [--workload cfg3|cfg3w] [--steps K] [--warmup W]

cfg3 (strong scaling): every rank generates the 1 GB text (seed 43) and passes its pinned, token-balanced shard with
local_shard semantics.  cfg3w (weak scaling): every rank generates its own 1 GB shard (seed 43 + 1000 * rank), the
corpus is their concatenation.  A step alternates the two ways in:

* text: bpe_add_text_stage on every rank, the exchange of the new characters (sharded.text_ingest_collective, the
  protocol ShardedBPETokenizer.addTextBatch runs), bpe_add_text_commit, then K1 + the pair-count exchange, mergeUntil;
* ids: bpe_add_documents from pinned host ids (4 B per character), K1 + exchange, mergeUntil -- bench.py's e2e step.

Phase times are host clocks around calls that end in a device synchronise, the maximum over the ranks, in ms; the
step time runs from a barrier to the end of mergeUntil.  The text path's merge-log SHA-1 must equal the golden for
cfg3 and the id path's for cfg3w.  Rank 0 prints one JSON line per timed step and a summary line with the card's
name and power limit (read, not set)."""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import bench  # noqa: E402
from bpe_tokenizer_b200 import _abi  # noqa: E402
from bpe_tokenizer_b200._abi import MERGE_DTYPE, p32, p64  # noqa: E402
from bpe_tokenizer_b200.sharded import exchange_pair_counts, shard_bounds, text_ingest_collective  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=10).stdout
        return q.strip().splitlines()
    except Exception as ex:
        return ["unknown: %r" % (ex,)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cfg3", choices=["cfg3", "cfg3w", "tiny", "tinyw"])
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")
        dist.init_process_group("nccl", device_id=dev)
    train_bytes, merges, _ = bench.WORKLOADS[args.workload]
    weak = args.workload.endswith("w")
    lib = _abi.load_library()

    # ---- inputs: this rank's shard as UTF-8 bytes and, for the id path, as token ids ----
    if weak:
        head, _ = bench.synth(None, 1_000_000, bench.TRAIN_SEED)
        lut, alphabet = bench.alphabet_lut(head)  # (bench.py's id path: rank 0's first megabyte holds the alphabet)
        text, off = bench.synth(None, train_bytes, bench.TRAIN_SEED + 1000 * rank)
        assert (lut[np.unique(text)] >= 0).all(), "shard uses a character outside the head's alphabet"
        lo, hi = 0, len(off) - 1
    else:
        text, off = bench.synth(None, train_bytes, bench.TRAIN_SEED)
        lut, alphabet = bench.alphabet_lut(text)
        b = shard_bounds(np.diff(off), world)
        lo, hi = b[rank], b[rank + 1]
    text_host = torch.from_numpy(np.ascontiguousarray(text[off[lo]:off[hi]])).pin_memory()
    ids_host = torch.from_numpy(lut[text[off[lo]:off[hi]]]).pin_memory()
    off_host = np.ascontiguousarray(off[lo:hi + 1] - off[lo])
    n_docs = len(off_host) - 1
    n0_total = int(text.size) if not weak else None
    del text
    if weak:
        t = torch.tensor([int(text_host.numel())], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(t)
        n0_total = int(t.item())

    h = C.c_void_p()
    assert lib.bpe_create(local, C.byref(h)) == 0
    if world > 1:
        handle = C.create_string_buffer(64)
        assert lib.bpe_mg_init(h, rank, world, handle) == 0, lib.bpe_last_error(h)
        hs = [b""] * world
        dist.all_gather_object(hs, bytes(handle.raw))
        assert lib.bpe_mg_connect(h, b"".join(hs)) == 0, lib.bpe_last_error(h)
        dist.barrier()
    len16 = np.ones(len(alphabet), dtype=np.int32)
    log = np.zeros(merges, dtype=MERGE_DTYPE)
    n_done = C.c_int64()

    def check(rc):
        if rc != 0:
            raise _abi.BpeError(rc, lib.bpe_last_error(h).decode())

    def now():
        return time.perf_counter() * 1e3

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def train(t):
        a = now()
        exchange_pair_counts(lib, h, rank, world, dev)  # K1 (the index build) + the sum of the shards' pair histograms
        torch.cuda.synchronize()
        b_ = now()
        check(lib.bpe_merge_until(h, 2, 0, merges, log.ctypes.data_as(C.c_void_p), merges, C.byref(n_done)))
        t["k1_exchange"], t["merge_until"] = b_ - a, now() - b_
        return hashlib.sha1(log[: n_done.value].tobytes()).hexdigest()

    def text_step():
        check(lib.bpe_clear_corpus(h))
        check(lib.bpe_set_tokens(h, None, 0))
        check(lib.bpe_set_chars(h, None, None, 0))
        check(lib.bpe_load_merges(h, None, 0))
        t = {}
        cps = np.zeros(1 << 16, dtype=np.int32)
        pos = np.zeros(1 << 16, dtype=np.int64)
        n = C.c_int32()

        def stage():
            a = now()
            check(lib.bpe_add_text_stage(h, C.cast(text_host.data_ptr(), _abi.u8p), p64(off_host), n_docs, p32(cps), p64(pos), cps.size, C.byref(n)))
            t["stage"] = now() - a
            return cps[: n.value], pos[: n.value]

        def commit(new):
            a = now()
            c = np.asarray(new, dtype=np.int32)
            check(lib.bpe_add_text_commit(h, p32(c), c.size, None, 0))
            t["commit"] = now() - a
            return np.zeros(c.size, dtype=np.int64)  # (the benchmark needs no character counts on the host)

        sync_all()
        t0 = now()
        new, _ = text_ingest_collective(stage, commit, 0, world, None, dev)
        t["exchange"] = now() - t0 - t["stage"] - t["commit"]
        assert new == list(alphabet), "the text path found another alphabet"
        sha = train(t)
        t["step"] = now() - t0
        return t, sha

    def id_step():
        check(lib.bpe_clear_corpus(h))
        check(lib.bpe_set_tokens(h, p32(len16), len(len16)))
        check(lib.bpe_load_merges(h, None, 0))
        t = {}
        sync_all()
        t0 = now()
        check(lib.bpe_add_documents(h, C.cast(ids_host.data_ptr(), _abi.i32p), p64(off_host), n_docs))
        t["ingest"] = now() - t0
        sha = train(t)
        t["step"] = now() - t0
        return t, sha

    def max_over_ranks(t):
        if world == 1:
            return t
        keys = sorted(t)
        v = torch.tensor([t[k] for k in keys], dtype=torch.float64, device=dev)
        dist.all_reduce(v, op=dist.ReduceOp.MAX)
        return dict(zip(keys, v.tolist()))

    for _ in range(args.warmup):
        text_step()
        id_step()
    golden = bench.merge_log_golden(args.workload, n0_total, merges)
    rows = []
    for step in range(args.steps):
        tt, sha_t = text_step()
        ti, sha_i = id_step()
        tt, ti = max_over_ranks(tt), max_over_ranks(ti)
        want = golden["sha1"] if golden else sha_i
        ok = sha_t == want and (golden is None or sha_i == want)
        rows.append((tt, ti, ok))
        if rank == 0:
            print(json.dumps({"step": step, "world": world, "workload": args.workload, "merges": n_done.value,
                              "text_ms": {k: round(v, 2) for k, v in tt.items()}, "ids_ms": {k: round(v, 2) for k, v in ti.items()},
                              "text_sha1": sha_t, "ids_sha1": sha_i, "checked_against": "golden " + golden["file"] if golden else "id path",
                              "sha1_ok": ok}), flush=True)
        assert ok, "merge log differs: text %s, ids %s, want %s" % (sha_t, sha_i, want)
    if rank == 0:
        med = lambda xs: float(np.median(xs))  # noqa: E731
        text_ms, ids_ms = [r[0]["step"] for r in rows], [r[1]["step"] for r in rows]
        print(json.dumps({"summary": True, "world": world, "workload": args.workload, "corpus_bytes": n0_total, "merges": merges,
                          "card": card(), "steps": args.steps, "warmup": args.warmup,
                          "e2e_text_merges_per_s": [round(merges / (x / 1e3)) for x in text_ms],
                          "e2e_ids_merges_per_s": [round(merges / (x / 1e3)) for x in ids_ms],
                          "median_text_ms": {k: round(med([r[0][k] for r in rows]), 2) for k in rows[0][0]},
                          "median_ids_ms": {k: round(med([r[1][k] for r in rows]), 2) for k in rows[0][1]}}), flush=True)
    lib.bpe_destroy(h)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
