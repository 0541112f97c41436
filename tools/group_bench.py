"""A device group (bpe_create_group: N GPUs driven from one process) against one process per GPU (tools/mg_bench.py), in one run:
    python tools/group_bench.py [--sizes 2,4,8] [--rounds 2] [--reps 2]

Training, cfg3 (1 GB of synthetic text, seed 43, 32 000 merges).  For every N the two set-ups alternate, `--rounds` times:
* group: bpe_add_documents from pinned host ids (split over the members), the in-process pair-count exchange (triggered by a
  sizing bpe_pair_counts call), then bpe_merge_until -- one warm-up step, then `--reps` timed steps;
* mg_bench.py under torch.distributed.run with N processes: bpe_add_documents_dev, the NCCL count exchange, bpe_merge_until --
  REPS = reps + 1 steps, the first one is the warm-up.
The figure is the host clock around bpe_merge_until alone (it ends in a device synchronise on every member), as mg_bench.py
times it; every line carries the merge-log SHA-1, which must be the CPU oracle's (tests/golden/cfg3_full_check.json).

Encode, cfg4 (the 1 GB encode text, seed 44, with the 32 000 merges just learned) on the largest group: bpe_encode_batch from
pinned host ids and bpe_encode_text_batch from pinned UTF-8 bytes into a pinned output, GB/s of input characters, host clock
around the call; the output is checked against the CPU restatement's golden (bench.full_encode_check).

--share-device puts every member on GPU 0 (BPE_GROUP_SHARE_DEVICE=1, each member with its share of the SMs) and skips mg_bench.py:
on a host with one GPU it runs the group end to end at full size and checks its results; its times say nothing about N GPUs.

One JSON line per measurement; the first line holds the cards' names and power limits (read, not set)."""
import argparse
import ctypes as C
import hashlib
import json
import os
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from bpe_tokenizer_b200 import _abi  # noqa: E402
from bpe_tokenizer_b200._abi import MERGE_DTYPE, p32, p64  # noqa: E402

GOLDEN_SHA1 = "add92aa1a96c276f03b63e3a952370ef04cb60f0"


def emit(d):
    print(json.dumps(d), flush=True)


def cards():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=10).stdout
        return q.strip().splitlines()
    except Exception as ex:
        return ["unknown: %r" % (ex,)]


def mg_bench(n, reps, size, merges):
    env = dict(os.environ, SIZE=str(size), MERGES=str(merges), REPS=str(reps + 1), NCCL_DEBUG="WARN")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr", "127.0.0.1",
           "--master-port", "29541", os.path.join(ROOT, "tools", "mg_bench.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=ROOT)
    pat = re.compile(r"rep (\d+) rc (-?\d+) world (\d+) ingest\+K1\+exchange ([\d.]+) ms merge_until ([\d.]+) ms merges (\d+) sha (\w+)")
    got = [m.groups() for m in pat.finditer(r.stdout)]
    if r.returncode != 0 or not got:
        emit({"setup": "processes", "n": n, "failed": r.returncode, "tail": (r.stdout + r.stderr)[-2000:]})
    for rep, rc, world, ingest, mu, done, sha in got:
        if int(rep) == 0:
            continue  # warm-up
        emit({"setup": "processes", "n": int(world), "rc": int(rc), "ingest_k1_exchange_ms": float(ingest), "merge_until_ms": float(mu),
              "merges": int(done), "merges_per_s": int(done) / (float(mu) / 1e3), "sha1_12": sha, "sha1_is_golden": GOLDEN_SHA1.startswith(sha)})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="2,4,8")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--size", type=int, default=1_000_000_000)
    ap.add_argument("--merges", type=int, default=32000)
    ap.add_argument("--encode-bytes", type=int, default=1_000_000_000)
    ap.add_argument("--share-device", action="store_true")
    args = ap.parse_args()
    have = torch.cuda.device_count()
    if args.share_device:
        os.environ["BPE_GROUP_SHARE_DEVICE"] = "1"
    sizes = [n for n in (int(s) for s in args.sizes.split(",")) if 2 <= n <= (8 if args.share_device else have)]
    setup = "group sharing GPU 0" if args.share_device else "group"
    emit({"cards": cards(), "devices": have, "sizes": sizes, "setup": setup})
    if not sizes:
        raise SystemExit("needs at least 2 GPUs")
    lib = _abi.load_library()
    text, off = bench.synth(None, args.size, bench.TRAIN_SEED)
    lut, alphabet = bench.alphabet_lut(text)
    ids_host = torch.from_numpy(lut[text]).pin_memory()
    n_docs = len(off) - 1
    del text
    len16 = np.ones(len(alphabet), dtype=np.int32)
    log = np.zeros(args.merges, dtype=MERGE_DTYPE)
    nd, npairs = C.c_int64(), C.c_int64()

    def check(h, rc):
        if rc != 0:
            raise RuntimeError("bpe error %d: %s" % (rc, lib.bpe_last_error(h).decode()))

    def train(h):
        check(h, lib.bpe_clear_corpus(h))
        check(h, lib.bpe_set_tokens(h, p32(len16), len(len16)))
        check(h, lib.bpe_load_merges(h, None, 0))
        t0 = time.time()
        check(h, lib.bpe_add_documents(h, C.cast(ids_host.data_ptr(), _abi.i32p), p64(off), n_docs))
        rc = lib.bpe_pair_counts(h, None, None, None, 0, C.byref(npairs))  # sums the histograms; BPE_E_CAPACITY = the size answer
        if rc not in (_abi.BPE_OK, _abi.BPE_E_CAPACITY):
            check(h, rc)
        t1 = time.time()
        check(h, lib.bpe_merge_until(h, 2, 0, args.merges, log.ctypes.data_as(C.c_void_p), args.merges, C.byref(nd)))
        t2 = time.time()
        return (t1 - t0) * 1e3, (t2 - t1) * 1e3

    def group(n):
        h = C.c_void_p()
        devs = (C.c_int * n)(*([0] * n if args.share_device else range(n)))
        assert lib.bpe_create_group(devs, n, C.byref(h)) == 0, "bpe_create_group failed"
        return h

    for rnd in range(args.rounds):
        for n in sizes:
            h = group(n)
            train(h)  # warm-up
            for _ in range(args.reps):
                ingest, mu = train(h)
                sha = hashlib.sha1(log[:nd.value].tobytes()).hexdigest()
                emit({"setup": setup, "n": n, "round": rnd, "ingest_k1_exchange_ms": ingest, "merge_until_ms": mu, "merges": nd.value,
                      "merges_per_s": nd.value / (mu / 1e3), "sha1_12": sha[:12], "sha1_is_golden": sha == GOLDEN_SHA1})
            lib.bpe_destroy(h)
            if not args.share_device:
                mg_bench(n, args.reps, args.size, args.merges)

    # ---- encode on the largest group, with the merges it learns here ----
    n = sizes[-1]
    h = group(n)
    train(h)
    done = nd.value
    del ids_host
    text2, off2 = bench.synth(None, args.encode_bytes, bench.ENCODE_SEED)
    chars, n_docs2 = int(text2.size), len(off2) - 1
    text2_host = torch.from_numpy(text2).pin_memory()
    ids2_host = torch.from_numpy(lut[text2]).pin_memory()
    del text2
    out_host = torch.empty(chars, dtype=torch.int32).pin_memory()
    ooff = np.zeros(n_docs2 + 1, dtype=np.int64)
    tvi = np.arange(len(alphabet) + done, dtype=np.int32)  # raw-index-equivalent map without holes, as bench.py
    cps = np.array(alphabet, dtype=np.int32)
    check(h, lib.bpe_set_chars(h, p32(cps), p32(np.arange(len(alphabet), dtype=np.int32)), len(alphabet)))
    n_out = C.c_int64()

    def enc_ids():
        check(h, lib.bpe_encode_batch(h, C.cast(ids2_host.data_ptr(), _abi.i32p), p64(off2), n_docs2, p32(tvi), len(tvi),
                                      C.cast(out_host.data_ptr(), _abi.i32p), chars, p64(ooff), None, C.byref(n_out)))

    def enc_text():
        check(h, lib.bpe_encode_text_batch(h, C.cast(text2_host.data_ptr(), _abi.u8p), p64(off2), n_docs2, p32(tvi), len(tvi),
                                           C.cast(out_host.data_ptr(), _abi.i32p), chars, p64(ooff), None, C.byref(n_out), None, None))

    for name, fn in (("host ids", enc_ids), ("raw text", enc_text)):
        fn()  # warm-up
        check_out = bench.full_encode_check(out_host.numpy()[: n_out.value], ooff, chars, done,
                                            table_is_golden=hashlib.sha1(log[:done].tobytes()).hexdigest() == GOLDEN_SHA1)
        for _ in range(args.reps + 1):
            t0 = time.time()
            fn()
            ms = (time.time() - t0) * 1e3
            emit({"setup": setup, "n": n, "encode_from": name, "chars": chars, "docs": n_docs2, "tokens_out": n_out.value, "ms": ms,
                  "gb_per_s": chars / (ms / 1e3) / 1e9, "output": check_out})
    lib.bpe_destroy(h)


if __name__ == "__main__":
    main()
