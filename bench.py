#!/usr/bin/env python
"""bench.py -- the reference's headline path on B200: `mergeUntil` merges/s and `encodeToVector` GB/s on
seeded Zipf text (BASELINE.json), through the C ABI of include/bpe_b200.h.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA engine
  python bench.py --impl reference --steps K --warmup W    # CPU restatement of core.ts (Node is not in the image)

One step = one full pass of the hot path over the workload: ingest the corpus (addToCorpus -> K1 pair
histogram + occurrence lists) and run mergeUntil to the configured number of merges.  `value` is measured
with the corpus ids already resident in HBM; `e2e` runs the same step from pinned HOST buffers through
bpe_add_documents / bpe_merge_until (H2D copy and log read-back inside the timed region).  The encode leg
(bpe_encode_batch*) is timed the same way and reported under "encode".

--dump-outputs DIR writes what the last timed steps returned, so that two builds can be compared output for output
on the same seeded inputs: merge_log.npy (float64 [merges, 4]: a, b, c, weight of bpe_merge_until) and, on one GPU, a
seeded sample of the device-resident encode (encode_docs.npy, encode_doc_lengths.npy: float64; encode_tokens.npy: float32).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

_OUT = sys.stdout

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the tree as it found it (it may be read-only)

WORKLOADS = {
    # name: (train bytes, merges, encode bytes)
    "cfg2": (10_000_000, 4000, 10_000_000),
    "cfg3": (1_000_000_000, 32000, 1_000_000_000),
    # weak scaling, reported BESIDE cfg3 (SURVEY 8(f) row 4: a corpus larger than one GPU's HBM lives as document shards on N GPUs):
    # every rank generates its own 1 GB shard (seed 43 + 1000 * rank; rank 0's is cfg3's corpus), the corpus is their concatenation
    "cfg3w": (1_000_000_000, 32000, 1_000_000_000),
    "tiny": (200_000, 200, 200_000),
    "tinyw": (200_000, 200, 200_000),
}
WORD_SEED, TRAIN_SEED, ENCODE_SEED, VOCAB = 42, 43, 44, 50000
# --dump-outputs: documents of the encode text drawn with DUMP_SEED, as many as fit in DUMP_CHARS characters (a character
# encodes to at most one token, so the sample stays under 32 MB of float32 and is the same set of documents for every build)
DUMP_SEED, DUMP_CHARS = 45, 8_000_000


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def synth(lib, target, seed):
    """Seeded Zipf text from the stand-alone generator library (libbpe_synth.so: host code only).  `lib` is unused and kept
    for the tools that pass it: neither arm needs the CUDA product library to make its input."""
    from bpe_tokenizer_b200.synth import native_corpus

    return native_corpus(target, seed, VOCAB, WORD_SEED)


def alphabet_lut(text):
    """first-appearance order, as addToCorpus assigns indices (core.ts:186-199)"""
    first = np.full(256, np.iinfo(np.int64).max, dtype=np.int64)
    step = 1 << 24
    seen = np.zeros(256, dtype=bool)
    for s in range(0, text.size, step):
        chunk = text[s:s + step]
        vals, idx = np.unique(chunk, return_index=True)
        for v, i in zip(vals.tolist(), idx.tolist()):
            if not seen[v]:
                seen[v] = True
                first[v] = s + i
        if seen.sum() >= 29 and s > 0:
            break
    order = np.argsort(first, kind="stable")[: int(seen.sum())]
    lut = np.full(256, -1, dtype=np.int32)
    lut[order] = np.arange(order.size, dtype=np.int32)
    return lut, [int(x) for x in order]


class ClockSampler:
    def __init__(self, device_index):
        self.idx = device_index
        self.samples = []
        self.reasons = set()
        self._stop = threading.Event()
        self._th = None

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append((float(out[0]), float(out[1])))
                for n, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self._th = threading.Thread(target=self._run, daemon=True)
        self._th.start()

    def stop(self):
        self._stop.set()
        if self._th:
            self._th.join(timeout=6)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": sorted(self.reasons)}
        sm = sorted(s[0] for s in self.samples)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(s[1] for s in self.samples), "reasons": sorted(self.reasons), "samples": len(sm)}


def scan_equivalent_bytes(n0, weights):
    """SURVEY.md 8(d): the reference algorithm reads N_t ids to count, reads N_t and writes N_{t+1} to replace."""
    n, total = int(n0), 0
    for w in weights:
        total += 4 * (2 * n + (n - int(w)))
        n -= int(w)
    return total


# ------------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist

    from bpe_tokenizer_b200 import _abi
    from bpe_tokenizer_b200._abi import MERGE_DTYPE, bpe_stats, p32, p64

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")  # (keeps NCCL's version banner off stdout: one JSON line only)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = _abi.load_library()
    train_bytes, merges, encode_bytes = WORKLOADS[args.workload]
    if args.merges:
        merges = args.merges
    peak, peak_src = measured_peak()

    # ---- synthetic inputs: ONE corpus (BASELINE.json config), sharded by document over the ranks (strong scaling) ----
    # every rank generates the same seeded text and keeps a contiguous, token-balanced range of its documents
    # (ranks in document order: global scan order = (rank, local position), see bpe_tokenizer_b200/sharded.py).
    from bpe_tokenizer_b200.sharded import exchange_pair_counts, shard_bounds

    t0 = time.time()
    weak = args.workload.endswith("w")
    if weak:
        # token indices follow first appearance in the concatenated corpus = in rank 0's shard; its first megabyte holds the
        # whole alphabet (checked), so every rank derives the same table without seeing rank 0's gigabyte
        head, _ = synth(lib, 1_000_000, TRAIN_SEED)
        lut, alphabet = alphabet_lut(head)
        text, off = synth(lib, train_bytes, TRAIN_SEED + 1000 * rank)
        assert (lut[np.unique(text)] >= 0).all(), "shard uses a character outside the head's alphabet"
        lo, hi = 0, len(off) - 1
        tot = torch.tensor([int(text.size), len(off) - 1], device="cuda", dtype=torch.int64)
        if world > 1:
            dist.all_reduce(tot)
        n0_total, n_docs_total = int(tot[0].item()), int(tot[1].item())
    else:
        text, off = synth(lib, train_bytes, TRAIN_SEED)
        lut, alphabet = alphabet_lut(text)
        n0_total, n_docs_total = int(text.size), len(off) - 1
        b = shard_bounds(np.diff(off), world)
        lo, hi = b[rank], b[rank + 1]
    ids_host = torch.from_numpy(lut[text[off[lo]:off[hi]]]).pin_memory()
    # the same shard as raw UTF-8 bytes (ASCII: 1 B per character), for the end-to-end step that enters through the text front end
    text_host = torch.from_numpy(np.ascontiguousarray(text[off[lo]:off[hi]])).pin_memory() if world == 1 else None
    off_host = np.ascontiguousarray(off[lo:hi + 1] - off[lo])
    del text
    text2, off2 = synth(lib, encode_bytes, ENCODE_SEED)
    c2_total = int(text2.size)
    b2 = shard_bounds(np.diff(off2), world)
    lo2, hi2 = b2[rank], b2[rank + 1]
    text2_host = torch.from_numpy(np.ascontiguousarray(text2[off2[lo2]:off2[hi2]])).pin_memory()  # the raw UTF-8 bytes (ASCII here)
    ids2_host = torch.from_numpy(lut[text2[off2[lo2]:off2[hi2]]]).pin_memory()
    off2 = np.ascontiguousarray(off2[lo2:hi2 + 1] - off2[lo2])
    del text2
    n0, n_docs = ids_host.numel(), len(off_host) - 1
    c2, n_docs2 = ids2_host.numel(), len(off2) - 1
    gen_s = time.time() - t0
    ids_dev = ids_host.cuda(non_blocking=True)
    ids2_dev = ids2_host.cuda(non_blocking=True)
    off2_dev = torch.from_numpy(off2).cuda()
    max_doc2 = int(np.max(np.diff(off2))) if n_docs2 else 0
    torch.cuda.synchronize()

    h = C.c_void_p()
    assert lib.bpe_create(local, C.byref(h)) == 0, "bpe_create failed"
    stream = torch.cuda.current_stream()
    assert lib.bpe_set_stream(h, C.c_void_p(stream.cuda_stream)) == 0
    dev = torch.device("cuda", local)
    if world > 1:  # mailboxes of the sharded merge loop: exchange the cudaIpc handles once
        handle = C.create_string_buffer(64)
        assert lib.bpe_mg_init(h, rank, world, handle) == 0, lib.bpe_last_error(h)
        handles = [b""] * world
        dist.all_gather_object(handles, bytes(handle.raw))
        assert lib.bpe_mg_connect(h, b"".join(handles)) == 0, lib.bpe_last_error(h)
        dist.barrier()
    len16 = np.ones(len(alphabet), dtype=np.int32)
    log = np.zeros(merges, dtype=MERGE_DTYPE)
    n_done = C.c_int64()

    def check(rc):
        if rc != 0:
            raise RuntimeError("bpe error %d: %s" % (rc, lib.bpe_last_error(h).decode()))

    def reset():
        check(lib.bpe_clear_corpus(h))
        check(lib.bpe_set_tokens(h, p32(len16), len(len16)))
        check(lib.bpe_load_merges(h, None, 0))

    def train_step(from_host: bool):
        reset()
        if from_host:
            check(lib.bpe_add_documents(h, C.cast(ids_host.data_ptr(), _abi.i32p), p64(off_host), n_docs))
        else:
            check(lib.bpe_add_documents_dev(h, C.c_void_p(ids_dev.data_ptr()), p64(off_host), n_docs))
        exchange_pair_counts(lib, h, rank, world, dev)  # world > 1: K1 histograms of all shards summed (NCCL all-gather)
        check(lib.bpe_merge_until(h, 2, 0, merges, log.ctypes.data_as(C.c_void_p), merges, C.byref(n_done)))
        return n_done.value

    def stats():
        s = bpe_stats()
        check(lib.bpe_get_stats(h, C.byref(s)))
        return s

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            tms = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            ms = float(tms.item())
        return ms

    # ---- train: device-resident value ---------------------------------------------------------------
    for _ in range(args.warmup):
        done = train_step(False)
    l0 = stats().kernel_launches
    sampler = ClockSampler(local)
    sampler.start()
    ms_train = timed(lambda: train_step(False), args.steps)
    l1 = stats().kernel_launches
    done = n_done.value
    weights = log["weight"][:done].copy()
    dumps = {}
    if args.dump_outputs:  # (the later steps overwrite `log`)
        dumps["merge_log"] = np.stack([log[f][:done].astype(np.float64) for f in ("a", "b", "c", "weight")], axis=1)
    k1_ms = None
    s_before = stats()
    # K1 alone (ingest + histogram + lists), for its own roofline line
    reset()
    check(lib.bpe_add_documents_dev(h, C.c_void_p(ids_dev.data_ptr()), p64(off_host), n_docs))
    if world == 1:
        m, found = _abi.bpe_merge(), C.c_int()
        check(lib.bpe_find_next_merge(h, 2, 0, C.byref(m), C.byref(found)))  # builds the index
    else:  # (single steps are refused on a sharded engine) sizing the export builds this shard's index
        npairs = C.c_int64()
        check(lib.bpe_mg_export_counts(h, None, None, 0, C.byref(npairs)))
    k1_ms = stats().ms_index_build - s_before.ms_index_build
    if world > 1:  # every rank must hold the same merge log
        import hashlib

        digest = hashlib.sha1(log[:done].tobytes()).hexdigest()
        digests = [None] * world
        dist.all_gather_object(digests, digest)
        assert all(d == digest for d in digests), "ranks disagree on the merge log: %r" % (digests,)
    import hashlib

    log_sha1_early = hashlib.sha1(log[:done].tobytes()).hexdigest()
    # ---- train: end to end from host buffers ----------------------------------------------------------
    e2e_steps = max(1, args.steps)
    train_step(True)
    ms_train_e2e = timed(lambda: train_step(True), e2e_steps)

    # ... and from raw text, the form the reference's addToCorpus takes (core.ts:182-207): UTF-8 bytes in, code point -> token index,
    # first-appearance token creation and weights on the device (bpe_add_text), then the same mergeUntil.  One GPU only (a sharded
    # engine takes ids).  The merge log must be the one the id path produced.
    e2e_text = None
    if world == 1:
        try:
            new_cps = np.zeros(1 << 16, dtype=np.int32)
            n_new = C.c_int32()

            def train_step_text():
                check(lib.bpe_clear_corpus(h))
                check(lib.bpe_set_tokens(h, None, 0))
                check(lib.bpe_set_chars(h, None, None, 0))
                check(lib.bpe_load_merges(h, None, 0))
                check(lib.bpe_add_text(h, C.cast(text_host.data_ptr(), _abi.u8p), p64(off_host), n_docs, p32(new_cps), new_cps.size, C.byref(n_new), None, 0))
                assert n_new.value == len(alphabet) and new_cps[: n_new.value].tolist() == list(alphabet), "text front end found other characters"
                check(lib.bpe_set_tokens(h, p32(len16), len(len16)))
                check(lib.bpe_merge_until(h, 2, 0, merges, log.ctypes.data_as(C.c_void_p), merges, C.byref(n_done)))

            train_step_text()
            assert n_done.value == done and hashlib.sha1(log[:done].tobytes()).hexdigest() == log_sha1_early, "text path learned another merge log"
            ms_text = timed(train_step_text, e2e_steps)
            e2e_text = {"value": done * e2e_steps / (ms_text / 1e3), "unit": "merges/s", "h2d_bytes_per_step": int(text_host.numel() + off_host.nbytes),
                        "d2h_bytes_per_step": int(done * MERGE_DTYPE.itemsize), "ms_per_step": ms_text / e2e_steps,
                        "note": "bpe_add_text + bpe_merge_until: UTF-8 bytes in (1 B/char), characters -> token indices in first-appearance order on the device; same merge log"}
        except Exception as ex:  # never take the line down
            e2e_text = {"failed": repr(ex)}

    # ---- encode with the table just learned -------------------------------------------------------------
    tvi = np.arange(len(alphabet) + done, dtype=np.int32)  # raw-index-equivalent map without holes
    tvi_dev = torch.from_numpy(tvi).cuda()
    out_dev = torch.empty(max(c2, 1), dtype=torch.int32, device="cuda")
    ooff_dev = torch.empty(n_docs2 + 1, dtype=torch.int64, device="cuda")
    n_out = C.c_int64()

    def encode_step_dev():
        check(lib.bpe_encode_batch_dev(h, C.c_void_p(ids2_dev.data_ptr()), C.c_void_p(off2_dev.data_ptr()), n_docs2, c2, max_doc2,
                                       C.c_void_p(tvi_dev.data_ptr()), len(tvi), C.c_void_p(out_dev.data_ptr()),
                                       C.c_void_p(ooff_dev.data_ptr()), None, C.byref(n_out)))

    out_host = torch.empty(max(c2, 1), dtype=torch.int32).pin_memory()
    ooff_host = np.zeros(n_docs2 + 1, dtype=np.int64)

    def encode_step_host():
        check(lib.bpe_encode_batch(h, C.cast(ids2_host.data_ptr(), _abi.i32p), p64(off2), n_docs2, p32(tvi), len(tvi),
                                   C.cast(out_host.data_ptr(), _abi.i32p), out_host.numel(), p64(ooff_host), None, C.byref(n_out)))

    for _ in range(args.warmup):
        encode_step_dev()
    le0 = stats().kernel_launches
    ms_enc = timed(encode_step_dev, args.steps)
    le1 = stats().kernel_launches
    k_out = n_out.value
    if args.dump_outputs and world == 1:  # (at N > 1 every rank holds only its shard of the vectors)
        dumps.update(encode_sample(out_dev[:k_out].cpu().numpy(), ooff_dev.cpu().numpy(), off2))
    enc_kernel_ms = stats().ms_encode
    encode_step_host()
    ms_enc_e2e = timed(encode_step_host, e2e_steps)

    # text in (UTF-8 bytes, 1 B/char over PCIe), vectors out: char -> index on the device (csrc/text_kernels.cuh)
    cps = np.array(alphabet, dtype=np.int32)
    check(lib.bpe_set_chars(h, p32(cps), p32(np.arange(len(alphabet), dtype=np.int32)), len(alphabet)))

    def encode_step_text():
        check(lib.bpe_encode_text_batch(h, C.cast(text2_host.data_ptr(), _abi.u8p), p64(off2), n_docs2, p32(tvi), len(tvi),
                                        C.cast(out_host.data_ptr(), _abi.i32p), out_host.numel(), p64(ooff_host), None, C.byref(n_out), None, None))

    encode_step_text()
    assert n_out.value == k_out, "text front end disagrees with the id path"
    ms_enc_text = timed(encode_step_text, e2e_steps)
    clocks = sampler.stop()

    # ---- aggregate over ranks -----------------------------------------------------------------------------
    def allsum(x):
        if world == 1:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t)
        return float(t.item())

    def max_over_ranks(x):
        t = torch.tensor([float(x)], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    import hashlib

    log_sha1 = hashlib.sha1(log[:done].tobytes()).hexdigest()
    golden_log = merge_log_golden(args.workload, n0_total, done)
    if golden_log is not None:  # a wrong merge sequence must not print a throughput
        assert log_sha1 == golden_log["sha1"], "merge log differs from the CPU oracle's (%s vs %s)" % (log_sha1, golden_log["sha1"])
    step_s = ms_train / 1e3 / args.steps
    value = done * args.steps / (ms_train / 1e3)  # ONE merge sequence for the whole (sharded) corpus
    e2e_value = done * e2e_steps / (ms_train_e2e / 1e3)
    scan_bytes = scan_equivalent_bytes(n0_total, weights)
    achieved = scan_bytes / step_s / 1e9 / world  # per GPU
    enc_gbs = allsum(c2 * args.steps) / (ms_enc / 1e3) / 1e9
    enc_e2e_gbs = allsum(c2 * e2e_steps) / (ms_enc_e2e / 1e3) / 1e9
    enc_text_gbs = allsum(c2 * e2e_steps) / (ms_enc_text / 1e3) / 1e9
    enc_text_h2d = int(allsum(c2 + off2.nbytes + tvi.nbytes))
    enc_alg_bytes = 4 * c2 + 4 * k_out  # this rank's shard, against this rank's kernel time
    enc_achieved = enc_alg_bytes / (enc_kernel_ms / 1e3) / 1e9
    h2d_total = int(allsum(n0 * 4 + off_host.nbytes))
    k_out_total = int(allsum(k_out))
    n_docs2_total = int(allsum(n_docs2))
    enc_h2d_total = int(allsum(c2 * 4 + off2.nbytes + tvi.nbytes))
    enc_d2h_total = int(allsum(k_out * 4 + off2.nbytes))

    # (out_host / ooff_host hold the result of the last host-buffer encode call: raw token indices, tvi being the identity)
    enc_full = None
    if world > 1:
        # the shards' vectors, gathered on rank 0 in document order (ranks own contiguous document ranges), are hashed exactly
        # like the single-GPU output and compared with the CPU golden of the whole text
        kmax = int(max_over_ranks(k_out))
        dmax = int(max_over_ranks(n_docs2 + 1))
        pad_v = torch.zeros(kmax, dtype=torch.int32, device="cuda")
        pad_v[:k_out] = out_host[:k_out].cuda()
        pad_o = torch.zeros(dmax, dtype=torch.int64, device="cuda")
        pad_o[:n_docs2 + 1] = torch.from_numpy(ooff_host).cuda()
        meta = torch.tensor([k_out, n_docs2], dtype=torch.int64, device="cuda")
        gv = [torch.empty_like(pad_v) for _ in range(world)] if rank == 0 else None
        go = [torch.empty_like(pad_o) for _ in range(world)] if rank == 0 else None
        gm = [torch.empty_like(meta) for _ in range(world)] if rank == 0 else None
        dist.gather(pad_v, gv, dst=0)
        dist.gather(pad_o, go, dst=0)
        dist.gather(meta, gm, dst=0)
        if rank == 0:
            vals, offs, base = [], [np.zeros(1, dtype=np.int64)], 0
            for q in range(world):
                kq, dq = (int(x) for x in gm[q].tolist())
                vals.append(gv[q][:kq].cpu().numpy())
                oq = go[q][:dq + 1].cpu().numpy()
                offs.append(oq[1:] - oq[0] + base)
                base += kq
            enc_full = full_encode_check(np.concatenate(vals), np.concatenate(offs), c2_total, done, golden_log is not None)
            del gv, go, vals
    st_final = stats()
    rounds = {"barrier_rounds": int(st_final.loop_rounds), "merges_committed": int(st_final.loop_round_merges), "site_passes_run": int(st_final.loop_round_tried),
              "rounds_that_dropped_a_tail": int(st_final.loop_rounds_cut),
              "merges_per_round": (st_final.loop_round_merges / st_final.loop_rounds) if st_final.loop_rounds else None,
              "note": "cumulative over every mergeUntil call of this process (warm-up, timed and end-to-end steps): bpe_merge_until commits several exact "
                      "merges per pair of grid barriers (csrc/round_kernels.cuh); merges above 2^20 sites run one per iteration in k_merge_loop and are not counted"}
    traffic = measured_traffic(args.workload, world, done)
    if rank == 0:
        cpu = cpu_baseline(args, merges_sample=8) if world == 1 else None  # timed on rank 0 at N=1 only
        cpu_inc = cpu_incremental_baseline(args) if world == 1 else None
        enc_cpu = cpu_encode_baseline(log, done, ids2_host.numpy(), off2, out_host.numpy(), ooff_host) if world == 1 else None
        if enc_cpu is not None:
            enc_cpu["full_output"] = full_encode_check(out_host.numpy(), ooff_host, c2, done, golden_log is not None)
        if enc_full is not None and enc_full.get("matches_cpu_golden") is False:
            raise AssertionError("encode output of the %d shards differs from the CPU golden: %r" % (world, enc_full))
        line = {
            "metric": "mergeUntil merges/sec",
            "value": value,
            "unit": "merges/s",
            "n_gpus": world,
            "steps": args.steps,
            "warmup": args.warmup,
            "ms_per_step": ms_train / args.steps,
            "higher_is_better": True,
            "scaling": "weak" if weak else "strong",
            "vs_baseline": None,
            "dtype": "u32",
            "data": "synthetic",
            "config": {
                "workload": "%s: %d B Zipf-word corpus (seed %d, %d docs), addToCorpus + mergeUntil to %d merges"
                            % (args.workload, n0_total, TRAIN_SEED, n_docs_total, merges),
                "merges_done": done,
                "merge_log_sha1": log_sha1,
                "merge_log_matches_cpu_golden": (None if golden_log is None else True),
                "merge_log_golden": (None if golden_log is None else golden_log["file"]),
                "sharding": (("corpus sharded by document over %d GPUs (contiguous, token-balanced); global pair counts replicated, "
                              "count deltas of a round of merges exchanged GPU-to-GPU over NVLink inside the persistent kernel" % world)
                             + ("; WEAK: every rank holds its own %d B shard, the corpus is their concatenation" % train_bytes if weak else "")) if world > 1 else "single GPU",
                "l2": "corpus (4 B/char) and occurrence pool are larger than the 126 MB L2" if n0 * 4 > 126e6 else "inputs smaller than L2; every step re-ingests and rebuilds the index (cold tables)",
            },
            "e2e": {"value": e2e_value, "unit": "merges/s", "h2d_bytes_per_step": h2d_total, "d2h_bytes_per_step": int(done * MERGE_DTYPE.itemsize * world),
                    "ms_per_step": ms_train_e2e / e2e_steps},
            "e2e_text": e2e_text,
            "gpu_launches": int(l1 - l0),
            "clocks": clocks,
            "rounds": rounds,
            "roofline": {
                "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": (traffic["bytes"] if traffic else None),
                "real_frac": (traffic["bytes"] / step_s / 1e9 / peak if traffic else None),
                "traffic_note": (traffic["note"] if traffic else "no ncu capture of this workload / GPU count is committed"),
                "kernel": "k_merge_rounds (persistent cooperative mergeUntil kernel, several merges per barrier round) + k_merge_loop for the merges above 2^20 sites; "
                          "the step also contains k_ingest_ids + K1",
                "note": "achieved = reference-algorithm bytes sum_t 4*(2*N_t+N_{t+1}) / step time ('x of reference-algorithm roofline', SURVEY 8d): the reference rescans "
                        "the corpus per merge, an incremental design exceeds 1.0 by construction; real_frac = DRAM bytes the kernels actually move (ncu) / step time / "
                        "peak -- random 32-byte sectors, not streams; peak from " + peak_src,
            },
            "roofline_k1": {"bound": "hbm", "achieved": 4 * n0 / (k1_ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                            "frac": 4 * n0 / (k1_ms / 1e3) / 1e9 / peak, "ms": k1_ms, "kernel": "k_hist + k_alloc_lists + k_scatter",
                            "traffic_note": "ncu at N=1 (profiles/r02b_traffic_cfg3.json): k_hist reads 4.0 GB in 3.3 ms (1.22 TB/s), k_scatter moves 11.7 GB read + "
                                            "9.0 GB written for 4 + 4 GB algorithmic in 25.7 ms"},
            "encode": {
                "metric": "encodeToVector GB/s of input text", "value": enc_gbs, "unit": "GB/s", "ms_per_step": ms_enc / args.steps,
                "chars": c2_total, "tokens_out": k_out_total, "docs": n_docs2_total, "gpu_launches": int(le1 - le0),
                "e2e": {"value": enc_e2e_gbs, "unit": "GB/s", "h2d_bytes_per_step": enc_h2d_total, "d2h_bytes_per_step": enc_d2h_total},
                "e2e_text": {"value": enc_text_gbs, "unit": "GB/s", "h2d_bytes_per_step": enc_text_h2d, "d2h_bytes_per_step": enc_d2h_total,
                             "note": "bpe_encode_text_batch: UTF-8 bytes in (1 B/char), char->index on the device, vectors out"},
                "roofline": {"bound": "hbm", "achieved": enc_achieved, "peak": peak, "unit": "GB/s", "frac": enc_achieved / peak, "traffic": 1.072 * enc_alg_bytes,
                             "traffic_note": "ncu --set full on a 100 MB launch: dram read+write = 1.072 x algorithmic bytes (profiles/r01b_encode_lanes.md), scaled to this shard",
                             "kernel": "k_range_starts + k_encode_lanes + scan + k_gather_map (ms_encode of the engine, rank 0 shard)", "alg_bytes": enc_alg_bytes},
            },
            "setup": {"synth_s": gen_s},
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if cpu_inc is not None:
            line["cpu_baseline_incremental"] = cpu_inc
        if enc_full is not None:
            line["encode"]["full_output"] = enc_full
        if enc_cpu is not None:
            line["encode"]["cpu_baseline"] = enc_cpu
        if args.dump_outputs:
            write_dumps(args.dump_outputs, dumps)
        print(json.dumps(line), file=_OUT, flush=True)
    lib.bpe_destroy(h)
    if world > 1:
        dist.destroy_process_group()


def encode_sample(values, offsets, in_offsets):
    """The encoded vectors of a seeded sample of documents: values / offsets = the encode output, in_offsets = its input's."""
    order = np.random.default_rng(DUMP_SEED).permutation(len(in_offsets) - 1)
    keep = int(np.searchsorted(np.cumsum(np.diff(in_offsets)[order]), DUMP_CHARS, side="right"))
    docs = np.sort(order[:keep])
    lo, lens = offsets[docs], offsets[docs + 1] - offsets[docs]
    idx = np.repeat(lo - (np.cumsum(lens) - lens), lens) + np.arange(int(lens.sum()))
    return {"encode_docs": docs.astype(np.float64), "encode_doc_lengths": lens.astype(np.float64), "encode_tokens": values[idx].astype(np.float32)}


def write_dumps(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20, "outputs larger than 64 MB"
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------------
def cpu_sample(args, merges_sample):
    """The CPU restatement of core.ts (oracle/int_oracle.cpp, 1 thread) on a bounded slice of the same workload."""
    from oracle.int_oracle import IntOracle

    train_bytes, merges, encode_bytes = WORKLOADS[args.workload]
    sample_bytes = min(train_bytes, 16_000_000)
    text, off = synth(None, sample_bytes, TRAIN_SEED)
    lut, alphabet = alphabet_lut(text)
    ids = lut[text]
    o = IntOracle()
    o.set_len16(np.ones(len(alphabet) + merges_sample + 1, dtype=np.int32))
    o.add_documents(ids, off)
    t0 = time.perf_counter()
    la, lb, lw = o.merge_until(2, 0, merges_sample, len(alphabet), merges_sample)
    dt = time.perf_counter() - t0
    rate_sample = len(la) / dt
    scale = ids.size / train_bytes
    return rate_sample, scale, ids.size, len(la), dt


def cpu_incremental_baseline(args, sample_bytes=16_000_000, merges_sample=2000):
    """A second CPU point: the INCREMENTAL oracle (oracle/fast_oracle.cpp -- same results, work per merge proportional to the
    occurrences touched; not the reference's algorithm) timed live on a bounded slice, next to the committed full-size figure."""
    try:
        from oracle.fast_oracle import FastOracle

        train_bytes, merges, _ = WORKLOADS[args.workload]
        text, off = synth(None, min(train_bytes, sample_bytes), TRAIN_SEED)
        lut, alphabet = alphabet_lut(text)
        ids = lut[text]
        o = FastOracle()
        o.set_len16(np.ones(len(alphabet), dtype=np.int32))
        t0 = time.perf_counter()
        o.add_documents(ids, off)
        la, _, _ = o.merge_until(2, 0, merges_sample, len(alphabet), merges_sample)
        dt = time.perf_counter() - t0
        out = {"value": len(la) / dt, "unit": "merges/s", "cores": 1, "kind": "port (incremental algorithm, not core.ts's)",
               "sample": "oracle/fast_oracle.cpp, 1 thread of %d: index build + first %d merges on the first %d chars took %.2f s"
                         % (os.cpu_count() or 1, len(la), ids.size, dt)}
        try:
            with open(os.path.join(ROOT, "tests", "golden", "cfg3_full_check.json")) as f:
                g = json.load(f)
            out["full_size_committed"] = {"value": g["merges"] / g["oracle_seconds"], "unit": "merges/s",
                                          "note": "the same oracle over the whole cfg3 workload, offline: %d merges in %.0f s (%s)"
                                                  % (g["merges"], g["oracle_seconds"], "tests/golden/cfg3_full_check.json")}
        except Exception:
            pass
        return out
    except Exception as e:  # never take the GPU line down
        return {"value": None, "unit": "merges/s", "cores": 1, "kind": "port", "sample": "failed: %r" % (e,)}


def cpu_baseline(args, merges_sample=8):
    try:
        rate, scale, n, done, dt = cpu_sample(args, merges_sample)
    except Exception as e:  # the baseline must never take the GPU line down
        return {"value": None, "unit": "merges/s", "cores": 1, "kind": "port", "sample": "failed: %r" % (e,)}
    return {
        "value": rate * scale, "unit": "merges/s", "cores": 1, "kind": "port",
        "sample": "C++ restatement of core.ts (Node/V8 absent), 1 thread of %d: first %d merges on the first %d chars took %.2f s (%.3f merges/s); "
                  "per-merge cost is linear in corpus size, value = that x %.4f (sample/workload size)" % (os.cpu_count() or 1, done, n, dt, rate, scale),
    }


def measured_traffic(workload, world, done):
    """DRAM bytes one step moves, from the committed ncu capture of the same workload (profiles/r02b_traffic_cfg3.json,
    tools/ncu_traffic.sh): per-launch dram__bytes_read + dram__bytes_write summed over every kernel of the step."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02b_traffic_cfg3.json")) as f:
            t = json.load(f)
        if t["workload"] != workload or t["n_gpus"] != world or done != 32000:
            return None
        b = int(t["step_read_bytes"]) + int(t["step_write_bytes"])
        return {"bytes": b, "note": "ncu, application replay over one full step, every launch (profiles/r02b_traffic_cfg3.json): %.0f GB read + %.0f GB written, of which "
                                    "the mergeUntil kernels %.0f GB" % (t["step_read_bytes"] / 1e9, t["step_write_bytes"] / 1e9, t["merge_kernels_bytes"] / 1e9)}
    except Exception:
        return None


def merge_log_golden(workload, n0_total, done):
    """SHA-1 of the CPU oracle's merge log for this exact workload, when a committed fixture holds one: cfg3 = the incremental
    oracle's full 32 000-merge run (tests/golden/cfg3_full_check.json), cfg2 = the literal restatement's (cfg2_merge_log.json)."""
    try:
        name = {"cfg3": "cfg3_full_check.json", "cfg2": "cfg2_merge_log.json"}.get(workload)
        if not name:
            return None
        with open(os.path.join(ROOT, "tests", "golden", name)) as f:
            g = json.load(f)
        if int(g.get("merges", -1)) != int(done) or ("%d B" % n0_total) not in g.get("workload", ""):
            return None
        return {"sha1": g["sha1"], "file": "tests/golden/" + name}
    except Exception:
        return None


def stream_sha1(values, offsets, block_docs=65536):
    """SHA-1 over the per-block SHA-1 digests of an int32 token stream (blocks of `block_docs` documents): the form in which
    tests/golden/make_cfg4_encode_golden.py records the CPU restatement's encoding of the whole 1 GB text."""
    import hashlib

    h = hashlib.sha1()
    n_docs = len(offsets) - 1
    for d0 in range(0, n_docs, block_docs):
        d1 = min(n_docs, d0 + block_docs)
        h.update(hashlib.sha1(np.ascontiguousarray(values[offsets[d0]:offsets[d1]], dtype=np.int32).tobytes()).digest())
    return h.hexdigest()


def full_encode_check(gpu_out, gpu_off, chars, merges_done, table_is_golden=True):
    """The GPU's vectors for the WHOLE encode text against what the CPU restatement produced offline for the same text and merge table
    (tests/golden/cfg4_encode.json, ~3.5 core-hours; BASELINE config 4): token count, per-document lengths and the token stream."""
    try:
        import hashlib

        path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "tests", "golden", "cfg4_encode.json")
        out = {"output_sha1": stream_sha1(gpu_out, gpu_off),
               "doc_lengths_sha1": hashlib.sha1(np.diff(gpu_off).astype(np.int32).tobytes()).hexdigest()}
        if os.path.exists(path):
            with open(path) as f:
                golden = json.load(f)
            # (the golden was made with cfg3's merge table: it only speaks about runs whose merge log equals that table's)
            if table_is_golden and ("%d B" % chars) in golden["workload"] and merges_done == 32000:
                out["matches_cpu_golden"] = bool(golden["output_sha1"] == out["output_sha1"] and golden["doc_lengths_sha1"] == out["doc_lengths_sha1"]
                                                 and golden["tokens_out"] == int(gpu_off[-1] - gpu_off[0]))
        return out
    except Exception as e:  # never take the GPU line down
        return {"failed": repr(e)}


def cpu_encode_baseline(log, done, ids, off, gpu_out, gpu_off, sample_bytes=1_000_000):
    """encodeToCode (core.ts:404-406: every merge in training order, replaceAll over the document) by the CPU restatement, one call per
    document, on the first ~1 MB of the encode text -- and the check that the vectors the GPU produced for those documents are identical."""
    try:
        from oracle.int_oracle import IntOracle

        o = IntOracle()
        o.load_merges(np.stack([log["a"][:done], log["b"][:done], log["c"][:done]], axis=1).astype(np.int32))
        d = max(1, min(int(np.searchsorted(off, off[0] + sample_bytes, side="left")), len(off) - 1))
        same, k = True, 0
        t0 = time.perf_counter()
        for i in range(d):
            want = o.encode(ids[off[i]:off[i + 1]])
            k += want.size
            same = same and np.array_equal(want, gpu_out[gpu_off[i]:gpu_off[i + 1]])
        dt = time.perf_counter() - t0
        chars = int(off[d] - off[0])
        return {"value": chars / dt / 1e9, "unit": "GB/s", "cores": 1, "kind": "port", "matches_gpu_output": bool(same),
                "sample": "C++ restatement of core.ts encodeToCode (Node/V8 absent), 1 thread of %d: the first %d documents (%d chars -> %d tokens) of the "
                          "encode text with the %d merges just learned took %.2f s" % (os.cpu_count() or 1, d, chars, k, done, dt)}
    except Exception as e:  # the baseline must never take the GPU line down
        return {"value": None, "unit": "GB/s", "cores": 1, "kind": "port", "sample": "failed: %r" % (e,)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    train_bytes, merges, _ = WORKLOADS[args.workload]
    for _ in range(max(0, min(args.warmup, 1))):
        cpu_sample(args, 2)
    rates, info = [], None
    t0 = time.perf_counter()
    for _ in range(args.steps):
        info = cpu_sample(args, 8)
        rates.append(info[0] * info[1])
    wall = time.perf_counter() - t0
    value = float(np.mean(rates))
    cpu = {"value": value, "unit": "merges/s", "cores": 1, "kind": "port",
           "sample": "oracle/int_oracle.cpp (literal C++ restatement of core.ts; Node is not in the image), 1 thread of %d: first %d merges on the first %d chars, "
                     "scaled by %.4f to the %d-char workload" % (os.cpu_count() or 1, info[3], info[2], info[1], train_bytes)}
    print(json.dumps({
        "impl": "reference", "metric": "mergeUntil merges/sec", "value": value, "unit": "merges/s", "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": wall / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": "%s: %d B Zipf-word corpus, mergeUntil to %d merges (bounded CPU sample, see cpu_baseline.sample)" % (args.workload, train_bytes, merges)},
        "cpu_baseline": cpu,
        "e2e": {"value": value, "unit": "merges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), file=_OUT, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=os.environ.get("BPE_BENCH_WORKLOAD", "cfg3"), choices=sorted(WORKLOADS))
    ap.add_argument("--merges", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the outputs of the last timed steps to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA engine (--impl b200)")
    # stdout carries ONE JSON line: anything native code writes to descriptor 1 on the way (NCCL's version banner) goes to stderr
    global _OUT
    sys.stdout.flush()
    _OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
