"""One engine, one GPU, a corpus larger than the 32-bit occurrence pool allowed: the synthetic Zipf text of bench.py (seed 43)
at --bytes characters (default 4.0e9), 32 000 merges.  Prints one JSON line: the GPU and its power limit, N0, the time of
mergeUntil (ingest from device ids included, as bench.py's step) and of K1, the pool cells used, the peak device memory seen by
cudaMemGetInfo around the step, and the merge log's SHA-1.  A step that fails reports the error code, its message and the merges
it had committed.

    python tools/large_corpus.py [--bytes 4.0e9] [--merges 32000] [--out profiles/x.json]

Host memory stays near the size of the text: the bytes go to the device as they are and are mapped to token ids there, in chunks.
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_identity(index):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip().split(",")
        return out[0].strip(), out[1].strip()
    except Exception:
        return None, None


def device_ids(text, chunk=1 << 28):
    """uint8 text (host) -> int32 token ids (device) in first-appearance order, the host holding nothing but the text."""
    import torch

    from bench import alphabet_lut

    lut, alphabet = alphabet_lut(text)
    lut_dev = torch.from_numpy(lut).cuda()
    ids = torch.empty(text.size, dtype=torch.int32, device="cuda")
    for s in range(0, text.size, chunk):
        part = torch.from_numpy(text[s:s + chunk]).cuda()
        ids[s:s + part.numel()] = lut_dev[part.long()]
    torch.cuda.synchronize()
    assert int(ids.min().item()) >= 0
    return ids, alphabet


def run(n_bytes, merges, seed=43):
    import torch

    from bench import synth
    from bpe_tokenizer_b200 import _abi
    from bpe_tokenizer_b200._abi import MERGE_DTYPE, bpe_stats, p32, p64

    t0 = time.time()
    text, off = synth(None, n_bytes, seed)
    gen_s = time.time() - t0
    torch.cuda.set_device(0)
    ids, alphabet = device_ids(text)
    n0, n_docs = int(text.size), len(off) - 1
    del text
    lib = _abi.load_library()
    h = C.c_void_p()
    assert lib.bpe_create(0, C.byref(h)) == 0, "bpe_create failed"
    len16 = np.ones(len(alphabet), dtype=np.int32)
    log = np.zeros(merges, dtype=MERGE_DTYPE)
    done = C.c_int64()
    name, power = gpu_identity(0)
    res = {"tool": "large_corpus", "gpu": name, "power_limit": power, "bytes": n_bytes, "seed": seed, "n0": n0, "docs": n_docs,
           "merges": merges, "gen_s": round(gen_s, 1)}

    def stats():
        s = bpe_stats()
        lib.bpe_get_stats(h, C.byref(s))
        return s

    free0, total = torch.cuda.mem_get_info()
    torch.cuda.synchronize()
    t1 = time.time()
    rc = lib.bpe_set_tokens(h, p32(len16), len(len16))
    if rc == 0:
        rc = lib.bpe_add_documents_dev(h, C.c_void_p(ids.data_ptr()), p64(np.ascontiguousarray(off)), n_docs)
    if rc == 0:
        rc = lib.bpe_merge_until(h, 2, 0, merges, log.ctypes.data_as(C.c_void_p), merges, C.byref(done))
    torch.cuda.synchronize()
    ms = (time.time() - t1) * 1e3
    free1, _ = torch.cuda.mem_get_info()
    s = stats()
    res.update({"rc": rc, "merges_done": int(done.value), "ms_merge_until": round(ms, 1),
                "merges_per_s": round(done.value / ms * 1e3, 1) if ms > 0 else None, "k1_ms": round(s.ms_index_build, 1),
                "pool_used": int(s.pool_used), "pool_used_gb": round(s.pool_used * 4 / 1e9, 2),
                "device_mem_used_gb": round((total - free1) / 1e9, 2), "device_mem_before_gb": round((total - free0) / 1e9, 2),
                "device_mem_total_gb": round(total / 1e9, 2),
                "merge_log_sha1": hashlib.sha1(log[:done.value].tobytes()).hexdigest()})
    if rc != 0:
        res["error"] = lib.bpe_last_error(h).decode()
    lib.bpe_destroy(h)
    return res, log[:done.value].copy()


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--bytes", type=float, default=4.0e9)
    ap.add_argument("--merges", type=int, default=32000)
    ap.add_argument("--seed", type=int, default=43)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    res, _ = run(int(a.bytes), a.merges, a.seed)
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")
    return 0 if res["rc"] == 0 else 1


if __name__ == "__main__":
    sys.exit(main())
