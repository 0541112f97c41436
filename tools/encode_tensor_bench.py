"""Encode into CUDA tensors against the host round trip, on tools/bench_encode.py's workload: the committed cfg3 merge table
(tools/data/merges_cfg3_abc.npy, 32 000 merges) and seed-44 Zipf text, 1 GB by default (ENC bytes) so that the working set is
far larger than the 126 MB L2.  Four paths, warmed up first, then timed in alternation (REPS rounds, host clock ending in a
device synchronise):
  host_to_host       encodeTextBatch: host bytes in, numpy values out (the pipelined host-buffer encode)
  tensor_to_ragged   encodeTextTensor(uint8 CUDA tensor, int64 CUDA offsets) -> ragged CUDA tensors
  bytes_to_padded    encodeTextTensor(host bytes, host offsets, pad_to=512) -> int32[B, 512] CUDA tensor (one pageable copy in)
  ids_dev            bpe_encode_batch_dev from single-character ids already on the device (the reference point: no front end)
Every path encodes with the vector index (all tokens have weight 1, so it is the identity).  Prints one JSON line: the card's
name and power limit (read, not set), per path the median / min / max ms per call and GB/s of text, and whether each tensor
path's values equal encodeTextBatch's."""
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from bpe_tokenizer_b200 import BPETokenizer, _abi  # noqa: E402
from bpe_tokenizer_b200.synth import native_corpus  # noqa: E402

WIDTH = 512


def gpu_identity():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=20)
        name, power = [x.strip() for x in q.stdout.strip().split(",")]
        return name, power
    except Exception as ex:
        return torch.cuda.get_device_name(0), "unknown: %r" % (ex,)


def cfg3_tokenizer():
    """The cfg3 vocabulary as a snapshot: the 29 byte characters, then every merge's token; weight 1 everywhere."""
    abc = np.load(os.path.join(ROOT, "tools", "data", "merges_cfg3_abc.npy"))
    alphabet = np.load(os.path.join(ROOT, "tools", "data", "alphabet_cfg3.npy"))
    chars = [chr(int(c)) for c in alphabet]
    for a, b, _ in abc.tolist():
        chars.append(chars[a] + chars[b])
    t = BPETokenizer(0)
    t.fromJSON({"version": 2, "char_count": len(alphabet), "token_table": [[c, 1, 1] for c in chars],
                "merge_codes": [[chr(a + 1), chr(b + 1), chr(c + 1)] for a, b, c in abc.tolist()]})
    return t, alphabet, len(abc)


def main():
    n_target = int(float(os.environ.get("ENC", 1e9)))
    reps = int(os.environ.get("REPS", 5))
    name, power = gpu_identity()
    t, alphabet, n_merges = cfg3_tokenizer()
    text, off = native_corpus(n_target, seed=44)
    n_bytes, n_docs = int(text.size), len(off) - 1
    text_bytes = text.tobytes()
    dev = torch.device("cuda", 0)
    text_d, off_d = torch.from_numpy(text).to(dev), torch.from_numpy(off).to(dev)
    lut = np.full(256, -1, dtype=np.int32)
    lut[alphabet] = np.arange(len(alphabet), dtype=np.int32)
    ids_d = torch.from_numpy(lut[text]).to(dev)
    tvi_d = torch.from_numpy(t._tvi_array()).to(dev)
    max_doc = int(np.diff(off).max())
    ids_out = torch.empty(n_bytes, dtype=torch.int32, device=dev)
    ids_ooff = torch.empty(n_docs + 1, dtype=torch.int64, device=dev)

    def ids_dev():
        n = C.c_int64()
        rc = t._lib.bpe_encode_batch_dev(t._h, C.c_void_p(ids_d.data_ptr()), C.c_void_p(off_d.data_ptr()), n_docs, n_bytes, max_doc, C.c_void_p(tvi_d.data_ptr()),
                                         tvi_d.numel(), C.c_void_p(ids_out.data_ptr()), C.c_void_p(ids_ooff.data_ptr()), None, C.byref(n))
        assert rc == 0, t._lib.bpe_last_error(t._h)
        return ids_out[: n.value], ids_ooff

    paths = {
        "host_to_host": lambda: t.encodeTextBatch(text_bytes, off),
        "tensor_to_ragged": lambda: t.encodeTextTensor(text_d, off_d),
        "bytes_to_padded": lambda: t.encodeTextTensor(text_bytes, off, pad_to=WIDTH),
        "ids_dev": ids_dev,
    }
    results = {}
    for k, fn in paths.items():  # warm-up, and the outputs the checks compare
        results[k] = fn()
        torch.cuda.synchronize()
    host_vals, host_off, host_bad = results["host_to_host"]
    assert not np.any(host_bad >= 0)
    ragged_vals, ragged_off = results["tensor_to_ragged"]
    equal = {"tensor_to_ragged": bool(np.array_equal(ragged_vals.cpu().numpy(), host_vals) and np.array_equal(ragged_off.cpu().numpy(), host_off))}
    ids_vals, ids_off = results["ids_dev"]
    equal["ids_dev"] = bool(np.array_equal(ids_vals.cpu().numpy(), host_vals) and np.array_equal(ids_off.cpu().numpy(), host_off))
    dense, lengths = results["bytes_to_padded"]
    lens_want = torch.clamp(ragged_off[1:] - ragged_off[:-1], max=WIDTH)
    col = torch.arange(WIDTH, device=dev)
    idx = torch.clamp(ragged_off[:-1, None] + col[None, :], max=max(ragged_vals.numel() - 1, 0))
    want = torch.where(col[None, :] < lens_want[:, None], ragged_vals[idx], torch.full_like(dense, -1))
    equal["bytes_to_padded"] = bool(torch.equal(dense, want) and torch.equal(lengths, lens_want))
    del results, want, idx

    times = {k: [] for k in paths}
    enc_ms = []
    for _ in range(reps):
        for k, fn in paths.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = fn()
            torch.cuda.synchronize()
            times[k].append((time.perf_counter() - t0) * 1e3)
            if k == "tensor_to_ragged":
                enc_ms.append(t.stats()["ms_encode"])
            del r
    out = {"tool": "encode_tensor_bench", "gpu": name, "power_limit": power, "bytes": n_bytes, "docs": n_docs, "longest_doc": max_doc,
           "tokens": int(host_vals.size), "merges": n_merges, "seed": 44, "reps": reps, "pad_width": WIDTH, "paths": {}, "equal": equal,
           "tensor_to_ragged_encode_kernels_ms_median": round(float(np.median(enc_ms)), 2)}
    for k, v in times.items():
        v = np.array(v)
        med = float(np.median(v))
        out["paths"][k] = {"ms_median": round(med, 2), "ms_min": round(float(v.min()), 2), "ms_max": round(float(v.max()), 2),
                           "spread_pct": round(100.0 * float(v.max() - v.min()) / med, 1), "gbps_median": round(n_bytes / med / 1e6, 2)}
    print(json.dumps(out), flush=True)
    if not all(equal.values()):
        sys.exit(1)


if __name__ == "__main__":
    main()
