"""CPU: the measurement contract of bench.py that needs no GPU.

* `bench.py --impl reference` (the CPU restatement timed on host cores) prints exactly one JSON line on stdout with the keys the
  driver reads, and the process never maps the CUDA product library (the reference arm must not depend on the thing it is
  compared with).
* The committed bench lines of this round (profiles/r02_bench_n*.json, produced on B200s by the same script) carry the merge
  log's SHA-1 of the CPU oracle (tests/golden/cfg3_full_check.json) at every GPU count, the roofline / cpu_baseline / e2e objects
  and a value that does not fall with N.
"""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_and_never_loads_the_product_library():
    code = (
        "import sys, runpy\n"
        "sys.argv = ['bench.py', '--impl', 'reference', '--steps', '1', '--warmup', '0', '--workload', 'tiny']\n"
        "try:\n"
        "    runpy.run_path(%r, run_name='__main__')\n"
        "finally:\n"
        "    maps = open('/proc/self/maps').read()\n"
        "    sys.stderr.write('PRODUCT_LIB_MAPPED=%%d\\n' %% ('libbpe_b200.so' in maps))\n" % os.path.join(ROOT, "bench.py")
    )
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "mergeUntil merges/sec" and d["unit"] == "merges/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 1 and d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "merges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "PRODUCT_LIB_MAPPED=0" in r.stderr, r.stderr[-500:]


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step_and_steps_sets_the_timed_steps(tmp_path):
    """`--dump-outputs DIR`: the merge log of the last timed step (the CPU oracle's) and a seeded sample of the encode output (the
    oracle's encoding of those documents), float .npy files, identical for any --steps; the timed launches scale with --steps."""
    import numpy as np

    from bpe_tokenizer_b200.synth import first_appearance_ids, synth_corpus
    from oracle.fast_oracle import FastOracle
    from oracle.int_oracle import IntOracle

    lines, dumps = {}, {}
    for steps in (1, 2):
        out = tmp_path / ("steps%d" % steps)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--workload", "tiny", "--steps", str(steps), "--warmup", "1",
                            "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        lines[steps] = json.loads(r.stdout)
        dumps[steps] = {f[:-4]: np.load(out / f) for f in sorted(os.listdir(out))}
    assert lines[1]["steps"] == 1 and lines[2]["steps"] == 2
    assert lines[2]["gpu_launches"] == 2 * lines[1]["gpu_launches"] > 0
    d = dumps[2]
    assert sorted(d) == ["encode_doc_lengths", "encode_docs", "encode_tokens", "merge_log"] and sorted(dumps[1]) == sorted(d)
    assert all(np.array_equal(d[k], dumps[1][k]) for k in d)
    assert all(a.dtype in (np.float32, np.float64) for a in d.values()) and sum(a.nbytes for a in d.values()) <= 64 << 20

    text, off = synth_corpus(200_000, seed=43)
    ids, alphabet = first_appearance_ids(text)
    o = FastOracle()
    o.set_len16(np.ones(len(alphabet), dtype=np.int32))
    o.add_documents(ids, off)
    la, lb, lw = o.merge_until(2, 0, 200, len(alphabet), 200)
    want = np.stack([la, lb, len(alphabet) + np.arange(len(la)), lw], axis=1).astype(np.float64)
    assert len(la) == 200 and np.array_equal(d["merge_log"], want)

    text2, off2 = synth_corpus(200_000, seed=44)
    lut = np.full(256, -1, dtype=np.int32)
    lut[alphabet] = np.arange(len(alphabet), dtype=np.int32)
    enc = IntOracle()
    enc.load_merges(want[:, :3].astype(np.int32))
    docs, lens = d["encode_docs"].astype(np.int64), d["encode_doc_lengths"].astype(np.int64)
    assert docs.size == len(off2) - 1  # 200 kB of text: the sample is every document
    got = np.split(d["encode_tokens"].astype(np.int32), np.cumsum(lens)[:-1])
    for doc, vec in zip(docs, got):
        assert np.array_equal(vec, enc.encode(lut[text2[off2[doc]:off2[doc + 1]]])), doc


@pytest.mark.parametrize("n", [1, 2, 4, 8])
def test_committed_bench_lines_of_this_round(n):
    with open(os.path.join(ROOT, "profiles", "r02_bench_n%d.json" % n)) as f:
        d = json.load(f)
    with open(os.path.join(ROOT, "tests", "golden", "cfg3_full_check.json")) as f:
        golden = json.load(f)
    assert d["n_gpus"] == n and d["metric"] == "mergeUntil merges/sec" and d["scaling"] == "strong"
    assert d["config"]["merges_done"] == 32000
    assert d["config"]["merge_log_sha1"] == golden["sha1"] and d["config"]["merge_log_matches_cpu_golden"] is True
    assert d["gpu_launches"] > 0 and d["clocks"]["reasons"] == []
    assert d["e2e"]["h2d_bytes_per_step"] > 4_000_000_000 and 0 < d["e2e"]["value"] <= d["value"]
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["peak"] > 0 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    enc = d["encode"]
    assert enc["tokens_out"] == 176384677
    full = enc["cpu_baseline"]["full_output"] if n == 1 else enc["full_output"]
    assert full["matches_cpu_golden"] is True
    if n == 1:
        assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline_incremental"]["value"] > d["cpu_baseline"]["value"]
        assert 0 < r["real_frac"] < 1 and r["traffic"] > 1e11
    else:
        with open(os.path.join(ROOT, "profiles", "r02_bench_n1.json")) as f:
            one = json.load(f)
        # (run-to-run spread of the one-GPU value on this pool: 65.5 k .. 66.4 k over five runs; N = 2 sits inside it, N = 4 and 8 above)
        assert d["value"] >= 0.98 * one["value"], "sharding must not make training slower than one GPU"
        if n >= 4:
            assert d["value"] > 1.1 * one["value"]
