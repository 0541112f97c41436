"""GPU: encodeTextTensor / decodeTensor and the C entry points under them (bpe_encode_text_batch_dev, bpe_pad_batch_dev).
Text as str, host bytes or CUDA tensors encodes to the same values, offsets and first holes as encodeTextBatch; padded rows
equal the ragged output padded in numpy; errors, offset shapes, streams and device groups behave as the header says."""
import ctypes as C
import random

import numpy as np
import pytest

from bpe_tokenizer_b200 import _abi

pytestmark = pytest.mark.gpu

# characters of 1 to 4 UTF-8 bytes, and a lone surrogate (written in its generalised 3-byte form)
EXTRA = ["héllo wörld ÿ", "中文字 中文", "emoji \U0001F600\U0001F600 end", "lone \ud800 and \udfff", "max \U0010FFFF!", "\x7f\x80߿ࠀ￿\U00010000"]


def _utf8_batch(docs):
    chunks = [d.encode("utf-8", "surrogatepass") for d in docs]
    off = np.zeros(len(chunks) + 1, dtype=np.int64)
    np.cumsum([len(c) for c in chunks], out=off[1:])
    return b"".join(chunks), off


def _docs(text, off):
    return [bytes(text[off[d]:off[d + 1]]).decode() for d in range(len(off) - 1)]


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


@pytest.fixture(scope="module")
def trained():
    """A tokenizer trained on 3 MB of Zipf text plus the non-ASCII documents (3000 merges), its training documents and
    held-out seed-44 documents."""
    from bpe_tokenizer_b200 import BPETokenizer
    from bpe_tokenizer_b200.synth import synth_corpus

    text, off = synth_corpus(3_000_000, seed=43)
    t = BPETokenizer()
    t.addTextBatch(bytes(text), off)
    for d in EXTRA * 3:
        t.addToCorpus(d)
    assert t.mergeUntil({"max_iterations": 3000}) == 3000
    t.compactVectorIndex()
    text2, off2 = synth_corpus(300_000, seed=44)
    held = _docs(text2, off2)
    rng = random.Random(5)
    for d in rng.sample(range(len(held)), 20):
        held[d] = held[d] + rng.choice(EXTRA)
    train = _docs(text, off)[:200] + EXTRA
    return t, train, held


def _want(t, docs, vector):
    return t.encodeTextBatch(*_utf8_batch(docs), vector=vector)


def _dev_encode(t, text_d, off_d, vector, n_bytes=None):
    """bpe_encode_text_batch_dev through ctypes: -> (rc, values, offsets, first_bad) as numpy."""
    import torch

    n_docs = off_d.numel() - 1
    n_bytes = text_d.numel() if n_bytes is None else n_bytes
    tvi = torch.from_numpy(t._tvi_array()).cuda() if vector else None
    out = torch.full((max(n_bytes, 1),), 0x5A5A5A5A, dtype=torch.int32, device="cuda")
    ooff = torch.full((n_docs + 1,), -7, dtype=torch.int64, device="cuda")
    bad = torch.full((max(n_docs, 1),), -7, dtype=torch.int64, device="cuda")
    n, upos, ucp = C.c_int64(), C.c_int64(), C.c_int32()
    rc = t._lib.bpe_encode_text_batch_dev(t._h, _ptr(text_d), n_bytes, _ptr(off_d), n_docs, _ptr(tvi), tvi.numel() if vector else 0, _ptr(out), _ptr(ooff),
                                          _ptr(bad), C.byref(n), C.byref(upos), C.byref(ucp))
    torch.cuda.synchronize()
    return rc, out.cpu().numpy(), ooff.cpu().numpy(), bad.cpu().numpy()[:n_docs], n.value, upos.value, ucp.value


def _same(t, docs, *args, vector):
    """encodeTextTensor(*args) (default: the docs as str) against encodeTextBatch of the docs: the same values and offsets, or,
    with vector=True and a hole, encodeToVector's error for the first document that has one."""
    args = args or (docs,)
    vals, voff, bad = _want(t, docs, vector)
    if vector and np.any(bad >= 0):
        with pytest.raises(ValueError) as ei:
            t.encodeTextTensor(*args)
        with pytest.raises(ValueError) as ej:
            t.encodeToVector(docs[int(np.flatnonzero(bad >= 0)[0])])
        assert str(ei.value) == str(ej.value)
        return
    got = t.encodeTextTensor(*args, vector=vector)
    assert got[0].dtype.itemsize == 4 and got[1].dtype.itemsize == 8 and got[0].is_cuda and got[1].is_cuda
    assert np.array_equal(got[0].cpu().numpy(), vals) and np.array_equal(got[1].cpu().numpy(), voff)


def test_parity_every_input_kind(trained):
    import torch

    t, _, held = trained
    text, off = _utf8_batch(held)
    for vector in (False, True):
        vals, voff, bad = _want(t, held, vector)
        # the C entry point: values, offsets and first holes bit for bit
        rc, o, oo, b, n, _, _ = _dev_encode(t, torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda(), torch.from_numpy(off).cuda(), vector)
        assert rc == 0 and n == vals.size
        assert np.array_equal(o[:n], vals) and np.array_equal(oo, voff)
        if vector:
            assert np.array_equal(b, bad)
        # the three input kinds of encodeTextTensor
        inputs = [(held, None), (text, off), (torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda(), torch.from_numpy(off).cuda())]
        for args in inputs:
            _same(t, held, *args, vector=vector)
    # a sample against the literal oracle
    from oracle import LiteralTokenizer

    lit = LiteralTokenizer()
    lit.fromJSON(t.toJSON())
    raw, roff = t.encodeTextTensor(held, vector=False)
    raw, roff = raw.cpu().numpy(), roff.cpu().numpy()
    for d in random.Random(9).sample(range(len(held)), 12):
        assert raw[roff[d]:roff[d + 1]].tolist() == [ord(ch) - 1 for ch in lit.encodeToCode(held[d])], d


def test_offset_shapes(trained):
    import torch

    t, train, _ = trained
    docs = ["", train[0], "", train[1], EXTRA[2], ""]
    text, off = _utf8_batch(docs)
    for vector in (False, True):
        # offsets that start past 0, trailing bytes after the last document
        shifted = b"\xff\xfejunk" + text + b"tail \xf0"
        off2 = off + 6
        for args in ((shifted, off2), (torch.frombuffer(bytearray(shifted), dtype=torch.uint8).cuda(), torch.from_numpy(off2).cuda())):
            _same(t, docs, *args, vector=vector)
    # only empty documents
    v, o = t.encodeTextTensor(["", "", ""])
    assert v.shape == (0,) and o.cpu().tolist() == [0, 0, 0, 0]
    # an empty batch
    for args in (([],), (b"", np.zeros(1, dtype=np.int64)), (torch.zeros(0, dtype=torch.uint8, device="cuda"), torch.zeros(1, dtype=torch.int64, device="cuda")),
                 (torch.zeros(4, dtype=torch.uint8, device="cuda"), torch.full((1,), 3, dtype=torch.int64, device="cuda"))):
        v, o = t.encodeTextTensor(*args)
        assert v.shape == (0,) and o.shape == (1,) and o.cpu().tolist() == [0]
        ids, lens = t.encodeTextTensor(*args, pad_to=7)
        assert ids.shape == (0, 7) and lens.shape == (0,)
        ids, lens = t.encodeTextTensor(*args, pad_to="longest")
        assert ids.shape == (0, 0)


def test_utf8_widths_and_long_documents(trained):
    t, train, _ = trained
    docs = EXTRA + ["a\ud800b", "\udfff", "ÿ" * 3, "\U0001F600"]
    for vector in (False, True):
        _same(t, docs, vector=vector)
    # documents longer than one lane batch (1536 characters at the widest) go to the per-document kernel
    long_doc = " ".join(train[:400])
    assert len(long_doc) > 5000
    docs = train[:50] + [long_doc] + EXTRA + [long_doc[:2000] + EXTRA[3]] + train[50:80]
    for vector in (False, True):
        _same(t, docs, vector=vector)
    # the long documents against the literal oracle as well: the host path above shares the encode kernels
    from oracle import LiteralTokenizer

    lit = LiteralTokenizer()
    lit.fromJSON(t.toJSON())
    longs = [long_doc, long_doc[:2000] + EXTRA[3]]
    raw, roff = t.encodeTextTensor(train[:5] + longs, vector=False)
    raw, roff = raw.cpu().numpy(), roff.cpu().numpy()
    for d, doc in enumerate(longs, start=5):
        assert raw[roff[d]:roff[d + 1]].tolist() == [ord(ch) - 1 for ch in lit.encodeToCode(doc)], d


def test_unknown_character_and_holes(trained):
    import torch

    from bpe_tokenizer_b200 import BPETokenizer

    t, train, _ = trained
    docs = [train[0], "ab☃c", "☂"]
    with pytest.raises(ValueError) as ei:
        t.encodeTextTensor(docs)
    with pytest.raises(ValueError) as ej:
        t.encodeTextBatch(*_utf8_batch(docs))
    assert str(ei.value) == str(ej.value) == "unknown token, char: \"☃\""
    # unknown_pos and the code point are the host path's
    text, off = _utf8_batch(docs)
    rc, _, _, _, _, upos, ucp = _dev_encode(t, torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda(), torch.from_numpy(off).cuda(), False)
    buf = np.frombuffer(text, dtype=np.uint8)
    out, ooff, n, hpos, hcp = np.zeros(len(text), dtype=np.int32), np.zeros(len(docs) + 1, dtype=np.int64), C.c_int64(), C.c_int64(), C.c_int32()
    hrc = t._lib.bpe_encode_text_batch(t._h, buf.ctypes.data_as(_abi.u8p), _abi.p64(off), len(docs), None, 0, _abi.p32(out), out.size, _abi.p64(ooff), None,
                                       C.byref(n), C.byref(hpos), C.byref(hcp))
    assert rc == hrc == _abi.BPE_E_INVALID and upos == hpos.value == len(train[0]) + 2 and ucp == hcp.value == ord("☃")
    # a zero-weight token: "a" and "b" were merged away; the first hole in document order is reported
    s = BPETokenizer()
    s.addToCorpus("abab")
    s.addToCorpus("c")
    assert s.mergeUntil({"max_iterations": 1}) == 1
    s.compactVectorIndex()
    with pytest.raises(ValueError) as ei:
        s.encodeTextTensor(["ab", "cb", "ca"])
    with pytest.raises(ValueError) as ej:
        s.encodeToVector("cb")
    assert str(ei.value) == str(ej.value) == "unknown token index: 1"
    assert s.encodeTextTensor(["ab", "cb", "ca"], vector=False)[0].cpu().tolist() == [3, 2, 1, 2, 0]
    assert s.encodeTextTensor(["abc", "cab"])[0].cpu().tolist() == [1, 0, 0, 1]


def test_bad_device_offsets_write_nothing(trained):
    import torch

    t, train, _ = trained
    text, _ = _utf8_batch(train[:3])
    text_d = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    nb = len(text)
    for bad in ([0, 5, 3, nb], [-1, 3, nb], [0, 3, nb + 1], [nb + 1], [0, nb, 2]):
        rc, o, oo, b, n, upos, _ = _dev_encode(t, text_d, torch.tensor(bad, dtype=torch.int64, device="cuda"), True)
        assert rc == _abi.BPE_E_INVALID, bad
        assert np.all(o == 0x5A5A5A5A) and np.all(oo == -7) and np.all(b == -7) and n == 0 and upos == -1, bad
        with pytest.raises(_abi.BpeError) as ei:
            t.encodeTextTensor(text_d, torch.tensor(bad, dtype=torch.int64, device="cuda"))
        assert ei.value.code == _abi.BPE_E_INVALID
    # inputs that are not on the engine's device, or of the wrong type
    with pytest.raises(ValueError):
        t.encodeTextTensor(torch.frombuffer(bytearray(text), dtype=torch.uint8), torch.tensor([0, nb]))
    with pytest.raises(ValueError):
        t.encodeTextTensor(text_d, torch.tensor([0, nb], dtype=torch.int32, device="cuda"))
    for pad_to in (-1, 2.0, "short"):
        with pytest.raises(ValueError):
            t.encodeTextTensor(train[:2], pad_to=pad_to)
    with pytest.raises(ValueError):
        t.encodeTextTensor(train[0])  # one str is not a batch of documents


def _pad_numpy(vals, off, width, pad):
    n = len(off) - 1
    ids = np.full((n, width), pad, dtype=np.int32)
    lens = np.minimum(np.diff(off), width)
    for d in range(n):
        ids[d, : lens[d]] = vals[off[d]:off[d] + lens[d]]
    return ids, lens


def test_padding(trained):
    import torch

    t, train, _ = trained
    docs = train[:40] + [""] + EXTRA
    vals, voff, _ = _want(t, docs, True)
    longest = int(np.diff(voff).max())
    for pad_to, pad in ((longest // 2, -1), (longest, 0), ("longest", 12345), (np.int64(longest + 37), -9), (0, -1), (1, 7)):
        ids, lens = t.encodeTextTensor(docs, pad_to=pad_to, pad_value=pad)
        width = longest if isinstance(pad_to, str) else int(pad_to)
        assert ids.shape == (len(docs), width) and ids.dtype == torch.int32 and lens.dtype == torch.int64
        want_ids, want_lens = _pad_numpy(vals, voff, width, pad)
        assert np.array_equal(ids.cpu().numpy(), want_ids) and np.array_equal(lens.cpu().numpy(), want_lens), pad_to
    # bpe_pad_batch_dev on bpe_encode_batch_dev's output (ids in) gives the same rows
    ids_in = np.concatenate([t._char_ids(d, create=False) for d in docs])
    off_in = np.zeros(len(docs) + 1, dtype=np.int64)
    np.cumsum([len(d) for d in docs], out=off_in[1:])
    ids_d, off_d = torch.from_numpy(ids_in).cuda(), torch.from_numpy(off_in).cuda()
    out = torch.empty(ids_in.size, dtype=torch.int32, device="cuda")
    ooff = torch.empty(len(docs) + 1, dtype=torch.int64, device="cuda")
    n = C.c_int64()
    assert t._lib.bpe_encode_batch_dev(t._h, _ptr(ids_d), _ptr(off_d), len(docs), ids_in.size, int(np.diff(off_in).max()), None, 0, _ptr(out), _ptr(ooff), None,
                                       C.byref(n)) == 0
    width = longest // 2
    dense = torch.full((len(docs), width), 99, dtype=torch.int32, device="cuda")
    lens = torch.empty(len(docs), dtype=torch.int64, device="cuda")
    assert t._lib.bpe_pad_batch_dev(t._h, _ptr(out), _ptr(ooff), len(docs), width, -3, _ptr(dense), _ptr(lens)) == 0
    raw, roff, _ = _want(t, docs, False)
    want_ids, want_lens = _pad_numpy(raw, roff, width, -3)
    assert np.array_equal(dense.cpu().numpy(), want_ids) and np.array_equal(lens.cpu().numpy(), want_lens)
    ids2, _ = t.encodeTextTensor(docs, vector=False, pad_to=width, pad_value=-3)
    assert torch.equal(ids2, dense)


def test_round_trip(trained):
    import torch

    t, train, _ = trained
    docs = train[:60] + ["", EXTRA[3]] + EXTRA
    vals, off = t.encodeTextTensor(docs)
    assert t.decodeTensor(vals, off) == docs
    v, o = vals.cpu().numpy(), off.cpu().numpy()
    assert [t.decodeVector(v[o[d]:o[d + 1]].tolist()) for d in range(len(docs))] == docs
    ids, lens = t.encodeTextTensor(docs, pad_to="longest")
    assert t.decodeTensor(ids, lengths=lens) == docs
    raw, roff = t.encodeTextTensor(docs, vector=False)
    assert t.decodeTensor(raw, roff, vector=False) == docs
    with pytest.raises(ValueError, match="unknown vector index: 1000000"):
        t.decodeTensor(vals[:3].clone().fill_(1_000_000), torch.tensor([0, 3]))
    assert t.decodeTensor(vals[:0], off[:1]) == []


def test_default_stream_input_from_queued_kernels(trained):
    """Text and offsets written by kernels queued on torch's default stream behind a long-running kernel, with no
    synchronisation before the call: the encode must run after them on that stream (torch's default stream has the handle 0,
    which alone would name the engine's own, unordered stream)."""
    import torch

    t, train, _ = trained
    docs = train[:150] + EXTRA
    text, off = _utf8_batch(docs)
    raw, roff, _ = _want(t, docs, False)
    src = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    lens = torch.from_numpy(np.diff(off)).cuda()
    for pad_to in (None, 96):
        text_d = torch.zeros_like(src)
        off_d = torch.zeros(len(off), dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()
        with torch.cuda.stream(torch.cuda.default_stream()):
            torch.cuda._sleep(200_000_000)  # keeps the default stream busy for a tenth of a second or so
            text_d.copy_(src)
            torch.cumsum(lens, 0, out=off_d[1:])
            got = t.encodeTextTensor(text_d, off_d, vector=False, pad_to=pad_to)
        if pad_to is None:
            assert np.array_equal(got[0].cpu().numpy(), raw) and np.array_equal(got[1].cpu().numpy(), roff)
        else:
            want_ids, want_lens = _pad_numpy(raw, roff, pad_to, -1)
            assert np.array_equal(got[0].cpu().numpy(), want_ids) and np.array_equal(got[1].cpu().numpy(), want_lens)


def test_streams():
    import torch

    from bpe_tokenizer_b200 import BPETokenizer
    from bpe_tokenizer_b200.synth import synth_corpus

    text, off = synth_corpus(400_000, seed=43)
    a, b = BPETokenizer(), BPETokenizer()
    for x in (a, b):
        x.addTextBatch(bytes(text), off)
        x.mergeUntil({"max_iterations": 300})
    docs = _docs(*synth_corpus(100_000, seed=44))
    want = a.encodeTextTensor(docs, vector=False)
    # the input is produced on a side stream, and the encode runs there
    s = torch.cuda.Stream()
    tb, ob = _utf8_batch(docs)
    with torch.cuda.stream(s):
        host = torch.frombuffer(bytearray(tb), dtype=torch.uint8).pin_memory()
        text_d = torch.empty(len(tb), dtype=torch.uint8, device="cuda")
        text_d.copy_(host, non_blocking=True)
        off_d = torch.from_numpy(ob).cuda()
        got = a.encodeTextTensor(text_d, off_d, vector=False)
        ids, lens = a.encodeTextTensor(text_d, off_d, vector=False, pad_to=64)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    assert np.array_equal(ids.cpu().numpy(), _pad_numpy(want[0].cpu().numpy(), want[1].cpu().numpy(), 64, -1)[0])
    # a stream the tokenizer was given before the call is its stream again afterwards: training and host encode carry on
    s2 = torch.cuda.Stream()
    a.set_stream(s2.cuda_stream)
    a.encodeTextTensor(docs[:10], vector=False)
    for x in (a, b):
        x.mergeUntil({"max_iterations": 200})
    assert a.toJSON() == b.toJSON()
    ha, hb = a.encodeTextBatch(tb, ob), b.encodeTextBatch(tb, ob)
    assert all(np.array_equal(p, q) for p, q in zip(ha, hb))
    a.set_stream(0)
    a.close()
    b.close()


def test_device_group_refuses(monkeypatch):
    import torch

    from bpe_tokenizer_b200 import BPETokenizer, BpeError

    if torch.cuda.device_count() >= 2 and torch.cuda.can_device_access_peer(0, 1):
        devs = [0, 1]
    else:
        monkeypatch.setenv("BPE_GROUP_SHARE_DEVICE", "1")  # (read by bpe_create_group when it is called)
        devs = [0, 0]
    g = BPETokenizer(devices=devs)
    g.addTextBatch(*_utf8_batch(["abcab", "bcabc"]))
    g.mergeUntil({"max_iterations": 2})
    text, off = _utf8_batch(["abc"])
    text_d, off_d = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda(), torch.from_numpy(off).cuda()
    rc, *_ = _dev_encode(g, text_d, off_d, False)
    assert rc == _abi.BPE_E_INVALID
    out = torch.zeros((1, 4), dtype=torch.int32, device="cuda")
    vals = torch.zeros(3, dtype=torch.int32, device="cuda")
    assert g._lib.bpe_pad_batch_dev(g._h, _ptr(vals), _ptr(off_d), 1, 4, -1, _ptr(out), None) == _abi.BPE_E_INVALID
    for args in ((["abc"],), (text_d, off_d)):
        with pytest.raises(BpeError):
            g.encodeTextTensor(*args)
    # the group still encodes from host buffers
    assert g.encodeTextBatch(text, off, vector=False)[0].size > 0
    g.close()
