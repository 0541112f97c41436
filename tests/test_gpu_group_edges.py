"""GPU: the sharded merge kernels (k_merge_rounds and k_merge_loop with mg_on) at the limits test_gpu_block_cells and
test_gpu_loop_stage pin for one GPU: staged cells and their exchange, a full list of touched cells (locally, or only once the
ranks' records are summed), the records of a round against the inbox, position tie-breaks across ranks, the tie mailbox, the
hand-off of merges above R_HUGE global sites, the born-pair cut and the last token indices.  A device group (bpe_create_group)
trains each corpus; its merge log (a, b, weight) and corpus must equal one engine's and the incremental CPU oracle's
(oracle/fast_oracle.py).  On a host with fewer GPUs than members, the members share GPU 0 (BPE_GROUP_SHARE_DEVICE=1).

Layouts: "split" uploads the corpus once, so it is balanced over the members; "last" uploads the first document, then the
rest, which goes whole to the last member (a group partitions only its first upload).  Every case checks on the corpus, or
in the stats, that it reaches the limit it is named after."""
import numpy as np
import pytest

from test_gpu_block_cells import STAGE, _alphabet, _mixed
from test_gpu_loop_stage import _giant_corpus

pytestmark = pytest.mark.gpu

R_HUGE = 1 << 20        # round_kernels.cuh: a merge with more counted occurrences runs in k_merge_loop(_mg)
R_LISTCAP = 32768       # touched cells one block lists per round
INBOX_RECORDS = (1 << 20) - 64  # records one rank can send per exchange (MG_INBOX_STRIDE - MGR_HDR)
TIE_CAP = 4096          # candidates the tie mailbox holds
MAX_TOKENS = 56319      # BPE_MAX_TOKENS
LOOPS = pytest.mark.parametrize("loop_rounds", [None, "0"], ids=["rounds", "loop"])


def _devices(members, monkeypatch):
    import torch

    n = torch.cuda.device_count()
    if n >= members and all(torch.cuda.can_device_access_peer(a, b) for a in range(members) for b in range(members) if a != b):
        return list(range(members))
    monkeypatch.setenv("BPE_GROUP_SHARE_DEVICE", "1")  # (read by bpe_create_group when it is called)
    return [0] * members


def _set(monkeypatch, **env):
    for k, v in env.items():
        if v is None:
            monkeypatch.delenv(k, raising=False)
        else:
            monkeypatch.setenv(k, v)


def _engine(devs, chars):
    from bpe_tokenizer_b200 import BPETokenizer

    t = BPETokenizer(devices=devs) if devs is not None else BPETokenizer()
    t.addToCorpus("".join(chr(c) for c in chars))
    t.corpus_in_code = []
    for tk in t.token_table:
        tk.weight = tk.original_weight = 0
    return t


def _upload(t, ids, off, layout):
    if layout == "split":
        t.addDocuments(ids, off)
    else:  # the first document alone, then the body: a later upload goes whole to the last member
        t.addDocuments(ids[: off[1]], off[:2] - off[0])
        t.addDocuments(ids[off[1]:], off[1:] - off[1])


def _shards(off, n):
    """First document of each member after a first upload (bpe_b200.cu, shard_bounds: balanced by ids)."""
    total = int(off[-1] - off[0])
    b, d = [0], 0
    for r in range(1, n):
        cut = (total * r + n - 1) // n
        while d < len(off) - 1 and off[d] - off[0] < cut:
            d += 1
        b.append(d)
    return b + [len(off) - 1]


def _log(t):
    return [[a.index, b.index, c.original_weight] for a, b, c in t.merge_tokens]


def _first_bad(got, want):
    return next((i for i, (g, w) in enumerate(zip(got, want)) if g != w), None)


def _oracle(ids, off, chars, merges):
    from oracle.fast_oracle import FastOracle

    o = FastOracle()
    o.set_len16(np.ones(len(chars), dtype=np.int32))
    o.add_documents(ids, off)
    la, lb, lw = o.merge_until(2, 0, merges, len(chars), merges)
    return o, [[int(a), int(b), int(w)] for a, b, w in zip(la, lb, lw)]


def _check_group(ids, off, n_alpha, merges, devs, layout, chars=None):
    """Trains a group on `devs`, one engine and the oracle on the same ids; merge logs and corpora must be equal.  -> the
    group's stats() and the one engine's."""
    chars = _alphabet(n_alpha) if chars is None else chars
    o, want = _oracle(ids, off, chars, merges)
    stats = []
    for d in (devs, None):
        t = _engine(d, chars)
        _upload(t, ids, off, layout)
        n = t.mergeUntil({"max_iterations": merges})
        got = _log(t)
        bad = _first_bad(got, want)
        assert bad is None, ("group" if d else "one engine", bad, got[bad], want[bad])
        assert n == len(got) == len(want)
        assert np.array_equal(t.corpusIds()[0], o.corpus())
        stats.append(t.stats())
        t.close()
    return stats[0], stats[1]


def _docs(rows):
    """documents given as equal-length rows of a 2-d array -> (ids, offsets)"""
    rows = np.asarray(rows, dtype=np.int32)
    return rows.ravel(), np.arange(0, rows.size + 1, rows.shape[1], dtype=np.int64)


def _cat(*parts):
    ids = np.concatenate([p[0] for p in parts])
    offs, base = [np.zeros(1, np.int64)], 0
    for i, o in parts:
        offs.append(o[1:] - o[0] + base)
        base += int(o[-1] - o[0])
    return ids, np.concatenate(offs)


def _sites(ids, off, a, b, lo=0, hi=None):
    """occurrences of (a, b), a != b, inside documents lo .. hi - 1"""
    hi = len(off) - 1 if hi is None else hi
    s, e = int(off[lo]), int(off[hi])
    x = ids[s:e]
    start = np.zeros(e - s + 1, bool)
    start[(off[lo:hi + 1] - s).astype(np.int64)] = True
    return int(np.count_nonzero((x[:-1] == a) & (x[1:] == b) & ~start[1:e - s]))


# ---- staged cells and the summing of the ranks' records (mgr_collect) ----
@pytest.mark.parametrize("members", [2, 4])
@pytest.mark.parametrize("stage", ["on", "off"])
def test_group_staged_cells_equal_the_oracle(stage, members, monkeypatch):
    devs = _devices(members, monkeypatch)
    _set(monkeypatch, BPE_BLOCK_CELLS_MIN_SITES=STAGE[stage], BPE_LOOP_ROUNDS=None, BPE_LOOP_BLOCKS=None)
    ids, off = _mixed(1, 3_000_000)
    st, _ = _check_group(ids, off, 600, 1500, devs, "split")
    assert st["loop_round_merges"] > 1.5 * st["loop_rounds"], st  # rounds of several merges that share neighbours


# ---- a full list of touched cells: on one member (the row scan of round_emit_records) or only globally (goverflow) ----
def _full_list_corpus():
    n = 17_000
    x = np.arange(2, 2 + n, dtype=np.int32)
    head = _docs(np.stack([x, np.zeros(n, np.int32), np.ones(n, np.int32), x[::-1]], axis=1))
    return _cat(head, _mixed(3, 40_000)), n


@pytest.mark.parametrize("layout", ["split", "last"])
@pytest.mark.parametrize("stage", ["on", "off"])
def test_group_full_cell_list(stage, layout, monkeypatch):
    """One block per member; the first merge (0, 1) has 17 000 sites with a different neighbour on either side: 34 000 cells,
    over R_LISTCAP.  Split over two members, each member's list holds its half (the exchange's GLOBAL list is full); with the
    head on the last member, that member's own list is full too and it sends its records from a scan of the rows."""
    devs = _devices(2, monkeypatch)
    _set(monkeypatch, BPE_BLOCK_CELLS_MIN_SITES=STAGE[stage], BPE_LOOP_BLOCKS="1", BPE_LOOP_ROUNDS=None)
    (ids, off), n = _full_list_corpus()
    assert 2 * n > R_LISTCAP
    if layout == "split":
        b = _shards(off, 2)
        local = [2 * min(max(0, min(b[r + 1], n) - b[r]), n) for r in range(2)]  # head documents of member r, two cells each
        assert sum(local) == 2 * n and max(local) < R_LISTCAP, local
    else:
        assert 2 * (n - 1) > R_LISTCAP  # every head document but the first is on the last member
    _check_group(ids, off, 2 + n, 300, devs, layout)


# ---- the records of a round against the peers' inboxes ----
def _inbox_corpus(pairs, sites, seed):
    """`pairs` pairs (a_j, b_j) of pairwise disjoint tokens 0 .. 2 pairs - 1, pair j in `sites` - j documents [x, a_j, b_j, y]
    whose x differ from each other, and so do the y: every touched cell of a round is a record of its own."""
    rng = np.random.default_rng(seed)
    rows = []
    for j in range(pairs):
        m = sites - j
        x = 2 * pairs + rng.permutation(m)
        y = 2 * pairs + rng.permutation(m)
        rows.append(np.stack([x, np.full(m, 2 * j), np.full(m, 2 * j + 1), y], axis=1))
    rows = np.concatenate(rows)[rng.permutation(sum(sites - j for j in range(pairs)))]
    return _docs(rows), 2 * pairs + sites


def _records_bound(pairs, sites, n_alpha):
    """records a rank can send for a batch of the first k merges, k = 1 .. pairs: sum of 2 min(w_i, c_i + 1)"""
    return np.cumsum([2 * min(sites - j, n_alpha + j + 1) for j in range(pairs)])


@pytest.mark.parametrize("sites", [53_000, 30_000], ids=["over", "fits"])
def test_group_round_records_fit_the_inbox(sites, monkeypatch):
    """16 pairs on the last member.  At 53 000 sites a batch of ten or more of their merges would send more records than a
    peer's inbox holds; at 30 000 all 16 would fit.  A round's records are at most the keys its born pairs may add, so the
    room of the hot list (at least 4 x 32 768 keys) ends these batches first: one merge per round at 53 000 (two merges would
    add up to 212 004 keys), two at 30 000.  The decisions on the group equal one engine's."""
    devs = _devices(2, monkeypatch)
    _set(monkeypatch, BPE_LOOP_ROUNDS=None, BPE_LOOP_BLOCKS=None, BPE_BLOCK_CELLS_MIN_SITES=None)
    (ids, off), n_alpha = _inbox_corpus(16, sites, 5)
    bound = _records_bound(16, sites, n_alpha)
    if sites == 53_000:
        assert bound[8] <= INBOX_RECORDS < bound[9], bound  # nine merges fit, ten do not
    else:
        assert bound[-1] <= INBOX_RECORDS, bound
    g, one = _check_group(ids, off, n_alpha, 16, devs, "last")
    assert g["loop_round_merges"] == g["loop_round_tried"] == 16, g
    assert g["loop_rounds"] == one["loop_rounds"] == (16 if sites == 53_000 else 8), (g, one)


# ---- position tie-breaks across ranks (mg_tie_winner: (rank, last local position)) ----
def _tie_corpus():
    """Four quarters of 4 000 ids each (the members' shards at 2 and at 4 members); documents [50] only pad a quarter.
    Tied groups (same count, same a + b), settled by the last counted occurrence in (rank, local position) order:
      (5, 10) / (6, 9), 3 000 each: (5, 10) only in quarters 0-1 (absent from the highest rank), (6, 9) last in quarter 3.
      (21, 29) / (20, 30), 500 each: (21, 29)'s last occurrence opens quarter 3 (local position 0 of rank 3 of 4), (20, 30)'s
      last is in quarter 2, so (20, 30) wins -- it would lose if the occurrence at position 0 were missed.
      (40, 40) / (39, 41), 400 counted each: quarter 2 opens with the run 40 40 40 (two raw occurrences, one counted)."""
    q = [
        [[5, 10]] * 1500 + [[6, 9]] * 300 + [[21, 29]] * 200,
        [[5, 10]] * 1500 + [[21, 29]] * 299 + [[39, 41]] * 150 + [[50]] * 102,
        [[40, 40, 40]] + [[40, 40]] * 399 + [[6, 9]] * 1099 + [[20, 30]] * 500 + [[50]],
        [[21, 29]] + [[6, 9]] * 1601 + [[39, 41]] * 250 + [[50]] * 296,
    ]
    parts = []
    for docs in q:
        ids = np.concatenate([np.asarray(d, np.int32) for d in docs])
        off = np.concatenate([[0], np.cumsum([len(d) for d in docs])]).astype(np.int64)
        parts.append((ids, off))
    return _cat(*parts), [len(p[0]) for p in parts]


def test_tie_corpus_layout():
    (ids, off), lens = _tie_corpus()
    assert _sites(ids, off, 5, 10) == _sites(ids, off, 6, 9) == 3000
    assert _sites(ids, off, 21, 29) == _sites(ids, off, 20, 30) == 500
    assert _sites(ids, off, 39, 41) == 400 and lens == [4000] * 4


@LOOPS
@pytest.mark.parametrize("members", [2, 4])
def test_group_ties_across_ranks(members, loop_rounds, monkeypatch):
    devs = _devices(members, monkeypatch)
    _set(monkeypatch, BPE_LOOP_ROUNDS=loop_rounds, BPE_LOOP_BLOCKS=None, BPE_BLOCK_CELLS_MIN_SITES=None)
    (ids, off), lens = _tie_corpus()
    b = _shards(off, members)
    starts = [int(off[d]) for d in b[:-1]]
    quarters = np.concatenate([[0], np.cumsum(lens)])[:4].tolist()
    assert starts == quarters[:: 4 // members], (starts, quarters)  # every member holds whole quarters
    g, _ = _check_group(ids, off, 64, 40, devs, "split")
    assert g["tie_breaks"] > 0, g


# ---- the tie mailbox: 4 096 candidates at most ----
def _mailbox_corpus(n_tied):
    """(9000, 9001) in three documents, then n_tied pairs (x, S - x) in two documents each: after the first merge, n_tied
    candidates tie on (2, S)."""
    s = 2 * n_tied + 1
    x = np.arange(1, n_tied + 1, dtype=np.int32)
    tied = np.stack([x, s - x], axis=1)
    rows = np.concatenate([np.array([[9000, 9001]] * 3, np.int32), tied, tied])
    return _docs(rows), 9002


def test_group_tie_mailbox(monkeypatch):
    from bpe_tokenizer_b200 import BpeError
    from bpe_tokenizer_b200._abi import BPE_E_DOMAIN

    devs = _devices(2, monkeypatch)
    _set(monkeypatch, BPE_LOOP_ROUNDS=None, BPE_LOOP_BLOCKS=None, BPE_BLOCK_CELLS_MIN_SITES=None)
    # as many candidates as the mailbox holds: equal to the oracle (the first 60 merges: every one a tie-break)
    (ids, off), n_alpha = _mailbox_corpus(TIE_CAP - 96)
    g, _ = _check_group(ids, off, n_alpha, 60, devs, "split")
    assert g["tie_breaks"] >= 59, g
    # one more than it holds: the group refuses the tie, after the merges before it; one engine takes it (a documented difference)
    (ids, off), n_alpha = _mailbox_corpus(TIE_CAP + 1)
    chars = _alphabet(n_alpha)
    _, want = _oracle(ids, off, chars, 3)
    grp = _engine(devs, chars)
    _upload(grp, ids, off, "split")
    with pytest.raises(BpeError) as ex:
        grp.mergeUntil({"max_iterations": 3})
    assert ex.value.code == BPE_E_DOMAIN and "tie mailbox" in str(ex.value), str(ex.value)
    assert _log(grp) == want[:1]  # (9000, 9001), then the tie
    one = _engine(None, chars)
    _upload(one, ids, off, "split")
    assert one.mergeUntil({"max_iterations": 3}) == 3 and _log(one) == want
    one.close()
    # the group trains again after its corpus is cleared
    grp.corpus_in_code = []
    (ids, off), n_alpha = _mailbox_corpus(TIE_CAP - 96)
    grp.addDocuments(ids, off)
    _, want = _oracle(ids, off, chars, 5)
    assert grp.mergeUntil({"max_iterations": 5}) == 5
    assert _log(grp)[1:] == want
    grp.close()


# ---- merges above R_HUGE global sites: the decision on global counts, the sharded k_merge_loop, and back ----
def test_group_giant_merge_on_global_counts(monkeypatch):
    """1.1 M sites of (0, 1) split over two members: neither holds more than R_HUGE, the corpus does."""
    devs = _devices(2, monkeypatch)
    _set(monkeypatch, BPE_LOOP_ROUNDS=None, BPE_LOOP_BLOCKS=None, BPE_BLOCK_CELLS_MIN_SITES=None)
    ids, off = _giant_corpus(7, 1_100_000)
    b = _shards(off, 2)
    local = [_sites(ids, off, 0, 1, b[r], b[r + 1]) for r in range(2)]
    assert max(local) <= R_HUGE < sum(local), local
    g, one = _check_group(ids, off, 600, 300, devs, "split")
    assert 0 < g["loop_round_merges"] < 300, g  # the rounds take every merge but the giant
    assert g["loop_round_merges"] == one["loop_round_merges"], (g, one)


@pytest.mark.parametrize("extra", [0, 1], ids=["2^20", "2^20+1"])
@pytest.mark.parametrize("kind", ["pair", "run"])
def test_group_r_huge_boundary(kind, extra, monkeypatch):
    """One pair with exactly R_HUGE (+ extra) counted occurrences, every site with the same left and the same right
    neighbour, so one delta cell counts all of them (a 21-bit field at its largest); all on the last member.  At R_HUGE the
    rounds take every merge; one more occurrence sends exactly that merge to the one-merge kernel."""
    devs = _devices(2, monkeypatch)
    _set(monkeypatch, BPE_LOOP_ROUNDS=None, BPE_LOOP_BLOCKS=None, BPE_BLOCK_CELLS_MIN_SITES=None)
    if kind == "pair":
        body = _docs(np.tile(np.array([[5, 0, 1, 6]], np.int32), (R_HUGE, 1)))
        first, a, b = [0, 1], 0, 1
    else:  # (0, 0) in runs of three: two raw occurrences, one counted
        body = _docs(np.tile(np.array([[5, 0, 0, 0, 6]], np.int32), (R_HUGE, 1)))
        first, a, b = [0, 0], 0, 0
    head = _docs(np.array([[7, 8]], np.int32))  # (the first upload: one document)
    parts = [head, body] + ([_docs(np.array([first], np.int32))] if extra else [])
    ids, off = _cat(*parts)
    _, want = _oracle(ids, off, _alphabet(10), 3)
    assert want[0][:2] == [a, b] and want[0][2] == R_HUGE + extra and all(w[2] == R_HUGE for w in want[1:]), want
    g, one = _check_group(ids, off, 10, 3, devs, "last")
    for s in (g, one):
        assert s["loop_round_merges"] == 3 - extra, s


# ---- the born-pair bound cuts a batch ----
def test_group_born_pair_cut(monkeypatch):
    """(10, 11) with 1 000 sites, 900 of them followed by 12; then (2, 3) with 900 and (11, 12) with 900 (larger a + b).  The
    batch [(10, 11), (2, 3)] is cut after its first merge: the born pair (c, 12) reaches 900, (2, 3)'s count."""
    devs = _devices(2, monkeypatch)
    _set(monkeypatch, BPE_LOOP_ROUNDS=None, BPE_LOOP_BLOCKS=None, BPE_BLOCK_CELLS_MIN_SITES=None)
    rows = [[10, 11, 12]] * 900 + [[10, 11, 13]] * 100 + [[2, 3, 14]] * 900
    rng = np.random.default_rng(3)
    rows = np.array(rows, np.int32)[rng.permutation(len(rows))]
    ids, off = _docs(rows)
    g, one = _check_group(ids, off, 20, 6, devs, "split")
    assert g["loop_rounds_cut"] > 0 and one["loop_rounds_cut"] > 0, (g, one)


# ---- the last token indices: rows near ND_STRIDE, and mergeUntil up to BPE_MAX_TOKENS ----
def _wide_alphabet(n):
    """n single-character tokens from U+4E00 on, without the surrogates U+D800..U+DFFF"""
    cps = [c for c in range(0x4E00, 0x4E00 + n + 0x800) if not 0xD800 <= c <= 0xDFFF]
    return cps[:n]


@pytest.mark.parametrize("members", [None, 2], ids=["one", "group"])
def test_merge_until_up_to_the_last_token(members, monkeypatch):
    from bpe_tokenizer_b200 import BpeError
    from bpe_tokenizer_b200._abi import BPE_E_DOMAIN

    devs = _devices(members, monkeypatch) if members else None
    _set(monkeypatch, BPE_LOOP_ROUNDS=None, BPE_LOOP_BLOCKS=None, BPE_BLOCK_CELLS_MIN_SITES=None)
    n_alpha = MAX_TOKENS - 300
    chars = _wide_alphabet(n_alpha)
    rng = np.random.default_rng(9)
    top = np.arange(n_alpha - 400, n_alpha, dtype=np.int32)  # the neighbours: the highest ids of the alphabet
    p = 1.0 / np.arange(1, top.size + 1)
    ids = rng.choice(top, size=400_000, p=p / p.sum()).astype(np.int32)
    cuts = np.cumsum(rng.integers(2, 40, size=ids.size // 8))
    off = np.concatenate([[0], cuts[cuts < ids.size], [ids.size]]).astype(np.int64)
    o, want = _oracle(ids, off, chars, 300)
    assert len(want) == 300
    t = _engine(devs, chars)
    _upload(t, ids, off, "split")
    assert len(t.token_table) == n_alpha
    assert t.mergeUntil() == 300  # exactly the room left
    assert _log(t) == want
    assert np.array_equal(t.corpusIds()[0], o.corpus())
    with pytest.raises(BpeError) as ex:
        t.mergeUntil()
    assert ex.value.code == BPE_E_DOMAIN
    t.close()
