// TEST INFRASTRUCTURE ONLY -- a second, INCREMENTAL CPU oracle for mergeUntil (core.ts:365-383).
//
// int_oracle.cpp restates the reference literally (count every pair of the whole corpus, rewrite every document, per
// merge) and cannot reach BASELINE config 3 (1 GB x 32 000 merges).  This file computes the same merge sequence with
// work proportional to the occurrences a merge touches, so that the FULL cfg3 run of the GPU can be checked on a CPU
// (BASELINE.md section 2: "a separate fast (incremental) CPU oracle that is itself proven equal to the literal one").
// It is pinned by fuzzing against the literal oracles (tests/test_oracle_golden.py) and shares no code and no
// bookkeeping scheme with the CUDA engine:
//   * the corpus is a doubly linked list over positions (a merged token keeps the position of its left half);
//   * counts are NOT updated by hand-derived deltas: around every merge site the literal counting rule of
//     core.ts:265-310 (adjacent pairs inside a document; inside a run of identical tokens every other pair, :285-290)
//     is re-applied to a window that starts and ends on run boundaries -- once before the replacement (subtract) and
//     once after it (add);
//   * the arg-max is a lazy max-heap on (count, -(a.index + b.index)); among pairs that tie on both, the winner is
//     the one whose LAST counted occurrence comes first in scan order (the consequence of the running maximum of
//     core.ts:294-305, SURVEY.md A.2), found by walking the tied pairs' occurrence lists from the back.
// Nothing here is linked into, or called by, the product library.
//
// Build: see oracle/Makefile  (g++ -O2 -shared -fPIC).
#include <algorithm>
#include <cstdint>
#include <queue>
#include <tuple>
#include <unordered_map>
#include <vector>

namespace {

constexpr uint32_t NONE = 0xFFFFFFFFu;

struct PairInfo {
  int64_t count = 0;
  uint32_t touched = 0;          // merge number + 1 of the last change (one heap entry per change)
  std::vector<uint32_t> occ;     // position of the left token of every adjacency this pair ever had, ascending
};

struct Fast {
  std::vector<int32_t> tok;      // token at a position; -1: the position no longer starts a token
  std::vector<uint32_t> nxt, prv;
  std::vector<uint8_t> first;    // the position starts a document (no pair reaches across, core.ts:265-267)
  std::vector<uint32_t> doc_start;  // first position of every document, empty ones included (they hold no position)
  std::vector<int32_t> len16;    // UTF-16 length of token.chars (the max_length test, core.ts:270-273)
  std::unordered_map<uint64_t, PairInfo> pairs;
  typedef std::tuple<int64_t, int64_t, uint64_t> Entry;  // count, -(a + b), key
  std::priority_queue<Entry> heap;
  bool built = false;
  uint32_t merge_no = 0;
  std::vector<uint64_t> changed;
};

inline uint64_t key_of(int32_t a, int32_t b) { return ((uint64_t)(uint32_t)a << 32) | (uint32_t)b; }

// right neighbour inside the same document, or NONE
inline uint32_t right_of(const Fast& F, uint32_t p) {
  uint32_t q = F.nxt[p];
  return (q == NONE || F.first[q]) ? NONE : q;
}
inline uint32_t left_of(const Fast& F, uint32_t p) { return F.first[p] ? NONE : F.prv[p]; }

uint32_t run_start(const Fast& F, uint32_t p) {
  for (;;) {
    uint32_t l = left_of(F, p);
    if (l == NONE || F.tok[l] != F.tok[p]) return p;
    p = l;
  }
}
uint32_t run_end(const Fast& F, uint32_t p) {
  for (;;) {
    uint32_t r = right_of(F, p);
    if (r == NONE || F.tok[r] != F.tok[p]) return p;
    p = r;
  }
}

void note_change(Fast& F, uint64_t key, PairInfo& pi) {
  if (pi.touched != F.merge_no + 1) {
    pi.touched = F.merge_no + 1;
    F.changed.push_back(key);
  }
}

// The literal counting rule over the tokens lo..hi (lo starts a run, hi ends one): sign = -1 takes the window's pairs out
// of the counts, sign = +1 puts them in.  new_tok >= 0 (only with +1): adjacencies that involve the token the current
// merge creates are new, their left positions join the pair's occurrence list.
void count_window(Fast& F, uint32_t lo, uint32_t hi, int sign, int32_t new_tok) {
  uint32_t p = lo, k = 0;  // k: index of p inside its run of identical tokens
  while (p != hi) {
    uint32_t q = F.nxt[p];
    if (F.first[q]) {      // (cannot happen inside a window: windows never span documents)
      k = 0;
      p = q;
      continue;
    }
    int32_t a = F.tok[p], b = F.tok[q];
    bool counted = (a != b) || ((k & 1u) == 0);  // core.ts:285-290: every other pair of a run
    uint64_t key = key_of(a, b);
    if (counted || (sign > 0 && (a == new_tok || b == new_tok))) {
      PairInfo& pi = F.pairs[key];
      if (counted) {
        pi.count += sign;
        note_change(F, key, pi);
      }
      if (sign > 0 && (a == new_tok || b == new_tok)) pi.occ.push_back(p);
    }
    k = (a == b) ? k + 1 : 0;
    p = q;
  }
}

void build(Fast& F) {
  F.pairs.clear();
  while (!F.heap.empty()) F.heap.pop();
  const size_t n = F.tok.size();
  uint32_t k = 0;
  for (size_t p = 0; p + 1 < n; p++) {
    if (F.first[p]) k = 0;
    if (F.first[p + 1]) continue;
    int32_t a = F.tok[p], b = F.tok[p + 1];
    PairInfo& pi = F.pairs[key_of(a, b)];
    if (a != b || (k & 1u) == 0) pi.count++;
    pi.occ.push_back((uint32_t)p);
    k = (a == b) ? k + 1 : 0;
  }
  for (auto& kv : F.pairs)
    if (kv.second.count > 0) F.heap.emplace(kv.second.count, -(int64_t)((kv.first >> 32) + (kv.first & 0xFFFFFFFFu)), kv.first);
  F.built = true;
}

bool occurs_at(const Fast& F, uint32_t p, int32_t a, int32_t b) {
  if (F.tok[p] != a) return false;
  uint32_t q = right_of(F, p);
  return q != NONE && F.tok[q] == b;
}

// position of the last COUNTED occurrence of (a, b), or NONE
uint32_t last_counted(const Fast& F, const PairInfo& pi, int32_t a, int32_t b) {
  for (size_t i = pi.occ.size(); i-- > 0;) {
    uint32_t p = pi.occ[i];
    if (!occurs_at(F, p, a, b)) continue;
    if (a != b) return p;
    uint32_t k = 0;  // index of p inside its run
    for (uint32_t l = left_of(F, p); l != NONE && F.tok[l] == a; l = left_of(F, l)) k++;
    if ((k & 1u) == 0) return p;
  }
  return NONE;
}

struct Window {
  uint32_t lo, hi;
  size_t site_begin, site_end;
};

// core.ts:332-360: replace (a, b) by c left to right, non-overlapping; counts follow
int64_t apply_merge(Fast& F, int32_t a, int32_t b, int32_t c) {
  auto it = F.pairs.find(key_of(a, b));
  if (it == F.pairs.end()) return 0;
  std::vector<uint32_t> occ = it->second.occ;  // (the map may rehash below)
  if (!std::is_sorted(occ.begin(), occ.end())) std::sort(occ.begin(), occ.end());
  std::vector<uint32_t> sites;
  uint32_t blocked = NONE;  // the right half of the site just taken cannot start another one (runs of a == b)
  for (uint32_t p : occ) {
    if (!sites.empty() && p == sites.back()) continue;
    if (p == blocked || !occurs_at(F, p, a, b)) continue;
    sites.push_back(p);
    blocked = F.nxt[p];
  }
  // windows: from the start of the run that holds the left neighbour to the end of the run that holds the right one
  std::vector<Window> win;
  for (size_t i = 0; i < sites.size(); i++) {
    uint32_t p = sites[i], q = F.nxt[p];
    uint32_t x = left_of(F, p), y = right_of(F, q);
    uint32_t lo = x == NONE ? p : run_start(F, x), hi = y == NONE ? q : run_end(F, y);
    if (!win.empty() && lo <= win.back().hi) {
      win.back().hi = std::max(win.back().hi, hi);
      win.back().site_end = i + 1;
    } else {
      win.push_back(Window{lo, hi, i, i + 1});
    }
  }
  for (const Window& w : win) {
    count_window(F, w.lo, w.hi, -1, -1);
    uint32_t hi = w.hi;
    for (size_t i = w.site_begin; i < w.site_end; i++) {
      uint32_t p = sites[i], q = F.nxt[p], r = F.nxt[q];
      F.tok[p] = c;
      F.tok[q] = -1;
      F.nxt[p] = r;
      if (r != NONE) F.prv[r] = p;
      if (hi == q) hi = p;
    }
    count_window(F, w.lo, hi, +1, c);
  }
  return (int64_t)sites.size();
}

}  // namespace

extern "C" {

void* fast_create() { return new Fast(); }
void fast_destroy(void* h) { delete static_cast<Fast*>(h); }

void fast_set_len16(void* h, const int32_t* len16, int32_t n) { static_cast<Fast*>(h)->len16.assign(len16, len16 + n); }

// documents in addToCorpus order (core.ts:182-207); ids = single-character token indices
int fast_add_documents(void* h, const int32_t* ids, const int64_t* off, int64_t n_docs) {
  Fast& F = *static_cast<Fast*>(h);
  if (n_docs <= 0) return 0;
  const size_t want = F.tok.size() + (size_t)(off[n_docs] - off[0]);
  if (want >= NONE) return -1;
  F.tok.reserve(want);
  F.first.reserve(want);
  F.prv.reserve(want);
  F.nxt.reserve(want);
  for (int64_t d = 0; d < n_docs; d++) {
    F.doc_start.push_back((uint32_t)F.tok.size());
    for (int64_t i = off[d]; i < off[d + 1]; i++) {
      uint32_t p = (uint32_t)F.tok.size();
      F.tok.push_back(ids[i]);
      F.first.push_back(i == off[d] ? 1 : 0);
      F.prv.push_back(p == 0 ? NONE : p - 1);
      F.nxt.push_back(NONE);
      if (p > 0) F.nxt[p - 1] = p;
    }
  }
  F.built = false;
  return 0;
}

int64_t fast_total_tokens(void* h) {
  Fast& F = *static_cast<Fast*>(h);
  int64_t n = 0;
  for (int32_t t : F.tok) n += t >= 0;
  return n;
}

// current tokens of the whole corpus, documents back to back (out holds fast_total_tokens values)
void fast_get_corpus(void* h, int32_t* out) {
  Fast& F = *static_cast<Fast*>(h);
  if (F.tok.empty()) return;
  size_t k = 0;
  for (uint32_t p = 0; p != NONE; p = F.nxt[p]) out[k++] = F.tok[p];
}

int64_t fast_num_documents(void* h) { return (int64_t) static_cast<Fast*>(h)->doc_start.size(); }

// current number of tokens of every document, in addition order (out holds fast_num_documents values)
void fast_document_lengths(void* h, int64_t* out) {
  Fast& F = *static_cast<Fast*>(h);
  const size_t nd = F.doc_start.size();
  for (size_t d = 0; d < nd; d++) {
    const uint32_t end = d + 1 < nd ? F.doc_start[d + 1] : (uint32_t)F.tok.size();
    int64_t n = 0;
    for (uint32_t p = F.doc_start[d]; p < end; p++) n += F.tok[p] >= 0;
    out[d] = n;
  }
}

// mergeUntil (core.ts:365-383): falsy options mean the defaults (min_weight 2, no max_length, no iteration limit).
// Token c of merge i is first_new_index + i.  Returns the number of merges; la/lb/lw receive pair and weight.
int64_t fast_merge_until(void* h, int64_t min_weight, int32_t max_length, int64_t max_iterations, int32_t first_new_index, int32_t* la,
                         int32_t* lb, int64_t* lw, int64_t cap) {
  Fast& F = *static_cast<Fast*>(h);
  if (!F.built) build(F);
  if (min_weight <= 0) min_weight = 2;
  int64_t done = 0;
  // entries of pairs that this call's max_length excludes: set aside, not dropped, because a later call may allow them
  std::vector<Fast::Entry> too_long_kept;
  while (done < cap && (max_iterations <= 0 || done < max_iterations)) {
    // ---- findNextMerge (core.ts:247-326) ----
    std::vector<Fast::Entry> tied;
    while (!F.heap.empty()) {
      Fast::Entry e = F.heap.top();
      uint64_t key = std::get<2>(e);
      int32_t a = (int32_t)(key >> 32), b = (int32_t)(key & 0xFFFFFFFFu);
      auto it = F.pairs.find(key);
      bool stale = it == F.pairs.end() || it->second.count != std::get<0>(e);
      bool too_long = max_length > 0 && F.len16[a] + F.len16[b] > max_length;  // core.ts:270-273: never eligible
      if (!tied.empty() && !(std::get<0>(e) == std::get<0>(tied[0]) && std::get<1>(e) == std::get<1>(tied[0]))) break;
      F.heap.pop();
      if (stale) continue;
      if (too_long) {
        too_long_kept.push_back(e);
        continue;
      }
      bool dup = false;
      for (const Fast::Entry& t : tied) dup = dup || std::get<2>(t) == key;
      if (!dup) tied.push_back(e);
    }
    if (tied.empty() || std::get<0>(tied[0]) < min_weight) {  // core.ts:312-313
      for (const Fast::Entry& t : tied) F.heap.push(t);
      break;
    }
    size_t win = 0;
    if (tied.size() > 1) {  // the pair whose last counted occurrence comes first (core.ts:294-305)
      uint32_t best = NONE;
      for (size_t i = 0; i < tied.size(); i++) {
        uint64_t key = std::get<2>(tied[i]);
        uint32_t p = last_counted(F, F.pairs[key], (int32_t)(key >> 32), (int32_t)(key & 0xFFFFFFFFu));
        if (p < best) {
          best = p;
          win = i;
        }
      }
    }
    for (size_t i = 0; i < tied.size(); i++)
      if (i != win) F.heap.push(tied[i]);
    uint64_t key = std::get<2>(tied[win]);
    int32_t a = (int32_t)(key >> 32), b = (int32_t)(key & 0xFFFFFFFFu), c = first_new_index + (int32_t)done;
    la[done] = a;
    lb[done] = b;
    lw[done] = std::get<0>(tied[win]);
    // ---- applyMerge (core.ts:332-360) ----
    if ((int32_t)F.len16.size() <= c) F.len16.resize((size_t)c + 1, 0);
    F.len16[c] = F.len16[a] + F.len16[b];
    F.changed.clear();
    apply_merge(F, a, b, c);
    for (uint64_t k : F.changed) {
      const PairInfo& pi = F.pairs[k];
      if (pi.count > 0) F.heap.emplace(pi.count, -(int64_t)((k >> 32) + (k & 0xFFFFFFFFu)), k);
    }
    F.merge_no++;
    done++;
  }
  for (const Fast::Entry& e : too_long_kept) F.heap.push(e);
  return done;
}

}  // extern "C"
