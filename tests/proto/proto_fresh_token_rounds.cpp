// PROTOTYPE / MEASUREMENT ONLY (test infrastructure, never linked into the product).
//
// What refusing tokens of the previous round costs k_merge_rounds: the batcher "K16 disjoint-tokens (adjacency handled)" of
// proto_batch_stats.cpp, replayed over the exact merge sequence of the incremental CPU oracle, once as the device now builds
// its batches and once with the rule it no longer has -- merges 1.. of a round may not hold a token the previous round
// created (their occurrence lists were still being written).  Prints both batchers' small merges, rounds and batch ends.
//
//   g++ -O2 -std=c++17 -pthread -o /tmp/proto_fresh_token_rounds tests/proto/proto_fresh_token_rounds.cpp bpe_tokenizer_b200/csrc/synth.cpp
//   /tmp/proto_fresh_token_rounds <bytes> <merges> [max_length]
#define main proto_batch_stats_main
#include "proto_batch_stats.cpp"
#undef main

namespace {

enum FreshReason { F_ORDER = 0, F_TIE, F_TOKENS, F_BIG, F_CAP, F_FRESH, F_N };
const char* fresh_reason_name[F_N] = {"not-the-next-candidate", "tie-on-primary", "shares-a-token", "big-merge", "cap-K",
                                      "token-of-the-previous-round"};

struct FreshBatcher {
  const char* name;
  bool forbid_fresh;
  std::vector<Cand> cands;
  size_t i = 0;
  int32_t c_first = INT32_MAX, prev_c_first = INT32_MAX;  // first token of the current / previous round
  std::set<int32_t> toks;
  int64_t merges_small = 0, rounds_small = 0, merges_big = 0;
  int64_t ends[F_N] = {0};
};

}  // namespace

int main(int argc, char** argv) {
  const size_t K = 16;
  const int64_t small_limit = 16384;
  int64_t bytes = argc > 1 ? atoll(argv[1]) : 16000000;
  int64_t M = argc > 2 ? atoll(argv[2]) : 4000;
  int32_t max_length = argc > 3 ? atoi(argv[3]) : 0;
  int64_t nb = 0, nd = 0;
  bpe_synth_corpus(bytes, 43, 50000, 42, nullptr, 0, nullptr, 0, &nb, &nd);
  std::vector<uint8_t> text(nb);
  std::vector<int64_t> off(nd + 1);
  bpe_synth_corpus(bytes, 43, 50000, 42, text.data(), nb, off.data(), nd + 1, &nb, &nd);
  std::vector<int32_t> ids(nb);
  int32_t map[256];
  for (int i = 0; i < 256; i++) map[i] = -1;
  int32_t T = 0;
  for (int64_t i = 0; i < nb; i++) {
    if (map[text[i]] < 0) map[text[i]] = T++;
    ids[i] = map[text[i]];
  }
  Fast F;
  fast_add_documents(&F, ids.data(), off.data(), nd);
  F.len16.assign(T, 1);
  build(F);
  fprintf(stderr, "corpus %lld bytes, %lld docs, %d chars\n", (long long)nb, (long long)nd, T);

  FreshBatcher B[2] = {{"K16 disjoint-tokens (adjacency handled)", false}, {"K16 disjoint-tokens, no token of the previous round", true}};
  int64_t done = 0;
  while (done < M) {
    std::vector<Cand> snap = topk(F, 18, max_length);
    uint64_t key;
    int64_t cnt;
    bool tie;
    if (!find_next(F, 2, max_length, &key, &cnt, &tie)) break;
    const int32_t a = (int32_t)(key >> 32), b = (int32_t)(key & 0xFFFFFFFFu), c = T + (int32_t)done;
    for (FreshBatcher& x : B) {
      const bool big = cnt > small_limit;
      int reason = -1;
      if (x.i == 0) reason = -2;  // nothing open
      else if (big) reason = F_BIG;
      else if (x.i >= K) reason = F_CAP;
      else if (x.i >= x.cands.size() || x.cands[x.i].key != key || x.cands[x.i].count != cnt) reason = F_ORDER;
      else if (tie || (x.i + 1 < x.cands.size() && x.cands[x.i + 1].count == cnt && x.cands[x.i + 1].negsum == x.cands[x.i].negsum)) reason = F_TIE;
      else if (a >= x.c_first || b >= x.c_first || x.toks.count(a) || x.toks.count(b)) reason = F_TOKENS;
      else if (x.forbid_fresh && (a >= x.prev_c_first || b >= x.prev_c_first)) reason = F_FRESH;
      if (reason != -1) {  // this merge opens a new round
        if (reason >= 0) x.ends[reason]++;
        x.cands = snap;
        x.i = 0;
        x.prev_c_first = x.c_first;
        x.c_first = c;
        x.toks.clear();
        if (big) {  // a big merge runs alone and is not counted as a round of the latency-bound regime
          x.merges_big++;
          continue;
        }
        x.rounds_small++;
      }
      x.merges_small++;
      x.toks.insert(a);
      x.toks.insert(b);
      x.i++;
    }
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
  printf("after %lld merges\n", (long long)done);
  for (const FreshBatcher& x : B) {
    printf("%-52s small merges %lld in %lld rounds = %.2f per round; big %lld; ends:", x.name, (long long)x.merges_small, (long long)x.rounds_small,
           x.rounds_small ? (double)x.merges_small / x.rounds_small : 0.0, (long long)x.merges_big);
    for (int r = 0; r < F_N; r++) printf(" %s=%lld", fresh_reason_name[r], (long long)x.ends[r]);
    printf("\n");
  }
  return 0;
}
