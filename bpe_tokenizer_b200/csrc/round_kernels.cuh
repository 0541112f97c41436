// round_kernels.cuh -- mergeUntil (core.ts:365-383) as ROUNDS of several exact merges per pair of grid barriers.
//
// k_merge_loop (train_kernels.cuh) pays ~26 us of dependent L2/DRAM round trips and two grid barriers for EVERY merge,
// however small.  93 % of the merges of a 1 GB run are that small, and the next winner is almost always the runner-up of
// the current decision (tests/proto/proto_batch_stats.cpp: with the rules below a decision of the 1 GB-style Zipf corpus
// yields 6.3 exact merges on average when up to 8 are tried, 8.8 when up to 16).  This kernel therefore takes the best K
// pairs of ONE decision and runs their site passes side by side:
//
//   decide      every block folds the per-block top-2 partials into the exact, strictly ordered list of the best pairs
//               (exact down to the largest "second best" any block published) and builds the same batch m_0 .. m_{k-1}:
//               strictly decreasing (count, -(a+b)) keys, no tie inside the batch, pairwise disjoint tokens, capacities.
//               A pair with a token born in the previous round has its occurrence list still being written; its site pass
//               walks the site records of the merge of that round whose row holds the pair instead (RoundSm::src).
//   P1          site passes of all k merges over the corpus as it was at the decision.  A merge changes counts only of
//               pairs that contain a, b or c, so ALL its count deltas live in dense per-token rows (no hashing in P1): one
//               packed 64-bit cell per (merge, side, other token x) = decrements of the old pair (x,a) / (b,x) | occurrences
//               of the born pair (x,c) / (c,x) << 21 | its counted occurrences << 42; one ATOM.64 per warp and distinct
//               neighbour carries all three, and the thread that finds a cell empty appends it to its block's list, so
//               that P2 visits exactly the touched cells.  Token sets are disjoint, so the sites of m_j are the same
//               before and after m_0..m_{j-1}; only a NEIGHBOUR of a site can have been rewritten by an earlier merge of the
//               batch, and the site pass of m_j looks for exactly that: a left neighbour b_i preceded by a_i, or a right
//               neighbour a_i followed by b_i (i < j), is the token c_i there (virtual neighbour), its pair with a_j / b_j
//               is the born pair (c_i, a_j) / (b_j, c_i) of merge i, and the new adjacency is (c_i, c_j) / (c_j, c_i).
//               Per merge and side the pass also sums, over its warps, the largest number of lanes that share one
//               neighbour: an upper bound U of the count of ANY pair born by that merge (fire-and-forget adds).
//   -- barrier --
//   P2          every block computes the same valid prefix v: m_j is the exact next winner iff its count did not move
//               (true by token disjointness), every older pair outside the batch ranks below it (the list was exact) and no
//               pair born by m_0..m_{j-1} reaches its count (U_i < W_j for all i < j -- conservative).  Merges >= v are
//               dropped: they only ever wrote to their own rows.  For the v valid merges, side by side: the born pairs
//               enter the table (count minus what later valid merges took from them), the decrements are applied -- one
//               thread per (pair), which hands the pair's new key to the arg-max --, the corpus is rewritten, and the
//               arg-max runs over the old hot pairs that no valid merge touches.  -> per-block top-2 partials.
//   -- barrier --
//   The occurrence lists of the born pairs are filled next to P1 of the following round (as in k_merge_loop) on the helper
//   warps, which also zero the cells the round touched (from the same lists; cells are double-buffered by round parity).
//
// Sharded corpus (mg_on): P1 runs on the local shard into local cells; after its barrier every block sends the cells it
// listed as records to every rank (NVLink stores) and reports to a per-(receiver, parity, sender) arrival counter; every
// block sums the records of the senders that are complete into the GLOBAL cells (mgr_collect), P2 runs over those.  The
// decisions are replicated: U bounds and site counts are sums over the ranks, capacities minima (headers of the messages).
// The header, its fold, the waits on the peers' flags and the tie-break are mg_kernels.cuh's, shared with k_merge_loop.
//
// Exactness argument for the order inside a batch (SURVEY.md A.2, core.ts:294-305): counts of existing pairs never grow
// under merging, so an old pair that ranked below m_j at the decision still does; born pairs are bounded by U; m_j's own
// count is unchanged; equal keys never enter a batch (position tie-breaks run alone: phase_tie, as in k_merge_loop, or
// mg_tie_winner on a sharded corpus).
#pragma once
#include "train_kernels.cuh"
#include "mg_kernels.cuh"

namespace bpe {

#ifndef BPE_RD_THREADS
#define BPE_RD_THREADS 512
#endif
constexpr int RD_THREADS = BPE_RD_THREADS;  // threads per block of k_merge_rounds (one block per SM)
constexpr int RB = 16;                   // merges per round at most
#ifndef BPE_R_SMALL_LOG
#define BPE_R_SMALL_LOG 20
#endif
#ifndef BPE_R_BATCH_LOG
#define BPE_R_BATCH_LOG 21
#endif
// (measured on cfg3, one GPU: 2^18 / 2^19 -> 498 ms per step, 2^19 / 2^20 -> 485, 2^20 / 2^21 -> 475: batching the big merges saves
// their rounds' fixed costs, the dropped tails cost less than that)
constexpr uint32_t R_SMALL = 1u << BPE_R_SMALL_LOG;   // a merge with more counted occurrences than this runs alone (<= R_HUGE)
constexpr uint32_t R_BATCH_SITES = 1u << BPE_R_BATCH_LOG;  // ... and a batch stops growing past this many sites (a dropped tail wastes its site pass)
constexpr uint32_t R_LAT = 16384;        // below this many sites a merge is latency bound (profile classes, warp splits)

// One 64-bit cell per (merge of the round, side, other token): decrements of the old pair | occurrences of the born pair
// << 21 | counted occurrences of the born pair << 42 -- ONE atomic per warp and distinct neighbour carries all three.
constexpr uint32_t R_FIELD = 21;
constexpr unsigned long long R_FMASK = (1ull << R_FIELD) - 1ull;
static_assert(BPE_R_SMALL_LOG <= 20, "a batched merge must fit the 21-bit fields of the delta cells (R_HUGE)");
constexpr uint32_t R_HUGE = 1u << 20;    // merges with more counted occurrences overflow the fields: they run through k_merge_loop
constexpr uint32_t R_POOL_CHUNK = 1u << 16;  // occurrence-pool cells a block reserves at a time
constexpr uint32_t R_LISTCAP = 32768;    // touched cells a block can list per round (more: the round falls back to scanning the rows)
// Per-block staging of the cells of frequent neighbours (R_STAGE_T, train_kernels.cuh): in P1 of a merge whose occurrence list
// is longer than LoopArgs::stage_min, their cells are summed in shared memory and added to the global cells ONCE per block
// before P1's barrier (round_flush_stage), instead of by one returning ATOM per warp-iteration on a few hot L2 lines.
constexpr uint32_t R_STAGE_CELLS = RB * 2u * R_STAGE_T;  // [RB][2][R_STAGE_T] u64 cells, then as many u16 list entries
constexpr size_t R_STAGE_BYTES = (size_t)R_STAGE_CELLS * (sizeof(unsigned long long) + sizeof(uint16_t));
static_assert(R_STAGE_CELLS <= 65536u, "a staged cell's index must fit the 16-bit entries of the block's list");
__host__ __device__ __forceinline__ uint32_t cell_dec(unsigned long long v) { return (uint32_t)(v & R_FMASK); }
__host__ __device__ __forceinline__ uint32_t cell_len(unsigned long long v) { return (uint32_t)((v >> R_FIELD) & R_FMASK); }
__host__ __device__ __forceinline__ uint32_t cell_cnt(unsigned long long v) { return (uint32_t)((v >> (2 * R_FIELD)) & R_FMASK); }
constexpr uint32_t MGR_HDR = 64;          // sharded: u64 words of header in front of the records of a round's message
static_assert(2u * ND_STRIDE <= MG_INBOX_STRIDE - MGR_HDR, "the records of a round's first merge always fit a message");
constexpr uint32_t R_QCAP = 512;         // per-block partial entries a decision can fold (RT x blocks)

constexpr uint32_t ERR_ROUND_MISMATCH = 2048u;  // a merge of a round found a different number of sites than its count

struct RoundState {
  // counters the site passes bump once per warp-iteration: one 128-byte line each, so that they spread over L2 slices instead
  // of queueing at one (same-sector atomics serialise)
  struct alignas(128) Line {
    uint32_t v;
    uint32_t pad[31];
  };
  struct alignas(128) Line64 {
    unsigned long long v;  // U bound of the left born pairs | of the right born pairs << 32
    unsigned long long pad[15];
  };
  Line n_sites[2][RB];
  Line64 ub[2][RB];
  uint32_t overflow[2];   // a block's list of touched cells was full: the round scans the rows instead
  // sharded corpus: what the exchange of a round folds out of the ranks' message headers (same values on every rank)
  uint32_t goverflow[2];            // a block's list of GLOBAL cells was full
  uint32_t mg_n[MG_MAX_WORLD];      // records each rank sent
  unsigned long long mg_ub[RB];     // sum over ranks of the U bounds (left | right << 32): bounds of the global counts
  uint32_t mg_ns[RB];               // sites of merge j on all ranks
  uint32_t mg_k;                    // merges every rank tried (the smallest batch)
  uint32_t mg_pad;
  unsigned long long rounds, round_merges, rounds_cut_born, rounds_single, tried;
  unsigned long long stop_reason[8];
  unsigned long long iters_small, iters_big, cells_small, cells_big, sites_small, sites_big;  // P1 warp-iterations, touched cells, sites  // why a batch was not extended: 0 cap, 1 no exact candidate, 2 tie, 3 big, 4 token, 5 (none: fresh tokens join), 6 limits
};

struct RoundArgs {
  LoopArgs L;
  unsigned long long* cells;  // [2][RB][2][ND_STRIDE] packed delta cells (see R_FIELD)
  uint32_t* slotrows;         // [2][RB][2][ND_STRIDE] table slot of the born pair (tok, c) / (c, tok), for the list filling
  uint32_t* lists;            // [2][blocks][R_LISTCAP] cells each block touched first: (merge * 2 + side) << 16 | token
  SiteRec* bsites;   // [2][RB][R_SMALL]: merges 1.. of a round (merge 0 uses L.A.sites / L.sites2, which the host sizes)
  int bar_mode;      // 0: k_merge_loop's barrier (two sequentially consistent fences); 1: release arrival + acquire poll
  uint4* gp;         // [RT * blocks] per-block top groups: (primary lo, primary hi, slot, mult)
  uint32_t* gk;      // [RT * blocks] ... and the pair key of that slot
  RoundState* rs;
  uint32_t kmax;     // merges per round (1 .. RB)
  // corpus sharded by document over several GPUs (L.mg_on, mg_kernels.cuh): the counts of the pair table are global and
  // replicated, the cells above hold THIS shard's deltas; once per round every rank stores its non-empty cells as records into
  // every rank's inbox over NVLink, and every rank sums all records into gcells -- the global deltas P2 then works from
  unsigned long long* gcells;  // [2][RB][2][ND_STRIDE]: decrements | counted occurrences << 21, summed over the ranks
  uint32_t* glists;            // [2][blocks][R_LISTCAP]: global cells each block touched first while summing
};

__device__ __forceinline__ unsigned long long* round_cells(const RoundArgs& R, uint32_t par, uint32_t j, uint32_t side) {
  return R.cells + (((size_t)par * RB + j) * 2u + side) * ND_STRIDE;
}
__device__ __forceinline__ uint32_t* round_slotrow(const RoundArgs& R, uint32_t par, uint32_t j, uint32_t side) {
  return R.slotrows + (((size_t)par * RB + j) * 2u + side) * ND_STRIDE;
}
__device__ __forceinline__ uint32_t* round_list(const RoundArgs& R, uint32_t par) {
  return R.lists + ((size_t)par * gridDim.x + blockIdx.x) * R_LISTCAP;
}
// decrements of the old pair a later merge holds in ITS cell of token `tok` (cross-reads of P2: nobody writes the cells then)
__device__ __forceinline__ unsigned long long* round_gcells(const RoundArgs& R, uint32_t par, uint32_t j, uint32_t side) {
  return R.gcells + (((size_t)par * RB + j) * 2u + side) * ND_STRIDE;
}
__device__ __forceinline__ uint32_t* round_glist(const RoundArgs& R, uint32_t par) {
  return R.glists + ((size_t)par * gridDim.x + blockIdx.x) * R_LISTCAP;
}
__device__ __forceinline__ uint32_t round_dec_of(const RoundArgs& R, uint32_t par, uint32_t j, uint32_t side, uint32_t tok) {
  return cell_dec(ld_cg((R.L.mg_on ? round_gcells(R, par, j, side) : round_cells(R, par, j, side)) + tok));  // (both layouts keep it in the low bits)
}

// Site record of a round: x = p, y = position of the left token of the born left adjacency (NOPOS: none),
// z = left token | right token << 16 of the born pairs (R_NOTOK: none), w = what the rewrite needs without walking the corpus
// again: DOCSTART of p << 31 | overflow << 30 | (q - p) << 15 | (e - p)   (q = start of b, e = last slot of b).
constexpr uint32_t R_NOTOK = 0xFFFFu;
constexpr uint32_t R_SRC_LIST = 0xFFFFFFFFu;  // RoundSm::src: the merge's sites are in its occurrence list
__device__ __forceinline__ uint32_t round_pack_span(uint32_t w, uint32_t p, uint32_t q, uint32_t e) {
  const uint32_t dq = q - p, de = e - p;
  const uint32_t doc = (w & DOCSTART) ? 0x80000000u : 0u;
  if (de >= 32768u) return doc | 0x40000000u;
  return doc | (dq << 15) | de;
}

// grid barrier with a release arrival and an acquire poll (no sequentially consistent fence): everything the block wrote
// before its __syncthreads is ordered before thread 0's release; what thread 0 acquires is ordered before the reads of the
// block after the second __syncthreads (acquire at gpu scope invalidates L1)
__device__ __forceinline__ void grid_barrier_ra(unsigned long long* ctr, unsigned long long target, uint32_t max_ns) {
  __syncthreads();
  if (threadIdx.x == 0) {
    asm volatile("red.release.gpu.global.add.u64 [%0], 1;" ::"l"(ctr) : "memory");
    uint32_t ns = 32;
    for (;;) {
      unsigned long long v;
      asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(ctr) : "memory");
      if (v >= target) break;
      __nanosleep(ns);
      if (ns < max_ns) ns <<= 1;
    }
  }
  __syncthreads();
}

// 256-bit filter over token indices (bit = index mod 256): "is this token the a / the b of a merge of the batch?" costs one
// shared-memory word for the 15 of 16 tokens that are not
__device__ __forceinline__ bool role_maybe(const uint32_t* filt, uint32_t tok) { return (filt[(tok >> 5) & 7u] >> (tok & 31u)) & 1u; }

// ---- top-N groups: the RT largest DISTINCT primaries, each with the number of pairs that share it and the smallest slot ----
// (what a block publishes for the next decision: the more groups per block, the deeper the exact candidate list reaches)
#ifndef BPE_RT
#define BPE_RT 2
#endif
constexpr int RT = BPE_RT;  // (3 reaches deeper -- 10 % fewer rounds on cfg3 -- but its reduction costs more than that saves: measured)
struct Top2 {
  unsigned long long p[RT];
  uint32_t s[RT], m[RT], k[RT];
};
__device__ __forceinline__ Top2 top2_empty() {
  Top2 t;
#pragma unroll
  for (int i = 0; i < RT; i++) {
    t.p[i] = 0ull;
    t.s[i] = NOSLOT;
    t.m[i] = 0u;
    t.k[i] = 0u;
  }
  return t;
}
__device__ __forceinline__ void top2_add(Top2& t, unsigned long long p, uint32_t slot, uint32_t mult, uint32_t key) {
  if (!p) return;
  bool done = false;
#pragma unroll
  for (int i = 0; i < RT; i++) {
    if (!done && p == t.p[i]) {
      t.m[i] += mult;
      if (slot < t.s[i]) {
        t.s[i] = slot;
        t.k[i] = key;
      }
      done = true;
    }
    if (!done && p > t.p[i]) {  // insert here, the smaller groups move down (the last one drops out)
#pragma unroll
      for (int j = RT - 1; j > i; j--) {
        t.p[j] = t.p[j - 1];
        t.s[j] = t.s[j - 1];
        t.m[j] = t.m[j - 1];
        t.k[j] = t.k[j - 1];
      }
      t.p[i] = p;
      t.s[i] = slot;
      t.m[i] = mult;
      t.k[i] = key;
      done = true;
    }
  }
}
__device__ __forceinline__ Top2 top2_warp_reduce(Top2 v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    Top2 w;
#pragma unroll
    for (int i = 0; i < RT; i++) {
      w.p[i] = __shfl_xor_sync(0xFFFFFFFFu, v.p[i], o);
      w.s[i] = __shfl_xor_sync(0xFFFFFFFFu, v.s[i], o);
      w.m[i] = __shfl_xor_sync(0xFFFFFFFFu, v.m[i], o);
      w.k[i] = __shfl_xor_sync(0xFFFFFFFFu, v.k[i], o);
    }
#pragma unroll
    for (int i = 0; i < RT; i++) top2_add(v, w.p[i], w.s[i], w.m[i], w.k[i]);
  }
  return v;
}
// a block's groups -> its RT entries of the partial arrays
__device__ __forceinline__ void top2_publish(const Top2& v, uint4* gp, uint32_t* gk, uint32_t bid) {
#pragma unroll
  for (int i = 0; i < RT; i++) {
    gp[RT * bid + i] = make_uint4((uint32_t)v.p[i], (uint32_t)(v.p[i] >> 32), v.s[i], v.m[i]);
    gk[RT * bid + i] = v.k[i];
  }
}

// shared memory of one block of k_merge_rounds
struct RoundSm {
  // the batch of the current round (same in every block)
  uint32_t k, status, mult0, pad0;
  uint32_t a[RB], b[RB], w[RB], slot[RB], llen[RB], lenc[RB];
  unsigned long long lstart[RB];  // where each merge's occurrence list starts in the pool
  uint32_t src[RB];        // where P1 finds each merge's sites: R_SRC_LIST, or merge i of the previous round << 1 | side of its row
  uint32_t iter0[RB + 1];  // warp-iterations of P1: merge j owns [iter0[j], iter0[j+1])
  uint32_t fill_n[RB];     // sites of the previous round's merges whose born adjacencies are not in their lists yet
  // decision scratch
  uint32_t qn;
  unsigned long long qp[R_QCAP];
  uint32_t qs[R_QCAP], qm[R_QCAP], qk[R_QCAP];
  unsigned long long cp[RB];
  uint32_t cs[RB], cm[RB], ck[RB], cll[RB], clen[RB];
  unsigned long long cls[RB];
  LoopCaps caps;  // this GPU's, or sharded: the minima over the ranks (loop_caps_folded)
  uint32_t g_n_keys, g_snap_err, g_abort;
  uint32_t ncell[2];  // cells this block touched first in the round of either parity (entries of its list)
  uint32_t nstage;    // staged cells this block touched in the current P1 (entries of r_stage_list)
  uint32_t gncell[2]; // sharded: global cells this block touched first while summing the ranks' records
  uint32_t rec_base, rec_cnt;  // sharded: where this block's records go in the inboxes, how many they are
  uint32_t mg_mask, mg_cnt[MG_MAX_WORLD];  // sharded: senders whose message is complete and not summed yet, their records
  unsigned long long pool_base;  // this block's private chunk of the occurrence pool (list space without a grid-wide atomic) ...
  uint32_t pool_next, pool_end;  // ... and the bump cursor / end inside it (32-bit offsets: a 64-bit shared atomic is a CAS loop)
  uint32_t keys_ins;             // keys this block inserted in the current P2 (one n_keys atomic per block and round)
  uint32_t filt_a[8], filt_b[8]; // role_maybe filters: the a's / the b's of the batch
  Top2 t2[32];
  unsigned long long red[32];
  uint32_t s_max[32];
  uint32_t rslot;
};

__device__ __forceinline__ unsigned long long block_max_u64(unsigned long long v, unsigned long long* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    unsigned long long u = __shfl_xor_sync(0xFFFFFFFFu, v, o);
    v = u > v ? u : v;
  }
  __syncthreads();
  if (lane_id() == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  const uint32_t nw = blockDim.x >> 5;
  unsigned long long u = lane_id() < nw ? red[lane_id()] : 0ull;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    unsigned long long x = __shfl_xor_sync(0xFFFFFFFFu, u, o);
    u = x > u ? x : u;
  }
  return u;
}

__device__ __forceinline__ Top2 top2_block_reduce(Top2 v, Top2* s_t2) {
  v = top2_warp_reduce(v);
  __syncthreads();
  if (lane_id() == 0) s_t2[threadIdx.x >> 5] = v;
  __syncthreads();
  const uint32_t nw = blockDim.x >> 5;
  Top2 u = lane_id() < nw ? s_t2[lane_id()] : top2_empty();
  return top2_warp_reduce(u);
}

// the block's staged cells (dynamic shared memory of k_merge_rounds, R_STAGE_BYTES): [RB][2][R_STAGE_T] packed cells, then the
// list of those the block touched in the current P1 (index (merge * 2 + side) * R_STAGE_T + token)
extern __shared__ __align__(16) unsigned long long r_stage[];
__device__ __forceinline__ uint16_t* r_stage_list() { return reinterpret_cast<uint16_t*>(r_stage + R_STAGE_CELLS); }

// All 32 lanes call; each `first` lane found the global cell of (js = merge * 2 + side, tok) empty: it lists the cell for P2
// (one shared-memory counter bump per warp).  c is the merge's new token, partner its a (side 0) or b (side 1).
__device__ __forceinline__ void cell_list_first(const RoundArgs& R, RoundSm& S, uint32_t par, uint32_t js, uint32_t tok, bool first, uint32_t c,
                                                uint32_t partner) {
  const uint32_t lane = lane_id();
  const uint32_t fm = __ballot_sync(0xFFFFFFFFu, first);
  if (!fm) return;
  uint32_t base = 0;
  const int src = __ffs(fm) - 1;
  if ((int)lane == src) base = atomicAdd(&S.ncell[par], (uint32_t)__popc(fm));
  base = __shfl_sync(0xFFFFFFFFu, base, src);
  if (first) {
    const uint32_t k = base + __popc(fm & ((1u << lane) - 1u));
    if (k < R_LISTCAP) round_list(R, par)[k] = (js << 16) | tok;
    else R.rs->overflow[par] = 1;
    // P2 will probe the pair table for the born pair (tok, c) / (c, tok) and for the old pair (tok, a) / (b, tok): ask for
    // their home slots now, so that they sit in L2 by then (hints only)
    const PairTable& t = R.L.A.t;
    const uint32_t side = js & 1u;
    prefetch_l2(t.keys + tbl_hash(t, side ? pair_key(c, tok) : pair_key(tok, c)));
    const uint32_t h2 = tbl_hash(t, side ? pair_key(partner, tok) : pair_key(tok, partner));
    prefetch_l2(t.keys + h2);
    prefetch_l2(t.cnt + h2);
  }
}

// All 32 lanes call; `has` lanes contribute to the cell of `tok`: a decrement (dec), an occurrence of the born pair (newp),
// a counted occurrence (counted).  Lanes that agree on tok elect a leader which issues ONE 64-bit atomic for all of them: into
// the block's staged cell when the merge stages (`staged`, warp-uniform) and tok < R_STAGE_T -- the first toucher appends it
// to the block's list, round_flush_stage lists it globally --, else into the global cell, whose first toucher lists it.
// Returns the leader's counted occurrences (0 elsewhere): the ingredient of the born-pair bound.
__device__ __forceinline__ uint32_t cell_add_warp(const RoundArgs& R, RoundSm& S, uint32_t par, uint32_t js, unsigned long long* cells, uint32_t tok, bool has,
                                                  bool dec, bool newp, bool counted, uint32_t c, uint32_t partner, bool staged) {
  const uint32_t lane = lane_id();
  const uint32_t peers = __match_any_sync(0xFFFFFFFFu, has ? tok : (0xFFFFFF00u + lane));
  const uint32_t dmask = __ballot_sync(0xFFFFFFFFu, has && dec);
  const uint32_t nmask = __ballot_sync(0xFFFFFFFFu, has && newp);
  const uint32_t cmask = __ballot_sync(0xFFFFFFFFu, has && newp && counted);
  const bool leader = has && lane == (uint32_t)(__ffs(peers) - 1);
  uint32_t nc = 0, nd = 0;
  bool first = false;
  if (leader) {
    nc = (uint32_t)__popc(peers & cmask);
    nd = (uint32_t)__popc(peers & dmask);
    const unsigned long long add = (unsigned long long)nd | ((unsigned long long)__popc(peers & nmask) << R_FIELD) | ((unsigned long long)nc << (2 * R_FIELD));
    if (staged && tok < R_STAGE_T) {
      const uint32_t e = js * R_STAGE_T + tok;
      if (atomicAdd(&r_stage[e], add) == 0ull) r_stage_list()[atomicAdd(&S.nstage, 1u)] = (uint16_t)e;
    } else {
      first = atomicAdd(cells + tok, add) == 0ull;
    }
  }
  cell_list_first(R, S, par, js, tok, first, c, partner);
  return nc;
}

// End of P1 in this block (all its threads call): every staged cell the block touched goes into its global cell with one
// atomic, and is zeroed for the next round; the block that finds a global cell empty lists it, as cell_add_warp does -- so
// P2 and the exchange of the sharded engine see the same cells and lists as without staging.  (Per-block sums of a merge's
// counts fit the 21-bit fields: its totals do, R_HUGE.)
__device__ __forceinline__ void round_flush_stage(const RoundArgs& R, RoundSm& S, uint32_t par, uint32_t c_first) {
  __syncthreads();
  const uint32_t ns = S.nstage;
  const uint16_t* list = r_stage_list();
  for (uint32_t i0 = threadIdx.x & ~31u; i0 < ns; i0 += blockDim.x) {
    const uint32_t i = i0 + lane_id();
    const bool has = i < ns;
    const uint32_t e = has ? list[i] : 0u;
    const uint32_t js = e / R_STAGE_T, tok = e - js * R_STAGE_T, j = js >> 1;
    bool first = false;
    if (has) {
      const unsigned long long v = r_stage[e];
      r_stage[e] = 0ull;
      first = atomicAdd(round_cells(R, par, j, js & 1u) + tok, v) == 0ull;
    }
    cell_list_first(R, S, par, js, tok, first, c_first + j, (js & 1u) ? S.b[j] : S.a[j]);
  }
}

// ---- sharded corpus: the message of a round ----
// u64 words of one (parity, sender) area of an inbox: MGR_HDR words of header, then the records.
//   [0..5]   the twelve u32 of mg_store_header (H_N records, H_ERR, capacities)
//   [8 + j]  U bounds of merge j on the sender (left | right << 32)       [24 + j]  sites of merge j on the sender
//   [40]     merges the sender tried (its batch; every rank commits at most the smallest)
// record: ((merge * 2 + side) << 16 | token) << 42 | counted occurrences << 21 | decrements    (one per warp and distinct
// neighbour of a site pass, written while the pass runs)

// arrival counter of (receiver dst, parity, sender): words 2 and 3 of the sender's flag line on the receiver.  Every block of
// the sender adds 1 << 32 | its records once its part of the message is out (fenced); the receiver resets it after use.
__device__ __forceinline__ unsigned long long* mgr_counter(const MgArgs& M, int dst, uint32_t epar, int sender) {
  return M.flag_data[dst] + 16 * sender + 2 + epar;
}

__device__ __forceinline__ void mgr_send_warp(const RoundArgs& R, uint32_t par, uint32_t epar, uint32_t k, unsigned long long epoch, bool with_flag);

// After the site passes of a round (grid barrier): every block turns the cells of ITS list -- the cells it touched first, now
// complete -- into records in every rank's inbox: ONE record per touched cell and rank, one slot reservation per block,
// coalesced NVLink stores.  (Records written while the passes run -- one per warp and neighbour -- were measured: the
// frequent neighbours then receive hundreds of records each and the summing on the other side queues on those cells.)
__device__ __forceinline__ void round_emit_records(const RoundArgs& R, RoundSm& S, uint32_t par, uint32_t epar, uint32_t k, uint32_t c_hi, unsigned long long epoch) {
  const MgArgs& M = R.L.mg;
  DevState* st = R.L.A.st;
  const uint32_t cap = M.inbox_stride - MGR_HDR;
  // (block 0: its last warp -- the records of a round keep the first warps busy, not that one -- also writes this rank's header)
  const bool hdr_warp = blockIdx.x == 0 && (threadIdx.x >> 5) == (blockDim.x >> 5) - 1u;
  if (threadIdx.x == 0) S.rec_cnt = 0;
  if (!ld_cg(&R.rs->overflow[par])) {
    const uint32_t n = min(S.ncell[par], R_LISTCAP);
    if (threadIdx.x == 0) {
      S.rec_base = n ? atomicAdd(&st->n_out, n) : 0u;
      S.rec_cnt = n;
    }
    __syncthreads();
    if (hdr_warp) mgr_send_warp(R, par, epar, k, epoch, false);
    const uint32_t base = S.rec_base;
    const uint32_t* list = round_list(R, par);
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
      const uint32_t ent = ld_cg(list + i);
      const uint32_t js = (ent >> 16) & (2u * RB - 1u), tok = ent & 0xFFFFu;
      const unsigned long long cellv = ld_cg(round_cells(R, par, js >> 1, js & 1u) + tok);
      const unsigned long long rec = ((unsigned long long)ent << 42) | ((unsigned long long)cell_cnt(cellv) << R_FIELD) | cell_dec(cellv);
      const uint32_t at = base + i;
      if (at < cap) {
        for (int q = 0; q < M.world; q++) mg_area(M, q, epar, M.rank)[MGR_HDR + at] = rec;
      } else {
        atomicOr(&st->err, ERR_INBOX_OVERFLOW);
      }
    }
  } else {
    // a list was full: every non-empty cell of the round's rows (slots one by one: rare)
    __syncthreads();
    if (hdr_warp) mgr_send_warp(R, par, epar, k, epoch, false);
    const uint32_t T = (c_hi + 31u) & ~31u;
    const uint32_t total = k * 2u * T;
    uint32_t mine = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
      const uint32_t js = i / T, tok = i - js * T;
      const unsigned long long cellv = ld_cg(round_cells(R, par, js >> 1, js & 1u) + tok);
      if (!cellv) continue;
      const uint32_t at = atomicAdd(&st->n_out, 1u);
      mine++;
      if (at < cap) {
        const unsigned long long rec = ((unsigned long long)((js << 16) | tok) << 42) | ((unsigned long long)cell_cnt(cellv) << R_FIELD) | cell_dec(cellv);
        for (int q = 0; q < M.world; q++) mg_area(M, q, epar, M.rank)[MGR_HDR + at] = rec;
      } else {
        atomicOr(&st->err, ERR_INBOX_OVERFLOW);
      }
    }
    if (mine) atomicAdd(&S.rec_cnt, mine);
  }
  // this block's part of the message is out: one remote add per rank says so -- arrivals in the upper half of the counter, the
  // block's records in the lower (the receiver needs their total, and only the sum over the blocks knows it)
  __syncthreads();
  if (threadIdx.x < (unsigned)M.world) {
    __threadfence_system();  // (after the barrier: cumulative over the stores of the whole block, as in a grid barrier's arrive)
    atomicAdd_system(mgr_counter(M, (int)threadIdx.x, epar, M.rank), (1ull << 32) | (unsigned long long)S.rec_cnt);
  }
}

// warp 0 of block 0, lane q talks to rank q: header of this rank's message, then the flag
__device__ __forceinline__ void mgr_send_warp(const RoundArgs& R, uint32_t par, uint32_t epar, uint32_t k, unsigned long long epoch, bool with_flag) {
  const MgArgs& M = R.L.mg;
  const LoopArgs& L = R.L;
  DevState* st = L.A.st;
  const int q = (int)lane_id();
  // lane j fetches merge j's figures once; the lanes that write a header read them out of each other's registers
  const unsigned long long ub_lane = ((uint32_t)q < k) ? ld_cg(&R.rs->ub[par][q].v) : 0ull;
  const uint32_t ns_lane = ((uint32_t)q < k) ? ld_cg(&R.rs->n_sites[par][q].v) : 0u;
  if (q < M.world) {
    unsigned long long* dst = mg_area(M, q, epar, M.rank);
    mg_store_header(L, dst, min(ld_cg(&st->n_out), M.inbox_stride - MGR_HDR), 0xFFFFFFFFu);
    dst[40] = k;
  }
  for (uint32_t j = 0; j < RB; j++) {  // (every lane takes part in the shuffles; the lanes that talk to a rank store)
    const unsigned long long u = __shfl_sync(0xFFFFFFFFu, ub_lane, j);
    const uint32_t n = __shfl_sync(0xFFFFFFFFu, ns_lane, j);
    if (q < M.world) {
      unsigned long long* dst = mg_area(M, q, epar, M.rank);
      dst[8 + j] = u;
      dst[24 + j] = (unsigned long long)n;
    }
  }
  // (no fence: lane q wrote rank q's header itself and its release store orders that; the records were fenced at system scope
  // by the blocks that wrote them, before the grid barrier this warp came through)
  __syncwarp();
  if (with_flag && q < M.world) st_release_sys(M.flag_data[q] + 16 * M.rank, epoch);  // (own rank included: every block of every rank polls all flags)
}

// fold the headers of all senders (their messages are complete): st->g_vals (mg_fold_headers_warp), sums of the per-merge
// bounds and site counts, the smallest batch
__device__ __forceinline__ void mgr_fold_warp(const RoundArgs& R, uint32_t epar) {
  const MgArgs& M = R.L.mg;
  RoundState* rs = R.rs;
  const int q = (int)lane_id();
  uint32_t kq = (q < M.world) ? (uint32_t)ld_cg(mg_area(M, M.rank, epar, q) + 40) : 0xFFFFFFFFu;
  const uint32_t n = mg_fold_headers_warp(M, R.L.A.st, epar);
  if (q < M.world) rs->mg_n[q] = n;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) kq = min(kq, __shfl_xor_sync(0xFFFFFFFFu, kq, o));
  if (q == 0) rs->mg_k = kq;
  if (q < RB) {  // lane j sums merge j's bounds and sites over the senders
    unsigned long long ul = 0, ur = 0;
    uint32_t nsum = 0;
#pragma unroll
    for (int s = 0; s < MG_MAX_WORLD; s++) {  // (unrolled: the loads of all senders are in flight together)
      if (s < M.world) {
        const unsigned long long* hs = mg_area(M, M.rank, epar, s);
        const unsigned long long u = ld_cg(hs + 8 + q);
        ul += (uint32_t)u;
        ur += (uint32_t)(u >> 32);
        nsum += (uint32_t)ld_cg(hs + 24 + q);
      }
    }
    rs->mg_ub[q] = min(ul, 0xFFFFFFFFull) | (min(ur, 0xFFFFFFFFull) << 32);
    rs->mg_ns[q] = nsum;
  }
}


// X2 of a round: the messages are summed as they complete.  Warp 0 of the block watches the arrival counters of all senders;
// whenever some are complete (every block of the sender has reported) the whole block adds ITS share of those senders'
// records to the global cells -- so what is left to do when the slowest rank reports is that rank's records alone.  The thread
// that finds a cell empty lists it.  Sender q's records start at thread q * (threads / world) of the grid: a round's few
// thousand records per sender spread over all blocks instead of queueing on the first ones.
__device__ __forceinline__ void mgr_collect(const RoundArgs& R, RoundSm& S, uint32_t par, uint32_t epar) {
  const MgArgs& M = R.L.mg;
  DevState* st = R.L.A.st;
  RoundState* rs = R.rs;
  const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
  const uint32_t G = gridDim.x * blockDim.x, gtid = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t shift = (G / (uint32_t)M.world) & ~31u;
  const uint32_t cap = M.inbox_stride - MGR_HDR;
  const uint32_t all = (1u << M.world) - 1u;
  uint32_t done = 0;
  const unsigned long long t0 = now_ns();
  while (done != all) {
    if (warp == 0) {
      uint32_t mask = 0, ns = 16;
      for (;;) {
        unsigned long long v = 0;
        if (lane < (uint32_t)M.world) v = ld_acquire_sys(mgr_counter(M, M.rank, epar, (int)lane));
        const bool here = (uint32_t)(v >> 32) == gridDim.x && !((done >> lane) & 1u);
        mask = __ballot_sync(0xFFFFFFFFu, here);
        if (here) {
          const uint32_t n = (uint32_t)v;
          if (n > cap) atomicOr(&st->err, ERR_INBOX_OVERFLOW);
          S.mg_cnt[lane] = min(n, cap);
        }
        if (mask) break;
        __nanosleep(ns);
        if (ns < 128) ns <<= 1;
        if (now_ns() - t0 > MG_TIMEOUT_NS) {
          atomicOr(&st->err, ERR_PEER_TIMEOUT);
          st->mg_abort = 1;
          mask = all & ~done;  // (leave the loop; the caller sees mg_abort)
          if (lane < (uint32_t)M.world) S.mg_cnt[lane] = 0;
          break;
        }
      }
      if (lane == 0) S.mg_mask = mask;
    }
    __syncthreads();
    const uint32_t mask = S.mg_mask;
    for (int q = 0; q < M.world; q++) {
      if (!((mask >> q) & 1u)) continue;
      const uint32_t n = S.mg_cnt[q];
      const unsigned long long* recs = mg_area(M, M.rank, epar, q) + MGR_HDR;
      uint32_t jx = gtid + G - (uint32_t)q * shift;
      if (jx >= G) jx -= G;
      for (; jx < ((n + 31u) & ~31u); jx += G) {
        bool first = false;
        uint32_t ent = 0;
        if (jx < n) {
          const unsigned long long rec = ld_cg(recs + jx);
          ent = (uint32_t)(rec >> 42);
          const uint32_t js = (ent >> 16) & (2u * RB - 1u), tok = ent & 0xFFFFu;
          // (bit 42 up counts the records of the cell: the sum is never zero once a record arrived, whatever it carried)
          first = atomicAdd(round_gcells(R, par, js >> 1, js & 1u) + tok, (rec & ((1ull << (2 * R_FIELD)) - 1ull)) + (1ull << (2 * R_FIELD))) == 0ull;
        }
        const uint32_t fm = __ballot_sync(0xFFFFFFFFu, first);
        if (fm) {
          uint32_t base = 0;
          const int src = __ffs(fm) - 1;
          if ((int)lane == src) base = atomicAdd(&S.gncell[par], (uint32_t)__popc(fm));
          base = __shfl_sync(0xFFFFFFFFu, base, src);
          if (first) {
            const uint32_t at = base + __popc(fm & ((1u << lane) - 1u));
            if (at < R_LISTCAP) round_glist(R, par)[at] = ent;
            else rs->goverflow[par] = 1;
          }
        }
      }
    }
    done |= mask;
    __syncthreads();  // (S.mg_mask and S.mg_cnt are rewritten by the next look at the counters)
  }
  if (warp == 0) mgr_fold_warp(R, epar);
}

__device__ __forceinline__ SiteRec* round_sites_buf(const RoundArgs& R, uint32_t par, uint32_t j) {
  if (j == 0) return par ? R.L.sites2 : R.L.A.sites;
  return R.bsites + ((size_t)par * RB + j) * R_SMALL;
}

// What a site record of merge i gives the pair merge i created on `side` (0: (tok, c_i), 1: (c_i, tok)): tok (R_NOTOK: none),
// and the entry of that pair's occurrence list -- the position of its left token.  The list fill of the following round and
// its site passes of pairs that contain c_i share this definition.
__device__ __forceinline__ uint32_t round_rec_tok(const uint4& rv, uint32_t side) { return side ? rv.z >> 16 : rv.z & 0xFFFFu; }
__device__ __forceinline__ uint32_t round_rec_pos(const uint4& rv, uint32_t side) { return side ? rv.x : rv.y; }

// One warp-iteration of the site pass of merge j of the round: 32 entries of its occurrence list, or -- when the pair contains
// a token the previous round created (S.src[j]) -- 32 site records of that round's merge whose row holds the pair.
// The logic of the neighbourhoods is phase_sites' (train_kernels.cuh); what differs is where the deltas go (the merge's
// dense rows) and the virtual neighbours c_i of the earlier merges of the batch.
__device__ __forceinline__ void round_sites_iter(const RoundArgs& R, RoundSm& S, uint32_t par, uint32_t fpar, uint32_t j, uint32_t c_first,
                                                 uint32_t i, SiteRec* site_out, uint32_t sites_cap) {
  const ApplyArgs& A = R.L.A;
  const uint32_t* slots = A.slots;
  const uint32_t n = A.n;
  DevState* st = A.st;
  const uint32_t a = S.a[j], b = S.b[j], c = c_first + j;
  const uint32_t total = S.llen[j];
  const bool staged = total > R.L.stage_min;
  const uint32_t lane = lane_id();
  unsigned long long* const cells_l = round_cells(R, par, j, 0);
  unsigned long long* const cells_r = round_cells(R, par, j, 1);
  bool site = false;
  uint32_t p = 0, w = 0, q = 0, koff = 0;
  bool has = i < total;
  if (has) {
    const uint32_t src = S.src[j];
    if (src == R_SRC_LIST) {
      p = A.pool[S.lstart[j] + i];
    } else {  // record i of merge src >> 1 of the previous round: an entry of this pair's list iff its token on that side matches
      const uint4 rv = ld_cg4(reinterpret_cast<const uint4*>(round_sites_buf(R, fpar, src >> 1)) + i);
      const uint32_t side = src & 1u;
      has = round_rec_tok(rv, side) == (side ? b : a);
      p = round_rec_pos(rv, side);
    }
  }
  if (has) {
    w = ld_slot(slots + p);
    if (slot_is_id(w) && slot_val(w) == a && right_token(slots, n, p, &q) == (int)b) {
      site = true;
      if (a == b) {
        koff = run_left(slots, p, w, (int)a);
        if (koff & 1u) site = false;  // overlaps the occurrence to its left (replaceAll is non-overlapping)
      }
    }
  }
  const uint32_t smask = __ballot_sync(0xFFFFFFFFu, site);
  if (!smask) return;
  uint32_t site_base = 0;
  if (lane == (uint32_t)(__ffs(smask) - 1)) site_base = atomicAdd(&R.rs->n_sites[par][j].v, (uint32_t)__popc(smask));
  SiteRec rec{p, NOPOS, R_NOTOK, R_NOTOK};
  // ---- adjacency on the left of the new token ----
  uint32_t dec1_tok = 0, new1_tok = 0;
  bool dec1 = false, new1 = false, new1_counted = true;
  if (site) {
    uint32_t lpos;
    int x = left_token(slots, p, w, &lpos);
    if (x != NOTOK) {
      bool chained = false;
      uint32_t chain_j = 0, llpos = NOPOS;
      if (a == b) {
        chained = koff >= 2;
        chain_j = koff >> 1;
        if (chained) left_token(slots, lpos, ld_slot(slots + lpos), &llpos);
      } else if ((uint32_t)x == b) {
        int xx = left_token(slots, lpos, ld_slot(slots + lpos), &llpos);
        if (xx == (int)a) {  // the pair to the left is itself a site: ... a b a b
          chained = true;
          chain_j = 1;
          uint32_t cur = llpos;
          for (;;) {  // index of this site within its chain of back-to-back sites
            uint32_t l1, l2;
            if (left_token(slots, cur, ld_slot(slots + cur), &l1) != (int)b) break;
            if (left_token(slots, l1, ld_slot(slots + l1), &l2) != (int)a) break;
            chain_j++;
            cur = l2;
          }
        }
      }
      new1 = true;
      if (chained) {
        if (a != b) {
          dec1 = true;
          dec1_tok = b;  // the pair (b,a)
        }
        new1_tok = c;  // the pair (c,c): runs of c count every other pair (:285-290)
        new1_counted = (chain_j & 1u) != 0;
        rec.lpos = llpos;
      } else {
        // is the left neighbour the right half of a site of an EARLIER merge of this batch?  Then it is c_i by now.
        int vi = -1;
        uint32_t vpos = NOPOS;
        for (uint32_t i2 = 0; i2 < (role_maybe(S.filt_b, (uint32_t)x) ? j : 0u); i2++) {
          if ((uint32_t)x != S.b[i2]) continue;
          const uint32_t wl = ld_slot(slots + lpos);
          if (S.a[i2] != S.b[i2]) {
            uint32_t l2;
            if (left_token(slots, lpos, wl, &l2) == (int)S.a[i2]) {
              vi = (int)i2;
              vpos = l2;
            }
          } else if (run_left(slots, lpos, wl, x) & 1u) {  // odd offset inside its run: the second half of a replaced pair
            vi = (int)i2;
            left_token(slots, lpos, wl, &vpos);
          }
          break;  // token sets are disjoint: at most one merge owns x as its b
        }
        if (vi >= 0) {
          dec1 = true;
          dec1_tok = c_first + (uint32_t)vi;  // the born pair (c_i, a) of merge i loses this adjacency
          new1_tok = c_first + (uint32_t)vi;  // ... and (c_i, c) is born
          rec.lpos = vpos;
        } else if ((uint32_t)x == a) {  // (a != b here) the run of a's ending at p loses its last element
          uint32_t Lr = 1 + run_left(slots, p, w, (int)a);
          dec1 = (Lr & 1u) == 0;
          dec1_tok = a;  // the pair (a,a)
          new1_tok = (uint32_t)x;
          rec.lpos = lpos;
        } else {
          dec1 = true;
          dec1_tok = (uint32_t)x;  // the pair (x,a)
          new1_tok = (uint32_t)x;  // the pair (x,c)
          rec.lpos = lpos;
        }
      }
    }
  }
  // one atomic per distinct left neighbour: the born pair (new1_tok, c), with the decrement when it concerns the same token
  // (it does unless the site is chained to the one on its left: then the decrement is (b,a)'s and goes out on its own)
  const bool dec1_same = dec1 && dec1_tok == new1_tok;
  const uint32_t nc1 = cell_add_warp(R, S, par, j * 2u, cells_l, new1_tok, new1, dec1_same, true, new1_counted, c, a, staged);
  if (__any_sync(0xFFFFFFFFu, dec1 && !dec1_same)) cell_add_warp(R, S, par, j * 2u, cells_l, dec1_tok, dec1 && !dec1_same, true, false, false, c, a, staged);
  rec.lslot = new1 ? new1_tok : R_NOTOK;

  // ---- adjacency on the right of the new token (left to the next site when that one is chained) ----
  uint32_t dec2_tok = 0, new2_tok = 0, span_word = 0;
  bool dec2 = false, new2 = false;
  if (site) {
    uint32_t r;
    int y = right_token(slots, n, q, &r);
    span_word = round_pack_span(w, p, q, r - 1u);  // r = first slot after b (n when b ends the corpus)
    if (y != NOTOK) {
      bool chained_right = false;
      if ((uint32_t)y == a) {
        uint32_t r2;
        chained_right = right_token(slots, n, r, &r2) == (int)b;
      }
      if (!chained_right) {
        int vi = -1;
        for (uint32_t i2 = 0; i2 < (role_maybe(S.filt_a, (uint32_t)y) ? j : 0u); i2++) {
          if ((uint32_t)y != S.a[i2]) continue;
          uint32_t r2;
          if (right_token(slots, n, r, &r2) == (int)S.b[i2]) vi = (int)i2;  // y starts a site of merge i (for a_i == b_i: offset 0 of its run)
          break;
        }
        if (vi >= 0) {
          dec2 = true;
          dec2_tok = c_first + (uint32_t)vi;  // the born pair (b, c_i) of merge i
          new2_tok = c_first + (uint32_t)vi;  // (c, c_i)
        } else if ((uint32_t)y == b && a != b) {  // the run of b's starting at q loses its first element
          uint32_t Lr = 1 + run_right(slots, n, q, (int)b);
          dec2 = (Lr & 1u) == 0;
          dec2_tok = b;  // the pair (b,b)
          new2_tok = (uint32_t)y;
        } else {
          if (!(a == b && (uint32_t)y == a)) {  // (a,a) itself is zeroed in P2
            dec2 = true;
            dec2_tok = (uint32_t)y;  // the pair (b,y)
          }
          new2_tok = (uint32_t)y;  // the pair (c,y)
        }
        new2 = true;
      }
    }
  }
  const bool dec2_same = dec2 && new2 && dec2_tok == new2_tok;  // (always, when there is a decrement: kept general)
  const uint32_t nc2 = cell_add_warp(R, S, par, j * 2u + 1u, cells_r, new2_tok, new2, dec2_same, true, true, c, b, staged);
  if (__any_sync(0xFFFFFFFFu, dec2 && !dec2_same)) cell_add_warp(R, S, par, j * 2u + 1u, cells_r, dec2_tok, dec2 && !dec2_same, true, false, false, c, b, staged);
  rec.rslot = new2 ? new2_tok : R_NOTOK;
  // upper bounds of the born pairs' counts: the largest group of lanes that share a neighbour, summed over the warps
  const uint32_t u1 = __reduce_max_sync(0xFFFFFFFFu, nc1), u2 = __reduce_max_sync(0xFFFFFFFFu, nc2);
  if (lane == 0) {
    if (u1 | u2) atomicAdd(&R.rs->ub[par][j].v, (unsigned long long)u1 | ((unsigned long long)u2 << 32));
  }
  // ---- record the site ----
  const uint32_t base = __shfl_sync(0xFFFFFFFFu, site_base, __ffs(smask) - 1);
  if (site) {
    const uint32_t k = base + __popc(smask & ((1u << lane) - 1u));
    if (k < sites_cap) reinterpret_cast<uint4*>(site_out)[k] = make_uint4(rec.p, rec.lpos, rec.lslot | (rec.rslot << 16), span_word);
    else atomicOr(&st->err, ERR_SITE_OVERFLOW);
  }
}

struct RoundFill {  // what the previous round left to do
  uint32_t v, par, k, c_first;  // merges committed / row parity / merges tried (rows to clear) / first token it created
  uint32_t overflow;            // a list of touched cells overflowed in that round: clear by scanning
  uint32_t goverflow;           // sharded: the same for the lists of global cells
};

// the lists of the pairs born by the previous round's merges, as ONE index space over all their sites (32-aligned per merge),
// so that the threads of the job share the work evenly whatever the sizes of the merges (runs on the helper warps next to
// P1, or on everybody)
__device__ __forceinline__ void round_fill_all(const RoundArgs& R, const RoundSm& S, const RoundFill& F, uint32_t vt, uint32_t nvt) {
  const ApplyArgs& A = R.L.A;
  const PairTable& t = A.t;
  uint32_t total = 0;
  for (uint32_t j = 0; j < F.v; j++) total += (S.fill_n[j] + 31u) & ~31u;
  for (uint32_t i = vt; i < total; i += nvt) {
    uint32_t j = 0, off = i;  // (warp-uniform: merge boundaries are 32-aligned)
    while (off >= ((S.fill_n[j] + 31u) & ~31u)) {
      off -= (S.fill_n[j] + 31u) & ~31u;
      j++;
    }
    const bool has = off < S.fill_n[j];
    const uint4 rv = has ? ld_cg4(reinterpret_cast<const uint4*>(round_sites_buf(R, F.par, j)) + off) : make_uint4(0, NOPOS, R_NOTOK | (R_NOTOK << 16), 0);
    const uint32_t ltok = round_rec_tok(rv, 0), rtok = round_rec_tok(rv, 1);
    const uint32_t lslot = (has && ltok != R_NOTOK) ? ld_cg(round_slotrow(R, F.par, j, 0) + ltok) : NOSLOT;
    const uint32_t rslot = (has && rtok != R_NOTOK) ? ld_cg(round_slotrow(R, F.par, j, 1) + rtok) : NOSLOT;
    const bool hl = has && lslot != NOSLOT && t.occ_len[lslot];
    const bool hr = has && rslot != NOSLOT && t.occ_len[rslot];
    const unsigned long long il = agg_cursor(t, lslot, hl);
    const unsigned long long ir = agg_cursor(t, rslot, hr);
    if (hl) A.pool[il] = round_rec_pos(rv, 0);
    if (hr) A.pool[ir] = round_rec_pos(rv, 1);
  }
}

// zero the cells a finished round touched: every block clears the cells of its own list (or, after an overflow, everybody
// scans the rows); runs next to the site pass of the following round -- which writes the cells of the OTHER parity -- or at exit
__device__ __forceinline__ void round_clear_cells(const RoundArgs& R, const RoundSm& S, const RoundFill& F, uint32_t lt, uint32_t nlt, uint32_t vt, uint32_t nvt) {
  if (!F.overflow) {
    const uint32_t n = min(S.ncell[F.par], R_LISTCAP);
    const uint32_t* list = round_list(R, F.par);
    for (uint32_t i = lt; i < n; i += nlt) {
      const uint32_t ent = ld_cg(list + i);
      round_cells(R, F.par, (ent >> 17) & (RB - 1u), (ent >> 16) & 1u)[ent & 0xFFFFu] = 0ull;
    }
  } else {
    const uint32_t T = F.c_first + F.k;
    const uint32_t total = F.k * 2u * T;
    for (uint32_t i = vt; i < total; i += nvt) {
      const uint32_t js = i / T, tok = i - js * T;
      round_cells(R, F.par, js >> 1, js & 1u)[tok] = 0ull;
    }
  }
  if (!R.L.mg_on) return;
  if (!F.goverflow) {  // sharded: the global cells this block listed while summing
    const uint32_t n = min(S.gncell[F.par], R_LISTCAP);
    const uint32_t* list = round_glist(R, F.par);
    for (uint32_t i = lt; i < n; i += nlt) {
      const uint32_t ent = ld_cg(list + i);
      round_gcells(R, F.par, (ent >> 17) & (RB - 1u), (ent >> 16) & 1u)[ent & 0xFFFFu] = 0ull;
    }
  } else {
    const uint32_t T = F.c_first + F.k;
    const uint32_t total = F.k * 2u * T;
    for (uint32_t i = vt; i < total; i += nvt) {
      const uint32_t js = i / T, tok = i - js * T;
      round_gcells(R, F.par, js >> 1, js & 1u)[tok] = 0ull;
    }
  }
}

__global__ void k_rounds_prepare(RoundState* rs) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    for (int p = 0; p < 2; p++)
      for (int j = 0; j < RB; j++) {
        rs->n_sites[p][j].v = 0;
        rs->ub[p][j].v = 0;
      }
    rs->overflow[0] = rs->overflow[1] = 0;
    rs->goverflow[0] = rs->goverflow[1] = 0;
  }
}

// how the warps of a block share three independent, latency-bound jobs whose items need q1/q2/q3 passes of ONE warp per
// block (q = items / (32 x blocks), rounded up) and whose dependent chains cost about l1/l2/l3 (same unit): greedy on the
// cost of each job, in float arithmetic (every thread of the grid runs this once per round: it has to be cheap)
__device__ __forceinline__ void round_split(float q1, float q2, float q3, float l1, float l2, float l3, uint32_t nwarps, uint32_t* w1, uint32_t* w2,
                                            uint32_t* w3) {
  float a = 1.f, b = 1.f, c = 1.f;
  for (uint32_t i = 3; i < nwarps; i++) {
    const float ca = ceilf(__fdividef(q1, a)) * l1, cb = ceilf(__fdividef(q2, b)) * l2, cc = ceilf(__fdividef(q3, c)) * l3;
    if (ca >= cb && ca >= cc) a += 1.f;
    else if (cb >= cc) b += 1.f;
    else c += 1.f;
  }
  *w1 = (uint32_t)a;
  *w2 = (uint32_t)b;
  *w3 = (uint32_t)c;
}

__global__ void __launch_bounds__(RD_THREADS, 1) k_merge_rounds(RoundArgs R) {
  __shared__ RoundSm S;
  const LoopArgs& L = R.L;
  const ApplyArgs& A = L.A;
  DevState* st = A.st;
  RoundState* rs = R.rs;
  const PairTable& t = A.t;
  const uint32_t bid = blockIdx.x, nblk = gridDim.x;
  const uint32_t tid = threadIdx.x;
  const uint32_t warp = tid >> 5, lane = tid & 31u;
  const uint32_t gt = bid * blockDim.x + tid, gn = nblk * blockDim.x;
  unsigned long long epoch = 0;
  const uint32_t n_tokens0 = ld_cg(&st->n_tokens);
  const uint32_t thresh = ld_cg(&st->hot_thresh);
  const bool lead = (bid == 0 && tid == 0);
#define RBARRIER()                                                        \
  do {                                                                    \
    ++epoch;                                                              \
    if (R.bar_mode) grid_barrier_ra(L.barrier, epoch * nblk, L.bar_ns);   \
    else grid_barrier(L.barrier, epoch * nblk, L.bar_ns);                 \
  } while (0)

  // ---- first partials: per-block top-2 over the hot list ----
  if (lead) st->snap_err = st->err;
  {
    Top2 mine = top2_empty();
    const uint32_t hn = ld_cg(&st->hot_n);
    for (uint32_t i = gt; i < hn; i += gn) {
      const uint32_t hs = L.hot[i];
      uint32_t hk;
      const unsigned long long pr = slot_primary_k(t, A.len16, hs, L.max_length, &hk);
      top2_add(mine, pr, hs, 1, hk);
    }
    const Top2 v = top2_block_reduce(mine, S.t2);
    if (tid == 0) {
      top2_publish(v, R.gp, R.gk, bid);
    }
    if (tid < RB) S.fill_n[tid] = 0;
    if (tid < 2) S.ncell[tid] = S.gncell[tid] = 0;
    if (tid == 0) S.pool_next = S.pool_end = S.keys_ins = S.nstage = 0;
    for (uint32_t i = tid; i < R_STAGE_CELLS; i += blockDim.x) r_stage[i] = 0ull;  // (each flush zeroes what it adds)
  }
  // sharded: exchanges completed so far (the peers' flags keep counting across launches), what the previous round may have
  // taken from the pool since the headers were written
  unsigned long long mg_epoch = R.L.mg_on ? ld_cg(&st->mg_epoch) : 0ull, tie_epoch = R.L.mg_on ? ld_cg(&st->mg_tie_epoch) : 0ull;
  unsigned long long mg_prev_alloc = 0;
  if (R.L.mg_on) {
    // hello exchange: headers only (capacities, errors), so that the first decision is taken on global minima
    if (lead) st->mg_abort = 0;
    if (bid == 0 && warp == 0) mgr_send_warp(R, 0, (uint32_t)((mg_epoch + 1) & 1u), 0, mg_epoch + 1, true);
    if (warp == 0) {  // (in EVERY block: wait for every rank's flag, own included, then fold the headers)
      if (lane < (uint32_t)R.L.mg.world) mg_wait_flag(R.L.mg.flag_data[R.L.mg.rank] + 16 * lane, mg_epoch + 1, now_ns(), 16, 128, st);
      __syncwarp();
      mgr_fold_warp(R, (uint32_t)((mg_epoch + 1) & 1u));
    }
    mg_epoch++;
  }
  RBARRIER();

  const bool prof = lead;
  unsigned long long tp0 = prof ? now_ns() : 0, tp1;
  // block 0's view, per phase (decide, P1, wait, P2, wait, -, -, tie path); fine_ns splits it into rounds of latency-bound
  // merges ([0..4], rounds in [5]) and rounds whose first merge has more than R_LAT sites ([6..10], rounds in [11])
  uint32_t prof_big = 0;
#define RPROF(i)                                              \
  if (prof) {                                                 \
    tp1 = now_ns();                                           \
    st->prof_ns[i] += tp1 - tp0;                              \
    if ((i) < 5) st->fine_ns[(prof_big ? 6 : 0) + (i)] += tp1 - tp0; \
    tp0 = tp1;                                                \
  }
  RoundFill F{0, 0, 0, 0, 0, 0};
  uint32_t it = 0;  // merges committed by this launch
  for (uint32_t round = 0;; round++) {
    const uint32_t par = round & 1u;
    const uint32_t c_first = n_tokens0 + it;
    const uint32_t hot_pre = ld_cg(&st->hot_n);
    // ================= decide =================
    {
      unsigned long long myp = 0;
      uint32_t mys = NOSLOT, mym = 0, myk = 0;
      if (tid < RT * nblk) {
        const uint4 v = ld_cg4(R.gp + tid);
        myp = (unsigned long long)v.x | ((unsigned long long)v.y << 32);
        mys = v.z;
        mym = v.w;
        myk = ld_cg(R.gk + tid);
      }
      if (tid == 0) S.qn = 0;
      if (tid < RB) {
        S.cp[tid] = 0;
        S.cm[tid] = 0;
      }
      if (tid == 1) S.ncell[par] = 0;  // (the cells the round before last listed were cleared next to the last P1)
      if (tid == 320) S.g_n_keys = ld_cg(&st->n_keys);  // (stable here: they only change in P2)
      if (tid == 321) {
        S.caps = R.L.mg_on ? loop_caps_folded(st) : loop_caps(L, ld_cg(&st->pool_cursor));
        S.caps.new_cap = 0xFFFFFFFFu;  // the rounds keep no list of born pairs (their message headers carry the same)
      }
      if (tid == 322) S.g_snap_err = ld_cg(&st->snap_err);
      if (tid == 323) S.g_abort = R.L.mg_on ? ld_cg(&st->mg_abort) : 0u;
      if (tid == 2) S.gncell[par] = 0;
      // the list of candidates is exact down to the largest LAST (RT-th best) primary any block published
      const unsigned long long Lcut = block_max_u64((tid % RT == RT - 1) ? myp : 0ull, S.red);  // (syncs inside: qn / cp are visible)
      if (myp && myp >= Lcut) {
        const uint32_t k = atomicAdd(&S.qn, 1u);
        S.qp[k] = myp;
        S.qs[k] = mys;
        S.qm[k] = mym;
        S.qk[k] = myk;
      }
      __syncthreads();
      const uint32_t qn = S.qn;
      if (tid < qn) {  // rank by counting; entries that share a primary form one group (sum of mults, smallest slot)
        const unsigned long long p = S.qp[tid];
        uint32_t rank = 0, mult = 0, slot = NOSLOT, key = 0;
        bool leader = true;
        for (uint32_t u = 0; u < qn; u++) {
          const unsigned long long pu = S.qp[u];
          rank += pu > p;
          if (pu == p) {
            mult += S.qm[u];
            if (S.qs[u] < slot) {
              slot = S.qs[u];
              key = S.qk[u];
            }
            if (u < tid) leader = false;
          }
        }
        if (leader && rank < RB) {
          S.cp[rank] = p;
          S.cs[rank] = slot;
          S.cm[rank] = mult;
          S.ck[rank] = key;
          // what the batch builder needs of this candidate, loaded side by side by the candidates' own threads
          S.cls[rank] = t.occ_start.get(slot);
          S.cll[rank] = t.occ_len[slot];
          S.clen[rank] = A.len16[key >> 16] + A.len16[key & 0xFFFFu];
        }
      }
      __syncthreads();
      if (warp == 0) {
        // lane j judges candidate j on its own; the batch is the longest prefix nobody objects to
        const uint32_t j = lane;
        const unsigned long long p0 = S.cp[0];
        const uint32_t w0 = (uint32_t)(p0 >> 20);
        uint32_t status = loop_stop(L, S.g_snap_err || S.g_abort || S.caps.err, p0, w0, thresh, it, c_first);
        if (status == LOOP_RUNNING && w0 > R_HUGE) status = LOOP_NEED_LEGACY;
        const unsigned long long pj = (j < RB) ? S.cp[j] : 0ull;
        const uint32_t wj = (uint32_t)(pj >> 20), key = (j < RB) ? S.ck[j] : 0u;
        const uint32_t aj = key >> 16, bj = key & 0xFFFFu, cj = c_first + j;
        // A pair with a token the previous round created is still having its list written (helper warps of this P1), but all
        // its occurrences are among that round's site records (double-buffered: intact), in exactly one row: (c_i, y) in merge
        // i's right row, (x, c_m) in merge m's left row, (c_i, c_m) in the row of the later merge (for i > m merge i's site
        // pass saw c_m as its virtual right neighbour; for i <= m merge m's saw c_i on its left).
        const bool fa = pj && F.v && aj >= F.c_first, fb = pj && F.v && bj >= F.c_first;
        const uint32_t src = (fa && (!fb || aj > bj)) ? (((aj - F.c_first) << 1) | 1u) : fb ? ((bj - F.c_first) << 1) : R_SRC_LIST;
        const uint32_t slen = (src != R_SRC_LIST) ? S.fill_n[src >> 1] : (j < RB ? S.cll[j] : 0u);  // entries P1 walks
        const unsigned long long new_keys = pj ? min(2ull * wj + 2ull, 2ull * (cj + 1ull) + 2ull) : 0ull;
        // cumulative over candidates 0..j (the batch is a prefix): new keys, counts, and the counts again with a pair's site
        // records in place of its count where P1 walks those (the batch limit: what a dropped tail's site pass costs)
        unsigned long long keys_incl = new_keys, w_incl = pj ? wj : 0u, s_incl = pj ? (src == R_SRC_LIST ? wj : slen) : 0u;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const unsigned long long x = __shfl_up_sync(0xFFFFFFFFu, keys_incl, o), y = __shfl_up_sync(0xFFFFFFFFu, w_incl, o),
                                   z = __shfl_up_sync(0xFFFFFFFFu, s_incl, o);
          if ((int)lane >= o) {
            keys_incl += x;
            w_incl += y;
            s_incl += z;
          }
        }
        // capacity the host guarantees, cumulative over the batch: 0 (LOOP_RUNNING) fine, else the status it would mean for
        // candidate 0.  Every block takes each round's list space from the pool in chunks.  Sharded: the headers' pool figure is
        // one round old, so what the previous round may have taken counts against it (mg_prev_alloc; this need is never 0).
        uint32_t cap_fail = loop_cap_status(S.caps, S.g_n_keys, keys_incl, 2ull * w_incl + (unsigned long long)nblk * R_POOL_CHUNK + mg_prev_alloc,
                                            j == 0 ? wj : 0u, (unsigned long long)hot_pre + keys_incl, cj);
        // sharded: a rank sends one record per touched cell, at most 2 min(w_i, c_i + 1) per merge: new_keys less 2, so the batch's
        // records are at most keys_incl - 2 (j + 1), and they must fit this rank's message area in every peer's inbox
        if (!cap_fail && R.L.mg_on && pj && keys_incl - 2ull * (j + 1u) > (unsigned long long)(R.L.mg.inbox_stride - MGR_HDR)) cap_fail = LOOP_NEED_HOST;
        const uint32_t mult0 = S.cm[0];
        if (status == LOOP_RUNNING) {
          const uint32_t cf0 = __shfl_sync(0xFFFFFFFFu, cap_fail, 0);
          if (cf0) status = cf0;
          else if (mult0 > 1 && mult0 > S.caps.cand_cap) status = LOOP_NEED_HOST;
        }
        // why candidate j >= 1 cannot join (0: it can); same codes as RoundState::stop_reason
        uint32_t stop = 0;
        if (j >= R.kmax) stop = 7;  // (the cap: reported as reason 0)
        else if (!pj) stop = 1;
        else if (cap_fail) stop = 6;
        else if (mult0 > 1 || S.cm[j] > 1) stop = 2;                                   // position tie-breaks run alone
        else if (w0 > R_SMALL || s_incl > R_BATCH_SITES) stop = 3;                     // a big merge keeps the whole grid
        else if (wj < thresh || wj < L.min_weight) stop = 6;                           // the next decision handles the status
        else if (it + j >= L.log_cap || cj >= L.max_tokens) stop = 6;
        else {
          for (uint32_t i2 = 0; i2 < j; i2++) {  // shares a token with an earlier candidate
            const uint32_t k2 = S.ck[i2], a2 = k2 >> 16, b2 = k2 & 0xFFFFu;
            if (aj == a2 || aj == b2 || bj == a2 || bj == b2) stop = 4;
          }
        }
        if (j == 0) stop = 0;
        const uint32_t objections = __ballot_sync(0xFFFFFFFFu, stop != 0);
        uint32_t k = objections ? (uint32_t)__ffs(objections) - 1u : 32u;  // first candidate that cannot join
        const uint32_t why = __shfl_sync(0xFFFFFFFFu, stop, k & 31u);
        if (status != LOOP_RUNNING) k = 0;
        if (j < 8) S.filt_a[j] = S.filt_b[j] = 0;
        __syncwarp();
        if (j < k) {
          atomicOr(&S.filt_a[(aj >> 5) & 7u], 1u << (aj & 31u));
          atomicOr(&S.filt_b[(bj >> 5) & 7u], 1u << (bj & 31u));
          S.a[j] = aj;
          S.b[j] = bj;
          S.w[j] = wj;
          S.slot[j] = S.cs[j];
          S.lstart[j] = S.cls[j];
          S.src[j] = src;
          S.llen[j] = slen;
          S.lenc[j] = S.clen[j];
        }
        uint32_t it_incl = (j < k) ? ((slen + 31u) >> 5) : 0u;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const uint32_t x = __shfl_up_sync(0xFFFFFFFFu, it_incl, o);
          if ((int)lane >= o) it_incl += x;
        }
        if (j < RB) S.iter0[j + 1] = it_incl;
        if (j == 0) {
          S.iter0[0] = 0;
          S.k = k;
          S.status = status;
          S.mult0 = mult0;
          if (bid == 0 && status == LOOP_RUNNING) {
            rs->rounds++;
            rs->tried += k;
            rs->stop_reason[why == 7 ? 0 : why]++;
            if (k == 1) rs->rounds_single++;
          }
        }
      }
      __syncthreads();
    }
    uint32_t status = S.status;
    uint32_t k = S.k;
    prof_big = (status == LOOP_RUNNING && S.w[0] > R_LAT) ? 1u : 0u;
    const bool prof_big_all = prof_big != 0;
    if (lead && status == LOOP_RUNNING) {
      if (prof_big) rs->iters_big += S.iter0[k];
      else rs->iters_small += S.iter0[k];
    }
    if (prof && status == LOOP_RUNNING) st->fine_ns[prof_big ? 11 : 5] += 1;
    RPROF(0)
    // ---- tie on (weight, a.index+b.index): the pair whose last counted occurrence comes first wins (core.ts:294-305) ----
    if (status == LOOP_RUNNING && S.mult0 > 1) {
      if (F.v) {  // the tie-break reads occurrence lists: those of the last round must be complete
        round_fill_all(R, S, F, gt, gn);
        __syncthreads();
        if (tid < RB) S.fill_n[tid] = 0;
        F.v = 0;  // (the rows of that round still wait for their clearing: F.k stays)
        RBARRIER();
      }
      phase_collect(t, A.len16, L.max_length, 1, L.hot, hot_pre, S.cp[0], L.cands, L.cand_cap, st, bid, nblk);
      RBARRIER();
      uint32_t tie_slot;
      if (!R.L.mg_on) {
        phase_tie(A.slots, A.n, t, A.pool, L.cands, ld_cg(&st->n_cand), st, S.s_max, bid, nblk);
        RBARRIER();
        const unsigned long long tp = ld_cg(&st->tie_pos);
        tie_slot = (tp == ~0ull) ? NOSLOT : (uint32_t)(tp & 0xFFFFFFFFu);
      } else {
        tie_slot = mg_tie_winner(L, S.s_max, tie_epoch, [&] { RBARRIER(); });  // (rank, local position) decides
      }
      __syncthreads();
      if (tie_slot == NOSLOT) {
        status = LOOP_ERROR;
      } else if (tid == 0) {
        const uint32_t s = tie_slot;
        const uint32_t key = t.keys[s];
        S.slot[0] = s;
        S.a[0] = key >> 16;
        S.b[0] = key & 0xFFFFu;
        for (int i = 0; i < 8; i++) S.filt_a[i] = S.filt_b[i] = 0;
        S.filt_a[((key >> 16) >> 5) & 7u] = 1u << ((key >> 16) & 31u);
        S.filt_b[((key & 0xFFFFu) >> 5) & 7u] = 1u << (key & 31u);
        S.lstart[0] = t.occ_start.get(s);
        S.src[0] = R_SRC_LIST;  // (the lists of the last round are complete: filled above)
        S.llen[0] = t.occ_len[s];
        S.lenc[0] = A.len16[key >> 16] + A.len16[key & 0xFFFFu];
        S.iter0[1] = (S.llen[0] + 31u) >> 5;
      }
      __syncthreads();
    }
    RPROF(7)
    if (status != LOOP_RUNNING) {
      // the kernel leaves every list complete and every row zero
      round_fill_all(R, S, F, gt, gn);
      if (F.k) round_clear_cells(R, S, F, tid, blockDim.x, gt, gn);
      if (lead) {
        const Best wb{S.cp[0], S.cp[0] ? S.cs[0] : NOSLOT, S.cm[0]};
        loop_exit(t, st, status, it, c_first, &wb, R.L.mg_on, mg_epoch, tie_epoch);
      }
      return;
    }
    // ================= P1: the site passes of the batch, next to the list filling of the previous round =================
    if (bid == 0 && warp == 0) {
      if (lane < k) A.len16[c_first + lane] = S.lenc[lane];  // chars = a.chars + b.chars (:318)
      if (lane < RB) {
        rs->n_sites[par ^ 1u][lane].v = 0;
        rs->ub[par ^ 1u][lane].v = 0;
      }
      if (lane == 0 && S.mult0 > 1) st->tie_breaks++;
    }
    {
      const uint32_t iters = S.iter0[k];
      uint32_t fill_total = 0;
      for (uint32_t j = 0; j < F.v; j++) fill_total += S.fill_n[j];
      // latency bound: some warps of every block walk the sites, the others fill the lists of the previous round's pairs and
      // zero the cells that round touched; throughput bound: everybody does everything
      const bool split = iters <= 3u * nblk * ((L.p1_sites * (blockDim.x >> 5)) / 16u) && fill_total <= 65536u;
      const uint32_t NW = blockDim.x >> 5;
      const uint32_t ws = split ? (L.p1_sites * NW) / 16u : NW, wh = NW - ws;
      if (warp < ws) {
        for (uint32_t wi = bid * ws + warp; wi < iters; wi += nblk * ws) {
          uint32_t j = 0;
          while (j + 1 < k && wi >= S.iter0[j + 1]) j++;
          round_sites_iter(R, S, par, F.par, j, c_first, (wi - S.iter0[j]) * 32u + lane, round_sites_buf(R, par, j), j == 0 ? A.sites_cap : R_SMALL);
        }
        if (!split) {
          if (F.v) round_fill_all(R, S, F, gt, gn);
          if (F.k) round_clear_cells(R, S, F, tid, blockDim.x, gt, gn);
        }
      } else {
        const uint32_t hvt = (bid * wh + warp - ws) * 32u + lane, hnvt = nblk * wh * 32u;
        if (F.v) round_fill_all(R, S, F, hvt, hnvt);
        if (F.k) round_clear_cells(R, S, F, (warp - ws) * 32u + lane, wh * 32u, hvt, hnvt);
        // Speculation: the candidates the batch left behind are the most likely members of the next one.  The helper warps
        // pull their occurrence lists and the corpus lines around the occurrences into L2, so that the next site pass -- a chain
        // of dependent loads -- finds them there instead of in DRAM.  Hints only: nothing depends on them.
        if (L.prefetch) {
          uint32_t budget = 32768u;
          for (uint32_t j = k; j < RB && budget; j++) {
            if (!S.cp[j]) break;
            const uint32_t len = min(S.cll[j], budget);
            const unsigned long long start = S.cls[j];
            for (uint32_t i = hvt; i < len; i += hnvt) {
              const uint32_t pp = ld_cg(A.pool + start + i);
              if (pp >= A.n) continue;
              const uint32_t* q = A.slots + pp;
              prefetch_l2(q);
              if (pp >= 12u) prefetch_l2(q - 12);
              if (pp + 28u < A.n) prefetch_l2(q + 28);
            }
            budget -= len;
          }
        }
      }
      bool staging = false;
      for (uint32_t j = 0; j < k; j++) staging |= S.llen[j] > R.L.stage_min;
      if (staging) round_flush_stage(R, S, par, c_first);
    }
    RPROF(1)
    RBARRIER();
    if (tid == 0) S.nstage = 0;  // (every thread of the block has read it: RBARRIER ends with __syncthreads)
    RPROF(2)
    if (R.L.mg_on) {
      // ================= sharded: one exchange per round =================
      // block 0 writes this rank's header (bounds, site counts, capacities, batch) into every rank's inbox, every block the
      // cells it listed as records; each block then reports to every rank's arrival counter.  No grid barrier on the way out:
      // a receiver knows a message is complete when all blocks of the sender have reported.
      const uint32_t epar = (uint32_t)((mg_epoch + 1) & 1u);
      unsigned long long xt0 = prof ? now_ns() : 0, xt1;
#define XPROF(i)                         \
  if (prof) {                            \
    xt1 = now_ns();                      \
    st->mg_prof_ns[5 + (i)] += xt1 - xt0; \
    xt0 = xt1;                           \
  }
      round_emit_records(R, S, par, epar, k, c_first + k, mg_epoch + 1);
      XPROF(0)
      mgr_collect(R, S, par, epar);  // all ranks' records summed into the global cells as they arrive, headers folded
      XPROF(1)
      mg_epoch++;
      if (ld_cg(&st->mg_abort)) {  // a peer did not answer: every block of every rank that still runs leaves
        if (lead) loop_exit(t, st, LOOP_ERROR, it, c_first, nullptr, true, mg_epoch, tie_epoch);
        return;
      }
      RBARRIER();
      if (bid == 0 && tid < (uint32_t)R.L.mg.world) {  // (used again two rounds on; the next round's records are reserved after more barriers)
        *mgr_counter(R.L.mg, R.L.mg.rank, epar, (int)tid) = 0ull;
        if (tid == 0) st->n_out = 0;
      }
      XPROF(2)
#undef XPROF
      RPROF(5)
    }
    // ================= P2 =================
    // valid prefix: no pair born by an earlier merge of the batch may reach the count of a later one
    // (sharded: every rank commits at most the smallest batch any rank tried, bounds and site counts are sums over the ranks)
    const uint32_t k_all = R.L.mg_on ? min(k, ld_cg(&rs->mg_k)) : k;
    uint32_t v = k_all;
    const uint32_t ns_all = (lane < k) ? ld_cg(&rs->n_sites[par][lane].v) : 0u;  // (requested together with the bounds and the flag)
    const uint32_t ns_glob = R.L.mg_on ? ((lane < k_all) ? ld_cg(&rs->mg_ns[lane]) : 0u) : ns_all;
    const uint32_t overflow = ld_cg(&rs->overflow[par]);                         // (set during P1 only)
    const uint32_t goverflow = R.L.mg_on ? ld_cg(&rs->goverflow[par]) : 0u;
    {
      const unsigned long long ub2 = (lane < k_all) ? (R.L.mg_on ? ld_cg(&rs->mg_ub[lane]) : ld_cg(&rs->ub[par][lane].v)) : 0ull;
      const uint32_t ubv = max((uint32_t)ub2, (uint32_t)(ub2 >> 32));  // lane j: the larger of merge j's two bounds
      uint32_t run = 0;
      for (uint32_t j = 0; j + 1 < k_all; j++) {
        run = max(run, __shfl_sync(0xFFFFFFFFu, ubv, j));
        if (run >= S.w[j + 1]) {
          v = j + 1;
          break;
        }
      }
    }
    // sites per merge (lane j of every warp holds merge j's), their sum
    const uint32_t ns_lane = (lane < v) ? ns_all : 0u;
    uint32_t sites_all = ns_lane;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sites_all += __shfl_xor_sync(0xFFFFFFFFu, sites_all, o);
    if (bid == 0 && warp == 0) {  // lane j commits merge j of the batch (a serial loop here would sit on every round's critical path)
      const bool mine_j = lane < v;
      if (mine_j) {
        MergeRec r;
        r.a = (int32_t)S.a[lane];
        r.b = (int32_t)S.b[lane];
        r.c = (int32_t)(c_first + lane);
        r.reserved = 0;
        r.weight = (long long)S.w[lane];
        L.log[it + lane] = r;
        t.cnt[S.slot[lane]] = 0;  // every counted occurrence of the winner is being replaced
      }
      const uint32_t bad = __ballot_sync(0xFFFFFFFFu, mine_j && ns_glob != S.w[lane]);
      if (lane == 0) {
        st->live_tokens -= sites_all;
        st->sites_total += sites_all;
        st->n_cand = 0;
        st->tie_pos = ~0ull;
        if (bad) atomicOr(&st->err, ERR_ROUND_MISMATCH);
        st->snap_err = st->err;
        rs->round_merges += v;
        if (S.w[0] > R_LAT) rs->sites_big += sites_all; else rs->sites_small += sites_all;
        if (v < k) rs->rounds_cut_born++;
      }
    }
    Top2 mine = top2_empty();
    if (tid == 0) {
      S.keys_ins = 0;
      if (S.pool_next + R_POOL_CHUNK / 4u > S.pool_end || S.pool_next > S.pool_end) {  // the chunk is (nearly) used up: take a fresh one
        const unsigned long long at = atomicAdd(&st->pool_cursor, (unsigned long long)R_POOL_CHUNK);
        if (at <= L.pool_cap && R_POOL_CHUNK <= L.pool_cap - at) {
          S.pool_base = at;
          S.pool_next = 0;
          S.pool_end = R_POOL_CHUNK;
        } else {
          S.pool_next = S.pool_end = 0;  // (the decision keeps this from happening; lists then come from the cursor and fail its check)
        }
      }
    }
    __syncthreads();
    const bool jprof = bid == 0 && lane == 0 && !prof_big_all;  // block 0, rounds of small merges: when each job of P2 ends
    const unsigned long long jt0 = jprof ? now_ns() : 0;
    {
      const bool split = sites_all <= (1u << 20);
      const uint32_t NW = blockDim.x >> 5;
      uint32_t wn = NW, wr = NW, wm = NW;
      if (split) {
        const float rg = __fdividef(1.f, (float)(nblk * 32u));
        round_split(ceilf((float)sites_all * 0.5f * rg), ceilf((float)sites_all * rg), ceilf((float)hot_pre * rg), 8.f, 2.f, 5.f, NW, &wn, &wr, &wm);
      }
      // ---- job 1: the cells the site passes touched -> born pairs and decrements of the valid merges.  Every block works
      // through the list of the cells IT touched first, one cell per lane (after a list overflow: everybody scans the rows) ----
      if (!split || warp < wn) {
        const uint32_t n1t = split ? wn * 32u : blockDim.x;  // threads of this block on the job (its first warps)
        const uint32_t lt = tid;
        // one touched cell: warp-collective (inactive lanes pass act = false)
        auto process = [&](bool act, uint32_t jj, uint32_t side, uint32_t tok, unsigned long long cellv) {
          const uint32_t cj = c_first + jj;
          const uint32_t ajj = S.a[jj], bjj = S.b[jj];
          const uint32_t dec = act ? cell_dec(cellv) : 0u, len = act ? cell_len(cellv) : 0u;
          uint32_t cntv = cell_cnt(cellv);
          // the old pair's home slot (key, count) is requested NOW: its round trip runs next to the born pair's insertion
          const bool has_dec = dec != 0 && tok < c_first;
          const uint32_t dpa = side ? bjj : tok, dpb = side ? tok : ajj;
          const uint32_t dkey = pair_key(dpa, dpb), dh = tbl_hash(t, dkey);
          uint32_t dk0 = EMPTY_KEY, dold = 0;
          if (has_dec) {
            dk0 = t.keys[dh];
            dold = t.cnt[dh];
          }
          // ---- a pair born by merge jj: (tok, c) or (c, tok) ----
          {
            const bool born = len != 0 || (act && cntv != 0);  // (sharded: counted on another shard only -> the key and its count, no list)
            // list space first (one cursor atomic per warp): its round trip overlaps the table probe below
            uint32_t mylen = len;
            uint32_t inc = mylen;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
              const uint32_t x = __shfl_up_sync(0xFFFFFFFFu, inc, o);
              if ((int)lane >= o) inc += x;
            }
            const uint32_t wtotal = __shfl_sync(0xFFFFFFFFu, inc, 31);
            // the warp's list cells come out of the block's private chunk of the pool (a shared-memory bump); only a warp that
            // needs more than a chunk holds, or finds the chunk used up, goes to the grid-wide cursor
            unsigned long long wbase = 0;
            if (lane == 31 && wtotal) {
              bool got = false;
              if (wtotal <= R_POOL_CHUNK / 4u) {
                const uint32_t at = atomicAdd(&S.pool_next, wtotal);
                if (at + wtotal <= S.pool_end) {
                  wbase = S.pool_base + at;
                  got = true;
                }
              }
              if (!got) {
                // (a failed bump leaves pool_next past pool_end: every later warp of the round takes this path too, and the
                // block fetches a fresh chunk at the start of its next P2)
                wbase = atomicAdd(&st->pool_cursor, (unsigned long long)wtotal);
              }
            }
            uint32_t s = NOSLOT, hot_s = NOSLOT, hot_key = 0;
            unsigned long long hot_pr = 0ull;
            bool ins = false;
            if (born) {
              // adjacencies a LATER valid merge of the batch took away again (its virtual neighbour c_jj)
              if (role_maybe(side ? S.filt_a : S.filt_b, tok)) {
                for (uint32_t j2 = jj + 1; j2 < v; j2++) {
                  if (side) {
                    if (tok == S.a[j2]) cntv -= round_dec_of(R, par, j2, 0, cj);
                  } else {
                    if (tok == S.b[j2]) cntv -= round_dec_of(R, par, j2, 1, cj);
                  }
                }
              }
              // the key is new (it holds a token this round creates): claim the home slot with one CAS, probe on only when taken
              const uint32_t key = side ? pair_key(cj, tok) : pair_key(tok, cj);
              const uint32_t h = tbl_hash(t, key);
              const uint32_t was = atomicCAS(t.keys + h, EMPTY_KEY, key);
              if (was == EMPTY_KEY) {
                s = h;
                ins = true;
              } else {
                s = tbl_find_or_insert_ex(t, key, &ins);
              }
              if (s == NOSLOT) atomicOr(&st->err, ERR_TABLE_FULL);
            }
            const uint32_t im = __ballot_sync(0xFFFFFFFFu, ins);
            if (im && lane == (uint32_t)(__ffs(im) - 1)) atomicAdd(&S.keys_ins, (uint32_t)__popc(im));
            wbase = __shfl_sync(0xFFFFFFFFu, wbase, 31);
            if (born && s != NOSLOT) {
              unsigned long long start = wbase + (inc - mylen);
              if (start > L.pool_cap || mylen > L.pool_cap - start) {
                atomicOr(&st->err, ERR_POOL_FULL);
                start = 0;
                mylen = 0;
              }
              t.occ_start.set(s, start);
              t.occ_len[s] = mylen;
              t.occ_fill[s] = 0;
              round_slotrow(R, par, jj, side)[tok] = s;
              t.cnt[s] = cntv;  // the key is new: nobody else touches its count in this phase
              const uint32_t pa = side ? cj : tok, pb = side ? tok : cj;
              const uint32_t la = (pa >= c_first) ? S.lenc[pa - c_first] : A.len16[pa], lb = (pb >= c_first) ? S.lenc[pb - c_first] : A.len16[pb];
              const unsigned long long pr = (cntv && !(L.max_length && la + lb > L.max_length)) ? make_primary(cntv, pa, pb) : 0ull;
              hot_pr = (pr && (uint32_t)(pr >> 20) >= thresh) ? pr : 0ull;
              hot_s = s;
              hot_key = pair_key(pa, pb);
            }
            // pairs that join the hot list: one hot_n atomic per warp
            const uint32_t hm = __ballot_sync(0xFFFFFFFFu, hot_pr != 0ull);
            if (hm) {
              uint32_t hbase = 0;
              const int src = __ffs(hm) - 1;
              if ((int)lane == src) hbase = atomicAdd(&st->hot_n, (uint32_t)__popc(hm));
              hbase = __shfl_sync(0xFFFFFFFFu, hbase, src);
              if (hot_pr) {
                const uint32_t hk = hbase + __popc(hm & ((1u << lane) - 1u));
                if (hk < L.hot_cap) L.hot[hk] = hot_s;
                else atomicOr(&st->err, ERR_HOT_OVERFLOW);
                top2_add(mine, hot_pr, hot_s, 1, hot_key);
              }
            }
          }
          // ---- decrements of an OLD pair: (tok, a_jj) on the left side, (b_jj, tok) on the right side ----
          if (has_dec) {
            uint32_t totald = dec;
            bool handle = true;
            if (side) {  // (b_jj, tok): also decremented from the left side of the valid merge whose a is tok
              if (role_maybe(S.filt_a, tok))
                for (uint32_t j2 = 0; j2 < v; j2++)
                  if (tok == S.a[j2]) totald += round_dec_of(R, par, j2, 0, bjj);
            } else {     // (tok, a_jj): when tok is the b of a valid merge whose right side holds the pair too, that side handles both
              if (role_maybe(S.filt_b, tok))
                for (uint32_t j2 = 0; j2 < v; j2++)
                  if (tok == S.b[j2] && round_dec_of(R, par, j2, 1, ajj) != 0) handle = false;
            }
            if (handle) {
              const uint32_t pa = dpa, pb = dpb, key = dkey, h = dh, k0 = dk0;
              uint32_t old = dold;
              uint32_t s = h;
              if (k0 != key) {
                s = (k0 == EMPTY_KEY) ? NOSLOT : tbl_find(t, key);
                if (s != NOSLOT) old = t.cnt[s];
              }
              if (s == NOSLOT) {
                atomicOr(&st->err, ERR_MISSING_KEY);
              } else {
                if (old < totald) atomicOr(&st->err, ERR_ROUND_MISMATCH);
                const uint32_t nv = old - totald;
                t.cnt[s] = nv;  // this thread is the only one that touches the pair in this phase
                if (nv && !(L.max_length && A.len16[pa] + A.len16[pb] > L.max_length)) top2_add(mine, make_primary(nv, pa, pb), s, 1, pair_key(pa, pb));
              }
            }
          }
        };
        // sharded: the global cell (decrements, counted occurrences: sums over the ranks) and this shard's (occurrences: its
        // list space) of one (merge, side, token), in the layout `process` reads
        auto cell_of = [&](uint32_t jj, uint32_t side, uint32_t tok) -> unsigned long long {
          if (!R.L.mg_on) return ld_cg(round_cells(R, par, jj, side) + tok);
          const unsigned long long g = ld_cg(round_gcells(R, par, jj, side) + tok), l = ld_cg(round_cells(R, par, jj, side) + tok);
          return (g & R_FMASK) | ((unsigned long long)cell_len(l) << R_FIELD) | (((g >> R_FIELD) & R_FMASK) << (2 * R_FIELD));
        };
        if (!(R.L.mg_on ? goverflow : overflow)) {
          const uint32_t ncell = R.L.mg_on ? S.gncell[par] : S.ncell[par];
          const uint32_t* list = R.L.mg_on ? round_glist(R, par) : round_list(R, par);
          if (lt == 0 && ncell) atomicAdd(S.w[0] > R_LAT ? &rs->cells_big : &rs->cells_small, (unsigned long long)ncell);
          for (uint32_t base = 0; base < ncell; base += n1t) {
            const uint32_t idx = base + lt;
            const uint32_t ent = idx < ncell ? ld_cg(list + idx) : 0u;
            const uint32_t jj = (ent >> 17) & (RB - 1u), side = (ent >> 16) & 1u, tok = ent & 0xFFFFu;
            const bool act = idx < ncell && jj < v;
            const unsigned long long cellv = act ? cell_of(jj, side, tok) : 0ull;
            process(act, jj, side, tok, cellv);
          }
        } else {
          // a list was full: every cell of the valid merges' rows, shared by the job's threads of the whole grid
          const uint32_t T = (c_first + k + 31u) & ~31u;
          const uint32_t total = v * 2u * T;
          for (uint32_t i = bid * n1t + lt; i < total; i += nblk * n1t) {
            const uint32_t js = i / T, tok = i - js * T;
            const unsigned long long cellv = cell_of(js >> 1, js & 1u, tok);
            if (!__any_sync(0xFFFFFFFFu, cellv != 0ull)) continue;
            process(cellv != 0ull, js >> 1, js & 1u, tok, cellv);
          }
        }
      }
      if (jprof && warp == 0) st->mg_prof_ns[0] += now_ns() - jt0;
      // ---- job 2: rewrite the corpus at the sites of the valid merges (the records carry the spans) ----
      if (!split || (warp >= wn && warp < wn + wr)) {
        const uint32_t vt = split ? (bid * wr + warp - wn) * 32u + lane : gt, nvt = split ? nblk * wr * 32u : gn;
        uint32_t* slots = A.slots;
        // one index space over the sites of all valid merges (32-aligned per merge): every thread of the job gets its share
        uint32_t total = 0;
        for (uint32_t j = 0; j < v; j++) total += (__shfl_sync(0xFFFFFFFFu, ns_lane, j) + 31u) & ~31u;
        for (uint32_t i = vt; i < total; i += nvt) {
          uint32_t j = 0, off = i;
          for (;;) {  // (warp-uniform)
            const uint32_t nj = (__shfl_sync(0xFFFFFFFFu, ns_lane, j) + 31u) & ~31u;
            if (off < nj) break;
            off -= nj;
            j++;
          }
          if (off >= __shfl_sync(0xFFFFFFFFu, ns_lane, j)) continue;
          const uint4 rv = ld_cg4(reinterpret_cast<const uint4*>(round_sites_buf(R, par, j)) + off);
          const uint32_t cj = c_first + j;
          const uint32_t p = rv.x;
          uint32_t q, e;
          if (rv.w & 0x40000000u) {  // span too long for the record: walk
            q = next_pos(slots, A.n, p);
            e = next_pos(slots, A.n, q) - 1;
          } else {
            q = p + ((rv.w >> 15) & 0x7FFFu);
            e = p + (rv.w & 0x7FFFu);
          }
          const uint32_t span = e - p + 1;
          if (span > VAL_MASK) atomicOr(&st->err, ERR_SPAN_OVERFLOW);
          slots[p] = (rv.w & DOCSTART) | cj;
          if (span == 2) {
            slots[p + 1] = mk_back(1);
          } else {
            if (q != p + 1 && q != e) slots[q] = mk_hole();
            slots[p + 1] = mk_span(span);
            slots[e] = mk_back(span - 1);
          }
        }
      }
      if (jprof && split && warp == wn) st->mg_prof_ns[1] += now_ns() - jt0;
      // ---- job 3: arg-max over the pairs that were already hot and that no valid merge touches ----
      if (!split || warp >= wn + wr) {
        const uint32_t vt = split ? (bid * wm + warp - wn - wr) * 32u + lane : gt, nvt = split ? nblk * wm * 32u : gn;
        for (uint32_t i = vt; i < hot_pre; i += nvt) {
          const uint32_t hs = L.hot[i];
          const uint32_t key = t.keys[hs];
          if (key == EMPTY_KEY) continue;
          const uint32_t cv = t.cnt[hs];  // (in flight next to the role test)
          const uint32_t x = key >> 16, y = key & 0xFFFFu;
          bool skip = false;
          if (role_maybe(S.filt_a, y) || role_maybe(S.filt_b, x) || role_maybe(S.filt_a, x)) {  // (a winner (a_j, b_j) passes the last test)
            for (uint32_t j2 = 0; j2 < v; j2++) {
              if (hs == S.slot[j2]) skip = true;  // a winner: its count is being zeroed
              if (y == S.a[j2] && round_dec_of(R, par, j2, 0, x) != 0) skip = true;  // job 1 hands in its new count
              if (x == S.b[j2] && round_dec_of(R, par, j2, 1, y) != 0) skip = true;
            }
          }
          if (skip || !cv) continue;
          if (L.max_length && A.len16[x] + A.len16[y] > L.max_length) continue;
          top2_add(mine, make_primary(cv, x, y), hs, 1, key);
        }
      }
    }
    if (jprof && warp == (blockDim.x >> 5) - 1u) st->mg_prof_ns[2] += now_ns() - jt0;
    {
      const Top2 tv = top2_block_reduce(mine, S.t2);
      if (tid == 0 && S.keys_ins) atomicAdd(&st->n_keys, S.keys_ins);
      if (tid < 2 && tv.p[0]) {  // the next decision reads the list fields of its candidates: ask for them now
        const uint32_t ps = tid == 0 ? tv.s[0] : tv.s[RT - 1];
        if (ps != NOSLOT) {
          prefetch_l2(t.occ_start.addr(ps));
          prefetch_l2(t.occ_len + ps);
        }
      }
      if (tid == 0) {
        top2_publish(tv, R.gp, R.gk, bid);
      }
      if (tid < RB) S.fill_n[tid] = (tid < v) ? ld_cg(&rs->n_sites[par][tid].v) : 0u;
    }
    if (jprof && warp == 0) {
      st->mg_prof_ns[3] += now_ns() - jt0;
      st->mg_prof_ns[4] += 1;
    }
    F.v = v;
    F.par = par;
    F.k = k;
    F.c_first = c_first;
    F.overflow = overflow;
    F.goverflow = goverflow;
    if (lead) rs->overflow[par ^ 1u] = rs->goverflow[par ^ 1u] = 0;  // (read by nobody before the next round's P2, set by nobody before its P1)
    if (R.L.mg_on) {  // what this round's P2 may take from the pool on any rank: the headers of the next exchange are written before
      unsigned long long wsum = 0;
      for (uint32_t j = 0; j < v; j++) wsum += S.w[j];
      mg_prev_alloc = 2ull * wsum + (unsigned long long)nblk * R_POOL_CHUNK;
    }
    it += v;
    RPROF(3)
    RBARRIER();
    RPROF(4)
  }
#undef RPROF
#undef RBARRIER
}

}  // namespace bpe
