// mg_kernels.cuh -- mergeUntil on a corpus sharded by document over several GPUs (one process per GPU).
//
// Reference semantics: the corpus is one list of documents (core.ts:106); findNextMerge counts pairs over ALL of them
// (core.ts:265-310) and applyMerge rewrites ALL of them (core.ts:356-359).  Documents never interact except through
// the global pair counts and the arg-max, so the corpus shards by document:
//   * rank r owns a contiguous range of documents (global scan order = (rank, local position), which is what the
//     reference's position tie-break needs, core.ts:294-305), its slots, occurrence lists and pool;
//   * the pair table's COUNTS are global and replicated: every merge, each rank stages its local count deltas
//     (cnt_delta), aggregates them per pair, and stores the (pair, delta) records straight into every peer's inbox
//     over NVLink (peer-mapped memory, cudaIpc); one flag store per peer publishes them.  Every rank then applies all
//     G record lists, so all tables hold the same counts and the arg-max needs NO collective: it is computed
//     redundantly and identically everywhere;
//   * only when several pairs tie on (weight, a.index + b.index) a second small exchange carries each rank's last
//     counted position per candidate (candidates in canonical key order); the highest rank holding a candidate owns its
//     last occurrence (mg_tie_winner).
// Everything runs inside a persistent cooperative kernel per GPU: compute and the exchange are fused, there is no host
// round trip and no NCCL call per merge.  k_merge_rounds with mg_on (round_kernels.cuh) runs almost every merge, several per
// exchange; k_merge_loop with mg_on (below: one kernel for one GPU and a sharded corpus) runs one merge per exchange: those above
// R_HUGE global sites, or all of them under BPE_LOOP_ROUNDS=0.  Their record formats differ; the steps every rank must run
// identically live here once, for both: the header of a message (mg_store_header) and its fold (mg_fold_headers_warp), the wait
// on a peer's flag (mg_wait_flag) and the tie-break.  Every decision that ends or interrupts the loop is taken from replicated values (or minima over ranks carried in
// the message headers: loop_caps_folded), with the stop chain and capacity test every loop kernel shares (loop_stop,
// loop_cap_status in train_kernels.cuh), so all ranks leave the kernel at the same merge with the same status.  Waits on peers are bounded
// (MG_TIMEOUT_NS) and abort the loop.
#pragma once
#include "train_kernels.cuh"

namespace bpe {

constexpr uint32_t MG_HDR = 16;  // u64 words of header in front of the records of one message
enum { H_N = 0, H_ERR, H_POOL_FREE, H_SITES_CAP, H_NEW_CAP, H_HOT_CAP, H_LEN16_CAP, H_TBL_CAP, H_CAND_CAP, H_STATUS };
constexpr unsigned long long MG_TIMEOUT_NS = 8000000000ull;
// u64 words of one (parity, sender) message area of an inbox, header included.  k_merge_loop sends at most 2 (c + 1) born-pair
// records and one per touched pair (< 4 BPE_MAX_TOKENS) per merge; k_merge_rounds bounds the records of a batch when it builds it.
constexpr uint32_t MG_INBOX_STRIDE = 1u << 20;
static_assert(2u * ND_STRIDE + 4u * BPE_MAX_TOKENS + 64u + MG_HDR <= MG_INBOX_STRIDE, "one merge of k_merge_loop must fit a message");

__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

// wait until a peer's flag `f` reaches `epoch`, sleeping `ns` ns between looks, doubled up to `ns_max`.  Still waiting
// MG_TIMEOUT_NS after t0: ERR_PEER_TIMEOUT, mg_abort set (the loop ends at its next check), false.
__device__ __forceinline__ bool mg_wait_flag(const unsigned long long* f, unsigned long long epoch, unsigned long long t0, uint32_t ns,
                                             uint32_t ns_max, DevState* st) {
  while (ld_acquire_sys(f) < epoch) {
    __nanosleep(ns);
    if (ns < ns_max) ns <<= 1;
    if (now_ns() - t0 > MG_TIMEOUT_NS) {
      atomicOr(&st->err, ERR_PEER_TIMEOUT);
      st->mg_abort = 1;
      return false;
    }
  }
  return true;
}

// thread 0 of block 0: publish `epoch` to every peer and wait until every peer has published it to us
__device__ __forceinline__ void mg_signal_and_wait(const MgArgs& M, unsigned long long* const* flags, unsigned long long epoch,
                                                   DevState* st) {
  for (int q = 0; q < M.world; q++)
    if (q != M.rank) st_release_sys(flags[q] + 16 * M.rank, epoch);
  const unsigned long long t0 = now_ns();
  for (int q = 0; q < M.world; q++)
    if (q != M.rank && !mg_wait_flag(flags[M.rank] + 16 * q, epoch, t0, 32, 1024, st)) return;
}

// ---- initial histogram exchange (host-driven, once per index build) ----------------------------------------------
__global__ void k_mg_export_counts(PairTable t, uint32_t* __restrict__ keys, uint32_t* __restrict__ cnts, uint32_t cap,
                                   uint32_t* __restrict__ n_out) {
  uint32_t tcap = t.mask + 1;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < tcap; i += gridDim.x * blockDim.x) {
    uint32_t key = t.keys[i];
    if (key == EMPTY_KEY) continue;
    uint32_t c = t.cnt[i];
    if (c == 0) continue;
    uint32_t k = atomicAdd(n_out, 1u);
    if (k < cap) {
      keys[k] = key;
      cnts[k] = c;
    }
  }
}

__global__ void k_mg_import_counts(PairTable t, const uint32_t* __restrict__ keys, const uint32_t* __restrict__ cnts, uint32_t n,
                                   DevState* st) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    uint32_t s = tbl_find_or_insert(t, keys[i], &st->n_keys);
    if (s == NOSLOT) {
      atomicOr(&st->err, ERR_TABLE_FULL);
    } else {
      const uint32_t old = atomicAdd(t.cnt + s, cnts[i]);
      if (old + cnts[i] < old) atomicOr(&st->err, ERR_COUNT_OVERFLOW);  // the global count does not fit 32 bits
    }
  }
}

// ---- the loop ----------------------------------------------------------------------------------------------------
// message of this rank for exchange `epoch`: header + n records (pair_key << 32 | (u32)delta) in every inbox
__device__ __forceinline__ unsigned long long* mg_area(const MgArgs& M, int dst, uint32_t par, int sender) {
  return M.inbox[dst] + ((size_t)par * M.world + sender) * M.inbox_stride;
}

// header of a message: 16 u32 (H_* indices) in the first 64 bytes of the area, moved with 128-bit accesses.  This rank's
// record count, error flags and capacities (its LoopCaps, H_N .. H_CAND_CAP, the pool figure clamped to 32 bits) into the header
// at `dst`; the pool figure only gates the next decision.
__device__ __forceinline__ void mg_store_header(const LoopArgs& L, unsigned long long* dst, uint32_t n_rec, uint32_t new_cap) {
  DevState* st = L.A.st;
  const LoopCaps g = loop_caps(L, ld_cg(&st->pool_cursor));
  uint32_t h[12];
#pragma unroll
  for (int i = 0; i < 12; i++) h[i] = 0;
  h[H_N] = n_rec;
  h[H_ERR] = ld_cg(&st->err);
  h[H_POOL_FREE] = (uint32_t)min(max(g.pool_free, 0ll), 0xFFFFFFFFll);
  h[H_SITES_CAP] = g.sites_cap;
  h[H_NEW_CAP] = new_cap;
  h[H_HOT_CAP] = g.hot_cap;
  h[H_LEN16_CAP] = g.len16_cap;
  h[H_TBL_CAP] = g.tbl_cap;
  h[H_CAND_CAP] = min(g.cand_cap, L.mg.tie_cap);
  uint4* d4 = reinterpret_cast<uint4*>(dst);
#pragma unroll
  for (int i = 0; i < 3; i++) d4[i] = make_uint4(h[4 * i], h[4 * i + 1], h[4 * i + 2], h[4 * i + 3]);
}

// One warp, lane q reads sender q's header in this rank's area `par` (the messages are complete): the G headers fold into
// st->g_vals (OR of the error flags, minima of the capacities; loop_caps_folded reads them), the same values on every rank.
// Returns sender q's H_N.
__device__ __forceinline__ uint32_t mg_fold_headers_warp(const MgArgs& M, DevState* st, uint32_t par) {
  const int q = (int)lane_id();
  uint32_t w[12];
#pragma unroll
  for (int i = 0; i < 12; i++) w[i] = (i == H_ERR) ? 0u : 0xFFFFFFFFu;
  if (q < M.world) {
    const uint4* hq = reinterpret_cast<const uint4*>(mg_area(M, M.rank, par, q));
    const uint4 v0 = ld_cg4(hq), v1 = ld_cg4(hq + 1), v2 = ld_cg4(hq + 2);
    w[0] = v0.x; w[1] = v0.y; w[2] = v0.z; w[3] = v0.w; w[4] = v1.x; w[5] = v1.y; w[6] = v1.z; w[7] = v1.w; w[8] = v2.x; w[9] = v2.y; w[10] = v2.z; w[11] = v2.w;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int i = H_ERR; i <= H_CAND_CAP; i++) {
      const uint32_t other = __shfl_xor_sync(0xFFFFFFFFu, w[i], o);
      w[i] = (i == H_ERR) ? (w[i] | other) : min(w[i], other);
    }
  }
  if (q == 0) {
    uint4* g = reinterpret_cast<uint4*>(st->g_vals);
    g[0] = make_uint4(w[H_ERR], w[H_POOL_FREE], w[H_SITES_CAP], w[H_NEW_CAP]);
    g[1] = make_uint4(w[H_HOT_CAP], w[H_LEN16_CAP], w[H_TBL_CAP], w[H_CAND_CAP]);
  }
  return w[H_N];
}

// Position tie-break on a sharded corpus (core.ts:294-305), shared by k_merge_loop and k_merge_rounds: from the candidates
// phase_collect listed (the same pairs on every rank) to the winner's table slot.  The last counted occurrence in GLOBAL scan
// order = (rank, local position) decides.  The candidates go in canonical (pair key) order so that every rank talks about the
// same one; each block takes one and stores its last counted LOCAL occurrence into every rank's tiebox; after the tie exchange
// the highest rank holding a candidate owns its last occurrence.  Every thread of the grid calls, after a grid barrier that
// follows phase_collect; `barrier` is the caller's grid barrier, s_max 32 words of shared scratch.  NOSLOT on a peer abort or
// when no rank holds a candidate.
template <class Bar>
__device__ __forceinline__ uint32_t mg_tie_winner(const LoopArgs& L, uint32_t* s_max, unsigned long long& tie_epoch, Bar barrier) {
  const MgArgs& M = L.mg;
  const ApplyArgs& A = L.A;
  DevState* st = A.st;
  const PairTable& t = A.t;
  const uint32_t bid = blockIdx.x, nblk = gridDim.x;
  const uint32_t gtid = bid * blockDim.x + threadIdx.x, gthreads = nblk * blockDim.x;
  const uint32_t tpar = (uint32_t)((tie_epoch + 1) & 1u);
  const uint32_t nc = ld_cg(&st->n_cand);  // == the winner's multiplicity, on every rank
  for (uint32_t i = gtid; i < nc; i += gthreads) {  // canonical order: by pair key
    const uint32_t si = ld_cg(&L.cands[i]);
    const uint32_t ki = t.keys[si];
    uint32_t r = 0;
    for (uint32_t j = 0; j < nc; j++) r += t.keys[ld_cg(&L.cands[j])] < ki;
    M.tie_sorted[r] = si;
  }
  barrier();
  for (uint32_t cnd = bid; cnd < nc; cnd += nblk) {  // one block per candidate: its last counted local occurrence
    const uint32_t s = ld_cg(&M.tie_sorted[cnd]);
    const uint32_t key = t.keys[s];
    const uint32_t a = key >> 16, b = key & 0xFFFFu;
    const unsigned long long start = t.occ_start.get(s);
    const uint32_t len = t.occ_len[s];
    uint32_t v = 0;
    for (uint32_t i = threadIdx.x; i < len; i += blockDim.x) {
      const uint32_t p = A.pool[start + i];
      if (counted_occurrence(A.slots, A.n, p, a, b)) v = max(v, p + 1);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xFFFFFFFFu, v, o));
    __syncthreads();
    if (lane_id() == 0) s_max[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t m = 0;
      for (uint32_t i = 0; i < (blockDim.x >> 5); i++) m = max(m, s_max[i]);
      for (int q = 0; q < M.world; q++) M.tiebox[q][((size_t)tpar * M.world + M.rank) * M.tie_cap + cnd] = m;
      __threadfence_system();
    }
  }
  barrier();
  if (bid == 0 && threadIdx.x == 0) {
    st->tie_pos = ~0ull;
    mg_signal_and_wait(M, M.flag_tie, tie_epoch + 1, st);
  }
  tie_epoch++;
  barrier();
  if (bid == 0) {
    const uint32_t* box = M.tiebox[M.rank] + (size_t)tpar * M.world * M.tie_cap;
    for (uint32_t i = threadIdx.x; i < nc; i += blockDim.x) {
      for (int q = M.world - 1; q >= 0; q--) {  // the highest rank holding the pair owns its last occurrence
        const uint32_t v = ld_cg(box + (size_t)q * M.tie_cap + i);
        if (v) {
          atomicMin(&st->tie_pos, ((((unsigned long long)q << 32) | (v - 1)) << 16) | i);
          break;
        }
      }
    }
  }
  barrier();
  const unsigned long long tp = ld_cg(&st->tie_pos);
  if (ld_cg(&st->mg_abort) || tp == ~0ull) return NOSLOT;
  return ld_cg(&M.tie_sorted[(uint32_t)(tp & 0xFFFFu)]);
}

// ---- exchange, executed by warp 0 of block 0: lane q talks to rank q, so its cost does not grow with the world size ----
__device__ __forceinline__ void mg_send_warp(const LoopArgs& L, uint32_t par, uint32_t n_rec, unsigned long long epoch,
                                             unsigned long long* const* flags) {
  const MgArgs& M = L.mg;
  const int q = (int)lane_id();
  if (q < M.world) {
    mg_store_header(L, mg_area(M, q, par, M.rank), n_rec, L.A.new_cap);
    __threadfence_system();
  }
  __syncwarp();
  if (q < M.world && q != M.rank) st_release_sys(flags[q] + 16 * M.rank, epoch);
}

// second half: wait for every peer's flag, then fold the G headers
__device__ __forceinline__ void mg_wait_fold_warp(const MgArgs& M, DevState* st, uint32_t par, unsigned long long epoch,
                                                  unsigned long long* const* flags) {
  const int q = (int)lane_id();
  if (q < M.world && q != M.rank) mg_wait_flag(flags[M.rank] + 16 * q, epoch, now_ns(), 16, 128, st);
  __syncwarp();
  mg_fold_headers_warp(M, st, par);
}

// ---- the one-merge kernel ----------------------------------------------------------------------------------------
// k_merge_loop (the scheme above LoopArgs, train_kernels.cuh) on one GPU and on every rank of a sharded corpus (MG = L.mg_on),
// where one merge is one exchange: the decision, the stop chain, the tie-break, the exit record and the merge log are the same code.
// What the two take the decision from is data: a sharded rank reads the capacities and error flags the last exchange folded
// (loop_caps_folded), which are one merge old, so the pool cells and hot-list entries of the previous merge count against them.
// One GPU pipelines the list filling (fill(t-1) next to P1(t)), splits the warps of small merges and stages the deltas of big
// ones; a sharded rank walks its sites with every thread and fills the lists in its own P2, next to the records' apply.
template <bool MG>  // (a template parameter, not a branch on L.mg_on: both paths keep the registers they need at 64 a thread)
__global__ void __launch_bounds__(ML_THREADS, ML_MIN_BLOCKS) k_merge_loop(LoopArgs L) {
  __shared__ Best s_best[ML_THREADS / 32];
  __shared__ uint32_t s_max[32];
  __shared__ __align__(8) uint32_t s_stage[LS_ROWS * R_STAGE_T];  // loop_flush_stage leaves it zero (phase_fill: u64 rows)
  __shared__ uint32_t s_rslot, s_wkey;
  for (uint32_t i = threadIdx.x; i < LS_ROWS * R_STAGE_T; i += blockDim.x) s_stage[i] = 0;
  const ApplyArgs& A = L.A;
  const MgArgs& M = L.mg;
  DevState* st = A.st;
  const PairTable& t = A.t;
  const uint32_t bid = blockIdx.x, nblk = gridDim.x;
  const uint32_t gt = bid * blockDim.x + threadIdx.x, gn = nblk * blockDim.x;
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
  const bool lead = (bid == 0 && threadIdx.x == 0);
  const bool replay = L.replay != nullptr;  // (one GPU only)
  const uint32_t n_tokens0 = ld_cg(&st->n_tokens);
  const uint32_t thresh = ld_cg(&st->hot_thresh);
  unsigned long long bar = 0;
  const auto barrier = [&] { grid_barrier(L.barrier, ++bar * nblk, L.bar_ns); };
  unsigned long long epoch = MG ? ld_cg(&st->mg_epoch) : 0ull, tie_epoch = MG ? ld_cg(&st->mg_tie_epoch) : 0ull;
  uint32_t wcnt_prev = 0;            // sharded: the previous merge's weight ...
  unsigned long long newk_prev = 0;  // ... and the hot-list entries its P3 may have appended (upper bound)

  if (lead) {
    st->snap_err = st->err;
    if (MG) {
      st->snap_n_keys = st->n_keys;
      st->snap_hot_n = st->hot_n;
      st->mg_abort = 0;
      st->n_newpair = 0;
    }
  }
  if (MG) {  // hello exchange: headers only (capacities, errors), so that the first decision is taken on global minima
    if (bid == 0 && threadIdx.x < 32) {
      mg_send_warp(L, (uint32_t)((epoch + 1) & 1u), 0, epoch + 1, M.flag_data);
      mg_wait_fold_warp(M, st, (uint32_t)((epoch + 1) & 1u), epoch + 1, M.flag_data);
    }
    epoch++;
  }
  if (!replay) {  // first arg-max partials
    Best v = best_block_reduce(argmax_stripe(t, A.len16, L.max_length, 1, L.hot, ld_cg(&st->hot_n), bid, nblk), s_best);
    if (threadIdx.x == 0) {
      L.partials[bid] = v;
      L.partial_keys[bid] = v.primary ? t.keys[v.slot] : 0u;
    }
  }
  barrier();

  // block 0's phase timers: one GPU's and a sharded rank's phases are listed at DevState::prof_ns and ::mg_prof_ns
  unsigned long long* const prof_ns = MG ? st->mg_prof_ns : st->prof_ns;
  unsigned long long tp0 = lead ? now_ns() : 0, tp1;
#define PROF(i)                      \
  if (lead) {                        \
    tp1 = now_ns();                  \
    prof_ns[i] += tp1 - tp0;         \
    tp0 = tp1;                       \
  }
  // deferred phase_fill (one GPU): the sites of the previous merge whose new adjacencies are not in their lists yet
  uint32_t fill_n = 0;
  const SiteRec* fill_sites = nullptr;
  for (uint32_t it = 0;; it++) {
    const uint32_t par = it & 1u;
    SiteRec* const my_sites = (par && !MG) ? L.sites2 : A.sites;
    // ---- every block (on every rank) folds the partials and takes the same decision ----
    // one GPU: n_keys, pool_cursor and hot_n only change in P2, err is snapshot by block 0 in P2: all stable here
    Best w{0ull, NOSLOT, 0};
    uint32_t wa = 0, wb = 0, wcnt = 0;
    const uint32_t c = n_tokens0 + it;
    const uint32_t hot_pre = ld_cg(&st->hot_n);  // entries before this merge's pairs join
    if (replay) {
      // the logged pair; it may not occur at all (a merge whose pair is absent still appends its token, core.ts:350-354)
      if (it < L.log_cap) {
        wa = (uint32_t)L.replay[2 * it];
        wb = (uint32_t)L.replay[2 * it + 1];
        __syncthreads();
        if (threadIdx.x == 0) s_rslot = tbl_find(t, pair_key(wa, wb));
        __syncthreads();
        w.slot = s_rslot;
        w.mult = 1;
        w.primary = 1;
        if (w.slot != NOSLOT) wcnt = max(t.cnt[w.slot], t.occ_len[w.slot]);  // bound on the sites (the list may hold stale entries)
      }
    } else {
      uint32_t my_key = 0;
      for (uint32_t i = threadIdx.x; i < nblk; i += blockDim.x) {
        Best pb;
        pb.primary = ld_cg(&L.partials[i].primary);
        pb.slot = ld_cg(&L.partials[i].slot);
        pb.mult = ld_cg(&L.partials[i].mult);
        const uint32_t pk = ld_cg(&L.partial_keys[i]);
        const uint32_t before = w.slot;
        w = best_merge(w, pb);
        if (w.slot != before) my_key = pk;
      }
      const Best mine_w = w;
      w = best_block_reduce(w, s_best);
      if (w.primary) {  // block-uniform: the thread that holds the winning partial hands out its key
        if (mine_w.primary == w.primary && mine_w.slot == w.slot) s_wkey = my_key;
        __syncthreads();
        const uint32_t key = s_wkey;
        wa = key >> 16;
        wb = key & 0xFFFFu;
        wcnt = (uint32_t)(w.primary >> 20);
      }
    }
    const LoopCaps g = MG ? loop_caps_folded(st) : loop_caps(L, ld_cg(&st->pool_cursor));
    uint32_t status, cap = LOOP_RUNNING;
    if (!replay) status = loop_stop(L, MG ? (ld_cg(&st->mg_abort) || g.err) : ld_cg(&st->snap_err) != 0, w.primary, wcnt, thresh, it, c);
    else if (ld_cg(&st->snap_err)) status = LOOP_ERROR;
    else status = (it >= L.log_cap) ? LOOP_LIMIT : (c >= L.max_tokens ? LOOP_NEED_HOST : LOOP_RUNNING);
    if (status == LOOP_RUNNING) {
      // sharded, against figures one merge old: the pool cells and hot-list entries the previous merge may have taken count
      // against them (2 wcnt >= 2 min_weight > 0, so this is 2 wcnt tested against the cells left after the previous merge,
      // saturated at 0).  One GPU tests against its live figures.  (Replayed merges do not feed the hot list.)
      const unsigned long long new_keys = min(2ull * wcnt + 2ull, 2ull * (c + 1ull) + 2ull);
      cap = loop_cap_status(g, MG ? ld_cg(&st->snap_n_keys) : ld_cg(&st->n_keys), new_keys, 2ull * wcnt + 2ull * wcnt_prev, wcnt,
                            replay ? 0ull : (MG ? ld_cg(&st->snap_hot_n) + newk_prev : hot_pre) + new_keys, c);
      if (MG) status = cap;  // (a sharded rank stops before the tie exchange, one GPU after its tie-break)
    }
    PROF(0)
    if (status == LOOP_RUNNING && w.mult > 1) {
      // tie on (weight, a.index+b.index): the pair whose last counted occurrence comes first wins (core.ts:294-305); on a
      // sharded corpus in GLOBAL scan order
      if (w.mult > g.cand_cap) status = LOOP_NEED_HOST;
      else {
        if (fill_n) {  // the tie-break reads occurrence lists: those of the last merge must be complete
          phase_fill(A, fill_n, gt, gn, fill_sites, fill_n > L.stage_min ? s_stage : nullptr);
          fill_n = 0;
          barrier();
        }
        phase_collect(t, A.len16, L.max_length, 1, L.hot, hot_pre, w.primary, L.cands, L.cand_cap, st, bid, nblk);
        barrier();
        uint32_t s;
        if (MG) {
          s = mg_tie_winner(L, s_max, tie_epoch, barrier);
        } else {
          phase_tie(A.slots, A.n, t, A.pool, L.cands, ld_cg(&st->n_cand), st, s_max, bid, nblk);
          barrier();
          const unsigned long long tp = ld_cg(&st->tie_pos);
          s = (tp == ~0ull) ? NOSLOT : (uint32_t)(tp & 0xFFFFFFFFu);
        }
        if (s == NOSLOT) status = LOOP_ERROR;
        else {
          const uint32_t key = t.keys[s];
          w.slot = s;
          wa = key >> 16;
          wb = key & 0xFFFFu;
        }
      }
    }
    PROF(MG ? 11 : 7)
    if (status == LOOP_RUNNING) status = cap;
    if (status != LOOP_RUNNING) {
      if (fill_n) phase_fill(A, fill_n, gt, gn, fill_sites, fill_n > L.stage_min ? s_stage : nullptr);  // the kernel leaves every list complete
      if (lead) {
        loop_exit(t, st, status, it, c, replay ? nullptr : &w, MG, epoch, tie_epoch);
        if (replay) {
          st->best_primary = 0;
          st->best_cnt = wcnt;  // what the host must make room for
          st->best_mult = 1;
        }
      }
      return;
    }
    if (fill_n && it && (wa == c - 1u || wb == c - 1u)) {
      // the winner was born by the previous merge: its list is exactly what fill(t-1) still has to write
      phase_fill(A, fill_n, gt, gn, fill_sites, fill_n > L.stage_min ? s_stage : nullptr);
      fill_n = 0;
      barrier();
    }
    // ---- P1: sites + deltas (one GPU: next to the list filling of the previous merge) ----
    if (lead) {
      A.len16[c] = A.len16[wa] + A.len16[wb];  // chars = a.chars + b.chars (:318)
      MergeRec r;
      r.a = (int32_t)wa;
      r.b = (int32_t)wb;
      r.c = (int32_t)c;
      r.reserved = 0;
      r.weight = (long long)wcnt;
      L.log[it] = r;
      st->n_sites[par ^ 1u] = 0;
      st->n_new[par ^ 1u] = 0;
      if (MG) {
        st->n_touched[par ^ 1u] = 0;
        st->n_newpair = 0;  // consumed by the previous merge's P3
      }
      if (w.mult > 1) st->tie_breaks++;
    }
    if (MG) {
      phase_sites(A, wa, wb, c, par, w.slot, gt, gn);  // local sites, staged count deltas
    } else if (fill_n <= 8192u && wcnt <= 16384u && blockDim.x == 512u) {
      // latency bound: 12 warps of every block walk the sites, 4 fill the lists of the last merge and then warm the L2
      // for the next one
      const uint32_t ws = L.p1_sites, wh = 16u - ws;
      if (warp < ws) {
        phase_sites(A, wa, wb, c, par, w.slot, (bid * ws + warp) * 32 + lane, nblk * ws * 32, my_sites);
      } else {
        if (fill_n) phase_fill(A, fill_n, (bid * wh + warp - ws) * 32 + lane, nblk * wh * 32, fill_sites);
        if (L.prefetch && !replay) prefetch_runner_up(L, w.slot, nblk, (bid * wh + warp - ws) * 32 + lane, nblk * wh * 32);
      }
    } else {
      // (the list length is block-uniform: nothing writes occ_len between P2's barrier and the next P2)
      const bool staged = w.slot != NOSLOT && t.occ_len[w.slot] > L.stage_min;
      if (fill_n) phase_fill(A, fill_n, gt, gn, fill_sites, fill_n > L.stage_min ? s_stage : nullptr);
      phase_sites(A, wa, wb, c, par, w.slot, gt, gn, my_sites, staged ? s_stage : nullptr);
      if (staged) loop_flush_stage(A, s_stage, wa, wb);
    }
    fill_n = 0;
#ifdef BPE_FINE_PROF
    const int bkt = 31 - __clz(wcnt | 1u);
    if (lead && !MG) {
      st->bucket_ns[bkt][0] += now_ns() - tp0;
      st->bucket_ns[bkt][3] += 1;
    }
#endif
    PROF(1)
    barrier();
    PROF(2)
    if (MG) {
      const uint32_t epar = (uint32_t)((epoch + 1) & 1u);
      // ---- M1: the counts of the pairs born by this merge (dense rows, one record per pair) and one (pair, delta) record per
      // touched pair -- stored into every rank's inbox ----
      {
        const uint32_t per_side = c + 1u, total2 = 2u * per_side;
        for (uint32_t i = gt; i < ((total2 + 31u) & ~31u); i += gn) {
          uint32_t cntv = 0, key = 0;
          if (i < total2) {
            uint32_t side = i >= per_side ? 1u : 0u, tok = i - side * per_side;
            cntv = ld_cg(A.nd + (size_t)(side ? ND_R_CNT : ND_L_CNT) * ND_STRIDE + tok);
            key = side ? pair_key(c, tok) : pair_key(tok, c);
          }
          uint32_t m = __ballot_sync(0xFFFFFFFFu, cntv != 0);
          if (!m) continue;
          uint32_t base = 0;
          int src = __ffs(m) - 1;
          if ((int)lane == src) base = atomicAdd(&st->n_out, (uint32_t)__popc(m));
          base = __shfl_sync(0xFFFFFFFFu, base, src);
          if (cntv) {
            uint32_t k = base + __popc(m & ((1u << lane) - 1u));
            if (MG_HDR + k >= M.inbox_stride) {
              atomicOr(&st->err, ERR_INBOX_OVERFLOW);
            } else {
              unsigned long long rec = ((unsigned long long)key << 32) | cntv;
              for (int q = 0; q < M.world; q++) mg_area(M, q, epar, M.rank)[MG_HDR + k] = rec;
            }
          }
        }
      }
      {
        const uint32_t nt = min(ld_cg(&st->n_touched[par]), A.touched_cap);
        for (uint32_t i = gt; i < nt; i += gn) {
          uint32_t s = ld_cg(&A.touched[i]);
          int32_t d = atomicExch(A.dlt + s, 0);
          if (d == 0) continue;
          uint32_t k = atomicAdd(&st->n_out, 1u);
          if (MG_HDR + k >= M.inbox_stride) {
            atomicOr(&st->err, ERR_INBOX_OVERFLOW);
            continue;
          }
          unsigned long long rec = ((unsigned long long)t.keys[s] << 32) | (uint32_t)d;
          for (int q = 0; q < M.world; q++) mg_area(M, q, epar, M.rank)[MG_HDR + k] = rec;
        }
      }
      __threadfence_system();
      PROF(3)
      barrier();
      PROF(4)
      // ---- send, then do the LOCAL half of P2 while the peers' messages travel: the pairs born on this shard enter the table
      // (their counts come with the records), the shard is rewritten.  The wait for the peers sits behind that work. ----
      if (bid == 0 && threadIdx.x < 32) mg_send_warp(L, epar, min(ld_cg(&st->n_out), M.inbox_stride - MG_HDR), epoch + 1, M.flag_data);
      const uint32_t n_sites_now = ld_cg(&st->n_sites[par]);
      phase_new_pairs(A, c, A.len16, L.max_length, 0, L.hot, L.hot_cap, L.pool_cap, true, gt, gn);
      phase_rewrite(A, c, n_sites_now, gt, gn);
      PROF(5)
      barrier();
      if (bid == 0 && threadIdx.x < 32) mg_wait_fold_warp(M, st, epar, epoch + 1, M.flag_data);
      if (lead) {
        st->n_out = 0;  // nobody appends before the next merge's P1
        st->n_cand = 0;
        st->tie_pos = ~0ull;
        t.cnt[w.slot] = 0;  // every counted occurrence of the winner, on every rank, is being replaced
        st->snap_hot_n = st->hot_n;  // stable: the appends of the previous merge are complete, the next ones come in P3
      }
      epoch++;
      PROF(6)
      barrier();
      if (ld_cg(&st->mg_abort)) {
        // the local shard was already rewritten for this merge; the engine is unusable after an abort
        if (lead) loop_exit(t, st, LOOP_ERROR, it + 1, c + 1, nullptr, true, epoch, tie_epoch);
        return;
      }
      // ---- P2 (second half): apply the deltas of all ranks to the replicated counts; the lists of the pairs born on this
      // shard are filled next to it (independent work: positions only) ----
      phase_fill(A, n_sites_now, gt, gn);
      {
        // all G record lists as ONE index space, so a thread walks a single record's chain whatever the world size
        uint32_t pre[MG_MAX_WORLD + 1];
        pre[0] = 0;
#pragma unroll
        for (int q = 0; q < MG_MAX_WORLD; q++)
          pre[q + 1] = pre[q] + (q < M.world ? ld_cg(reinterpret_cast<const uint32_t*>(mg_area(M, M.rank, epar, q)) + H_N) : 0u);
        const uint32_t total = pre[MG_MAX_WORLD];
        for (uint32_t j = gt; j < ((total + 31u) & ~31u); j += gn) {  // warp-uniform
          bool ins = false, born = false;
          uint32_t s = NOSLOT;
          if (j < total) {
            int q = 0;
#pragma unroll
            for (int r = 1; r < MG_MAX_WORLD; r++) q += (j >= pre[r]) ? 1 : 0;
            unsigned long long rec = ld_cg(mg_area(M, M.rank, epar, q) + MG_HDR + (j - pre[q]));
            uint32_t key = (uint32_t)(rec >> 32);
            s = tbl_find_or_insert_ex(t, key, &ins);
            if (s == NOSLOT) {
              atomicOr(&st->err, ERR_TABLE_FULL);
            } else {
              atomicAdd(t.cnt + s, (uint32_t)rec);
              born = ins;  // a pair born on another shard only: whoever inserts the key lists it for the hot-list test of P3
            }
          }
          uint32_t im = __ballot_sync(0xFFFFFFFFu, ins);
          if (im && lane == (uint32_t)(__ffs(im) - 1)) atomicAdd(&st->n_keys, (uint32_t)__popc(im));
          uint32_t bm = __ballot_sync(0xFFFFFFFFu, born);
          if (bm) {
            uint32_t base = 0;
            int src = __ffs(bm) - 1;
            if ((int)lane == src) base = atomicAdd(&st->n_newpair, (uint32_t)__popc(bm));
            base = __shfl_sync(0xFFFFFFFFu, base, src);
            if (born) {
              uint32_t k = base + __popc(bm & ((1u << lane) - 1u));
              if (k < A.newpair_cap) A.newpair[k] = s;
              else atomicOr(&st->err, ERR_HOT_OVERFLOW);
            }
          }
        }
      }
      PROF(7)
      barrier();
      PROF(8)
      // ---- P3: pairs born in this merge join the hot list; next arg-max partials ----
      if (lead) {
        st->snap_n_keys = st->n_keys;
        st->snap_pool_cursor = st->pool_cursor;
        st->snap_err = st->err;
      }
      const uint32_t hot_n0 = ld_cg(&st->snap_hot_n);
      Best mine{0ull, NOSLOT, 0};
      {
        const uint32_t nnp = min(ld_cg(&st->n_newpair), A.newpair_cap);
        for (uint32_t i = gt; i < nnp; i += gn) {
          uint32_t s = ld_cg(&A.newpair[i]);
          unsigned long long pr = slot_primary(t, A.len16, s, L.max_length);
          if (pr && (uint32_t)(pr >> 20) >= thresh) {
            uint32_t k = atomicAdd(&st->hot_n, 1u);
            if (k < L.hot_cap) L.hot[k] = s;
            else atomicOr(&st->err, ERR_HOT_OVERFLOW);
            mine = best_merge(mine, Best{pr, s, 1});
          }
        }
      }
      {
        Best stripe = argmax_stripe(t, A.len16, L.max_length, 1, L.hot, hot_n0, bid, nblk);
        Best v = best_block_reduce(best_merge(mine, stripe), s_best);
        if (threadIdx.x == 0) {
          L.partials[bid] = v;
          L.partial_keys[bid] = v.primary ? t.keys[v.slot] : 0u;
        }
      }
      PROF(9)
      barrier();
      PROF(10)
      wcnt_prev = wcnt;
      newk_prev = min(2ull * wcnt + 2ull, 2ull * (c + 1ull) + 2ull);
      continue;
    }
    // ---- P2: the born pairs (table, list space, hot list, arg-max), the corpus rewrite, the arg-max over the old hot pairs ----
    if (lead) {
      st->n_cand = 0;
      st->tie_pos = ~0ull;
      st->snap_err = st->err;  // what every block will act on at the next decision (errors of this phase: one merge later)
      if (w.slot != NOSLOT) t.cnt[w.slot] = 0;  // every counted occurrence of the winner is being replaced (no delta of P1
                                                // touches the winner's own pair); the arg-max below skips the slot
      if (replay) L.log[it].weight = (long long)st->n_sites[par];  // replacements performed (bpe_apply_merge's n_replaced)
    }
    const uint32_t n_sites_now = ld_cg(&st->n_sites[par]);
    Best mine{0ull, NOSLOT, 0};
    uint32_t mine_key = 0;
    {
      // Three independent jobs.  Small merges are latency bound, so the warps of every block split up (p2_new / p2_rw / rest) and the
      // three dependency chains run side by side; big merges keep every thread on every job.
      const bool split = n_sites_now <= 16384u && blockDim.x == 512u;
      const uint32_t wn = L.p2_new, wr = L.p2_rw, wm = 16u - wn - wr;
      if (!split || warp < wn)
        phase_new_pairs(A, c, A.len16, L.max_length, replay ? 0 : 1, L.hot, L.hot_cap, L.pool_cap, false,
                        split ? (bid * wn + warp) * 32 + lane : gt, split ? nblk * wn * 32 : gn, &mine, &mine_key);
      if (!split || (warp >= wn && warp < wn + wr))
        phase_rewrite(A, c, n_sites_now, split ? (bid * wr + warp - wn) * 32 + lane : gt, split ? nblk * wr * 32 : gn, my_sites);
      if (!replay && (!split || warp >= wn + wr)) {
        for (uint32_t i = split ? (bid * wm + warp - wn - wr) * 32 + lane : gt; i < hot_pre; i += split ? nblk * wm * 32 : gn) {
          uint32_t hs = L.hot[i], hk;
          if (hs == w.slot) continue;  // the winner's count is being zeroed
          unsigned long long pr = slot_primary_k(t, A.len16, hs, L.max_length, &hk);
          if (pr) {
            const uint32_t before = mine.slot;
            mine = best_merge(mine, Best{pr, hs, 1});
            if (mine.slot != before) mine_key = hk;
          }
        }
      }
    }
    if (!replay) {
      Best v = best_block_reduce(mine, s_best);
      if (threadIdx.x == 0) L.partials[bid] = v;
      if (mine.primary == v.primary && mine.slot == v.slot) L.partial_keys[bid] = mine_key;  // the owner of the block's best
    }
    fill_n = n_sites_now;
    fill_sites = my_sites;
#ifdef BPE_FINE_PROF
    if (lead) st->bucket_ns[bkt][1] += now_ns() - tp0;
#endif
    PROF(3)
    barrier();
    PROF(4)
  }
#undef PROF
}

}  // namespace bpe
