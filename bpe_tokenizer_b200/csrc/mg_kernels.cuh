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
// exchange; k_merge_loop_mg below runs one merge per exchange: those above R_HUGE global sites, or all of them under
// BPE_LOOP_ROUNDS=0.  Their record formats differ; the steps every rank must run identically live here once, for both: the
// header of a message (mg_store_header) and its fold (mg_fold_headers_warp), the wait on a peer's flag (mg_wait_flag) and the
// tie-break.  Every decision that ends or interrupts the loop is taken from replicated values (or minima over ranks carried in
// the message headers), so all ranks leave the kernel at the same merge with the same status.  Waits on peers are bounded
// (MG_TIMEOUT_NS) and abort the loop.
#pragma once
#include "train_kernels.cuh"

namespace bpe {

constexpr int MG_MAX_WORLD = 8;
constexpr uint32_t MG_HDR = 16;  // u64 words of header in front of the records of one message
enum { H_N = 0, H_ERR, H_POOL_FREE, H_SITES_CAP, H_NEW_CAP, H_HOT_CAP, H_LEN16_CAP, H_TBL_CAP, H_CAND_CAP, H_STATUS };
constexpr unsigned long long MG_TIMEOUT_NS = 8000000000ull;
constexpr uint32_t MG_DIRECT_MAX = 8192;  // merges with at most this many (global) occurrences push their deltas unstaged

struct MgArgs {
  int rank, world;
  uint32_t inbox_stride;  // u64 words per (parity, sender) message area, header included
  uint32_t tie_cap;       // candidates per tie message
  // mailboxes, indexed by rank; [rank] is this GPU's own (peers store into it), the others are peer-mapped
  unsigned long long* flag_data[MG_MAX_WORLD];  // [world] one 128-byte line per sender
  unsigned long long* flag_tie[MG_MAX_WORLD];
  unsigned long long* inbox[MG_MAX_WORLD];      // [2][world][inbox_stride]
  uint32_t* tiebox[MG_MAX_WORLD];               // [2][world][tie_cap]
  // local scratch
  uint32_t* tie_sorted;    // candidates (table slots) in canonical key order
  uint32_t* newpair;       // table slots of the pairs born in the current merge (any rank), deduplicated
  uint32_t newpair_cap;
};

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

struct LoopArgsMg {
  LoopArgs L;
  MgArgs M;
};

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
// record count, error flags and capacities (H_N .. H_CAND_CAP) into the header at `dst`; the pool figure only gates the next
// decision.
__device__ __forceinline__ void mg_store_header(const LoopArgs& L, const MgArgs& M, unsigned long long* dst, uint32_t n_rec, uint32_t new_cap) {
  DevState* st = L.A.st;
  const unsigned long long cur = ld_cg(&st->pool_cursor);
  uint32_t h[12];
#pragma unroll
  for (int i = 0; i < 12; i++) h[i] = 0;
  h[H_N] = n_rec;
  h[H_ERR] = ld_cg(&st->err);
  h[H_POOL_FREE] = (uint32_t)min(L.pool_cap > cur ? L.pool_cap - cur : 0ull, 0xFFFFFFFFull);
  h[H_SITES_CAP] = L.A.sites_cap;
  h[H_NEW_CAP] = new_cap;
  h[H_HOT_CAP] = min(L.hot_cap, L.hot_limit);
  h[H_LEN16_CAP] = L.len16_cap;
  h[H_TBL_CAP] = L.tbl_cap;
  h[H_CAND_CAP] = min(L.cand_cap, M.tie_cap);
  uint4* d4 = reinterpret_cast<uint4*>(dst);
#pragma unroll
  for (int i = 0; i < 3; i++) d4[i] = make_uint4(h[4 * i], h[4 * i + 1], h[4 * i + 2], h[4 * i + 3]);
}

// One warp, lane q reads sender q's header in this rank's area `par` (the messages are complete): the G headers fold into
// st->g_vals (OR of the error flags, minima of the capacities), the same values on every rank.  Returns sender q's H_N.
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

// Position tie-break on a sharded corpus (core.ts:294-305), shared by k_merge_loop_mg and k_merge_rounds: from the candidates
// phase_collect listed (the same pairs on every rank) to the winner's table slot.  The last counted occurrence in GLOBAL scan
// order = (rank, local position) decides.  The candidates go in canonical (pair key) order so that every rank talks about the
// same one; each block takes one and stores its last counted LOCAL occurrence into every rank's tiebox; after the tie exchange
// the highest rank holding a candidate owns its last occurrence.  Every thread of the grid calls, after a grid barrier that
// follows phase_collect; `barrier` is the caller's grid barrier, s_max 32 words of shared scratch.  NOSLOT on a peer abort or
// when no rank holds a candidate.
template <class Bar>
__device__ __forceinline__ uint32_t mg_tie_winner(const LoopArgs& L, const MgArgs& M, uint32_t* s_max, unsigned long long& tie_epoch,
                                                  Bar barrier) {
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
__device__ __forceinline__ void mg_send_warp(const LoopArgsMg& P, uint32_t par, uint32_t n_rec, unsigned long long epoch,
                                             unsigned long long* const* flags) {
  const MgArgs& M = P.M;
  const int q = (int)lane_id();
  if (q < M.world) {
    mg_store_header(P.L, M, mg_area(M, q, par, M.rank), n_rec, P.L.A.new_cap);
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

__global__ void __launch_bounds__(ML_THREADS, ML_MIN_BLOCKS) k_merge_loop_mg(LoopArgsMg P) {
  __shared__ Best s_best[ML_THREADS / 32];
  __shared__ uint32_t s_max[32];
  const LoopArgs& L = P.L;
  const MgArgs& M = P.M;
  const ApplyArgs& A = L.A;
  DevState* st = A.st;
  const PairTable& t = A.t;
  const uint32_t bid = blockIdx.x, nblk = gridDim.x;
  const uint32_t gtid = bid * blockDim.x + threadIdx.x, gthreads = nblk * blockDim.x;
  const bool lead = (bid == 0 && threadIdx.x == 0);
  unsigned long long bar = 0;
  const uint32_t n_tokens0 = ld_cg(&st->n_tokens);
  const uint32_t thresh = ld_cg(&st->hot_thresh);
  unsigned long long epoch = ld_cg(&st->mg_epoch);
  unsigned long long tie_epoch = ld_cg(&st->mg_tie_epoch);
#define GRID_BARRIER() grid_barrier(L.barrier, ++bar * nblk)

  // ---- hello exchange: headers only (capacities, errors), so that the first decision is taken on global minima ----
  if (lead) {
    st->snap_n_keys = st->n_keys;
    st->snap_hot_n = st->hot_n;
    st->mg_abort = 0;
    st->n_newpair = 0;
  }
  if (bid == 0 && threadIdx.x < 32) {
    mg_send_warp(P, (uint32_t)((epoch + 1) & 1u), 0, epoch + 1, M.flag_data);
    mg_wait_fold_warp(M, st, (uint32_t)((epoch + 1) & 1u), epoch + 1, M.flag_data);
  }
  epoch++;
  {
    Best v = best_block_reduce(argmax_stripe(t, A.len16, L.max_length, 1, L.hot, ld_cg(&st->hot_n), bid, nblk), s_best);
    if (threadIdx.x == 0) L.partials[bid] = v;
  }
  GRID_BARRIER();
  uint32_t wcnt_prev = 0;
  unsigned long long tp0 = lead ? now_ns() : 0, tp1;
#define MGPROF(i)                    \
  if (lead) {                        \
    tp1 = now_ns();                  \
    st->mg_prof_ns[i] += tp1 - tp0;  \
    tp0 = tp1;                       \
  }
  unsigned long long newk_prev = 0;  // upper bound of the hot-list entries appended by the previous merge's P3

  for (uint32_t it = 0;; it++) {
    const uint32_t par = it & 1u;
    // ---- every block (on every rank) folds the partials and takes the same decision ----
    Best w{0ull, NOSLOT, 0};
    for (uint32_t i = threadIdx.x; i < nblk; i += blockDim.x) {
      Best pb;
      pb.primary = ld_cg(&L.partials[i].primary);
      pb.slot = ld_cg(&L.partials[i].slot);
      pb.mult = ld_cg(&L.partials[i].mult);
      w = best_merge(w, pb);
    }
    w = best_block_reduce(w, s_best);
    uint32_t status = LOOP_RUNNING;
    uint32_t wa = 0, wb = 0, wcnt = 0;
    if (w.primary) {
      uint32_t key = t.keys[w.slot];
      wa = key >> 16;
      wb = key & 0xFFFFu;
      wcnt = (uint32_t)(w.primary >> 20);
    }
    const uint32_t c = n_tokens0 + it;
    const uint4 g0 = ld_cg4(reinterpret_cast<const uint4*>(st->g_vals)), g1 = ld_cg4(reinterpret_cast<const uint4*>(st->g_vals) + 1);
    const uint32_t g_err = g0.x, g_pool_free = g0.y, g_sites_cap = g0.z, g_new_cap = g0.w, g_hot_cap = g1.x, g_len16_cap = g1.y,
                   g_tbl_cap = g1.z, g_cand_cap = g1.w;
    const uint32_t snap_n_keys = ld_cg(&st->snap_n_keys), snap_hot_n = ld_cg(&st->snap_hot_n), aborted = ld_cg(&st->mg_abort);
    if (aborted || g_err) status = LOOP_ERROR;
    else if (!w.primary) status = (thresh <= 1) ? LOOP_EMPTY : LOOP_NEED_REBUILD;
    else if (wcnt < thresh) status = LOOP_NEED_REBUILD;
    else if (wcnt < L.min_weight) status = LOOP_DONE;  // core.ts:313
    else if (it >= L.log_cap) status = LOOP_LIMIT;
    else if (c >= L.max_tokens) status = LOOP_NEED_HOST;
    if (status == LOOP_RUNNING) {
      unsigned long long new_keys = min(2ull * wcnt + 2ull, 2ull * (c + 1ull) + 2ull);
      unsigned long long pool_free = g_pool_free;
      pool_free = pool_free > 2ull * wcnt_prev ? pool_free - 2ull * wcnt_prev : 0;  // headers are one merge old
      if ((unsigned long long)snap_n_keys + new_keys > (unsigned long long)(g_tbl_cap >> 1)) status = LOOP_NEED_HOST;
      else if (2ull * wcnt > pool_free) status = LOOP_NEED_HOST;
      else if (wcnt > g_sites_cap || new_keys > g_new_cap) status = LOOP_NEED_HOST;
      else if ((unsigned long long)snap_hot_n + newk_prev + new_keys > g_hot_cap) status = LOOP_NEED_REBUILD;
      else if (c + 1 > g_len16_cap) status = LOOP_NEED_HOST;
      else if (w.mult > 1 && w.mult > g_cand_cap) status = LOOP_NEED_HOST;
    }
    MGPROF(0)
    if (status == LOOP_RUNNING && w.mult > 1) {
      // ---- tie on (weight, a.index+b.index): last counted occurrence in GLOBAL scan order decides (core.ts:294-305) ----
      phase_collect(t, A.len16, L.max_length, 1, L.hot, ld_cg(&st->hot_n), w.primary, L.cands, L.cand_cap, st, bid, nblk);
      GRID_BARRIER();
      const uint32_t s = mg_tie_winner(L, M, s_max, tie_epoch, [&] { GRID_BARRIER(); });
      if (s == NOSLOT) status = LOOP_ERROR;
      else {
        const uint32_t key = t.keys[s];
        w.slot = s;
        wa = key >> 16;
        wb = key & 0xFFFFu;
      }
    }
    MGPROF(11)
    if (status != LOOP_RUNNING) {
      if (lead) {
        st->status = status;
        st->iters_done = it;
        st->n_tokens = n_tokens0 + it;
        publish_best(t, st, w);
        st->n_cand = 0;
        st->tie_pos = ~0ull;
        st->mg_epoch = epoch;
        st->mg_tie_epoch = tie_epoch;
      }
      return;
    }
    // ---- P1: local sites, staged count deltas ----
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
      st->n_touched[par ^ 1u] = 0;
      st->n_newpair = 0;  // consumed by the previous merge's P3
      if (w.mult > 1) st->tie_breaks++;
    }
    const uint32_t epar = (uint32_t)((epoch + 1) & 1u);
    // small merges: every warp-aggregated delta goes straight into all inboxes (no staging pass, one barrier less);
    // big merges stage per pair first (a handful of pairs get millions of deltas)
    const bool direct = wcnt <= MG_DIRECT_MAX;
    {
      ApplyArgs Ad = A;
      if (direct) {
        for (int q = 0; q < M.world; q++) Ad.push[q] = mg_area(M, q, epar, M.rank) + MG_HDR;
        Ad.push_world = M.world;
        Ad.push_cap = M.inbox_stride - MG_HDR;
      }
      phase_sites(Ad, wa, wb, c, par, w.slot, bid * blockDim.x + threadIdx.x, nblk * blockDim.x);
      if (direct) __threadfence_system();
    }
    MGPROF(1)
    GRID_BARRIER();
    MGPROF(2)
    // ---- M1 (staged mode; small merges pushed everything during P1): the counts of the pairs born by this merge (dense
    // rows, one record per pair) and one (pair, delta) record per touched pair -- stored into every rank's inbox ----
    if (!direct) {
      const uint32_t lane = lane_id();
      const uint32_t per_side = c + 1u, total2 = 2u * per_side;
      for (uint32_t i = gtid; i < ((total2 + 31u) & ~31u); i += gthreads) {
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
    if (!direct) {
      const uint32_t nt = min(ld_cg(&st->n_touched[par]), A.touched_cap);
      for (uint32_t i = gtid; i < nt; i += gthreads) {
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
    if (!direct) {
      __threadfence_system();
      MGPROF(3)
      GRID_BARRIER();
      MGPROF(4)
    }
    // ---- send, then do the LOCAL half of P2 while the peers' messages travel: the pairs born on this shard enter the table
    // (their counts come with the records), the shard is rewritten.  The wait for the peers sits behind that work. ----
    if (bid == 0 && threadIdx.x < 32) mg_send_warp(P, epar, min(ld_cg(&st->n_out), M.inbox_stride - MG_HDR), epoch + 1, M.flag_data);
    const uint32_t n_sites_now = ld_cg(&st->n_sites[par]);
    phase_new_pairs(A, c, A.len16, L.max_length, 0, L.hot, L.hot_cap, L.pool_cap, true, gtid, gthreads);
    phase_rewrite(A, c, n_sites_now, gtid, gthreads);
    MGPROF(5)
    GRID_BARRIER();
    if (bid == 0 && threadIdx.x < 32) mg_wait_fold_warp(M, st, epar, epoch + 1, M.flag_data);
    if (lead) {
      st->n_out = 0;  // nobody appends before the next merge's P1
      st->n_cand = 0;
      st->tie_pos = ~0ull;
      t.cnt[w.slot] = 0;  // every counted occurrence of the winner, on every rank, is being replaced
      st->snap_hot_n = st->hot_n;  // stable: the appends of the previous merge are complete, the next ones come in P3
    }
    epoch++;
    MGPROF(6)
    GRID_BARRIER();
    if (ld_cg(&st->mg_abort)) {
      if (lead) {
        st->status = LOOP_ERROR;
        st->iters_done = it + 1;  // the local shard was already rewritten for this merge; the engine is unusable after an abort
        st->n_tokens = n_tokens0 + it + 1;
        st->mg_epoch = epoch;
        st->mg_tie_epoch = tie_epoch;
      }
      return;
    }
    // ---- P2 (second half): apply the deltas of all ranks to the replicated counts; the lists of the pairs born on this
    // shard are filled next to it (independent work: positions only) ----
    phase_fill(A, n_sites_now, bid * blockDim.x + threadIdx.x, nblk * blockDim.x);
    {
      // all G record lists as ONE index space, so a thread walks a single record's chain whatever the world size
      uint32_t pre[MG_MAX_WORLD + 1];
      pre[0] = 0;
#pragma unroll
      for (int q = 0; q < MG_MAX_WORLD; q++)
        pre[q + 1] = pre[q] + (q < M.world ? ld_cg(reinterpret_cast<const uint32_t*>(mg_area(M, M.rank, epar, q)) + H_N) : 0u);
      const uint32_t total = pre[MG_MAX_WORLD];
      const uint32_t lane = lane_id();
      for (uint32_t j = gtid; j < ((total + 31u) & ~31u); j += gthreads) {  // warp-uniform
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
            if (k < M.newpair_cap) M.newpair[k] = s;
            else atomicOr(&st->err, ERR_HOT_OVERFLOW);
          }
        }
      }
    }
    MGPROF(7)
    GRID_BARRIER();
    MGPROF(8)
    // ---- P3: rewrite the local shard; pairs born in this merge join the hot list; next arg-max partials ----
    if (lead) {
      st->snap_n_keys = st->n_keys;
      st->snap_pool_cursor = st->pool_cursor;
      st->snap_err = st->err;
    }
    const uint32_t hot_n0 = ld_cg(&st->snap_hot_n);
    Best mine{0ull, NOSLOT, 0};
    {
      const uint32_t nnp = min(ld_cg(&st->n_newpair), M.newpair_cap);
      for (uint32_t i = gtid; i < nnp; i += gthreads) {
        uint32_t s = ld_cg(&M.newpair[i]);
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
      if (threadIdx.x == 0) L.partials[bid] = v;
    }
    MGPROF(9)
    GRID_BARRIER();
    MGPROF(10)
    wcnt_prev = wcnt;
    newk_prev = min(2ull * wcnt + 2ull, 2ull * (c + 1ull) + 2ull);
  }
#undef GRID_BARRIER
#undef MGPROF
}

}  // namespace bpe
