// train_kernels.cuh -- K1 (pair histogram + occurrence lists), K2 (arg-max with the reference's exact
// tie-break) and K3 (apply merge in place with count deltas) for sm_100a, plus the persistent
// cooperative kernel that runs the whole mergeUntil loop on the device.
//
// Reference semantics restated (SURVEY.md Appendix A; all citations are /root/reference/core.ts):
//   counting  :265-310  every adjacent pair inside a document; for a == b only every other pair of a
//                       run is counted (:285-290), i.e. count(X,X) = sum over runs floor(len/2)
//   arg-max   :294-305  running max => winner = max weight, then min a.index+b.index, then the pair
//                       whose LAST counted occurrence comes first in scan order
//   filter    :270-273  utf16len(a)+utf16len(b) <= max_length when max_length is truthy
//   apply     :356-359  replaceAll: left to right, non-overlapping
//
// Key structural fact used by the occurrence lists: all instances of a token index are created by the
// one merge that created the index, so every adjacency (p,q) is born in iteration max(birth p, birth q)
// -- each pair's occurrence list is written exactly once (contiguous in `pool`) and afterwards only
// goes stale, which is detected by re-reading the corpus.
//
// Every phase is a __device__ function over (block id, block count) so that the same code runs as a
// stand-alone kernel (findNextMerge / applyMerge called one at a time) and inside k_merge_loop.
#pragma once
#include "common.cuh"

namespace bpe {

struct DevState {
  // persistent
  uint32_t n_keys;
  unsigned long long pool_cursor;  // next free cell of the occurrence pool (64-bit: the pool may pass 2^32 cells)
  uint32_t err;
  uint32_t hot_n;
  uint32_t hot_thresh;
  // per iteration (double-buffered by iteration parity inside k_merge_loop; index 0 otherwise)
  uint32_t n_sites[2];
  uint32_t n_new[2];
  uint32_t n_cand;
  uint32_t blocks_done;
  // arg-max result
  unsigned long long best_primary;  // (count << 20) | (0xFFFFF - (a+b)); 0 = nothing
  uint32_t best_slot;
  uint32_t best_mult;  // number of pairs sharing best_primary
  uint32_t best_a, best_b, best_cnt;
  uint32_t list_len;
  unsigned long long tie_pos;  // (lastpos << 32 | slot) min over candidates
  unsigned long long live_tokens;
  unsigned long long _unused_barrier;
  // k_merge_loop bookkeeping
  uint32_t n_tokens;     // next free token index
  uint32_t iters_done;   // merges applied by the current launch
  uint32_t status;       // LOOP_* exit reason
  uint32_t tie_breaks;
  unsigned long long sites_total;
  // snapshot taken by block 0 while nothing changes these (start of P3), read by every block for its exit decision:
  // the decision must not depend on values a faster block may already be changing in the next phase
  uint32_t snap_n_keys, snap_hot_n, snap_err;
  unsigned long long snap_pool_cursor;
  unsigned long long prof_ns[8];  // block 0's view: decide, P1 work, P1 wait, P2 work, P2 wait, P3 work, P3 wait, tie path
  uint32_t bins[36];  // histogram of bit lengths of counts (hot-list threshold selection)
  // ---- sharded (multi-GPU) training, mg_kernels.cuh ----
  unsigned long long mg_epoch;      // count-delta exchanges completed (monotone across launches)
  unsigned long long mg_tie_epoch;  // tie exchanges completed
  uint32_t n_touched[2];            // pairs whose count changed on this rank in the current merge (by iteration parity)
  uint32_t n_out;                   // records in the outgoing delta message
  uint32_t n_newpair;               // distinct pairs born in the current merge on ANY rank (hot-list candidates)
  uint32_t mg_abort;                // a peer did not answer in time / a rank reported an error: every block leaves
  unsigned long long mg_prof_ns[12];  // block 0: decide, P1, wait, M1, wait, exchange, wait, P2, wait, P3, wait, tie path
  // folded message headers, read by every thread with two 128-bit loads: [0] OR of all ranks' error flags, then the
  // minima over ranks of pool_free, sites_cap, new_cap, hot_cap, len16_cap, tbl_cap, cand_cap
  alignas(16) uint32_t g_vals[8];
  unsigned long long fine_ns[12];  // BPE_FINE_PROF builds: block 0 / thread 0 sub-steps of phase_sites
  unsigned long long bucket_ns[32][4];  // BPE_FINE_PROF: per log2(weight) bucket: P1, P2, P3 work (block 0), merges
};

constexpr uint32_t LOOP_RUNNING = 0, LOOP_DONE = 1, LOOP_NEED_REBUILD = 2, LOOP_NEED_HOST = 3, LOOP_EMPTY = 4,
                   LOOP_ERROR = 5, LOOP_LIMIT = 6;

struct SiteRec {
  uint32_t p;      // position of the `a` being merged
  uint32_t lpos;   // position of the left token of the new left adjacency (NOPOS if none)
  uint32_t lslot;  // table slot of the new left adjacency's pair (NOSLOT if none)
  uint32_t rslot;  // table slot of the new right adjacency's pair (NOSLOT if none)
};

struct MergeRec {  // layout of bpe_merge (include/bpe_b200.h)
  int32_t a, b, c, reserved;
  long long weight;
};

__device__ __forceinline__ unsigned long long make_primary(uint32_t cnt, uint32_t a, uint32_t b) {
  return ((unsigned long long)cnt << 20) | (unsigned long long)(0xFFFFFu - (a + b));
}

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

// ------------------------------------------------------------------------------------------------
// ingest: int32 ids -> slots (vectorised 128-bit), then DOCSTART flags per document
// ------------------------------------------------------------------------------------------------
__global__ void k_ingest_ids(const int32_t* __restrict__ ids, uint32_t* __restrict__ slots, uint64_t n,
                             uint32_t max_id, uint32_t* __restrict__ err) {
  uint64_t i4 = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  uint64_t n4 = n >> 2;
  bool aligned = ((((uintptr_t)ids) | ((uintptr_t)slots)) & 15) == 0;
  uint32_t bad = 0;
  if (aligned) {
    for (uint64_t i = i4; i < n4; i += stride) {
      int4 v = __ldg(reinterpret_cast<const int4*>(ids) + i);
      bad |= ((uint32_t)v.x >= max_id) | ((uint32_t)v.y >= max_id) | ((uint32_t)v.z >= max_id) | ((uint32_t)v.w >= max_id);
      reinterpret_cast<uint4*>(slots)[i] = make_uint4((uint32_t)v.x, (uint32_t)v.y, (uint32_t)v.z, (uint32_t)v.w);
    }
    for (uint64_t i = (n4 << 2) + i4; i < n; i += stride) {
      uint32_t v = (uint32_t)ids[i];
      bad |= v >= max_id;
      slots[i] = v;
    }
  } else {
    for (uint64_t i = i4; i < n; i += stride) {
      uint32_t v = (uint32_t)ids[i];
      bad |= v >= max_id;
      slots[i] = v;
    }
  }
  if (bad) atomicOr(err, 1u);
}

// ids already sit in the slot array (host upload path): range check only
__global__ void k_validate_ids(const uint32_t* __restrict__ slots, uint64_t n, uint32_t max_id, uint32_t* __restrict__ err) {
  uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  uint32_t bad = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) bad |= slots[i] >= max_id;
  if (bad) atomicOr(err, 1u);
}

__global__ void k_mark_docstarts(uint32_t* __restrict__ slots, const int64_t* __restrict__ doc_off, int64_t n_docs,
                                 int64_t base) {
  int64_t d = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; d < n_docs; d += stride) {
    int64_t s = doc_off[d], e = doc_off[d + 1];
    if (e > s) slots[base + s] |= DOCSTART;
  }
}

// ------------------------------------------------------------------------------------------------
// K1: pair histogram.  128-bit coalesced loads of the slots, block-local shared-memory open-addressing
// hash for the counts (one global atomic per distinct pair per block instead of one per position).
// ------------------------------------------------------------------------------------------------
constexpr int K1_THREADS = 256;
constexpr int K1_SMEM_SLOTS = 2048;  // 24 KB
constexpr int K1_MAX_PROBE = 8;
// 2^15 positions: 96 KB of shared memory per block, two 1024-thread blocks per SM (9.1 ms for K1 on cfg3 against 10.1 ms
// with 2^16 and one block per SM; profiles/r04a_k1b_staged.md)
#ifndef BPE_K1B_CHUNK_LOG
#define BPE_K1B_CHUNK_LOG 15
#endif
static_assert(BPE_K1B_CHUNK_LOG >= 10 && BPE_K1B_CHUNK_LOG <= 16, "k_scatter stages 16-bit offsets within a chunk");
constexpr uint32_t K1B_CHUNK = 1u << BPE_K1B_CHUNK_LOG;  // positions per block iteration of the scatter
constexpr int K1B_THREADS = 1024;
static_assert(K1_SMEM_SLOTS % K1B_THREADS == 0 && K1B_THREADS % 32 == 0, "the prefix gives every thread whole slots");

struct SmemHist {
  uint32_t key[K1_SMEM_SLOTS];
  uint32_t a[K1_SMEM_SLOTS];  // k_hist: adjacencies seen        k_scatter: count, then staging cursor
  uint32_t b[K1_SMEM_SLOTS];  // k_hist: of which NOT counted    k_scatter: base cell in the pool, low word
};

// k_scatter's dynamic shared memory: the block-local table, where each slot's run starts in the staging buffer, and the
// staging buffer itself (the chunk's adjacencies as 16-bit offsets, grouped by slot)
struct SmemScatter {
  SmemHist h;
  uint32_t bhi[K1_SMEM_SLOTS];  // high word of the base cell (NOPOS: the pair is missing from the table)
  uint32_t start[K1_SMEM_SLOTS + 1];
  uint32_t warp_sum[K1B_THREADS / 32];
  uint16_t stage[K1B_CHUNK];
};
constexpr size_t K1B_SMEM_BYTES = sizeof(SmemScatter);

// slot of `key` in the block-local table (inserting it), or -1 when the neighbourhood is crowded
__device__ __forceinline__ int sh_slot(SmemHist& sh, uint32_t key, bool insert) {
  uint32_t h = (key * 0x9E3779B1u) >> (32 - 11);
#pragma unroll 1
  for (int probe = 0; probe < K1_MAX_PROBE; probe++) {
    uint32_t k = sh.key[h];
    if (k == EMPTY_KEY) {
      if (!insert) return -1;
      uint32_t old = atomicCAS(&sh.key[h], EMPTY_KEY, key);
      k = (old == EMPTY_KEY) ? key : old;
    }
    if (k == key) return (int)h;
    h = (h + 1) & (K1_SMEM_SLOTS - 1);
  }
  return -1;
}

// One adjacency starting at position p (slot value w).  Returns false when p starts no adjacency.
// counted (optional): the run-parity rule of core.ts:285-290.
__device__ __forceinline__ bool edge_at(const uint32_t* __restrict__ slots, uint32_t n, uint32_t p, uint32_t w,
                                        uint32_t wnext_hint, uint32_t* key, uint32_t* counted) {
  if (!slot_is_id(w)) return false;
  uint32_t a = slot_val(w);
  int b;
  if (slot_is_id(wnext_hint)) {
    b = (wnext_hint & DOCSTART) ? NOTOK : (int)slot_val(wnext_hint);
  } else {
    uint32_t q;
    b = right_token(slots, n, p, &q);
  }
  if (b == NOTOK) return false;
  *key = pair_key(a, (uint32_t)b);
  if (counted) {
    *counted = 1;
    if ((uint32_t)b == a) *counted = (run_left(slots, p, w, (int)a) & 1u) ? 0u : 1u;
  }
  return true;
}

// loads the 4 slots of group g plus the slot after them
__device__ __forceinline__ void load_group(const uint32_t* __restrict__ slots, uint32_t n, uint32_t g, uint32_t v[5]) {
  uint32_t p0 = g << 2;
  if (p0 + 4 <= n) {
    uint4 q = ld_slots4(slots + p0);
    v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
  } else {
#pragma unroll
    for (int j = 0; j < 4; j++) v[j] = (p0 + j < n) ? ld_slot(slots + p0 + j) : mk_hole();
  }
  v[4] = (p0 + 4 < n) ? ld_slot(slots + p0 + 4) : (DOCSTART);  // DOCSTART|ID(0): "no right neighbour"
}

__global__ void __launch_bounds__(K1_THREADS) k_hist(const uint32_t* __restrict__ slots, uint32_t n, PairTable t,
                                                      DevState* st) {
  __shared__ SmemHist sh;
  for (int i = threadIdx.x; i < K1_SMEM_SLOTS; i += K1_THREADS) {
    sh.key[i] = EMPTY_KEY;
    sh.a[i] = 0;
    sh.b[i] = 0;
  }
  __syncthreads();
  // contiguous chunk of 4-slot groups per block, so the shared table sees as few distinct pairs as possible
  uint32_t n4 = (n + 3) >> 2;
  uint32_t per_block = (n4 + gridDim.x - 1) / gridDim.x;
  uint32_t g_begin = blockIdx.x * per_block;
  uint32_t g_end = min(n4, g_begin + per_block);
  for (uint32_t g = g_begin + threadIdx.x; g < g_end; g += K1_THREADS) {
    uint32_t p0 = g << 2;
    uint32_t v[5];
    load_group(slots, n, g, v);
#pragma unroll
    for (int j = 0; j < 4; j++) {
      uint32_t key, counted;
      if (p0 + j < n && edge_at(slots, n, p0 + j, v[j], v[j + 1], &key, &counted)) {
        int h = sh_slot(sh, key, true);
        if (h >= 0) {
          atomicAdd(&sh.a[h], 1u);
          if (!counted) atomicAdd(&sh.b[h], 1u);
        } else {  // shared table crowded: straight to the global table
          uint32_t gs = tbl_find_or_insert(t, key, &st->n_keys);
          if (gs == NOSLOT) {
            atomicOr(&st->err, ERR_TABLE_FULL);
          } else {
            if (counted) atomicAdd(t.cnt + gs, 1u);
            atomicAdd(t.occ_len + gs, 1u);
          }
        }
      }
    }
  }
  __syncthreads();
  uint32_t n_ins = 0;
  for (int i = threadIdx.x; i < K1_SMEM_SLOTS; i += K1_THREADS) {
    uint32_t key = sh.key[i];
    if (key == EMPTY_KEY) continue;
    bool ins;
    uint32_t gs = tbl_find_or_insert_ex(t, key, &ins);
    if (gs == NOSLOT) {
      atomicOr(&st->err, ERR_TABLE_FULL);
      continue;
    }
    n_ins += ins ? 1u : 0u;
    if (sh.a[i] != sh.b[i]) atomicAdd(t.cnt + gs, sh.a[i] - sh.b[i]);
    if (sh.a[i]) atomicAdd(t.occ_len + gs, sh.a[i]);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) n_ins += __shfl_xor_sync(0xFFFFFFFFu, n_ins, o);
  if ((threadIdx.x & 31) == 0 && n_ins) atomicAdd(&st->n_keys, n_ins);  // one n_keys atomic per warp
}

// carve every pair's occurrence list out of the pool
__global__ void k_alloc_lists(PairTable t, DevState* st, unsigned long long pool_cap) {
  uint32_t cap = t.mask + 1;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += gridDim.x * blockDim.x) {
    if (t.keys[i] == EMPTY_KEY) continue;
    uint32_t len = t.occ_len[i];
    t.occ_fill[i] = 0;
    if (len == 0) continue;
    const unsigned long long start = atomicAdd(&st->pool_cursor, (unsigned long long)len);
    if (start > pool_cap || len > pool_cap - start) atomicOr(&st->err, ERR_POOL_FULL);
    t.occ_start.set(i, start);
  }
}

// K1b: scatter every adjacency's position into its pair's list.  Per chunk of K1B_CHUNK positions a block
//  1. counts the chunk's adjacencies per pair in its shared table;
//  2. lays the pairs' runs out back to back in a shared staging buffer (an exclusive prefix of the counts) and reserves
//     one range per pair in the pool with a single global atomic;
//  3. re-reads the chunk (from L2) and puts each adjacency's 16-bit offset into its pair's run with a shared ticket;
//  4. copies the staging buffer out with consecutive threads on consecutive cells of one range, so that a range leaves
//     as whole sectors plus at most two partial edges.  Stored one adjacency at a time, the cells of a range reach the
//     L2 spread over the whole time the block spends on the chunk, and partly written sectors go back to HBM as
//     read-modify-writes.
// A pair that found no room in the shared table takes one global cursor atomic per adjacency and stores directly.
// The order of the cells inside a range follows the tickets and is not deterministic; no reader of the lists depends on it.
__global__ void __launch_bounds__(K1B_THREADS) k_scatter(const uint32_t* __restrict__ slots, uint32_t n, PairTable t,
                                                          uint32_t* __restrict__ pool, DevState* st) {
  extern __shared__ __align__(16) unsigned char k1b_smem[];
  SmemScatter& sh = *reinterpret_cast<SmemScatter*>(k1b_smem);
  constexpr int PER = K1_SMEM_SLOTS / K1B_THREADS;  // slots per thread in the prefix
  constexpr int WARPS = K1B_THREADS / 32;
  const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
  const uint32_t n_chunks = (n + K1B_CHUNK - 1) / K1B_CHUNK;
  for (uint32_t chunk = blockIdx.x; chunk < n_chunks; chunk += gridDim.x) {
    for (int i = threadIdx.x; i < K1_SMEM_SLOTS; i += K1B_THREADS) {
      sh.h.key[i] = EMPTY_KEY;
      sh.h.a[i] = 0;
    }
    __syncthreads();
    const uint32_t c0 = chunk * K1B_CHUNK;
    const uint32_t g_begin = c0 >> 2;
    const uint32_t g_end = min((n + 3) >> 2, g_begin + (K1B_CHUNK >> 2));
    for (uint32_t g = g_begin + threadIdx.x; g < g_end; g += K1B_THREADS) {
      uint32_t p0 = g << 2;
      uint32_t v[5];
      load_group(slots, n, g, v);
#pragma unroll
      for (int j = 0; j < 4; j++) {
        uint32_t key;
        if (p0 + j < n && edge_at(slots, n, p0 + j, v[j], v[j + 1], &key, nullptr)) {
          int h = sh_slot(sh.h, key, true);
          if (h >= 0) atomicAdd(&sh.h.a[h], 1u);
        }
      }
    }
    __syncthreads();
    // exclusive prefix of the counts: thread i owns slots PER*i .. PER*i + PER-1
    const int i0 = threadIdx.x * PER;
    uint32_t cnt[PER], sum = 0;
#pragma unroll
    for (int e = 0; e < PER; e++) {
      cnt[e] = sh.h.a[i0 + e];
      sum += cnt[e];
    }
    uint32_t inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t y = __shfl_up_sync(0xFFFFFFFFu, inc, o);
      if (lane >= (uint32_t)o) inc += y;
    }
    if (lane == 31) sh.warp_sum[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      uint32_t w = lane < (uint32_t)WARPS ? sh.warp_sum[lane] : 0u, wi = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        uint32_t y = __shfl_up_sync(0xFFFFFFFFu, wi, o);
        if (lane >= (uint32_t)o) wi += y;
      }
      if (lane < (uint32_t)WARPS) sh.warp_sum[lane] = wi - w;
    }
    __syncthreads();
    uint32_t run = sh.warp_sum[warp] + inc - sum;
#pragma unroll
    for (int e = 0; e < PER; e++) {
      const int i = i0 + e;
      sh.start[i] = run;
      if (cnt[e]) {  // (every key in the table has a count)
        uint32_t gs = tbl_find(t, sh.h.key[i]);
        if (gs == NOSLOT) {
          atomicOr(&st->err, ERR_MISSING_KEY);
          sh.bhi[i] = NOPOS;
        } else {
          const unsigned long long base = t.occ_start.get(gs) + atomicAdd(t.occ_fill + gs, cnt[e]);
          sh.h.b[i] = (uint32_t)base;
          sh.bhi[i] = (uint32_t)(base >> 32);  // (< 4: the pool holds at most 3 * 2^32 cells)
        }
      }
      sh.h.a[i] = run;  // staging cursor
      run += cnt[e];
    }
    if (threadIdx.x == K1B_THREADS - 1) sh.start[K1_SMEM_SLOTS] = run;
    __syncthreads();
    for (uint32_t g = g_begin + threadIdx.x; g < g_end; g += K1B_THREADS) {
      uint32_t p0 = g << 2;
      uint32_t v[5];
      load_group(slots, n, g, v);
#pragma unroll
      for (int j = 0; j < 4; j++) {
        uint32_t key;
        if (p0 + j < n && edge_at(slots, n, p0 + j, v[j], v[j + 1], &key, nullptr)) {
          int h = sh_slot(sh.h, key, false);
          if (h >= 0) {
            sh.stage[atomicAdd(&sh.h.a[h], 1u)] = (uint16_t)(p0 + j - c0);
          } else {  // pair did not fit the block-local table: one global cursor atomic
            uint32_t gs = tbl_find(t, key);
            if (gs == NOSLOT) atomicOr(&st->err, ERR_MISSING_KEY);
            else pool[t.occ_start.get(gs) + atomicAdd(t.occ_fill + gs, 1u)] = p0 + j;
          }
        }
      }
    }
    __syncthreads();
    const uint32_t total = sh.start[K1_SMEM_SLOTS];
    for (uint32_t k = threadIdx.x; k < total; k += K1B_THREADS) {
      uint32_t s = 0;  // the last slot whose run starts at or before k: the slot whose run holds k
#pragma unroll
      for (uint32_t half = K1_SMEM_SLOTS / 2; half; half >>= 1)
        if (sh.start[s + half] <= k) s += half;
      const uint32_t hi = sh.bhi[s];
      if (hi != NOPOS) pool[(((unsigned long long)hi << 32) | sh.h.b[s]) + (k - sh.start[s])] = c0 + sh.stage[k];
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// K2: arg-max.  primary = (count, -(a+b)); the position tie-break runs only when best_mult > 1.
// ------------------------------------------------------------------------------------------------
struct Best {
  unsigned long long primary;
  uint32_t slot;
  uint32_t mult;
};

__device__ __forceinline__ Best best_merge(Best x, Best y) {
  if (x.primary > y.primary) return x;
  if (y.primary > x.primary) return y;
  Best r;
  r.primary = x.primary;
  r.slot = min(x.slot, y.slot);
  r.mult = x.mult + y.mult;
  return r;
}

__device__ __forceinline__ Best best_warp_reduce(Best v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    Best w;
    w.primary = __shfl_xor_sync(0xFFFFFFFFu, v.primary, o);
    w.slot = __shfl_xor_sync(0xFFFFFFFFu, v.slot, o);
    w.mult = __shfl_xor_sync(0xFFFFFFFFu, v.mult, o);
    v = best_merge(v, w);
  }
  return v;
}

// block-wide reduction; the result is valid in every thread.  s_best must hold blockDim.x/32 entries.
__device__ __forceinline__ Best best_block_reduce(Best v, Best* s_best) {
  v = best_warp_reduce(v);
  __syncthreads();
  if (lane_id() == 0) s_best[threadIdx.x >> 5] = v;
  __syncthreads();
  uint32_t nw = blockDim.x >> 5;
  Best u = (lane_id() < nw) ? s_best[lane_id()] : Best{0ull, NOSLOT, 0};
  u = best_warp_reduce(u);
  return u;
}

__device__ __forceinline__ unsigned long long slot_primary(const PairTable& t, const uint32_t* len16, uint32_t s,
                                                           uint32_t max_length) {
  uint32_t key = t.keys[s];
  if (key == EMPTY_KEY) return 0ull;
  uint32_t c = t.cnt[s];
  if (c == 0) return 0ull;
  uint32_t a = key >> 16, b = key & 0xFFFFu;
  if (max_length && len16[a] + len16[b] > max_length) return 0ull;
  return make_primary(c, a, b);
}

// the same, also handing out the pair's key
__device__ __forceinline__ unsigned long long slot_primary_k(const PairTable& t, const uint32_t* len16, uint32_t s, uint32_t max_length,
                                                             uint32_t* key_out) {
  uint32_t key = t.keys[s];
  *key_out = key;
  if (key == EMPTY_KEY) return 0ull;
  uint32_t c = t.cnt[s];
  if (c == 0) return 0ull;
  uint32_t a = key >> 16, b = key & 0xFFFFu;
  if (max_length && len16[a] + len16[b] > max_length) return 0ull;
  return make_primary(c, a, b);
}

// per-thread partial over this block's stripe of the hot list (use_hot) or of the whole table
__device__ __forceinline__ Best argmax_stripe(const PairTable& t, const uint32_t* len16, uint32_t max_length, int use_hot,
                                              const uint32_t* hot, uint32_t n, uint32_t bid, uint32_t nblk) {
  Best mine{0ull, NOSLOT, 0};
  for (uint32_t i = bid * blockDim.x + threadIdx.x; i < n; i += nblk * blockDim.x) {
    uint32_t s = use_hot ? hot[i] : i;
    unsigned long long pr = slot_primary(t, len16, s, max_length);
    if (pr) mine = best_merge(mine, Best{pr, s, 1});
  }
  return mine;
}

__device__ __forceinline__ void publish_best(const PairTable& t, DevState* st, Best u) {
  st->best_primary = u.primary;
  st->best_slot = u.slot;
  st->best_mult = u.mult;
  if (u.primary) {
    uint32_t key = t.keys[u.slot];
    st->best_a = key >> 16;
    st->best_b = key & 0xFFFFu;
    st->best_cnt = t.cnt[u.slot];
    st->list_len = t.occ_len[u.slot];
  } else {
    st->best_a = st->best_b = st->best_cnt = st->list_len = 0;
  }
}

constexpr int AM_THREADS = 256;

// Stand-alone K2 over the whole table.  The last block to finish folds the per-block partials and resets the per-iteration counters.
__global__ void __launch_bounds__(AM_THREADS) k_argmax(PairTable t, const uint32_t* __restrict__ len16,
                                                        uint32_t max_length, Best* __restrict__ partials, DevState* st) {
  __shared__ Best s_best[AM_THREADS / 32];
  __shared__ bool s_last;
  Best v = best_block_reduce(argmax_stripe(t, len16, max_length, 0, nullptr, t.mask + 1, blockIdx.x, gridDim.x), s_best);
  if (threadIdx.x == 0) {
    partials[blockIdx.x] = v;
    __threadfence();
    uint32_t done = atomicAdd(&st->blocks_done, 1u);
    s_last = (done == gridDim.x - 1);
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  Best w{0ull, NOSLOT, 0};
  for (uint32_t i = threadIdx.x; i < gridDim.x; i += blockDim.x) w = best_merge(w, partials[i]);
  w = best_block_reduce(w, s_best);
  if (threadIdx.x == 0) {
    publish_best(t, st, w);
    st->blocks_done = 0;
    st->n_sites[0] = st->n_sites[1] = 0;
    st->n_new[0] = st->n_new[1] = 0;
    st->n_cand = 0;
    st->tie_pos = ~0ull;
  }
}

// candidates = pairs whose primary equals `best`
__device__ __forceinline__ void phase_collect(const PairTable& t, const uint32_t* len16, uint32_t max_length, int use_hot,
                                              const uint32_t* hot, uint32_t n, unsigned long long best, uint32_t* cands,
                                              uint32_t cand_cap, DevState* st, uint32_t bid, uint32_t nblk) {
  for (uint32_t i = bid * blockDim.x + threadIdx.x; i < n; i += nblk * blockDim.x) {
    uint32_t s = use_hot ? hot[i] : i;
    if (slot_primary(t, len16, s, max_length) == best) {
      uint32_t k = atomicAdd(&st->n_cand, 1u);
      if (k < cand_cap) cands[k] = s;
      else atomicOr(&st->err, ERR_CAND_OVERFLOW);
    }
  }
}

__global__ void k_collect_cands(PairTable t, const uint32_t* __restrict__ len16, uint32_t max_length, uint32_t* __restrict__ cands,
                                uint32_t cand_cap, DevState* st) {
  phase_collect(t, len16, max_length, 0, nullptr, t.mask + 1, st->best_primary, cands, cand_cap, st, blockIdx.x, gridDim.x);
}

// Is position p a *counted* occurrence of (a,b) right now?
__device__ __forceinline__ bool counted_occurrence(const uint32_t* slots, uint32_t n, uint32_t p, uint32_t a, uint32_t b) {
  uint32_t w = ld_slot(slots + p);
  if (!slot_is_id(w) || slot_val(w) != a) return false;
  uint32_t q;
  if (right_token(slots, n, p, &q) != (int)b) return false;
  if (a == b && (run_left(slots, p, w, (int)a) & 1u)) return false;
  return true;
}

// one block per candidate: scan position of its last counted occurrence; global min of (pos, slot) wins
__device__ __forceinline__ void phase_tie(const uint32_t* slots, uint32_t n, const PairTable& t, const uint32_t* pool,
                                          const uint32_t* cands, uint32_t n_cand, DevState* st, uint32_t* s_max,
                                          uint32_t bid, uint32_t nblk) {
  for (uint32_t c = bid; c < n_cand; c += nblk) {
    uint32_t s = cands[c];
    uint32_t key = t.keys[s];
    uint32_t a = key >> 16, b = key & 0xFFFFu;
    const unsigned long long start = t.occ_start.get(s);
    uint32_t len = t.occ_len[s];
    uint32_t v = 0;  // 1 + max position, 0 = none
    for (uint32_t i = threadIdx.x; i < len; i += blockDim.x) {
      uint32_t p = pool[start + i];
      if (counted_occurrence(slots, n, p, a, b)) v = max(v, p + 1);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xFFFFFFFFu, v, o));
    __syncthreads();
    if (lane_id() == 0) s_max[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t m = 0;
      for (uint32_t i = 0; i < (blockDim.x >> 5); i++) m = max(m, s_max[i]);
      if (m) atomicMin(&st->tie_pos, ((unsigned long long)(m - 1) << 32) | s);
    }
  }
}

__global__ void __launch_bounds__(256) k_tie_break(const uint32_t* __restrict__ slots, uint32_t n, PairTable t,
                                                    const uint32_t* __restrict__ pool,
                                                    const uint32_t* __restrict__ cands, DevState* st) {
  __shared__ uint32_t s_max[32];
  phase_tie(slots, n, t, pool, cands, st->n_cand, st, s_max, blockIdx.x, gridDim.x);
}

__global__ void k_tie_finish(PairTable t, DevState* st) {
  if (threadIdx.x == 0 && blockIdx.x == 0 && st->tie_pos != ~0ull) {
    uint32_t s = (uint32_t)(st->tie_pos & 0xFFFFFFFFu);
    uint32_t key = t.keys[s];
    st->best_slot = s;
    st->best_a = key >> 16;
    st->best_b = key & 0xFFFFu;
    st->best_cnt = t.cnt[s];
    st->list_len = t.occ_len[s];
  }
}

// look a pair up for bpe_apply_merge called on its own (restoreMerge path)
__global__ void k_lookup_pair(PairTable t, uint32_t a, uint32_t b, DevState* st) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    uint32_t s = tbl_find(t, pair_key(a, b));
    st->best_slot = s;
    st->best_a = a;
    st->best_b = b;
    st->best_cnt = (s == NOSLOT) ? 0 : t.cnt[s];
    st->list_len = (s == NOSLOT) ? 0 : t.occ_len[s];
    st->n_sites[0] = st->n_sites[1] = 0;
    st->n_new[0] = st->n_new[1] = 0;
    st->n_cand = 0;
  }
}

// ------------------------------------------------------------------------------------------------
// hot list: pairs with count >= hot_thresh (and passing the length filter).  Counts of existing pairs
// never grow under merging, so between rebuilds only pairs created by a merge can enter.
// ------------------------------------------------------------------------------------------------
__global__ void k_count_bins(PairTable t, const uint32_t* __restrict__ len16, uint32_t max_length, DevState* st) {
  __shared__ uint32_t s_bins[36];
  if (threadIdx.x < 36) s_bins[threadIdx.x] = 0;
  __syncthreads();
  uint32_t cap = t.mask + 1;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += gridDim.x * blockDim.x) {
    unsigned long long pr = slot_primary(t, len16, i, max_length);
    if (pr) atomicAdd(&s_bins[32 - __clz((uint32_t)(pr >> 20))], 1u);
  }
  __syncthreads();
  if (threadIdx.x < 36 && s_bins[threadIdx.x]) atomicAdd(&st->bins[threadIdx.x], s_bins[threadIdx.x]);
}

__global__ void k_build_hot(PairTable t, const uint32_t* __restrict__ len16, uint32_t max_length,
                            uint32_t* __restrict__ hot, uint32_t hot_cap, DevState* st) {
  uint32_t cap = t.mask + 1;
  uint32_t thresh = st->hot_thresh;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += gridDim.x * blockDim.x) {
    unsigned long long pr = slot_primary(t, len16, i, max_length);
    if (pr && (uint32_t)(pr >> 20) >= thresh) {
      uint32_t k = atomicAdd(&st->hot_n, 1u);
      if (k < hot_cap) hot[k] = i;
      else atomicOr(&st->err, ERR_HOT_OVERFLOW);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// K3 phase 1: find the merge sites of (a,b) -> c, emit count deltas and size the new pairs' lists.
// Reads the corpus only (all writes happen in phase_apply), so every thread sees the pre-merge state.
// Count deltas and list sizing are warp-aggregated: lanes that touch the same pair elect one leader
// (__match_any_sync) which issues a single atomic for all of them -- early merges hit a handful of
// pairs millions of times.  scan_mode = 1 walks every slot instead of the pair's occurrence list.
// ------------------------------------------------------------------------------------------------
struct ApplyArgs {
  uint32_t* slots;
  uint32_t n;
  PairTable t;
  uint32_t* pool;
  DevState* st;
  SiteRec* sites;
  uint32_t sites_cap;
  uint32_t* newslots;
  uint32_t new_cap;
  uint32_t* len16;
  int scan_mode;
  // sharded training: count deltas are staged per pair (dlt) and listed (touched) instead of applied, see mg_kernels.cuh
  int32_t* dlt;
  uint32_t* touched;
  uint32_t touched_cap;
  // pairs born by a merge are (x,c) or (c,y): they are accumulated in dense per-token rows (L2-resident, RED atomics, no
  // hashing) and entered into the pair table once each by phase_new_pairs.  nd[ND_*][tok], row stride ND_STRIDE
  uint32_t* nd;
  // sharded training: table slots of the pairs born by the current merge on ANY rank (candidates for the hot list); a
  // pair is listed by whoever inserts its key -- phase_new_pairs for pairs born on this shard, the record pass otherwise
  uint32_t* newpair;
  uint32_t newpair_cap;
  // sharded training, small merges: every (pair, delta) goes straight into the record area of each rank's inbox
  unsigned long long* push[8];
  int push_world;  // 0: staged mode (or single GPU)
  uint32_t push_cap;
};

constexpr uint32_t ND_STRIDE = 56320;  // >= BPE_MAX_TOKENS + 1
enum { ND_L_LEN = 0, ND_L_CNT, ND_R_LEN, ND_R_CNT, ND_L_SLOT, ND_R_SLOT, ND_ROWS };
constexpr uint32_t NOTOKV = 0xFFFFFFFFu;

// Per-block staging of the deltas of frequent neighbours: in the site pass of a merge whose occurrence list is longer than
// LoopArgs::stage_min, the deltas whose other token is below R_STAGE_T -- on Zipf text the characters and the earliest merges,
// the neighbours of nearly every site of a big merge -- are summed in shared memory and added to their global word ONCE per
// block before P1's barrier, instead of by one atomic per warp-iteration on a few hot L2 lines (k_merge_rounds: profiles/r03a,
// k_merge_loop: profiles/r06a).
#ifndef BPE_STAGE_T
#define BPE_STAGE_T 256
#endif
constexpr uint32_t R_STAGE_T = BPE_STAGE_T;
constexpr uint32_t R_STAGE_MIN_DEFAULT = 16384;  // list entries above which a merge stages its deltas (measured: profiles/r03a)
// k_merge_loop's staged rows, [LS_ROWS][R_STAGE_T] u32 in shared memory: the four born-pair rows of nd (ND_L_LEN .. ND_R_CNT,
// same order), then the decrements of the old pairs (tok, a) and (b, tok)
enum { LS_DEC_L = ND_R_CNT + 1, LS_DEC_R, LS_ROWS };

constexpr uint32_t ERR_TOUCH_OVERFLOW = 128u, ERR_PEER_TIMEOUT = 256u, ERR_INBOX_OVERFLOW = 512u, ERR_PEER = 1024u;

__device__ __forceinline__ unsigned long long now_ns();
// non-blocking hints: the per-site chain of dependent DRAM round trips is what bounds a merge iteration, so the
// neighbourhood of a site and the table cells of its (up to four) pairs are requested before they are walked / updated
__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ void prefetch_pair(const PairTable& t, uint32_t key) {
  uint32_t h = tbl_hash(t, key);
  prefetch_l1(t.keys + h);
  prefetch_l2(t.cnt + h);
  prefetch_l2(t.occ_len + h);
}

// Count deltas, warp-collective (all 32 lanes call; `has` lanes carry one delta of pair slot s): applied to the table
// (single GPU), pushed into every rank's inbox (sharded, small merges) or staged per pair (sharded, big merges).
// Counters shared by the whole grid (n_out, n_touched) get ONE atomic per warp.
__device__ __forceinline__ void cnt_delta_warp(const ApplyArgs& A, bool has, uint32_t s, uint32_t key, int32_t d, uint32_t par) {
  const uint32_t lane = lane_id();
  if (A.push_world) {
    uint32_t m = __ballot_sync(0xFFFFFFFFu, has);
    if (!m) return;
    uint32_t base = 0;
    int src = __ffs(m) - 1;
    if ((int)lane == src) base = atomicAdd(&A.st->n_out, (uint32_t)__popc(m));
    base = __shfl_sync(0xFFFFFFFFu, base, src);
    if (has) {
      uint32_t k = base + __popc(m & ((1u << lane) - 1u));
      if (k < A.push_cap) {
        unsigned long long rec = ((unsigned long long)key << 32) | (uint32_t)d;
        for (int q = 0; q < A.push_world; q++) A.push[q][k] = rec;
      } else {
        atomicOr(&A.st->err, ERR_INBOX_OVERFLOW);
      }
    }
  } else if (A.dlt) {
    bool first = has && atomicAdd(A.dlt + s, d) == 0;  // first delta of this pair in this merge (deltas of a pair share a sign)
    uint32_t m = __ballot_sync(0xFFFFFFFFu, first);
    if (!m) return;
    uint32_t base = 0;
    int src = __ffs(m) - 1;
    if ((int)lane == src) base = atomicAdd(&A.st->n_touched[par], (uint32_t)__popc(m));
    base = __shfl_sync(0xFFFFFFFFu, base, src);
    if (first) {
      uint32_t i = base + __popc(m & ((1u << lane) - 1u));
      if (i < A.touched_cap) A.touched[i] = s;
      else atomicOr(&A.st->err, ERR_TOUCH_OVERFLOW);
    }
  } else if (has) {
    atomicAdd(A.t.cnt + s, (uint32_t)d);
  }
}

// all 32 lanes call; lanes with has == false pass any key
__device__ __forceinline__ void agg_dec(const ApplyArgs& A, uint32_t key, bool has, uint32_t par) {
  const PairTable& t = A.t;
  uint32_t lane = lane_id();
  uint32_t k = has ? key : (EMPTY_KEY - 1 - lane);
  uint32_t peers = __match_any_sync(0xFFFFFFFFu, k);
  bool leader = has && lane == (uint32_t)(__ffs(peers) - 1);
  uint32_t s = NOSLOT;
  if (leader) {
    s = tbl_find(t, key);
    if (s == NOSLOT) atomicOr(&A.st->err, ERR_MISSING_KEY);
  }
  cnt_delta_warp(A, leader && s != NOSLOT, s, key, -(int32_t)__popc(peers), par);
}

// Two decrements at once: both first probes are issued before either is consumed (one DRAM round trip instead of two).
// key1 is always (x, a) and key2 always (b, y) of the merge (a, b): with `stage` (single GPU, k_merge_loop), a decrement whose
// x / y is below R_STAGE_T goes into the block's staged row of that token instead, and loop_flush_stage applies it (single GPU
// only: see phase_sites).
__device__ __forceinline__ void agg_dec2(const ApplyArgs& A, uint32_t key1, bool has1, uint32_t key2, bool has2, uint32_t par,
                                         uint32_t* stage = nullptr) {
  const PairTable& t = A.t;
  uint32_t lane = lane_id();
  uint32_t peers1 = __match_any_sync(0xFFFFFFFFu, has1 ? key1 : (EMPTY_KEY - 1 - lane));
  uint32_t peers2 = __match_any_sync(0xFFFFFFFFu, has2 ? key2 : (EMPTY_KEY - 1 - lane));
  bool lead1 = has1 && lane == (uint32_t)(__ffs(peers1) - 1);
  bool lead2 = has2 && lane == (uint32_t)(__ffs(peers2) - 1);
  if (stage) {
    if (lead1 && (key1 >> 16) < R_STAGE_T) {
      atomicAdd(stage + LS_DEC_L * R_STAGE_T + (key1 >> 16), (uint32_t)__popc(peers1));
      lead1 = false;
    }
    if (lead2 && (key2 & 0xFFFFu) < R_STAGE_T) {
      atomicAdd(stage + LS_DEC_R * R_STAGE_T + (key2 & 0xFFFFu), (uint32_t)__popc(peers2));
      lead2 = false;
    }
  }
  uint32_t h1 = tbl_hash(t, key1), h2 = tbl_hash(t, key2);
  uint32_t k1 = lead1 ? t.keys[h1] : EMPTY_KEY;
  uint32_t k2 = lead2 ? t.keys[h2] : EMPTY_KEY;
  uint32_t s1 = NOSLOT, s2 = NOSLOT;
  if (lead1) {
    s1 = (k1 == key1) ? h1 : (k1 == EMPTY_KEY ? NOSLOT : tbl_find(t, key1));
    if (s1 == NOSLOT) atomicOr(&A.st->err, ERR_MISSING_KEY);
  }
  if (lead2) {
    s2 = (k2 == key2) ? h2 : (k2 == EMPTY_KEY ? NOSLOT : tbl_find(t, key2));
    if (s2 == NOSLOT) atomicOr(&A.st->err, ERR_MISSING_KEY);
  }
  cnt_delta_warp(A, lead1 && s1 != NOSLOT, s1, key1, -(int32_t)__popc(peers1), par);
  cnt_delta_warp(A, lead2 && s2 != NOSLOT, s2, key2, -(int32_t)__popc(peers2), par);
}

// One adjacency of a pair BORN by this merge -- (tok, c) for side 0, (c, tok) for side 1 -- per `has` lane: occurrences
// and counted occurrences go to the dense rows with fire-and-forget atomics (one per distinct token per warp), or, with
// `stage` and tok below R_STAGE_T, to the block's staged copy of those rows (single GPU only: see phase_sites).
__device__ __forceinline__ void agg_new_dense(const ApplyArgs& A, uint32_t side, uint32_t tok, uint32_t c, bool has, bool counted,
                                              uint32_t par, uint32_t* stage = nullptr) {
  uint32_t lane = lane_id();
  uint32_t k = has ? tok : (0xFFFFFF00u + lane);
  uint32_t peers = __match_any_sync(0xFFFFFFFFu, k);
  uint32_t cmask = __ballot_sync(0xFFFFFFFFu, has && counted);
  const bool leader = has && lane == (uint32_t)(__ffs(peers) - 1);
  uint32_t nc = 0;
  if (leader) {
    nc = __popc(peers & cmask);
    if (stage && tok < R_STAGE_T) {
      uint32_t* srow = stage + (side ? ND_R_LEN : ND_L_LEN) * R_STAGE_T;
      atomicAdd(srow + tok, (uint32_t)__popc(peers));
      if (nc) atomicAdd(srow + R_STAGE_T + tok, nc);
    } else {
      uint32_t* row = A.nd + (size_t)(side ? ND_R_LEN : ND_L_LEN) * ND_STRIDE;
      atomicAdd(row + tok, (uint32_t)__popc(peers));
      if (nc && !A.push_world) atomicAdd(row + ND_STRIDE + tok, nc);
    }
  }
  // sharded, small merges: the count goes straight to every rank's inbox (partial counts per warp add up on arrival)
  if (A.push_world) cnt_delta_warp(A, nc != 0, NOSLOT, side ? pair_key(c, tok) : pair_key(tok, c), (int32_t)nc, par);
}

// vt / nvt: virtual thread id and count (whole warps), so that a loop kernel can give the phase a subset of its warps;
// site_buf: where the site records go (the loop kernel alternates between two buffers), A.sites when null.
// stage: the block's staged rows ([LS_ROWS][R_STAGE_T] u32 in shared memory, zero) when every thread of the block runs the phase
// and the merge stages; loop_flush_stage must then follow, with every thread of the block.  Single GPU only (A.push_world == 0,
// A.dlt == nullptr, as in k_merge_loop): the staged words go to nd and the table counts, not to an inbox or the touched list.
__device__ __forceinline__ void phase_sites(const ApplyArgs& A, uint32_t a, uint32_t b, uint32_t c, uint32_t par,
                                            uint32_t pair_slot, uint32_t vt, uint32_t nvt, SiteRec* site_buf = nullptr,
                                            uint32_t* stage = nullptr) {
  SiteRec* const site_out = site_buf ? site_buf : A.sites;
  const uint32_t* slots = A.slots;
  const uint32_t n = A.n;
  const PairTable& t = A.t;
  DevState* st = A.st;
  unsigned long long list_start = 0;
  uint32_t total = n;
  if (!A.scan_mode) {
    uint32_t s = pair_slot;
    total = (s == NOSLOT) ? 0 : t.occ_len[s];
    list_start = (s == NOSLOT) ? 0 : t.occ_start.get(s);
  }
  uint32_t lane = lane_id();
  uint32_t total_round = (total + 31u) & ~31u;
#ifdef BPE_FINE_PROF
  const bool fine = (vt == 0);
  unsigned long long ft0 = fine ? now_ns() : 0, ft1;
#define FINE(k, dep)                                   \
  if (fine) {                                          \
    if ((uint32_t)(dep) == 0xDEADBEEFu) ft0++;         \
    ft1 = now_ns();                                    \
    st->fine_ns[k] += ft1 - ft0;                       \
    ft0 = ft1;                                         \
  }
#else
#define FINE(k, dep)
#endif
  for (uint32_t i = vt; i < total_round; i += nvt) {
    bool site = false;
    uint32_t p = 0, w = 0, q = 0, koff = 0;
    if (i < total) {
      p = A.scan_mode ? i : A.pool[list_start + i];
      FINE(0, p)
      w = ld_slot(slots + p);
      if (slot_is_id(w) && slot_val(w) == a && right_token(slots, n, p, &q) == (int)b) {
        site = true;
        if (a == b) {
          koff = run_left(slots, p, w, (int)a);
          if (koff & 1u) site = false;  // overlaps the occurrence to its left (replaceAll is non-overlapping)
        }
      }
    }
    FINE(1, w + q + koff)
    // reserve the warp's cells in the site list NOW: the counter's round trip overlaps the neighbour walks below
    const uint32_t smask = __ballot_sync(0xFFFFFFFFu, site);
    if (!smask) continue;
    uint32_t site_base = 0;
    if (lane == (uint32_t)(__ffs(smask) - 1)) site_base = atomicAdd(&st->n_sites[par], (uint32_t)__popc(smask));
    SiteRec rec{p, NOPOS, NOTOKV, NOTOKV};
    // ---- adjacency on the left of the new token ----
    uint32_t dec1_key = 0, new1_tok = 0;
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
            dec1_key = pair_key(b, a);
          }
          new1_tok = c;  // the pair (c,c): runs of c count every other pair (:285-290)
          new1_counted = (chain_j & 1u) != 0;
          rec.lpos = llpos;
        } else {
          if ((uint32_t)x == a) {  // (a != b here) the run of a's ending at p loses its last element
            uint32_t L = 1 + run_left(slots, p, w, (int)a);
            dec1 = (L & 1u) == 0;
            dec1_key = pair_key(a, a);
          } else {
            dec1 = true;
            dec1_key = pair_key((uint32_t)x, a);
          }
          new1_tok = (uint32_t)x;  // the pair (x,c)
          rec.lpos = lpos;
        }
      }
    }
    FINE(2, (uint32_t)dec1_key + new1_tok)
    FINE(3, 0)
    agg_new_dense(A, 0, new1_tok, c, new1, new1_counted, par, stage);
    rec.lslot = new1 ? new1_tok : NOTOKV;  // resolved to the pair's table slot by phase_apply (ND_L_SLOT)
    FINE(4, rec.lslot)

    // ---- adjacency on the right of the new token (left to the next site when that one is chained) ----
    uint32_t dec2_key = 0, new2_tok = 0;
    bool dec2 = false, new2 = false;
    if (site) {
      uint32_t r;
      int y = right_token(slots, n, q, &r);
      if (y != NOTOK) {
        bool chained_right = false;
        if ((uint32_t)y == a) {
          uint32_t r2;
          chained_right = right_token(slots, n, r, &r2) == (int)b;
        }
        if (!chained_right) {
          if ((uint32_t)y == b && a != b) {  // the run of b's starting at q loses its first element
            uint32_t L = 1 + run_right(slots, n, q, (int)b);
            dec2 = (L & 1u) == 0;
            dec2_key = pair_key(b, b);
          } else if (!(a == b && (uint32_t)y == a)) {  // (a,a) itself is zeroed by phase_apply
            dec2 = true;
            dec2_key = pair_key(b, (uint32_t)y);
          }
          new2 = true;
          new2_tok = (uint32_t)y;  // the pair (c,y)
        }
      }
    }
    FINE(5, (uint32_t)dec2_key + new2_tok)
    agg_dec2(A, dec1_key, dec1, dec2_key, dec2, par, stage);
    FINE(6, 0)
    agg_new_dense(A, 1, new2_tok, c, new2, true, par, stage);
    rec.rslot = new2 ? new2_tok : NOTOKV;
    FINE(7, rec.rslot)

    // ---- record the site ----
    uint32_t base = __shfl_sync(0xFFFFFFFFu, site_base, __ffs(smask) - 1);
    if (site) {
      uint32_t k = base + __popc(smask & ((1u << lane) - 1u));
      if (k < A.sites_cap) reinterpret_cast<uint4*>(site_out)[k] = make_uint4(rec.p, rec.lpos, rec.lslot, rec.rslot);
      else atomicOr(&st->err, ERR_SITE_OVERFLOW);
    }
    FINE(8, base)
  }
#undef FINE
}

// End of a staged site pass in this block (all its threads call): every non-zero staged word goes to its global word with one
// atomic -- the born-pair rows to nd, a decrement to the count of (tok, a) / (b, tok) after one table probe -- and is zeroed for
// the next merge.  The rows are scanned rather than listed: LS_ROWS x R_STAGE_T words of shared memory (1 536, three per thread
// at the defaults) take a few hundred cycles, which is nothing next to a pass over more than stage_min sites.
__device__ __forceinline__ void loop_flush_stage(const ApplyArgs& A, uint32_t* stage, uint32_t a, uint32_t b) {
  __syncthreads();
  for (uint32_t i = threadIdx.x; i < LS_ROWS * R_STAGE_T; i += blockDim.x) {
    const uint32_t v = stage[i];
    if (!v) continue;
    stage[i] = 0;
    const uint32_t row = i / R_STAGE_T, tok = i - row * R_STAGE_T;
    if (row < LS_DEC_L) {
      atomicAdd(A.nd + (size_t)row * ND_STRIDE + tok, v);
    } else {
      const uint32_t s = tbl_find(A.t, row == LS_DEC_L ? pair_key(tok, a) : pair_key(b, tok));
      if (s == NOSLOT) atomicOr(&A.st->err, ERR_MISSING_KEY);
      else atomicAdd(A.t.cnt + s, 0u - v);
    }
  }
}

// K3 phase 2: every pair born in this merge -- the non-empty cells of the dense rows -- enters the pair table ONCE:
// key, occurrence-list length, list space from the pool (one cursor atomic per warp), count (unless the counts travel
// through the sharded exchange), hot list.  The cells are cleared for the next merge; ND_*_SLOT keeps the table slot for
// phase_apply.
__device__ __forceinline__ void phase_new_pairs(const ApplyArgs& A, uint32_t c, const uint32_t* len16, uint32_t max_length,
                                                int hot_valid, uint32_t* hot, uint32_t hot_cap, unsigned long long pool_cap, bool counts_elsewhere,
                                                uint32_t vt, uint32_t nvt,  // virtual thread id / count (whole warps)
                                                Best* mine = nullptr,       // arg-max candidate of the caller: pairs that go onto the hot list join it
                                                uint32_t* mine_key = nullptr) {  // ... and the key of that candidate
  const PairTable& t = A.t;
  DevState* st = A.st;
  const uint32_t thresh = st->hot_thresh;
  const uint32_t lane = lane_id();
  const uint32_t per_side = c + 1u;            // tokens 0..c can be the other half of a new pair
  const uint32_t total = 2u * per_side;
  for (uint32_t i = vt; i < ((total + 31u) & ~31u); i += nvt) {
    uint32_t side = 0, tok = 0, len = 0, cnt = 0;
    uint32_t* row = nullptr;
    if (i < total) {
      side = i >= per_side ? 1u : 0u;
      tok = i - side * per_side;
      row = A.nd + (size_t)(side ? ND_R_LEN : ND_L_LEN) * ND_STRIDE;
      len = ld_cg(row + tok);
      cnt = ld_cg(row + ND_STRIDE + tok);  // both cells in flight together (the count is only used when len != 0)
    }
    const bool act = len != 0;
    uint32_t s = NOSLOT;
    bool ins = false;
    if (act) {
      row[tok] = 0;
      row[ND_STRIDE + tok] = 0;
      s = tbl_find_or_insert_ex(t, side ? pair_key(c, tok) : pair_key(tok, c), &ins);
      if (s == NOSLOT) atomicOr(&st->err, ERR_TABLE_FULL);
    }
    uint32_t im = __ballot_sync(0xFFFFFFFFu, ins);
    if (im && lane == (uint32_t)(__ffs(im) - 1)) atomicAdd(&st->n_keys, (uint32_t)__popc(im));
    // one pool_cursor atomic per warp: inclusive scan of the list lengths
    uint32_t mylen = (act && s != NOSLOT) ? len : 0u;
    uint32_t inc = mylen;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t v = __shfl_up_sync(0xFFFFFFFFu, inc, o);
      if ((int)lane >= o) inc += v;
    }
    uint32_t wtotal = __shfl_sync(0xFFFFFFFFu, inc, 31);
    unsigned long long wbase = 0;
    if (lane == 31 && wtotal) wbase = atomicAdd(&st->pool_cursor, (unsigned long long)wtotal);
    wbase = __shfl_sync(0xFFFFFFFFu, wbase, 31);
    if (!act || s == NOSLOT) continue;
    unsigned long long start = wbase + (inc - mylen);
    if (start > pool_cap || len > pool_cap - start) {
      atomicOr(&st->err, ERR_POOL_FULL);
      start = 0;
      len = 0;
    }
    t.occ_start.set(s, start);
    t.occ_len[s] = len;
    t.occ_fill[s] = 0;
    A.nd[(size_t)(side ? ND_R_SLOT : ND_L_SLOT) * ND_STRIDE + tok] = s;
    if (counts_elsewhere) {
      if (ins) {  // (the counts arrive with the records of the exchange; P3 tests the pair against the hot-list threshold)
        uint32_t k = atomicAdd(&st->n_newpair, 1u);
        if (k < A.newpair_cap) A.newpair[k] = s;
        else atomicOr(&st->err, ERR_HOT_OVERFLOW);
      }
    } else {
      t.cnt[s] = cnt;  // the key is new: nobody else touches its count in this phase
      if (hot_valid) {
        // = slot_primary(t, len16, s, max_length), from what this thread already holds (no re-read of the cells it just wrote)
        const uint32_t pa = side ? c : tok, pb = side ? tok : c;
        unsigned long long pr = (cnt && !(max_length && len16[pa] + len16[pb] > max_length)) ? make_primary(cnt, pa, pb) : 0ull;
        if (pr && (uint32_t)(pr >> 20) >= thresh) {
          uint32_t k = atomicAdd(&st->hot_n, 1u);
          if (k < hot_cap) hot[k] = s;
          else atomicOr(&st->err, ERR_HOT_OVERFLOW);
          if (mine) {
            const uint32_t before = mine->slot;
            *mine = best_merge(*mine, Best{pr, s, 1});
            if (mine_key && mine->slot != before) *mine_key = pair_key(pa, pb);
          }
        }
      }
    }
  }
}

// K3 phase 3: rewrite the corpus in place and fill the new pairs' occurrence lists.
__device__ __forceinline__ unsigned long long agg_cursor(const PairTable& t, uint32_t slot, bool has) {
  uint32_t lane = lane_id();
  uint32_t k = has ? slot : (0xFFFFFF00u + lane);
  uint32_t peers = __match_any_sync(0xFFFFFFFFu, k);
  uint32_t leader = __ffs(peers) - 1;
  unsigned long long base = 0;
  if (has && lane == leader) base = t.occ_start.get(slot) + atomicAdd(t.occ_fill + slot, (uint32_t)__popc(peers));
  base = __shfl_sync(0xFFFFFFFFu, base, leader);
  return base + __popc(peers & ((1u << lane) - 1u));
}

// K3 phase 3 comes in two independent halves, so that the loop kernels can run the first one next to phase_new_pairs
// (neither reads what the other writes): phase_rewrite puts c into the corpus, phase_fill writes the positions of the
// new adjacencies into the lists phase_new_pairs allocated.
__device__ __forceinline__ void phase_rewrite(const ApplyArgs& A, uint32_t c, uint32_t n_sites, uint32_t vt, uint32_t nvt,
                                              const SiteRec* site_buf = nullptr) {
  const SiteRec* const sites = site_buf ? site_buf : A.sites;
  uint32_t* slots = A.slots;
  const uint32_t n = A.n;
  if (vt == 0) {
    A.st->live_tokens -= n_sites;
    A.st->sites_total += n_sites;
  }
  for (uint32_t i = vt; i < n_sites; i += nvt) {
    uint32_t p = ld_cg(&sites[i].p);
    // own slots only: [p, e] where e is the last slot of b
    uint32_t q = next_pos(slots, n, p);
    uint32_t e = next_pos(slots, n, q) - 1;
    uint32_t span = e - p + 1;
    uint32_t w = ld_slot(slots + p);
    if (span > VAL_MASK) atomicOr(&A.st->err, ERR_SPAN_OVERFLOW);
    slots[p] = (w & DOCSTART) | c;
    if (span == 2) {
      slots[p + 1] = mk_back(1);
    } else {
      if (q != p + 1 && q != e) slots[q] = mk_hole();
      slots[p + 1] = mk_span(span);
      slots[e] = mk_back(span - 1);
    }
  }
}

// All 32 lanes call: lanes that agree on `key` elect a leader which adds their number to the shared-memory word ctr[key] once;
// returns each `has` lane's ticket (the word's old value plus its rank among its peers).
__device__ __forceinline__ uint32_t agg_smem_ticket(uint32_t* ctr, uint32_t key, bool has) {
  const uint32_t lane = lane_id();
  const uint32_t peers = __match_any_sync(0xFFFFFFFFu, has ? key : (0xFFFFFF00u + lane));
  const uint32_t leader = __ffs(peers) - 1;
  uint32_t base = 0;
  if (has && lane == leader) base = atomicAdd(ctr + key, (uint32_t)__popc(peers));
  base = __shfl_sync(0xFFFFFFFFu, base, leader);
  return base + __popc(peers & ((1u << lane) - 1u));
}

// stage: the block's staged rows (as for phase_sites, zero) when every thread of the block runs the phase (vt / nvt of the whole
// grid) and the merge whose sites these are had more than stage_min of them.  The adjacencies of born pairs whose other token is
// below R_STAGE_T then take their list cells in three steps instead of one returning occ_fill atomic per warp on a few words of
// the whole grid: the block counts them per (side, token) in shared memory, reserves each (pair, block) range with ONE occ_fill
// atomic, and a second pass over the sites hands out shared-memory tickets inside the ranges.  The rows are zero on return.
// (The order of the cells inside a list was never fixed; nothing reads it.)
__device__ __forceinline__ void phase_fill(const ApplyArgs& A, uint32_t n_sites, uint32_t vt, uint32_t nvt, const SiteRec* site_buf = nullptr,
                                           uint32_t* stage = nullptr) {
  const PairTable& t = A.t;
  const SiteRec* const sites = site_buf ? site_buf : A.sites;
  uint32_t* const scnt = stage;                      // [2][R_STAGE_T]: the block's cells per (side, token), then its tickets
  // [2][R_STAGE_T] u64 over the other four rows: start of the block's range in that list (FILL_NONE: no list)
  unsigned long long* const sbase = reinterpret_cast<unsigned long long*>(stage + 2u * R_STAGE_T);
  constexpr unsigned long long FILL_NONE = ~0ull;
  uint32_t round = (n_sites + 31u) & ~31u;
  for (uint32_t i = vt; i < round; i += nvt) {
    bool has = i < n_sites;
    uint4 rv = has ? ld_cg4(reinterpret_cast<const uint4*>(sites) + i) : make_uint4(0, NOPOS, NOTOKV, NOTOKV);
    uint32_t p = rv.x, lpos = rv.y;
    const bool sl = stage && has && rv.z < R_STAGE_T, sr = stage && has && rv.w < R_STAGE_T;  // (NOTOKV is not below it)
    if (stage) {
      agg_smem_ticket(scnt, rv.z, sl);
      agg_smem_ticket(scnt, R_STAGE_T + rv.w, sr);
    }
    uint32_t lslot = (has && !sl && rv.z != NOTOKV) ? ld_cg(A.nd + (size_t)ND_L_SLOT * ND_STRIDE + rv.z) : NOSLOT;
    uint32_t rslot = (has && !sr && rv.w != NOTOKV) ? ld_cg(A.nd + (size_t)ND_R_SLOT * ND_STRIDE + rv.w) : NOSLOT;
    bool hl = has && lslot != NOSLOT && t.occ_len[lslot];
    bool hr = has && rslot != NOSLOT && t.occ_len[rslot];
    const unsigned long long il = agg_cursor(t, lslot, hl);
    const unsigned long long ir = agg_cursor(t, rslot, hr);
    if (hl) A.pool[il] = lpos;
    if (hr) A.pool[ir] = p;
  }
  if (!stage) return;
  __syncthreads();
  for (uint32_t e = threadIdx.x; e < 2u * R_STAGE_T; e += blockDim.x) {
    const uint32_t v = scnt[e];
    if (!v) continue;
    scnt[e] = 0;
    const uint32_t side = e >= R_STAGE_T ? 1u : 0u, tok = e - side * R_STAGE_T;
    const uint32_t s = ld_cg(A.nd + (size_t)(side ? ND_R_SLOT : ND_L_SLOT) * ND_STRIDE + tok);
    sbase[e] = (s != NOSLOT && t.occ_len[s]) ? t.occ_start.get(s) + atomicAdd(t.occ_fill + s, v) : FILL_NONE;
  }
  __syncthreads();
  for (uint32_t i = vt; i < round; i += nvt) {
    const bool has = i < n_sites;
    const uint4 rv = has ? ld_cg4(reinterpret_cast<const uint4*>(sites) + i) : make_uint4(0, NOPOS, NOTOKV, NOTOKV);
    const bool sl = has && rv.z < R_STAGE_T, sr = has && rv.w < R_STAGE_T;
    const uint32_t kl = agg_smem_ticket(scnt, rv.z, sl);
    const uint32_t kr = agg_smem_ticket(scnt, R_STAGE_T + rv.w, sr);
    const unsigned long long bl = sl ? sbase[rv.z] : FILL_NONE, br = sr ? sbase[R_STAGE_T + rv.w] : FILL_NONE;
    if (bl != FILL_NONE) A.pool[bl + kl] = rv.y;
    if (br != FILL_NONE) A.pool[br + kr] = rv.x;
  }
  __syncthreads();
  for (uint32_t e = threadIdx.x; e < 6u * R_STAGE_T; e += blockDim.x) stage[e] = 0;
  __syncthreads();
}

__device__ __forceinline__ void phase_apply(const ApplyArgs& A, uint32_t a, uint32_t b, uint32_t c, uint32_t n_sites,
                                            bool zero_count, uint32_t bid, uint32_t nblk) {
  if (zero_count && bid == 0 && threadIdx.x == 0) {
    uint32_t s = tbl_find(A.t, pair_key(a, b));
    if (s != NOSLOT) A.t.cnt[s] = 0;  // every counted occurrence was replaced
  }
  phase_fill(A, n_sites, bid * blockDim.x + threadIdx.x, nblk * blockDim.x);
  phase_rewrite(A, c, n_sites, bid * blockDim.x + threadIdx.x, nblk * blockDim.x);
}

// ---- stand-alone K3 kernels (applyMerge / restoreMerge one at a time) ----
__global__ void __launch_bounds__(256) k_sites(ApplyArgs A, uint32_t a, uint32_t b, uint32_t c) {
  if (blockIdx.x == 0 && threadIdx.x == 0) A.len16[c] = A.len16[a] + A.len16[b];  // chars = a.chars + b.chars (:318)
  phase_sites(A, a, b, c, 0, tbl_find(A.t, pair_key(a, b)), blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
}

__global__ void __launch_bounds__(256) k_alloc_new(ApplyArgs A, uint32_t c, uint32_t max_length, int hot_valid, uint32_t* __restrict__ hot,
                                                    uint32_t hot_cap, unsigned long long pool_cap) {
  phase_new_pairs(A, c, A.len16, max_length, hot_valid, hot, hot_cap, pool_cap, false, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
}

__global__ void __launch_bounds__(256) k_apply(ApplyArgs A, uint32_t a, uint32_t b, uint32_t c) {
  phase_apply(A, a, b, c, A.st->n_sites[0], true, blockIdx.x, gridDim.x);
}

// ------------------------------------------------------------------------------------------------
// mergeUntil (core.ts:365-383) as ONE persistent cooperative kernel: every block runs the same loop,
// phases are separated by a grid barrier (2 per merge), every block takes the same exit decision from
// the same published state.  The host is only needed to grow buffers or rebuild the hot list.
//
//   decide(t)                      fold the arg-max partials; same winner, same status in every block
//   P1(t)  ||  fill(t-1)           sites + count deltas of merge t; the occurrence lists of the pairs BORN by merge t-1 are
//                                  written next to it (software pipelining: nothing before P1(t+1) reads those lists, unless
//                                  the winner of t contains the token merge t-1 created, or a tie must be broken by position
//                                  -- then fill(t-1) is finished, with a barrier of its own, first)
//   ---- barrier ----
//   P2(t)                          born pairs enter the table / get list space / join the hot list and the arg-max, the corpus
//                                  is rewritten, the arg-max runs over the pairs that were already hot -> partials
//   ---- barrier ----
// ------------------------------------------------------------------------------------------------
#ifndef BPE_ML_THREADS
#define BPE_ML_THREADS 512
#endif
constexpr int ML_THREADS = BPE_ML_THREADS;
constexpr int ML_MIN_BLOCKS = ML_THREADS >= 1024 ? 1 : 2;

struct LoopArgs {
  ApplyArgs A;
  unsigned long long pool_cap;  // cells of the occurrence pool
  uint32_t len16_cap;
  uint32_t* hot;
  uint32_t hot_cap;
  uint32_t hot_limit;  // rebuild the hot list with a higher threshold once it would pass this many entries
  uint32_t* cands;
  uint32_t cand_cap;
  Best* partials;
  uint32_t* partial_keys;       // key (a << 16 | b) of partials[i].slot: the decision does not have to go back to the table for it
  unsigned long long* barrier;  // arrival counter, zeroed before the launch
  MergeRec* log;       // device merge log for this launch
  uint32_t log_cap;    // max merges this launch may apply
  uint32_t max_length;
  uint32_t min_weight;
  uint32_t max_tokens;
  uint32_t tbl_cap;
  SiteRec* sites2;     // second site buffer (capacity A.sites_cap): merges alternate, so that the list filling of merge t
                       // can run next to the site pass of merge t+1
  // replay mode (batched restoreMerge, core.ts:477-494): the winners are GIVEN -- (a,b) of merge i at replay[2i..2i+1]
  // -- instead of found by the arg-max; the hot list is neither read nor fed
  const int32_t* replay;
  // how the 16 warps of a block share the latency-bound phases of small merges (tuning knobs, defaults in loop_args, bpe_b200.cu):
  // P1: p1_sites warps walk the sites, the others fill the previous merge's lists and prefetch; P2: p2_new warps enter the
  // born pairs, p2_rw warps rewrite the corpus, the others run the arg-max over the old hot pairs
  uint32_t p1_sites, p2_new, p2_rw;
  uint32_t bar_ns;  // longest back-off of a barrier poll
  int prefetch;  // speculative L2 prefetch of the sites of this many runner-ups (prefetch_runner_up); BPE_LOOP_PREFETCH=0..2
  uint32_t stage_min;  // a merge whose occurrence list is longer stages its frequent neighbours' deltas per block (R_STAGE_T);
                       // k_merge_loop and k_merge_rounds, BPE_BLOCK_CELLS_MIN_SITES
};

// Grid barrier for the co-resident (cooperative) launch.  The arrival counter lives in its own 128-byte line, away
// from the DevState counters the phases hit with atomics, and pollers back off so that they do not saturate the
// L2 slice that owns it.
__device__ __forceinline__ unsigned long long now_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

__device__ __forceinline__ void grid_barrier(unsigned long long* ctr, unsigned long long target, uint32_t max_ns = 256) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(ctr, 1ull);
    uint32_t ns = 32;
    while (ld_volatile_u64(ctr) < target) {
      __nanosleep(ns);
      if (ns < max_ns) ns <<= 1;
    }
    __threadfence();
  }
  __syncthreads();
}

// Speculation: the runner-up of a decision is the most likely next winner (its count only changes when it neighbours a site
// of the current merge; 97.6 % of the cfg3 winners are pairs that existed before the previous merge).  While a block walks
// the sites of the current merge, its spare warps pull the corpus lines around the runner-up's occurrences into L2, so that
// the next site pass -- a chain of dependent loads -- finds them there instead of in DRAM.  Hints only: nothing depends on them.
__device__ __forceinline__ void prefetch_runner_up(const LoopArgs& L, uint32_t winner_slot, uint32_t nblk, uint32_t vt, uint32_t nvt) {
  const PairTable& t = L.A.t;
  uint32_t skip = winner_slot;
  for (int cand = 0; cand < L.prefetch; cand++) {  // the best L.prefetch candidates below the winner
    Best r{0ull, NOSLOT, 0};
    for (uint32_t i = lane_id(); i < nblk; i += 32) {
      Best pb{ld_cg(&L.partials[i].primary), ld_cg(&L.partials[i].slot), 1};
      if (pb.slot != winner_slot && pb.slot != skip && pb.slot != NOSLOT) r = best_merge(r, pb);
    }
    r = best_warp_reduce(r);
    if (!r.primary || r.slot == NOSLOT) return;
    skip = r.slot;
    const unsigned long long start = t.occ_start.get(r.slot);
    const uint32_t len = t.occ_len[r.slot];
    if (len > 32768u) continue;  // a merge of that size is throughput bound
    for (uint32_t i = vt; i < len; i += nvt) {
      const uint32_t p = ld_cg(L.A.pool + start + i);
      if (p >= L.A.n) continue;
      const uint32_t* q = L.A.slots + p;  // the site, the token on its left, the two tokens on its right
      prefetch_l2(q);
      if (p >= 16u) prefetch_l2(q - 16);
      if (p + 24u < L.A.n) prefetch_l2(q + 24);
    }
  }
}

__global__ void k_loop_prepare(DevState* st, uint32_t n_tokens, unsigned long long* barrier) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    st->status = LOOP_RUNNING;
    *barrier = 0;
    st->n_tokens = n_tokens;
    st->iters_done = 0;
    st->n_sites[0] = st->n_sites[1] = 0;
    st->n_new[0] = st->n_new[1] = 0;
    st->n_cand = 0;
    st->blocks_done = 0;
    st->tie_pos = ~0ull;
    st->n_touched[0] = st->n_touched[1] = 0;
    st->n_out = 0;
    st->mg_abort = 0;
  }
}

__global__ void __launch_bounds__(ML_THREADS, ML_MIN_BLOCKS) k_merge_loop(LoopArgs L) {
  __shared__ Best s_best[ML_THREADS / 32];
  __shared__ uint32_t s_max[32];
  __shared__ __align__(8) uint32_t s_stage[LS_ROWS * R_STAGE_T];  // loop_flush_stage leaves it zero (phase_fill: u64 rows)
  for (uint32_t i = threadIdx.x; i < LS_ROWS * R_STAGE_T; i += blockDim.x) s_stage[i] = 0;
  const ApplyArgs& A = L.A;
  DevState* st = A.st;
  const PairTable& t = A.t;
  const uint32_t bid = blockIdx.x, nblk = gridDim.x;
  unsigned long long epoch = 0;
  const uint32_t n_tokens0 = ld_cg(&st->n_tokens);
  const uint32_t thresh = ld_cg(&st->hot_thresh);

  const bool replay = L.replay != nullptr;
  __shared__ uint32_t s_rslot, s_wkey;

  // first arg-max partials
  if (bid == 0 && threadIdx.x == 0) st->snap_err = st->err;
  if (!replay) {
    Best v = best_block_reduce(argmax_stripe(t, A.len16, L.max_length, 1, L.hot, ld_cg(&st->hot_n), bid, nblk), s_best);
    if (threadIdx.x == 0) {
      L.partials[bid] = v;
      L.partial_keys[bid] = v.primary ? t.keys[v.slot] : 0u;
    }
  }
  grid_barrier(L.barrier, ++epoch * nblk, L.bar_ns);

  const bool prof = (bid == 0 && threadIdx.x == 0);
  unsigned long long tp0 = prof ? now_ns() : 0, tp1;
#define PROF(i)                      \
  if (prof) {                        \
    tp1 = now_ns();                  \
    st->prof_ns[i] += tp1 - tp0;     \
    tp0 = tp1;                       \
  }
  const uint32_t gt = bid * blockDim.x + threadIdx.x, gn = nblk * blockDim.x;
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
  // deferred phase_fill: the sites of the previous merge whose new adjacencies are not in their lists yet
  uint32_t fill_n = 0;
  const SiteRec* fill_sites = nullptr;
  for (uint32_t it = 0;; it++) {
    const uint32_t par = it & 1u;
    SiteRec* const my_sites = par ? L.sites2 : A.sites;
    // ---- every block folds the partials and takes the same decision ----
    // n_keys, pool_cursor and hot_n only change in P2, err is snapshot by block 0 in P2: all stable here
    Best w{0ull, NOSLOT, 0};
    uint32_t status = LOOP_RUNNING;
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
    if (ld_cg(&st->snap_err)) status = LOOP_ERROR;
    else if (replay) status = (it >= L.log_cap) ? LOOP_LIMIT : (c >= L.max_tokens ? LOOP_NEED_HOST : LOOP_RUNNING);
    else if (!w.primary) status = (thresh <= 1) ? LOOP_EMPTY : LOOP_NEED_REBUILD;
    else if (wcnt < thresh) status = LOOP_NEED_REBUILD;
    else if (wcnt < L.min_weight) status = LOOP_DONE;  // core.ts:313
    else if (it >= L.log_cap) status = LOOP_LIMIT;
    else if (c >= L.max_tokens) status = LOOP_NEED_HOST;
    PROF(0)
    if (status == LOOP_RUNNING && w.mult > 1) {
      // tie on (weight, a.index+b.index): the pair whose last counted occurrence comes first wins (core.ts:294-305)
      if (w.mult > L.cand_cap) status = LOOP_NEED_HOST;
      else {
        if (fill_n) {  // the tie-break reads occurrence lists: those of the last merge must be complete
          phase_fill(A, fill_n, gt, gn, fill_sites, fill_n > L.stage_min ? s_stage : nullptr);
          fill_n = 0;
          grid_barrier(L.barrier, ++epoch * nblk, L.bar_ns);
        }
        phase_collect(t, A.len16, L.max_length, 1, L.hot, hot_pre, w.primary, L.cands, L.cand_cap, st, bid, nblk);
        grid_barrier(L.barrier, ++epoch * nblk, L.bar_ns);
        phase_tie(A.slots, A.n, t, A.pool, L.cands, ld_cg(&st->n_cand), st, s_max, bid, nblk);
        grid_barrier(L.barrier, ++epoch * nblk, L.bar_ns);
        unsigned long long tp = ld_cg(&st->tie_pos);
        if (tp == ~0ull) status = LOOP_ERROR;
        else {
          uint32_t s = (uint32_t)(tp & 0xFFFFFFFFu);
          uint32_t key = t.keys[s];
          w.slot = s;
          wa = key >> 16;
          wb = key & 0xFFFFu;
        }
      }
    }
    PROF(7)
    if (status == LOOP_RUNNING) {
      // capacity the host guarantees: sites = wcnt; new pairs are (x,c) or (c,y), so at most 2*(c+1) of them and
      // at most 2 per site; new list cells <= 2 per site
      unsigned long long new_keys = min(2ull * wcnt + 2ull, 2ull * (c + 1ull) + 2ull);
      if ((unsigned long long)ld_cg(&st->n_keys) + new_keys > (unsigned long long)(L.tbl_cap >> 1)) status = LOOP_NEED_HOST;
      else if ((unsigned long long)ld_cg(&st->pool_cursor) + 2ull * wcnt > L.pool_cap) status = LOOP_NEED_HOST;
      else if (wcnt > A.sites_cap || new_keys > A.new_cap) status = LOOP_NEED_HOST;
      else if (!replay && (unsigned long long)hot_pre + new_keys > min(L.hot_cap, L.hot_limit)) status = LOOP_NEED_REBUILD;
      else if (c + 1 > L.len16_cap) status = LOOP_NEED_HOST;
    }
    if (status != LOOP_RUNNING) {
      if (fill_n) phase_fill(A, fill_n, gt, gn, fill_sites, fill_n > L.stage_min ? s_stage : nullptr);  // the kernel leaves every list complete
      if (bid == 0 && threadIdx.x == 0) {
        st->status = status;
        st->iters_done = it;
        st->n_tokens = n_tokens0 + it;
        if (replay) {
          st->best_primary = 0;
          st->best_cnt = wcnt;  // what the host must make room for
          st->best_mult = 1;
        } else {
          publish_best(t, st, w);
        }
        st->n_cand = 0;
        st->tie_pos = ~0ull;
      }
      return;
    }
    if (fill_n && it && (wa == c - 1u || wb == c - 1u)) {
      // the winner was born by the previous merge: its list is exactly what fill(t-1) still has to write
      phase_fill(A, fill_n, gt, gn, fill_sites, fill_n > L.stage_min ? s_stage : nullptr);
      fill_n = 0;
      grid_barrier(L.barrier, ++epoch * nblk, L.bar_ns);
    }
    // ---- P1: sites + deltas, next to the list filling of the previous merge ----
    if (bid == 0 && threadIdx.x == 0) {
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
      if (w.mult > 1) st->tie_breaks++;
    }
    if (fill_n <= 8192u && wcnt <= 16384u && blockDim.x == 512u) {
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
    if (prof) {
      st->bucket_ns[bkt][0] += now_ns() - tp0;
      st->bucket_ns[bkt][3] += 1;
    }
#endif
    PROF(1)
    grid_barrier(L.barrier, ++epoch * nblk, L.bar_ns);
    PROF(2)
    // ---- P2: the born pairs (table, list space, hot list, arg-max), the corpus rewrite, the arg-max over the old hot pairs ----
    if (bid == 0 && threadIdx.x == 0) {
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
    if (prof) st->bucket_ns[bkt][1] += now_ns() - tp0;
#endif
    PROF(3)
    grid_barrier(L.barrier, ++epoch * nblk, L.bar_ns);
    PROF(4)
  }
#undef PROF
}

// ------------------------------------------------------------------------------------------------
// corpus read-back: compact ID slots of a slot range (two passes: count per block, then scatter)
// ------------------------------------------------------------------------------------------------
constexpr int CP_THREADS = 256;
constexpr int CP_ITEMS = 8;  // slots per thread
constexpr int CP_TILE = CP_THREADS * CP_ITEMS;

__global__ void __launch_bounds__(CP_THREADS) k_count_ids(const uint32_t* __restrict__ slots, uint64_t begin,
                                                           uint64_t end, uint32_t* __restrict__ block_counts) {
  __shared__ uint32_t s_w[CP_THREADS / 32];
  uint64_t base = begin + (uint64_t)blockIdx.x * CP_TILE;
  uint32_t c = 0;
#pragma unroll
  for (int j = 0; j < CP_ITEMS; j++) {
    uint64_t p = base + (uint64_t)j * CP_THREADS + threadIdx.x;
    if (p < end && slot_is_id(__ldg(slots + p))) c++;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
  if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t s = 0;
    for (int i = 0; i < CP_THREADS / 32; i++) s += s_w[i];
    block_counts[blockIdx.x] = s;
  }
}

// single-block exclusive scan of up to a few million block counts (u32 -> u64 offsets)
__global__ void __launch_bounds__(1024) k_scan_counts(const uint32_t* __restrict__ in, uint64_t* __restrict__ out,
                                                       uint32_t n) {
  __shared__ uint64_t s_part[1024];
  uint32_t per = (n + 1023) / 1024;
  uint32_t lo = min(n, threadIdx.x * per), hi = min(n, lo + per);
  uint64_t s = 0;
  for (uint32_t i = lo; i < hi; i++) s += in[i];
  s_part[threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint64_t acc = 0;
    for (int i = 0; i < 1024; i++) {
      uint64_t v = s_part[i];
      s_part[i] = acc;
      acc += v;
    }
    out[n] = acc;
  }
  __syncthreads();
  uint64_t acc = s_part[threadIdx.x];
  for (uint32_t i = lo; i < hi; i++) {
    out[i] = acc;
    acc += in[i];
  }
}

__global__ void __launch_bounds__(CP_THREADS) k_compact_ids(const uint32_t* __restrict__ slots, uint64_t begin,
                                                             uint64_t end, const uint64_t* __restrict__ block_off,
                                                             int32_t* __restrict__ out) {
  __shared__ uint32_t s_w[CP_THREADS / 32];
  uint64_t base = begin + (uint64_t)blockIdx.x * CP_TILE;
  uint64_t off = block_off[blockIdx.x];
  uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // order-preserving: item j of the tile is slot base + j*CP_THREADS + tid, processed j-major
  for (int j = 0; j < CP_ITEMS; j++) {
    uint64_t p = base + (uint64_t)j * CP_THREADS + threadIdx.x;
    uint32_t w = (p < end) ? __ldg(slots + p) : mk_hole();
    bool is = slot_is_id(w);
    uint32_t m = __ballot_sync(0xFFFFFFFFu, is);
    if (lane == 0) s_w[warp] = __popc(m);
    __syncthreads();
    uint32_t before = 0, total = 0;
    for (int i = 0; i < CP_THREADS / 32; i++) {
      uint32_t v = s_w[i];
      if (i < (int)warp) before += v;
      total += v;
    }
    if (is) out[off + before + __popc(m & ((1u << lane) - 1))] = (int32_t)slot_val(w);
    off += total;
    __syncthreads();
  }
}

// number of ID slots in [begin, pos) for each document boundary `pos`
__global__ void k_doc_ranks(const uint32_t* __restrict__ slots, uint64_t begin, const uint64_t* __restrict__ block_off,
                            const int64_t* __restrict__ doc_pos, int64_t n_bounds, int64_t* __restrict__ out_offsets) {
  // one warp per boundary
  int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  uint32_t lane = threadIdx.x & 31;
  int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t d = wid; d < n_bounds; d += nw) {
    uint64_t pos = (uint64_t)doc_pos[d];
    uint64_t blk = (pos - begin) / CP_TILE;
    uint64_t tile0 = begin + blk * CP_TILE;
    uint32_t c = 0;
    for (uint64_t p = tile0 + lane; p < pos; p += 32)
      if (slot_is_id(__ldg(slots + p))) c++;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
    if (lane == 0) out_offsets[d] = (int64_t)(block_off[blk] + c);
  }
}

// pair-count dump (debug / parity)
__global__ void k_dump_pairs(PairTable t, int32_t* __restrict__ a, int32_t* __restrict__ b, int64_t* __restrict__ cnt,
                             uint32_t cap, uint32_t* __restrict__ n_out) {
  uint32_t tcap = t.mask + 1;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < tcap; i += gridDim.x * blockDim.x) {
    uint32_t key = t.keys[i];
    if (key == EMPTY_KEY) continue;
    uint32_t c = t.cnt[i];
    if (c == 0) continue;
    uint32_t k = atomicAdd(n_out, 1u);
    if (k < cap) {
      a[k] = (int32_t)(key >> 16);
      b[k] = (int32_t)(key & 0xFFFFu);
      cnt[k] = (int64_t)c;
    }
  }
}

}  // namespace bpe
