// common.cuh -- corpus slot encoding, neighbour walks and the pair table.
//
// Device layout of corpus_in_code (reference core.ts:106), designed for merge-in-place:
//   one u32 "slot" per ORIGINAL position (= per character ingested by addToCorpus).  A token lives in
//   the slot of its first character; merging (a at p, b at q) -> c rewrites slot p and turns the
//   slots of b into filler, so positions never move and a position is a monotone scan-order key
//   (the reference's tie-break needs the scan position of a pair's last counted occurrence,
//   core.ts:294-305; merging never reorders tokens).
//
//   bit 31      DOCSTART  first token of a document (documents are merge-isolation units,
//                         core.ts:265-267).  Only ever set on ID slots.
//   bits 30:29  kind      ID   token index in bits 28:0, a token starts here
//                         SPAN second slot of a token covering `val` >= 3 slots
//                         BACK last slot of a token covering val+1 >= 2 slots (val = distance to its start)
//                         HOLE interior filler
//   Only the second and the last slot of a token are ever read as markers, so interior slots may
//   hold stale markers (never a stale ID).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace bpe {

constexpr uint32_t DOCSTART = 0x80000000u;
constexpr uint32_t KIND_SHIFT = 29;
constexpr uint32_t KIND_ID = 0u, KIND_SPAN = 1u, KIND_BACK = 2u, KIND_HOLE = 3u;
constexpr uint32_t VAL_MASK = 0x1FFFFFFFu;
constexpr uint32_t NOPOS = 0xFFFFFFFFu;
constexpr uint32_t NOSLOT = 0xFFFFFFFFu;
constexpr uint32_t EMPTY_KEY = 0xFFFFFFFFu;
constexpr int NOTOK = -1;

__host__ __device__ __forceinline__ uint32_t slot_kind(uint32_t v) { return (v >> KIND_SHIFT) & 3u; }
__host__ __device__ __forceinline__ uint32_t slot_val(uint32_t v) { return v & VAL_MASK; }
__host__ __device__ __forceinline__ bool slot_is_id(uint32_t v) { return slot_kind(v) == KIND_ID; }
__host__ __device__ __forceinline__ uint32_t mk_span(uint32_t s) { return (KIND_SPAN << KIND_SHIFT) | s; }
__host__ __device__ __forceinline__ uint32_t mk_back(uint32_t d) { return (KIND_BACK << KIND_SHIFT) | d; }
__host__ __device__ __forceinline__ uint32_t mk_hole() { return (KIND_HOLE << KIND_SHIFT); }
__host__ __device__ __forceinline__ uint32_t pair_key(uint32_t a, uint32_t b) { return (a << 16) | b; }

// Corpus slots are rewritten by other SMs during the SAME launch (persistent mergeUntil kernel), so they are never
// read through the non-coherent path (no __ldg / ld.global.nc).  Plain loads may be served by L1: within a phase
// nobody rewrites what a thread reads, and every grid barrier ends with a gpu-scope fence (which invalidates L1)
// before the next phase starts -- the same contract cooperative-groups grid.sync() gives.
// Control words polled or read right after a barrier use ld_cg (L2).
__device__ __forceinline__ uint32_t ld_slot(const uint32_t* p) { return *p; }
__device__ __forceinline__ uint4 ld_slots4(const uint32_t* p) { return *reinterpret_cast<const uint4*>(p); }
__device__ __forceinline__ uint32_t ld_cg(const uint32_t* p) { return __ldcg(p); }
__device__ __forceinline__ unsigned long long ld_cg(const unsigned long long* p) { return __ldcg(p); }
__device__ __forceinline__ uint4 ld_cg4(const uint4* p) { return __ldcg(p); }
__device__ __forceinline__ unsigned long long ld_volatile_u64(const unsigned long long* p) {
  return *reinterpret_cast<const volatile unsigned long long*>(p);
}

// Position of the token after the one starting at p, or n when there is none in the array.
__device__ __forceinline__ uint32_t next_pos(const uint32_t* slots, uint32_t n, uint32_t p) {
  uint32_t q = p + 1;
  if (q >= n) return n;
  uint32_t w = ld_slot(slots + q);
  uint32_t k = slot_kind(w);
  if (k == KIND_ID) return q;
  if (k == KIND_BACK) return q + 1;  // span-2 token: its second slot is also its last
  return p + slot_val(w);            // SPAN
}

// Token index of the right neighbour of the token at p inside the same document, or NOTOK.
__device__ __forceinline__ int right_token(const uint32_t* slots, uint32_t n, uint32_t p, uint32_t* pos) {
  uint32_t q = next_pos(slots, n, p);
  *pos = q;
  if (q >= n) return NOTOK;
  uint32_t w = ld_slot(slots + q);
  if (w & DOCSTART) return NOTOK;
  return (int)slot_val(w);
}

// Token index of the left neighbour of the token at p (whose slot value is `wp`), or NOTOK.
__device__ __forceinline__ int left_token(const uint32_t* slots, uint32_t p, uint32_t wp, uint32_t* pos) {
  if ((wp & DOCSTART) || p == 0) {
    *pos = NOPOS;
    return NOTOK;
  }
  uint32_t w = ld_slot(slots + p - 1);
  uint32_t l = p - 1;
  if (slot_kind(w) == KIND_BACK) {
    l = p - 1 - slot_val(w);
    w = ld_slot(slots + l);
  }
  *pos = l;
  return (int)slot_val(w);
}

// Number of consecutive tokens equal to `t` immediately to the left of position p (same document).
__device__ __forceinline__ uint32_t run_left(const uint32_t* slots, uint32_t p, uint32_t wp, int t) {
  uint32_t k = 0;
  for (;;) {
    uint32_t l;
    int x = left_token(slots, p, wp, &l);
    if (x != t) return k;
    k++;
    p = l;
    wp = ld_slot(slots + l);
  }
}

// Number of consecutive tokens equal to `t` immediately to the right of the token at p.
__device__ __forceinline__ uint32_t run_right(const uint32_t* slots, uint32_t n, uint32_t p, int t) {
  uint32_t k = 0;
  for (;;) {
    uint32_t q;
    int y = right_token(slots, n, p, &q);
    if (y != t) return k;
    k++;
    p = q;
  }
}

// ---- pair table: open addressing, linear probing, keys never deleted --------------------------
// (the reference rebuilds a Map<Token, Map<Token, number>> on every findNextMerge, core.ts:259;
//  here the histogram persists and is updated by count deltas.)
// One array per field (TBL_STRIDE = 1).  A 32-byte entry per slot (TBL_STRIDE = 8: key, count and list fields of a pair
// in one DRAM sector) was measured on the 1 GB corpus and LOST 8 %: linear probing then pays one sector per probe
// instead of one per eight, and the hot-list / threshold scans read four times the bytes.  TblField keeps the
// `t.cnt[i]` / `t.cnt + i` notation either way.
#ifndef BPE_TBL_STRIDE
#define BPE_TBL_STRIDE 1
#endif
constexpr uint32_t TBL_STRIDE = BPE_TBL_STRIDE;  // u32 words between consecutive slots of one field
struct TblField {
  uint32_t* p;
  __host__ __device__ __forceinline__ uint32_t& operator[](uint32_t i) const { return p[(size_t)i * TBL_STRIDE]; }
  __host__ __device__ __forceinline__ uint32_t* operator+(uint32_t i) const { return p + (size_t)i * TBL_STRIDE; }
};
// Where a pair's occurrence list starts in the pool.  The pool holds up to 3 cells per corpus position, so on one engine of
// more than ~1.4 G positions its cell indices pass 2^32: the start is 64-bit, one 8-byte word per slot (the words 6..7 of a
// 32-byte entry when TBL_STRIDE = 8).  Kernels read and write it through get / set only and never see the layout.
struct TblStart {
  unsigned long long* p;
  static constexpr uint32_t STRIDE = TBL_STRIDE == 1 ? 1u : TBL_STRIDE / 2u;  // u64 words between consecutive slots
  __host__ __device__ __forceinline__ unsigned long long get(uint32_t i) const { return p[(size_t)i * STRIDE]; }
  __host__ __device__ __forceinline__ void set(uint32_t i, unsigned long long v) const { p[(size_t)i * STRIDE] = v; }
  __host__ __device__ __forceinline__ const void* addr(uint32_t i) const { return p + (size_t)i * STRIDE; }  // (prefetch)
};
struct PairTable {
  TblField keys;       // pair_key(a,b) or EMPTY_KEY
  TblField cnt;        // counted occurrences (run-parity rule of core.ts:285-290 applied)
  TblStart occ_start;  // occurrence list = pool[occ_start .. occ_start+occ_len)
  TblField occ_len;    //   every adjacency (a,b) born in the iteration that created the pair
  TblField occ_fill;   //   scatter cursor
  uint32_t mask;       // capacity - 1
  uint32_t shift;      // 32 - log2(capacity)
};

__device__ __forceinline__ uint32_t tbl_hash(const PairTable& t, uint32_t key) { return (key * 0x9E3779B1u) >> t.shift; }

__device__ __forceinline__ uint32_t tbl_find(const PairTable& t, uint32_t key) {
  uint32_t i = tbl_hash(t, key);
  for (uint32_t probes = 0; probes <= t.mask; probes++) {
    uint32_t k = t.keys[i];
    if (k == key) return i;
    if (k == EMPTY_KEY) return NOSLOT;
    i = (i + 1) & t.mask;
  }
  return NOSLOT;
}

__device__ __forceinline__ uint32_t tbl_find_or_insert(const PairTable& t, uint32_t key, uint32_t* n_keys) {
  uint32_t i = tbl_hash(t, key);
  for (uint32_t probes = 0; probes <= t.mask; probes++) {
    uint32_t k = t.keys[i];
    if (k == key) return i;
    if (k == EMPTY_KEY) {
      uint32_t old = atomicCAS(t.keys + i, EMPTY_KEY, key);
      if (old == EMPTY_KEY) {
        atomicAdd(n_keys, 1u);
        return i;
      }
      if (old == key) return i;
    }
    i = (i + 1) & t.mask;
  }
  return NOSLOT;  // table full
}

// Same as tbl_find_or_insert, but the caller accounts for the new key (one n_keys atomic per warp / block instead of
// one per key: thousands of atomics on ONE address serialise in L2 and used to dominate a merge iteration).
__device__ __forceinline__ uint32_t tbl_find_or_insert_ex(const PairTable& t, uint32_t key, bool* inserted) {
  *inserted = false;
  uint32_t i = tbl_hash(t, key);
  for (uint32_t probes = 0; probes <= t.mask; probes++) {
    uint32_t k = t.keys[i];
    if (k == key) return i;
    if (k == EMPTY_KEY) {
      uint32_t old = atomicCAS(t.keys + i, EMPTY_KEY, key);
      if (old == EMPTY_KEY) {
        *inserted = true;
        return i;
      }
      if (old == key) return i;
    }
    i = (i + 1) & t.mask;
  }
  return NOSLOT;  // table full
}

// error flags raised by kernels (checked by the host after each phase)
constexpr uint32_t ERR_TABLE_FULL = 1u, ERR_MISSING_KEY = 2u, ERR_POOL_FULL = 4u, ERR_SITE_OVERFLOW = 8u,
                   ERR_SPAN_OVERFLOW = 16u, ERR_CAND_OVERFLOW = 32u, ERR_HOT_OVERFLOW = 64u, ERR_COUNT_OVERFLOW = 4096u;

}  // namespace bpe
