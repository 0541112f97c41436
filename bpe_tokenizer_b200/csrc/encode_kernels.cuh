// encode_kernels.cuh -- K4 (apply the learned merge list to new text) and K5 (vector-index map).
//
// Reference: encodeToCode applies every merge in training order with replaceAll over the whole
// string (core.ts:404-406).  Because a merge of rank r can only create pairs of rank > r, that is
// equivalent to "repeat: take the lowest-rank pair present, replace all its occurrences left to right
// without overlap" (SURVEY.md A.4(i), cross-checked against the literal form in tests).
//
// One warp owns one document (tokens + cached pair ranks in shared memory, global scratch above ENC_WARP_MAX
// tokens).  Instead of one round per distinct merge, every round merges ALL pairs that are provably merged as they
// stand by the sequential process (see below), then compacts the document in place.
#pragma once
#include "common.cuh"

namespace bpe {

constexpr uint32_t RK_NONE = 0xFFFFFFFFu;
constexpr unsigned long long MT_EMPTY = ~0ull;
constexpr int ENC_WARPS = 8;
constexpr int ENC_THREADS = ENC_WARPS * 32;
constexpr int ENC_WARP_MAX = 512;  // tokens per document handled in shared memory (10 B per token)

struct MergeTable {
  const unsigned long long* ent;  // (pair_key << 32) | (rank << 16) | c
  uint32_t mask;
  uint32_t shift;
};

__device__ __forceinline__ uint32_t mt_lookup(const MergeTable& mt, uint32_t a, uint32_t b) {
  uint32_t key = pair_key(a, b);
  uint32_t h = (key * 0x9E3779B1u) >> mt.shift;
  for (;;) {
    unsigned long long e = __ldg(mt.ent + h);
    if ((uint32_t)(e >> 32) == key) return (uint32_t)e;
    if (e == MT_EMPTY) return RK_NONE;
    h = (h + 1) & mt.mask;
  }
}

// ---- which pairs may be merged in the same round ---------------------------------------------------
// The sequential process (core.ts:404-406) merges pair (x,y) of rank r at "time" r iff both tokens are still
// there.  x can only disappear earlier by being consumed as the RIGHT operand of a lower-rank rule, y as the LEFT
// operand.  Let
//   SL[i] = largest r such that token i is certainly not consumed from its left strictly before time r
//         = max(minAsRight[tok i], min(rank(i-1,i), SL[i-1])),   SL[0] = inf
//   SR[i] = max(minAsLeft[tok i],  min(rank(i,i+1), SR[i+1])),   SR[n-1] = inf
// (no rule can take it earlier, or the neighbouring pair fires no earlier and the neighbour itself is stable).
// A pair with r <= SL[i] and r <= SR[i+1] is merged by the sequential process exactly as it stands, so it can be
// merged now; merging early cannot enable anything earlier because every rule involving the new token has rank > r.
// Runs x x x ... (replaceAll parity, core.ts:285-290) need both run ends stable and the run unable to GROW at its
// left end before time r.  The lowest rank present always qualifies, so every round makes progress.
// SL and SR are prefix scans of clamp functions x -> max(lo, min(hi, x)), which compose into clamps: one
// warp-shuffle scan per 32 tokens.  After each round the document is compacted in place, so the work shrinks with
// the token count.  Prototype + fuzz against the literal oracle: tests/proto/proto_encode_safe.py.
constexpr uint32_t RK_DIRTY = 0xFFFFFFFEu;
constexpr uint32_t RINF = 0xFFFFu;

struct EncTables {
  MergeTable mt;
  const uint32_t* minlr;  // per token: (lowest rank with the token as LEFT operand << 16) | lowest rank as RIGHT operand
};

constexpr int ENC_WALK = 16;  // bound of the stability walks

// token j is not consumed from its left strictly before time r (see above); contiguous layout: neighbours are j-1, j+1
template <typename TokT>
__device__ __forceinline__ bool stable_left(const TokT* tok, const uint32_t* rk, const uint32_t* minlr, uint32_t j, uint32_t r) {
#pragma unroll 1
  for (int s = 0; s <= ENC_WALK; s++) {
    if (j == 0 || (__ldg(minlr + tok[j]) & 0xFFFFu) >= r) return true;
    if ((rk[j - 1] >> 16) < r) return false;
    j--;
  }
  return false;
}

template <typename TokT>
__device__ __forceinline__ bool stable_right(const TokT* tok, const uint32_t* rk, const uint32_t* minlr, uint32_t j, uint32_t n,
                                             uint32_t r) {
#pragma unroll 1
  for (int s = 0; s <= ENC_WALK; s++) {
    if (j + 1 >= n || (__ldg(minlr + tok[j]) >> 16) >= r) return true;
    if ((rk[j] >> 16) < r) return false;
    j++;
  }
  return false;
}

// TokT/StT: uint16_t in shared memory (n <= ENC_WARP_MAX), uint32_t in global scratch.
// take_g: per-position selection marks for the global-scratch path (the shared path keeps them in a register).
template <typename TokT, typename StT>
__device__ __forceinline__ uint32_t encode_doc(TokT* tok, uint32_t* rk, StT* sl, StT* sr, uint32_t* take_g, uint32_t n,
                                               const EncTables& T, uint32_t lane) {
  constexpr bool kSmem = sizeof(TokT) == 2;
  const MergeTable& mt = T.mt;
  for (uint32_t i = lane; i < n; i += 32) rk[i] = (i + 1 < n) ? mt_lookup(mt, tok[i], tok[i + 1]) : RK_NONE;
  __syncwarp();
  for (;;) {
    const uint32_t rows = (n + 31) >> 5;
    // lowest rank present: always mergeable (progress), and the loop ends when there is none
    uint32_t m = RK_NONE;
    for (uint32_t i = lane; i < n; i += 32) m = min(m, rk[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = min(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
    if (m == RK_NONE) break;
    const uint32_t gmin = m >> 16;
    // ---- select (read-only): bounded walks evaluate SL / SR lazily, "unknown" counts as unstable ----
    uint32_t mask = 0;  // bit row: position 32*row + lane is merged with its right neighbour
    for (uint32_t row = 0; row < rows; row++) {
      uint32_t i = (row << 5) + lane;
      bool take = false;
      if (i + 1 < n) {
        uint32_t r = rk[i] >> 16;
        if (r != RINF) {
          TokT x = tok[i];
          if (x != tok[i + 1]) {
            take = (r == gmin) || (stable_left<TokT>(tok, rk, T.minlr, i, r) && stable_right<TokT>(tok, rk, T.minlr, i + 1, n, r));
          } else {
            uint32_t s = i;
            while (s > 0 && tok[s - 1] == x) s--;
            if (((i - s) & 1u) == 0) {
              if (r == gmin) {
                take = true;
              } else {
                uint32_t e = i + 1;
                while (e + 1 < n && tok[e + 1] == x) e++;
                take = stable_left<TokT>(tok, rk, T.minlr, s, r) && (s == 0 || stable_left<TokT>(tok, rk, T.minlr, s - 1, r)) &&
                       stable_right<TokT>(tok, rk, T.minlr, e, n, r);
              }
            }
          }
        }
      }
      if (kSmem) mask |= (take ? 1u : 0u) << row;
      else if (i < n) take_g[i] = take ? 1u : 0u;
    }
    __syncwarp();
    // ---- apply + compact in place (rows in order: writes never pass the row being read) ----
    uint32_t wr = 0, carry_sel = 0;
    for (uint32_t row = 0; row < rows; row++) {
      uint32_t i = (row << 5) + lane;
      uint32_t t = 0, v = RK_NONE;
      bool take = false;
      if (i < n) {
        t = tok[i];
        v = rk[i];
        take = kSmem ? ((mask >> row) & 1u) != 0 : take_g[i] != 0;
      }
      uint32_t S = __ballot_sync(0xFFFFFFFFu, take);
      uint32_t removed = (S << 1) | carry_sel;
      bool keep = (i < n) && !((removed >> lane) & 1u);
      uint32_t K = __ballot_sync(0xFFFFFFFFu, keep);
      if (keep) {
        uint32_t j = wr + __popc(K & ((1u << lane) - 1u));
        tok[j] = (TokT)(take ? (v & 0xFFFFu) : t);
        rk[j] = take ? RK_DIRTY : v;
      }
      wr += __popc(K);
      carry_sel = S >> 31;
      __syncwarp();
    }
    n = wr;
    // ---- refresh the ranks of pairs that touch a new token ----
    for (uint32_t base = 0; base < n; base += 32) {
      uint32_t i = base + lane;
      uint32_t r = (i < n) ? rk[i] : RK_NONE;
      uint32_t rn = (i + 1 < n) ? rk[i + 1] : RK_NONE;
      __syncwarp();
      if (i < n && (r == RK_DIRTY || rn == RK_DIRTY)) rk[i] = (i + 1 < n) ? mt_lookup(mt, tok[i], tok[i + 1]) : RK_NONE;
      __syncwarp();
    }
  }
  return n;
}

// One warp per document.  out_tmp holds each document's tokens at the document's INPUT offset.
__global__ void __launch_bounds__(ENC_THREADS) k_encode(const int32_t* __restrict__ ids,
                                                         const int64_t* __restrict__ doc_off, int64_t n_docs,
                                                         EncTables T, int32_t* __restrict__ out_tmp,
                                                         uint32_t* __restrict__ out_len, uint32_t* __restrict__ g_tok,
                                                         uint32_t* __restrict__ g_sl, uint32_t* __restrict__ g_sr,
                                                         uint32_t* __restrict__ g_rk, uint32_t* __restrict__ g_take,
                                                         int only_marked) {
  __shared__ uint16_t s_tok[ENC_WARPS][ENC_WARP_MAX];
  __shared__ uint16_t s_sl[ENC_WARPS][ENC_WARP_MAX];
  __shared__ uint16_t s_sr[ENC_WARPS][ENC_WARP_MAX];
  __shared__ uint32_t s_rk[ENC_WARPS][ENC_WARP_MAX];
  uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int64_t wid = (int64_t)blockIdx.x * ENC_WARPS + warp;
  int64_t nw = (int64_t)gridDim.x * ENC_WARPS;
  int64_t base0 = doc_off[0];
  for (int64_t d = wid; d < n_docs; d += nw) {
    if (only_marked && out_len[d] != 0xFFFFFFFFu) continue;  // the lane path (encode_lanes.cuh) left this one
    int64_t s = doc_off[d], e = doc_off[d + 1];
    uint32_t n = (uint32_t)(e - s);
    const int32_t* src = ids + s;
    int32_t* dst = out_tmp + s;
    if (n <= ENC_WARP_MAX) {
      for (uint32_t i = lane; i < n; i += 32) s_tok[warp][i] = (uint16_t)__ldg(src + i);
      __syncwarp();
      n = encode_doc<uint16_t, uint16_t>(s_tok[warp], s_rk[warp], s_sl[warp], s_sr[warp], nullptr, n, T, lane);
      for (uint32_t i = lane; i < n; i += 32) dst[i] = (int32_t)s_tok[warp][i];
    } else {
      uint32_t* tok = g_tok + (s - base0);
      for (uint32_t i = lane; i < n; i += 32) tok[i] = (uint32_t)__ldg(src + i);
      __syncwarp();
      n = encode_doc<uint32_t, uint32_t>(tok, g_rk + (s - base0), g_sl + (s - base0), g_sr + (s - base0), g_take + (s - base0), n, T, lane);
      for (uint32_t i = lane; i < n; i += 32) dst[i] = (int32_t)tok[i];
    }
    if (lane == 0) out_len[d] = n;
    __syncwarp();
  }
}

// K5: gather each document's tokens to its final offset, mapping through to_vector_index
// (core.ts:434-442); a hole (-1) marks the document's first_bad and is emitted as -(index+1).
__global__ void __launch_bounds__(128) k_gather_map(const int32_t* __restrict__ out_tmp,
                                                     const int64_t* __restrict__ doc_off,
                                                     const uint64_t* __restrict__ out_off, int64_t n_docs,
                                                     const int32_t* __restrict__ tvi, int32_t n_tvi,
                                                     int32_t* __restrict__ out, int64_t* __restrict__ out_offsets,
                                                     int64_t* __restrict__ first_bad) {
  uint32_t lane = threadIdx.x & 31;
  int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t d = wid; d <= n_docs; d += nw) {
    if (d == n_docs) {
      if (lane == 0) out_offsets[d] = (int64_t)out_off[d];
      continue;
    }
    const int32_t* src = out_tmp + doc_off[d];
    uint64_t o = out_off[d];
    uint32_t n = (uint32_t)(out_off[d + 1] - o);
    uint32_t bad = 0xFFFFFFFFu;
    for (uint32_t i = lane; i < n; i += 32) {
      int32_t t = __ldg(src + i);
      int32_t v = t;
      if (tvi) {
        v = (t < n_tvi) ? __ldg(tvi + t) : -1;
        if (v < 0) {
          bad = min(bad, i);
          v = -(t + 1);
        }
      }
      out[o + i] = v;
    }
    if (first_bad) {
#pragma unroll
      for (int s = 16; s > 0; s >>= 1) bad = min(bad, __shfl_xor_sync(0xFFFFFFFFu, bad, s));
      if (lane == 0) first_bad[d] = (bad == 0xFFFFFFFFu) ? -1 : (int64_t)bad;
    }
    if (lane == 0) out_offsets[d] = (int64_t)o;
  }
}

// Ragged -> dense (bpe_pad_batch_dev): row d of out[n_docs x width] = the first min(len_d, width) values of document d, then
// `pad`.  One warp per row: the warp's loads and stores are 32 consecutive values, and the pad tail goes out in the same pass.
__global__ void __launch_bounds__(256) k_pad_rows(const int32_t* __restrict__ values, const int64_t* __restrict__ off, int64_t n_docs,
                                                  int64_t width, int32_t pad, int32_t* __restrict__ out, int64_t* __restrict__ lengths) {
  const uint32_t lane = threadIdx.x & 31;
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t d = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; d < n_docs; d += nw) {
    const int64_t s = off[d];
    const int64_t len = max((int64_t)0, min(off[d + 1] - s, width));
    const int32_t* src = values + s;
    int32_t* dst = out + d * width;
#pragma unroll 4
    for (int64_t j = lane; j < width; j += 32) dst[j] = (j < len) ? __ldg(src + j) : pad;
    if (lengths && lane == 0) lengths[d] = len;
  }
}

// ---- exclusive scan of the per-document token counts (u32 -> u64 offsets), three launches: tile sums, scan of the
// tile sums (k_scan_counts, one block), tile-local scan + tile offset ----
constexpr int SC_THREADS = 256, SC_ITEMS = 16, SC_TILE = SC_THREADS * SC_ITEMS;

__global__ void __launch_bounds__(SC_THREADS) k_sum_tiles(const uint32_t* __restrict__ in, uint32_t n, uint32_t* __restrict__ tile_sums) {
  __shared__ uint32_t s_w[SC_THREADS / 32];
  uint32_t base = blockIdx.x * SC_TILE, s = 0;
#pragma unroll
  for (int j = 0; j < SC_ITEMS; j++) {
    uint32_t i = base + j * SC_THREADS + threadIdx.x;
    if (i < n) s += in[i];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
  if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t t = 0;
    for (int i = 0; i < SC_THREADS / 32; i++) t += s_w[i];
    tile_sums[blockIdx.x] = t;
  }
}

__global__ void __launch_bounds__(SC_THREADS) k_scan_tiles(const uint32_t* __restrict__ in, uint32_t n, const uint64_t* __restrict__ tile_off,
                                                            uint32_t n_tiles, uint64_t* __restrict__ out) {
  __shared__ uint32_t s_w[SC_THREADS / 32];
  uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t first = blockIdx.x * SC_TILE + threadIdx.x * SC_ITEMS;  // SC_ITEMS consecutive elements per thread
  uint32_t v[SC_ITEMS], s = 0;
#pragma unroll
  for (int j = 0; j < SC_ITEMS; j++) {
    v[j] = (first + j < n) ? in[first + j] : 0u;
    s += v[j];
  }
  uint32_t inc = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, o);
    if ((int)lane >= o) inc += t;
  }
  if (lane == 31) s_w[warp] = inc;
  __syncthreads();
  uint32_t wbase = 0;
  for (uint32_t i = 0; i < warp; i++) wbase += s_w[i];
  uint64_t acc = tile_off[blockIdx.x] + wbase + (inc - s);
#pragma unroll
  for (int j = 0; j < SC_ITEMS; j++) {
    if (first + j < n) out[first + j] = acc;
    acc += v[j];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) out[n] = tile_off[n_tiles];
}

// A few result words go to PINNED HOST memory straight from a kernel (unified addressing: the device writes through the
// mapped pointer).  A cudaMemcpyAsync of 8 bytes would queue on the device-to-host copy engine behind the tens of MB of
// vectors the encode pipeline is streaming out at the same time, and stall the host for that long at every chunk.
__global__ void k_copy_u64(unsigned long long* __restrict__ dst, const unsigned long long* __restrict__ src, int n) {
  if ((int)threadIdx.x < n) dst[threadIdx.x] = src[threadIdx.x];
}

// first position whose id lies outside [0, n_tokens): the reference throws at the FIRST offending character (core.ts:396-402)
__global__ void k_first_bad_id(const int32_t* __restrict__ ids, uint64_t n, uint32_t n_tokens, unsigned long long* __restrict__ first_bad) {
  unsigned long long best = ~0ull;
  uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    if ((uint32_t)__ldg(ids + i) >= n_tokens && i < best) best = i;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) best = min(best, __shfl_xor_sync(0xFFFFFFFFu, best, o));
  if ((threadIdx.x & 31) == 0 && best != ~0ull) atomicMin(first_bad, best);
}

// ---- decodeVector / decodeTokens (core.ts:447-471) on the device: vector index -> token -> its UTF-8 bytes ----
// lens[i] = byte length of value i (0 for an unknown vector index); bad values are reported per document
__global__ void k_decode_lens(const int32_t* __restrict__ values, uint64_t n, const int32_t* __restrict__ fvi, int32_t n_fvi,
                              const int64_t* __restrict__ tok_off, int32_t n_tokens, const int64_t* __restrict__ doc_off, int64_t n_docs,
                              uint32_t* __restrict__ lens, unsigned long long* __restrict__ first_bad) {
  uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    int32_t v = __ldg(values + i);
    int32_t tok = v;
    if (fvi) tok = (v >= 0 && v < n_fvi) ? __ldg(fvi + v) : -1;  // `vector_index in from_vector_index` (core.ts:463)
    uint32_t len = 0;
    if (tok >= 0 && tok < n_tokens) {
      len = (uint32_t)(tok_off[tok + 1] - tok_off[tok]);
    } else if (first_bad) {  // first offender of its document (core.ts:466-468 throws there)
      int64_t lo = 0, hi = n_docs;  // last d with doc_off[d] <= i (relative offsets, doc_off[0] == 0)
      while (lo + 1 < hi) {
        int64_t mid = (lo + hi) >> 1;
        if ((uint64_t)doc_off[mid] <= i) lo = mid;
        else hi = mid;
      }
      atomicMin(first_bad + lo, (unsigned long long)(i - (uint64_t)doc_off[lo]));
    }
    lens[i] = len;
  }
}

__global__ void k_decode_gather(const int32_t* __restrict__ values, uint64_t n, const int32_t* __restrict__ fvi, int32_t n_fvi,
                                const uint8_t* __restrict__ tok_bytes, const int64_t* __restrict__ tok_off, int32_t n_tokens,
                                const uint64_t* __restrict__ byte_off, uint8_t* __restrict__ out) {
  uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    int32_t v = __ldg(values + i);
    int32_t tok = v;
    if (fvi) tok = (v >= 0 && v < n_fvi) ? __ldg(fvi + v) : -1;
    if (tok < 0 || tok >= n_tokens) continue;
    int64_t s = tok_off[tok], e = tok_off[tok + 1];
    uint8_t* dst = out + byte_off[i];
    for (int64_t k = s; k < e; k++) dst[k - s] = __ldg(tok_bytes + k);
  }
}

// out_offsets[d] = byte offset of document d's first value (byte_off has n + 1 entries)
__global__ void k_decode_doc_offsets(const int64_t* __restrict__ doc_off, int64_t n_docs, const uint64_t* __restrict__ byte_off,
                                     int64_t* __restrict__ out_offsets) {
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t d = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; d <= n_docs; d += stride) out_offsets[d] = (int64_t)byte_off[doc_off[d]];
}

}  // namespace bpe
