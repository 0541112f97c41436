// text_kernels.cuh -- the text front end of addToCorpus / encodeToCode on the device (SURVEY.md 8(f) rank 1).
//
// Reference: `for (let char of content)` iterates CODE POINTS (core.ts:185, :396); every code point maps to its
// single-character token through char_to_token, unknown ones are created in first-appearance order by addToCorpus
// (core.ts:186-199) and throw in encodeToCode (core.ts:398-400).  Here the documents arrive as UTF-8 bytes (lone
// surrogates in their 3-byte generalised form, as Python's 'surrogatepass' writes them): one pass counts the lead
// bytes per tile, a scan gives every code point its index, a second pass decodes and looks the code point up in a
// dense device table (0x110000 x int32).  Unknown code points are written as -(cp + 1) and their first position is
// kept with an atomicMin, so the host can create the new tokens in the reference's order.
#pragma once
#include "common.cuh"

namespace bpe {

constexpr int TX_THREADS = 256, TX_ITEMS = 16, TX_TILE = TX_THREADS * TX_ITEMS;  // bytes per block
constexpr uint32_t CP_LIMIT = 0x110000u;

__device__ __forceinline__ bool utf8_is_lead(uint8_t b) { return (b & 0xC0u) != 0x80u; }

__global__ void __launch_bounds__(TX_THREADS) k_utf8_count(const uint8_t* __restrict__ text, uint64_t n, uint32_t* __restrict__ tile_counts) {
  __shared__ uint32_t s_w[TX_THREADS / 32];
  uint64_t base = (uint64_t)blockIdx.x * TX_TILE;
  uint32_t c = 0;
#pragma unroll
  for (int j = 0; j < TX_ITEMS; j++) {
    uint64_t i = base + (uint64_t)j * TX_THREADS + threadIdx.x;
    if (i < n && utf8_is_lead(__ldg(text + i))) c++;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
  if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t t = 0;
    for (int i = 0; i < TX_THREADS / 32; i++) t += s_w[i];
    tile_counts[blockIdx.x] = t;
  }
}

// ids[k] = token index of the k-th code point, or -(cp + 1) when the table does not know it
__global__ void __launch_bounds__(TX_THREADS) k_utf8_decode(const uint8_t* __restrict__ text, uint64_t n, const uint64_t* __restrict__ tile_off,
                                                             const int32_t* __restrict__ cpmap, int32_t* __restrict__ ids,
                                                             uint32_t* __restrict__ first_pos /* [CP_LIMIT], may be NULL */,
                                                             unsigned long long* __restrict__ first_unknown /* (pos << 32 | cp), may be NULL */) {
  __shared__ uint32_t s_w[TX_THREADS / 32];
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint64_t base = (uint64_t)blockIdx.x * TX_TILE;
  uint64_t out = tile_off[blockIdx.x];
  for (int j = 0; j < TX_ITEMS; j++) {  // j-major keeps the order of the bytes
    uint64_t i = base + (uint64_t)j * TX_THREADS + threadIdx.x;
    uint8_t b0 = (i < n) ? __ldg(text + i) : 0x80;
    bool lead = (i < n) && utf8_is_lead(b0);
    uint32_t m = __ballot_sync(0xFFFFFFFFu, lead);
    if (lane == 0) s_w[warp] = __popc(m);
    __syncthreads();
    uint32_t before = 0, total = 0;
    for (int w = 0; w < TX_THREADS / 32; w++) {
      uint32_t v = s_w[w];
      if (w < (int)warp) before += v;
      total += v;
    }
    if (lead) {
      uint32_t cp = b0;
      if (b0 >= 0xF0) {
        cp = ((b0 & 0x07u) << 18) | (((i + 1 < n ? __ldg(text + i + 1) : 0) & 0x3Fu) << 12) | (((i + 2 < n ? __ldg(text + i + 2) : 0) & 0x3Fu) << 6) |
             ((i + 3 < n ? __ldg(text + i + 3) : 0) & 0x3Fu);
      } else if (b0 >= 0xE0) {
        cp = ((b0 & 0x0Fu) << 12) | (((i + 1 < n ? __ldg(text + i + 1) : 0) & 0x3Fu) << 6) | ((i + 2 < n ? __ldg(text + i + 2) : 0) & 0x3Fu);
      } else if (b0 >= 0xC0) {
        cp = ((b0 & 0x1Fu) << 6) | ((i + 1 < n ? __ldg(text + i + 1) : 0) & 0x3Fu);
      }
      if (cp >= CP_LIMIT) cp = 0xFFFDu;
      uint64_t k = out + before + __popc(m & ((1u << lane) - 1u));
      int32_t id = __ldg(cpmap + cp);
      if (id < 0) {
        id = -(int32_t)(cp + 1);
        // (look before the atomic: the entries only ever decrease, so a stale cached value can only let a superfluous atomic
        // through, never hide a smaller position -- a fresh tokenizer's first gigabyte is ALL unknown characters, and 10^9
        // atomics on the few dozen addresses of its alphabet were 200 ms)
        const uint32_t k32 = (uint32_t)min(k, (uint64_t)0xFFFFFFFEu);
        if (first_pos && k32 < first_pos[cp]) atomicMin(first_pos + cp, k32);
        const unsigned long long fu = ((unsigned long long)k << 32) | cp;
        if (first_unknown && fu < *first_unknown) atomicMin(first_unknown, fu);
      }
      ids[k] = id;
    }
    out += total;
    __syncthreads();
  }
}

// code points per document: lead bytes inside the document's byte range (one warp per document; total work = n bytes)
__global__ void k_utf8_doc_counts(const uint8_t* __restrict__ text, const int64_t* __restrict__ doc_byte_off, int64_t n_docs,
                                  uint32_t* __restrict__ doc_chars) {
  int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  uint32_t lane = threadIdx.x & 31;
  int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t d = wid; d < n_docs; d += nw) {
    uint64_t b0 = (uint64_t)doc_byte_off[d], b1 = (uint64_t)doc_byte_off[d + 1];
    uint32_t c = 0;
    for (uint64_t p = b0 + lane; p < b1; p += 32)
      if (utf8_is_lead(__ldg(text + p))) c++;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
    if (lane == 0) doc_chars[d] = c;
  }
}

__global__ void k_u64_to_i64(const uint64_t* __restrict__ in, int64_t* __restrict__ out, int64_t n) {
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = (int64_t)in[i];
}

// offsets[i] += delta: rebases the caller's document offsets to the start of a chunk, and a chunk's output offsets to their
// place in the whole batch (the host-buffer encode pipeline of bpe_b200.cu)
__global__ void k_shift_i64(int64_t* __restrict__ p, int64_t n, int64_t delta) {
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) p[i] += delta;
}

// *out = max(*out, max of in[0..n))
__global__ void k_max_u32(const uint32_t* __restrict__ in, int64_t n, unsigned long long* __restrict__ out) {
  uint32_t m = 0;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) m = max(m, __ldg(in + i));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
  if ((threadIdx.x & 31) == 0 && m) atomicMax(out, (unsigned long long)m);
}

// unknown code points seen by the last decode, with their first positions
__global__ void k_collect_new_cps(uint32_t* __restrict__ first_pos, uint32_t* __restrict__ out_cp, uint32_t* __restrict__ out_pos, uint32_t cap,
                                  uint32_t* __restrict__ n_out) {
  for (uint32_t cp = blockIdx.x * blockDim.x + threadIdx.x; cp < CP_LIMIT; cp += gridDim.x * blockDim.x) {
    uint32_t p = first_pos[cp];
    if (p == 0xFFFFFFFFu) continue;
    first_pos[cp] = 0xFFFFFFFFu;  // ready for the next call
    uint32_t k = atomicAdd(n_out, 1u);
    if (k < cap) {
      out_cp[k] = cp;
      out_pos[k] = p;
    }
  }
}

__global__ void k_set_cpmap(int32_t* __restrict__ cpmap, const int32_t* __restrict__ cps, const int32_t* __restrict__ idx, uint32_t n) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    if ((uint32_t)cps[i] < CP_LIMIT) cpmap[cps[i]] = idx[i];
}

// the table's current entries for n code points (all < CP_LIMIT): bpe_add_text_commit refuses to reassign a known one
__global__ void k_get_cpmap(const int32_t* __restrict__ cpmap, const int32_t* __restrict__ cps, int32_t* __restrict__ out, uint32_t n) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) out[i] = cpmap[cps[i]];
}

constexpr uint32_t FIX_SMEM_TOKENS = 2048;
// resolve the -(cp + 1) placeholders after the new tokens got their indices; count every token (weights, core.ts:201-202)
__global__ void k_fix_and_count(int32_t* __restrict__ ids, uint64_t n, const int32_t* __restrict__ cpmap, unsigned long long* __restrict__ counts,
                                uint32_t n_tokens) {
  // the counts of the low token indices -- every character of ordinary text -- are gathered per block in shared memory: a
  // gigabyte of text would otherwise send some 10^8 atomics to the few dozen addresses of its alphabet
  __shared__ uint32_t s_cnt[FIX_SMEM_TOKENS];
  for (uint32_t t = threadIdx.x; t < FIX_SMEM_TOKENS; t += blockDim.x) s_cnt[t] = 0;
  __syncthreads();
  uint64_t stride = (uint64_t)gridDim.x * blockDim.x;  // a multiple of 32: the loop is warp-uniform
  const uint32_t lane = threadIdx.x & 31;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < ((n + 31) & ~31ull); i += stride) {
    int32_t id = -2 - (int32_t)lane;  // inactive lanes: distinct keys that match nobody
    if (i < n) {
      id = ids[i];
      if (id < 0) {
        id = __ldg(cpmap + (uint32_t)(-(id + 1)));
        ids[i] = id;
      }
    }
    uint32_t peers = __match_any_sync(0xFFFFFFFFu, id);  // one atomic per distinct token per warp
    if (lane == (uint32_t)(__ffs(peers) - 1) && id >= 0 && (uint32_t)id < n_tokens) {
      if ((uint32_t)id < FIX_SMEM_TOKENS) atomicAdd(&s_cnt[id], (uint32_t)__popc(peers));  // (a block sees far fewer than 2^32 characters)
      else atomicAdd(counts + id, (unsigned long long)__popc(peers));
    }
  }
  __syncthreads();
  for (uint32_t t = threadIdx.x; t < FIX_SMEM_TOKENS && t < n_tokens; t += blockDim.x)
    if (s_cnt[t]) atomicAdd(counts + t, (unsigned long long)s_cnt[t]);
}

}  // namespace bpe
