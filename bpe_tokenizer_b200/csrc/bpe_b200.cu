// bpe_b200.cu -- engine state, host orchestration and the C ABI declared in include/bpe_b200.h.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC (build.py).
#include "../../include/bpe_b200.h"

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <functional>
#include <string>
#include <condition_variable>
#include <mutex>
#include <thread>
#include <unordered_map>
#include <unordered_set>
#include <vector>

#include "encode_kernels.cuh"
#include "encode_lanes.cuh"
#include "train_kernels.cuh"
#include "mg_kernels.cuh"
#include "round_kernels.cuh"
#include "text_kernels.cuh"

using namespace bpe;

namespace {

template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t cap = 0;  // elements
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept : p(o.p), cap(o.cap) {
    o.p = nullptr;
    o.cap = 0;
  }
  DevBuf& operator=(DevBuf&& o) noexcept {
    if (this != &o) {
      release();
      p = o.p;
      cap = o.cap;
      o.p = nullptr;
      o.cap = 0;
    }
    return *this;
  }
  ~DevBuf() { release(); }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  // grow to at least n elements; keep_n elements are preserved (stream-ordered copy)
  cudaError_t reserve(size_t n, size_t keep_n = 0, cudaStream_t s = 0, double growth = 1.0) {
    if (n <= cap) return cudaSuccess;
    size_t want = std::max(n, (size_t)((double)cap * growth));
    T* q = nullptr;
    cudaError_t err = cudaMalloc(&q, want * sizeof(T));
    if (err != cudaSuccess) {
      (void)cudaGetLastError();  // the runtime keeps the failure as its "last error": the next launch check must not see it
      want = n;
      err = cudaMalloc(&q, want * sizeof(T));
      if (err != cudaSuccess) {
        (void)cudaGetLastError();
        return err;
      }
    }
    if (p && keep_n) {
      err = cudaMemcpyAsync(q, p, keep_n * sizeof(T), cudaMemcpyDeviceToDevice, s);
      if (err != cudaSuccess) {
        cudaFree(q);
        return err;
      }
      cudaStreamSynchronize(s);
    }
    if (p) cudaFree(p);
    p = q;
    cap = want;
    return cudaSuccess;
  }
};

// grow-only pinned host buffer (staging of the small per-document arrays of the encode pipeline)
template <typename T>
struct PinBuf {
  T* p = nullptr;
  size_t cap = 0;
  ~PinBuf() {
    if (p) cudaFreeHost(p);
  }
  cudaError_t reserve(size_t n) {
    if (n <= cap) return cudaSuccess;
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    cudaError_t err = cudaHostAlloc((void**)&p, n * sizeof(T), cudaHostAllocDefault);
    if (err == cudaSuccess) cap = n;
    else (void)cudaGetLastError();
    return err;
  }
};

uint32_t pow2_at_least(uint64_t x) {
  uint32_t p = 1;
  while (p < x && p < 0x80000000u) p <<= 1;
  return p;
}
int ilog2(uint32_t p) {
  int l = 0;
  while ((1u << l) < p) l++;
  return l;
}

}  // namespace

// Host rendezvous of a group's members before every launch of the sharded mergeUntil loop: no member starts a kernel that waits for
// its peers while another member still does host work between launches (buffer growth frees memory, and cudaFree waits for the
// device's kernels).  A member that leaves the loop drops out, so the others never wait for it here.
struct LaunchGate {
  std::mutex mu;
  std::condition_variable cv;
  int expected;
  int arrived = 0;
  uint64_t generation = 0;
  explicit LaunchGate(int n) : expected(n) {}
  void release() {
    arrived = 0;
    generation++;
    cv.notify_all();
  }
  void arrive() {
    std::unique_lock<std::mutex> lk(mu);
    const uint64_t g = generation;
    if (++arrived >= expected) release();
    else cv.wait(lk, [&] { return generation != g; });
  }
  void drop() {
    std::lock_guard<std::mutex> lk(mu);
    expected--;
    if (arrived > 0 && arrived >= expected) release();
  }
};

struct EncodeScratch {
  DevBuf<int32_t> out_tmp;
  DevBuf<uint32_t> out_len;
  DevBuf<uint64_t> out_off;
  DevBuf<uint32_t> g_tok, g_nxt, g_prv, g_rk, g_sel;
  DevBuf<uint32_t> range_first, tile_sums;
  DevBuf<uint64_t> tile_off;
  DevBuf<uint32_t> flags;  // [0] long documents left for the per-document kernel, [1] error, [2] next range to claim
};

struct bpe_engine {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr, own_stream = nullptr;
  std::string err;
  bool profiling = false;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;

  // corpus_in_code (core.ts:106): slots + document boundaries
  DevBuf<uint32_t> slots;
  uint64_t n_slots = 0;
  std::vector<int64_t> doc_off{0};
  uint64_t live_tokens = 0;

  // vocabulary
  std::vector<int32_t> h_len16;
  DevBuf<uint32_t> d_len16;
  int32_t n_tokens = 0;

  // merge list (core.ts:88-91) + device lookup table for encode
  std::vector<int32_t> h_merges;
  bool mt_dirty = true;
  DevBuf<unsigned long long> d_mt;
  DevBuf<uint32_t> d_minlr;  // per token: lowest rank as left operand << 16 | lowest rank as right operand
  uint32_t mt_cap = 0;
  // lane path (encode_lanes.cuh): pair table with spine bounds, dense table of the low ids, token of each rank
  bool lt_dirty = true;
  DevBuf<uint4> d_lt;
  DevBuf<uint2> d_lt_dense;
  DevBuf<uint16_t> d_rule_c;
  uint32_t lt_cap = 0;
  int32_t lt_c_affine = -1;
  int enc_lmax = 32;     // rows per lane of the lane path (32 or 48); BPE_ENC_LMAX overrides
  int enc_lmax_forced = 0;
  int enc_force_old = 0; // debug: BPE_ENC_OLD=1 routes every document through the per-document kernel

  // pair index
  bool index_valid = false;
  uint32_t tbl_cap = 0;
  DevBuf<uint32_t> t_ent;  // 6 words per slot: 4 u32 fields and the u64 list start (field-major when TBL_STRIDE == 1, common.cuh)
  DevBuf<uint32_t> u_ent;  // second buffer, target of the next rehash (kept at high water)
  DevBuf<uint32_t> pool;
  DevBuf<DevState> d_st;
  DevState* h_st = nullptr;  // pinned
  DevBuf<Best> partials;
  DevBuf<uint32_t> partial_keys;
  DevBuf<SiteRec> sites, sites2;  // k_merge_loop alternates between the two (deferred list filling)
  DevBuf<uint32_t> newslots;
  DevBuf<uint32_t> nd;  // dense accumulator of the pairs born by the current merge (train_kernels.cuh, ND_*)
  DevBuf<uint32_t> hot;
  bool hot_valid = false;
  uint32_t hot_max_length = 0;
  uint32_t hot_limit = 0;
  DevBuf<uint32_t> cands;
  DevBuf<MergeRec> dev_log;
  DevBuf<unsigned long long> barrier;  // own 128-byte line
  int loop_blocks = 0;   // co-resident grid of k_merge_loop
  // several exact merges per barrier round (round_kernels.cuh): dense delta rows, site buffers of merges 1.., per-block top-2 partials
  DevBuf<unsigned long long> r_cells;
  DevBuf<uint32_t> r_slotrows, r_lists;
  DevBuf<SiteRec> r_bsites;
  DevBuf<uint4> r_gp;
  DevBuf<uint32_t> r_gk;
  DevBuf<RoundState> r_state;
  DevBuf<unsigned long long> r_gcells;  // sharded rounds: the deltas summed over the ranks
  DevBuf<uint32_t> r_glists;
  int round_blocks = 0;  // co-resident grid of k_merge_rounds
  int scan_mode = 0;     // debug: walk all slots instead of occurrence lists

  // sharded training (mg_kernels.cuh): this rank's mailbox + the peers' mailboxes mapped through cudaIpc
  int mg_rank = 0, mg_world = 1;
  void* mg_mailbox = nullptr;            // cudaMalloc'ed, exported with cudaIpcGetMemHandle
  size_t mg_mailbox_bytes = 0;
  void* mg_peer[MG_MAX_WORLD] = {};      // [rank] == mg_mailbox
  bool mg_connected = false;
  bool mg_counts_global = false;         // the table's counts are the sum over all ranks (import done for this index)
  uint32_t mg_inbox_stride = 0, mg_tie_cap = 0;
  DevBuf<int32_t> mg_dlt;
  DevBuf<uint32_t> mg_mark, mg_touched, mg_tie_sorted, mg_export_n, mg_newpair;
  int mg_loop_blocks = 0;
  unsigned long long mg_epoch = 0, mg_tie_epoch = 0;
  bool mg_timed_out = false;             // the last sharded mergeUntil stopped because a peer did not answer
  LaunchGate* mg_gate = nullptr;         // group member inside the group's bpe_merge_until: the members' launch rendezvous

  // device group (bpe_create_group): the handle holds one member engine per device, member r initialised as rank r of the group
  // with its mailbox connected to the others' by pointer.  The handle itself owns no device state; the entry points forward to
  // the members (group_* below).
  std::vector<bpe_engine*> members;
  bool grp_uploaded = false;              // the corpus got its first, partitioned upload: later uploads go to the last member
  DevBuf<uint32_t> grp_keys, grp_counts;  // member: its pair histogram, exported for the other members to import over NVLink
  int64_t grp_n = 0;

  // text front end (text_kernels.cuh): code point -> single-character token index, -1 = unknown
  DevBuf<int32_t> d_cpmap;
  DevBuf<uint32_t> d_firstpos;
  DevBuf<uint8_t> x_text;
  DevBuf<uint32_t> x_tilecnt;
  DevBuf<uint64_t> x_tileoff;
  DevBuf<unsigned long long> x_counts;
  DevBuf<uint32_t> x_doccnt;
  DevBuf<uint64_t> x_docoff;
  // bpe_add_text_stage -> bpe_add_text_commit: the decoded batch waits in x_ids (placeholders for its new code points) with its
  // document boundaries in h_rel.  Every other call that reuses those buffers, or replaces the character table, drops it.
  bool txt_staged = false;
  int64_t txt_chars = 0, txt_docs = 0;
  std::vector<int32_t> txt_new;  // the staged batch's new code points, ascending

  // staging of the host-buffer encode / restore calls (grow-only, reused across calls)
  DevBuf<int32_t> x_ids, x_out, x_tvi;
  DevBuf<int64_t> x_off, x_ooff, x_ooff2, x_bad;
  DevBuf<unsigned long long> x_flag;
  std::vector<int64_t> h_rel;
  EncodeScratch x_scratch;
  EncodeScratch dev_scratch;             // scratch of bpe_encode_batch_dev (device buffers in, device buffers out)
  uint32_t lanes_attr_set = 0;           // bit per k_encode_lanes instantiation whose dynamic shared memory limit was raised on
                                         // THIS engine's device (the attribute is per device, not per process)
  // the host-buffer encode calls run as a three-stream pipeline over chunks of whole documents: copy in | encode | copy out
  cudaStream_t s_in = nullptr, s_out = nullptr;
  cudaEvent_t ev_in[3] = {nullptr, nullptr, nullptr}, ev_done = nullptr, ev_res[2] = {nullptr, nullptr};
  unsigned long long* h_pipe = nullptr;  // pinned: 3 slots x 4 words of per-chunk flags, [12..13] flags of the lane kernel
  PinBuf<int64_t> h_in_off, h_out_off, h_bad;  // pinned staging of document offsets in, output offsets and first offenders out
  int64_t enc_chunk = 128ll << 20;       // input units (ids or bytes) per full-size chunk; BPE_ENC_CHUNK overrides
  std::vector<int64_t> enc_parts;        // the last host-buffer encode, per chunk: where its vectors wait in x_out, how many
  int64_t enc_bad_id_pos = -1;           // the last host-buffer encode: input position of an id outside the token table

  // scratch
  DevBuf<int32_t> stage_ids;
  DevBuf<int64_t> stage_off;

  bpe_stats stats{};

  PairTable table() const {
    PairTable t;
    const size_t fs = (TBL_STRIDE == 1) ? (size_t)tbl_cap : 1;  // distance between fields
    t.keys.p = t_ent.p;
    t.cnt.p = t_ent.p + fs;
    t.occ_len.p = t_ent.p + 2 * fs;
    t.occ_fill.p = t_ent.p + 3 * fs;
    t.occ_start.p = reinterpret_cast<unsigned long long*>(t_ent.p + (TBL_STRIDE == 1 ? 4 * fs : 6));  // (8-byte aligned)
    t.mask = tbl_cap - 1;
    t.shift = 32 - ilog2(tbl_cap);
    return t;
  }
  int grid(int per_sm = 4) const { return sm_count * per_sm; }
};

namespace {

int fail(bpe_engine* e, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (e) e->err = buf;
  return code;
}

#define CK(call)                                                                                              \
  do {                                                                                                        \
    cudaError_t _err = (call);                                                                                \
    if (_err != cudaSuccess)                                                                                  \
      return fail(e, _err == cudaErrorMemoryAllocation ? BPE_E_NOMEM : BPE_E_CUDA, "%s:%d %s: %s", __FILE__, \
                  __LINE__, #call, cudaGetErrorString(_err));                                                 \
  } while (0)

#define CKL()                                \
  do {                                       \
    e->stats.kernel_launches++;              \
    CK(cudaGetLastError());                  \
  } while (0)

#define TRY(call)             \
  do {                        \
    int _rc = (call);         \
    if (_rc != BPE_OK) return _rc; \
  } while (0)

int fetch_state(bpe_engine* e) {
  CK(cudaMemcpyAsync(e->h_st, e->d_st.p, sizeof(DevState), cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  return BPE_OK;
}

int check_dev_err(bpe_engine* e) {
  uint32_t f = e->h_st->err & ~ERR_HOT_OVERFLOW;  // hot-list overflow is recoverable (rebuild), handled by the caller
  if (!f) return BPE_OK;
  if (f & ERR_POOL_FULL) return fail(e, BPE_E_INTERNAL, "occurrence pool exhausted (flags 0x%x)", f);
  if (f & ERR_MISSING_KEY) return fail(e, BPE_E_INTERNAL, "pair missing from the table (flags 0x%x)", f);
  if (f & ERR_SPAN_OVERFLOW) return fail(e, BPE_E_DOMAIN, "token span exceeds 2^29 positions");
  if (f & ERR_COUNT_OVERFLOW) return fail(e, BPE_E_DOMAIN, "a pair's count summed over the shards exceeds 2^32 - 1");
  return fail(e, BPE_E_INTERNAL, "device error flags 0x%x", f);
}

int sync_len16(bpe_engine* e) {
  size_t n = e->h_len16.size();
  CK(e->d_len16.reserve(std::max<size_t>(n + 1024, 4096), 0, e->stream, 2.0));
  if (n) {
    std::vector<uint32_t> tmp(e->h_len16.begin(), e->h_len16.end());
    CK(cudaMemcpyAsync(e->d_len16.p, tmp.data(), n * sizeof(uint32_t), cudaMemcpyHostToDevice, e->stream));
    CK(cudaStreamSynchronize(e->stream));
  }
  return BPE_OK;
}

// ---- pair table allocation / growth -------------------------------------------------------------
__global__ void k_init_table(uint4* __restrict__ ent, uint64_t cap) {  // key = EMPTY_KEY, every other field 0
  uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += stride) {
    ent[2 * i] = make_uint4(EMPTY_KEY, 0u, 0u, 0u);
    ent[2 * i + 1] = make_uint4(0u, 0u, 0u, 0u);
  }
}

int alloc_table(bpe_engine* e, uint32_t cap) {
  // buffers only ever grow (cudaFree / cudaMalloc of GBs costs up to seconds); the logical capacity is `cap`
  CK(e->t_ent.reserve((size_t)cap * (TBL_STRIDE == 1 ? 6 : TBL_STRIDE)));
  e->tbl_cap = cap;
  if (TBL_STRIDE == 1) {
    CK(cudaMemsetAsync(e->t_ent.p, 0xFF, (size_t)cap * 4, e->stream));
    CK(cudaMemsetAsync(e->t_ent.p + cap, 0, (size_t)cap * 20, e->stream));
  } else {
    k_init_table<<<e->grid(8), 256, 0, e->stream>>>(reinterpret_cast<uint4*>(e->t_ent.p), (uint64_t)cap);
    CKL();
  }
  if (e->mg_world > 1) {  // per-slot side arrays of the sharded loop follow the table (all zero between merges)
    CK(e->mg_dlt.reserve(cap));
    CK(cudaMemsetAsync(e->mg_dlt.p, 0, (size_t)cap * 4, e->stream));
  }
  return BPE_OK;
}

__global__ void k_rehash(PairTable src, PairTable dst, DevState* st) {
  uint32_t cap = src.mask + 1;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += gridDim.x * blockDim.x) {
    uint32_t key = src.keys[i];
    if (key == EMPTY_KEY) continue;
    uint32_t h = (key * 0x9E3779B1u) >> dst.shift;
    for (;;) {
      uint32_t old = atomicCAS(dst.keys + h, EMPTY_KEY, key);
      if (old == EMPTY_KEY) break;
      h = (h + 1) & dst.mask;
    }
    dst.cnt[h] = src.cnt[i];
    dst.occ_start.set(h, src.occ_start.get(i));
    dst.occ_len[h] = src.occ_len[i];
    dst.occ_fill[h] = src.occ_fill[i];
  }
}

int grow_table(bpe_engine* e, uint32_t new_cap) {
  PairTable old = e->table();
  std::swap(e->t_ent, e->u_ent);
  TRY(alloc_table(e, new_cap));  // the (former) alternate set becomes the live table
  k_rehash<<<e->grid(), 256, 0, e->stream>>>(old, e->table(), e->d_st.p);
  CKL();
  CK(cudaStreamSynchronize(e->stream));
  e->hot_valid = false;  // slot numbers changed
  return BPE_OK;
}

// ---- K1: build histogram + occurrence lists from the corpus -------------------------------------
// BPE_POOL_BASE (cells, default 0): index build starts the occurrence pool's cursor there, with real memory reserved below
// it, so that a corpus of a few MB puts its lists on both sides of cell 2^32 (tests of the 64-bit cell indices)
uint64_t pool_base_knob() {
  if (const char* v = getenv("BPE_POOL_BASE")) return (uint64_t)std::max(0ll, atoll(v));
  return 0;
}

int build_index(bpe_engine* e) {
  e->index_valid = false;
  e->hot_valid = false;
  if (!e->h_st) CK(cudaHostAlloc((void**)&e->h_st, sizeof(DevState), cudaHostAllocDefault));
  CK(e->d_st.reserve(1));
  CK(e->partials.reserve((size_t)e->grid(8)));
  if (!e->nd.p) CK(e->nd.reserve((size_t)ND_ROWS * ND_STRIDE));
  CK(cudaMemsetAsync(e->nd.p, 0, (size_t)ND_ROWS * ND_STRIDE * 4, e->stream));  // all rows zero between merges
  TRY(sync_len16(e));
  uint64_t n = e->n_slots;
  if (n >= 0xFFFFFFF0ull) return fail(e, BPE_E_DOMAIN, "corpus of %llu positions exceeds the 2^32 engine limit", (unsigned long long)n);
  // The pool holds K1's n cells and at most two per merge site, n + 2 * sites <= 3n (DESIGN.md section 1), plus the private
  // chunks the blocks of k_merge_rounds open and the sharded loop's one-round lag.  It is reserved here, once, so that a run
  // does not grow it: a growth copies the old pool into the new one and needs both resident.
  const uint64_t pool_base = pool_base_knob();
  const uint64_t pool_need = pool_base + 3 * n + 2ull * R_HUGE + 2ull * std::max(R_HUGE, R_BATCH_SITES) + 2ull * e->sm_count * R_POOL_CHUNK;
  if (e->pool.cap < pool_need) e->pool.release();  // (nothing in it survives the rebuild: never hold the old and the new pool together)
  CK(e->pool.reserve((size_t)pool_need));
  uint64_t t2 = (uint64_t)e->n_tokens * (uint64_t)e->n_tokens;
  uint32_t cap = pow2_at_least(std::min<uint64_t>(std::max<uint64_t>(2 * std::min(n, t2), 1u << 16), 1u << 24));
  {
    if (!e->ev0) {
      CK(cudaEventCreate(&e->ev0));
      CK(cudaEventCreate(&e->ev1));
    }
    CK(cudaEventRecord(e->ev0, e->stream));
  }
  for (;;) {
    TRY(alloc_table(e, cap));
    DevState init{};
    init.pool_cursor = pool_base;
    init.live_tokens = e->live_tokens;
    init.tie_pos = ~0ull;
    init.mg_epoch = e->mg_epoch;  // the peers' flags keep counting across index rebuilds
    init.mg_tie_epoch = e->mg_tie_epoch;
    CK(cudaMemcpyAsync(e->d_st.p, &init, sizeof init, cudaMemcpyHostToDevice, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    if (n) {
      k_hist<<<e->grid(4), K1_THREADS, 0, e->stream>>>(e->slots.p, (uint32_t)n, e->table(), e->d_st.p);
      CKL();
    }
    TRY(fetch_state(e));
    if (e->h_st->err & ERR_TABLE_FULL) {
      if (cap >= 0x80000000u) return fail(e, BPE_E_NOMEM, "pair table cannot grow further");
      cap <<= 2;
      continue;
    }
    TRY(check_dev_err(e));
    if ((uint64_t)e->h_st->n_keys * 2 > cap && cap < 0x80000000u) {  // keep the load factor <= 0.5
      cap <<= 1;
      continue;
    }
    break;
  }
  if (n) {
    k_alloc_lists<<<e->grid(4), 256, 0, e->stream>>>(e->table(), e->d_st.p, (unsigned long long)e->pool.cap);
    CKL();
    int k1b_per_sm = 0;
    CK(cudaFuncSetAttribute(k_scatter, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)K1B_SMEM_BYTES));  // the staging buffer
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&k1b_per_sm, k_scatter, K1B_THREADS, K1B_SMEM_BYTES));
    if (k1b_per_sm < 1) return fail(e, BPE_E_CUDA, "k_scatter does not fit on an SM");
    k_scatter<<<e->grid(k1b_per_sm), K1B_THREADS, K1B_SMEM_BYTES, e->stream>>>(e->slots.p, (uint32_t)n, e->table(), e->pool.p, e->d_st.p);
    CKL();
  }
  CK(cudaEventRecord(e->ev1, e->stream));
  TRY(fetch_state(e));
  TRY(check_dev_err(e));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, e->ev0, e->ev1));
  e->stats.ms_index_build += ms;
  e->stats.index_builds++;
  e->index_valid = true;
  e->mg_counts_global = false;
  return BPE_OK;
}

int ensure_index(bpe_engine* e) {
  if (e->index_valid) return BPE_OK;
  return build_index(e);
}

// ---- hot list -----------------------------------------------------------------------------------
constexpr uint32_t HOT_TARGET = 1u << 15;

// returns found=0 when no pair with a count exists at all
int rebuild_hot(bpe_engine* e, uint32_t max_length, bool* any) {
  PairTable t = e->table();
  CK(cudaMemsetAsync(&e->d_st.p->bins[0], 0, sizeof(uint32_t) * 36, e->stream));
  k_count_bins<<<e->grid(4), 256, 0, e->stream>>>(t, e->d_len16.p, max_length, e->d_st.p);
  CKL();
  TRY(fetch_state(e));
  uint64_t acc = 0;
  int pick = 0;
  for (int k = 32; k >= 1; k--) {
    uint64_t nk = e->h_st->bins[k];
    if (acc + nk > HOT_TARGET && acc > 0) break;
    acc += nk;
    if (nk) pick = k;
    if (acc > HOT_TARGET) break;
  }
  *any = pick != 0;
  e->hot_valid = false;
  if (!pick) return BPE_OK;
  // everything from bin `pick` up: counts >= 2^(pick-1); extend down to the lowest bin that adds nothing
  int lo = pick;
  while (lo > 1 && e->h_st->bins[lo - 1] == 0) lo--;
  uint32_t thresh = 1u << (lo - 1);
  CK(e->hot.reserve(std::max<size_t>((size_t)acc * 2 + 4096 + 2 * (size_t)BPE_MAX_TOKENS, 1u << 18)));
  e->h_st->hot_n = 0;
  e->h_st->hot_thresh = thresh;
  uint32_t two[2] = {0, thresh};
  CK(cudaMemcpyAsync(&e->d_st.p->hot_n, two, sizeof two, cudaMemcpyHostToDevice, e->stream));
  k_build_hot<<<e->grid(4), 256, 0, e->stream>>>(t, e->d_len16.p, max_length, e->hot.p, (uint32_t)e->hot.cap, e->d_st.p);
  CKL();
  e->hot_limit = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(4ull * HOT_TARGET, 2 * acc + 4096), 0xFFFFFFF0u);
  e->hot_max_length = max_length;
  e->hot_valid = true;
  e->stats.hot_rebuilds++;
  return BPE_OK;
}

// ---- K2 driver: leaves the winner in h_st (best_primary == 0: none) -------------------------------
int run_argmax(bpe_engine* e, uint32_t max_length) {
  PairTable t = e->table();
  int blocks = e->grid(4);
  k_argmax<<<blocks, AM_THREADS, 0, e->stream>>>(t, e->d_len16.p, max_length, e->partials.p, e->d_st.p);
  CKL();
  TRY(fetch_state(e));
  TRY(check_dev_err(e));
  if (e->h_st->best_primary && e->h_st->best_mult > 1) {
    // tie on (weight, a.index + b.index): the pair whose last counted occurrence comes first wins (core.ts:294-305)
    uint32_t mult = e->h_st->best_mult;
    CK(e->cands.reserve(std::max<size_t>(mult, 1024), 0, e->stream, 2.0));
    k_collect_cands<<<blocks, 256, 0, e->stream>>>(t, e->d_len16.p, max_length, e->cands.p, (uint32_t)e->cands.cap, e->d_st.p);
    CKL();
    k_tie_break<<<std::min<uint32_t>(mult, (uint32_t)e->grid(4)), 256, 0, e->stream>>>(e->slots.p, (uint32_t)e->n_slots, t, e->pool.p, e->cands.p, e->d_st.p);
    CKL();
    k_tie_finish<<<1, 32, 0, e->stream>>>(t, e->d_st.p);
    CKL();
    TRY(fetch_state(e));
    TRY(check_dev_err(e));
    e->stats.tie_breaks++;
  }
  return BPE_OK;
}

ApplyArgs apply_args(bpe_engine* e) {
  ApplyArgs A;
  A.slots = e->slots.p;
  A.n = (uint32_t)e->n_slots;
  A.t = e->table();
  A.pool = e->pool.p;
  A.st = e->d_st.p;
  A.sites = e->sites.p;
  A.sites_cap = (uint32_t)std::min<size_t>(e->sites.cap, 0xFFFFFFFFu);
  A.newslots = e->newslots.p;
  A.nd = e->nd.p;
  A.newpair = nullptr;
  A.newpair_cap = 0;
  A.new_cap = (uint32_t)std::min<size_t>(e->newslots.cap, 0xFFFFFFFFu);
  A.len16 = e->d_len16.p;
  A.scan_mode = e->scan_mode;
  A.dlt = nullptr;
  A.touched = nullptr;
  A.touched_cap = 0;
  return A;
}

// ---- K3 driver ------------------------------------------------------------------------------------
// bound = upper bound on the number of sites (count of the pair, or its list length)
int run_apply(bpe_engine* e, uint32_t a, uint32_t b, uint32_t c, uint32_t bound) {
  // capacity: new keys <= 2*bound, new list cells <= 2*bound
  uint64_t keys_after = (uint64_t)e->h_st->n_keys + std::min<uint64_t>(2ull * bound + 2, 2ull * ((uint64_t)e->n_tokens + 1) + 2);
  if (keys_after * 2 > e->tbl_cap) {
    uint64_t want = keys_after * 5 / 2;
    if (want > 0x80000000ull) want = 0x80000000ull;
    if (keys_after * 2 > pow2_at_least(want)) return fail(e, BPE_E_NOMEM, "pair table cannot grow further");
    TRY(grow_table(e, pow2_at_least(want)));
  }
  uint64_t pool_after = (uint64_t)e->h_st->pool_cursor + 2ull * bound;
  if (pool_after > e->pool.cap) CK(e->pool.reserve((size_t)pool_after, e->h_st->pool_cursor, e->stream, 1.5));
  CK(e->sites.reserve(std::max<size_t>(bound, 4096), 0, e->stream, 2.0));
  CK(e->newslots.reserve(std::max<size_t>(2ull * bound + 2, 8192), 0, e->stream, 2.0));
  if ((size_t)c + 1 > e->d_len16.cap) CK(e->d_len16.reserve((size_t)c + 1, (size_t)c, e->stream, 2.0));
  PairTable t = e->table();
  uint32_t work = e->scan_mode ? (uint32_t)e->n_slots : bound;
  int blocks = (int)std::min<uint64_t>((uint64_t)e->grid(8), std::max<uint64_t>(1, (work + 255) / 256));
  ApplyArgs A = apply_args(e);
  k_sites<<<blocks, 256, 0, e->stream>>>(A, a, b, c);
  CKL();
  int blocks2 = (int)std::min<uint64_t>((uint64_t)e->grid(8), std::max<uint64_t>(1, (2ull * bound + 255) / 256));
  k_alloc_new<<<blocks2, 256, 0, e->stream>>>(A, c, e->hot_max_length, e->hot_valid ? 1 : 0, e->hot.p, (uint32_t)e->hot.cap, (unsigned long long)e->pool.cap);
  CKL();
  int blocks3 = (int)std::min<uint64_t>((uint64_t)e->grid(8), std::max<uint64_t>(1, ((uint64_t)bound + 255) / 256));
  k_apply<<<blocks3, 256, 0, e->stream>>>(A, a, b, c);
  CKL();
  e->h_len16.push_back(e->h_len16[a] + e->h_len16[b]);
  e->h_merges.push_back((int32_t)a);
  e->h_merges.push_back((int32_t)b);
  e->h_merges.push_back((int32_t)c);
  e->mt_dirty = e->lt_dirty = true;
  e->n_tokens++;
  e->stats.merges_applied++;
  return BPE_OK;
}

// ---- merge lookup table for encode ------------------------------------------------------------------
int ensure_merge_table(bpe_engine* e) {
  if (!e->mt_dirty && e->d_mt.p) return BPE_OK;
  size_t m = e->h_merges.size() / 3;
  uint32_t cap = pow2_at_least(std::max<size_t>(4 * m, 1024));
  std::vector<unsigned long long> h(cap, MT_EMPTY);
  int shift = 32 - ilog2(cap);
  for (size_t r = 0; r < m; r++) {
    uint32_t a = (uint32_t)e->h_merges[3 * r], b = (uint32_t)e->h_merges[3 * r + 1], c = (uint32_t)e->h_merges[3 * r + 2];
    uint32_t key = pair_key(a, b);
    uint32_t i = (key * 0x9E3779B1u) >> shift;
    bool dup = false;
    while (h[i] != MT_EMPTY) {
      if ((uint32_t)(h[i] >> 32) == key) {
        dup = true;  // a second rule for the same pair can never fire (the first one removed every occurrence)
        break;
      }
      i = (i + 1) & (cap - 1);
    }
    if (!dup) h[i] = ((unsigned long long)key << 32) | ((unsigned long long)(uint32_t)r << 16) | c;
  }
  std::vector<uint32_t> minlr((size_t)std::max(e->n_tokens, 1), 0xFFFFFFFFu);
  for (size_t r = 0; r < m; r++) {
    uint32_t a = (uint32_t)e->h_merges[3 * r], b = (uint32_t)e->h_merges[3 * r + 1];
    if (a >= minlr.size() || b >= minlr.size()) return fail(e, BPE_E_INVALID, "merge %zu refers to a token outside the table", r);
    uint32_t rr = (uint32_t)std::min<size_t>(r, 0xFFFE);
    if ((minlr[a] >> 16) > rr) minlr[a] = (minlr[a] & 0xFFFFu) | (rr << 16);
    if ((minlr[b] & 0xFFFFu) > rr) minlr[b] = (minlr[b] & 0xFFFF0000u) | rr;
  }
  CK(e->d_minlr.reserve(minlr.size()));
  CK(cudaMemcpyAsync(e->d_minlr.p, minlr.data(), minlr.size() * 4, cudaMemcpyHostToDevice, e->stream));
  CK(e->d_mt.reserve(cap));
  CK(cudaMemcpyAsync(e->d_mt.p, h.data(), (size_t)cap * 8, cudaMemcpyHostToDevice, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  e->mt_cap = cap;
  e->mt_dirty = false;
  return BPE_OK;
}

// ---- pair table of the lane path: rank + spine bounds per pair (see encode_lanes.cuh) ---------------------------
// rank, token and spine bounds of every pair that is a rule or lies on a spine of one (encode_lanes.cuh) -- pure host work,
// also reachable without a device through bpe_debug_lane_table (CPU parity test against the prototype of the algorithm)
struct LaneEnt {
  uint16_t rk = 0xFFFF, c = 0, rs = 0xFFFF, ls = 0xFFFF;
};

int build_lane_entries(bpe_engine* e, const std::vector<int32_t>& merges, int32_t n_tokens, std::unordered_map<uint32_t, LaneEnt>& M,
                       std::vector<uint16_t>& rule_c) {
  size_t m = merges.size() / 3;
  if (m > EL_MAX_RANK + 1) return fail(e, BPE_E_DOMAIN, "merge list too long");
  const int32_t nt = std::max(n_tokens, 1);
  M.clear();
  M.reserve(m * 3 + 16);
  // definition of every merged token (core.ts:315-325: c is a fresh index, so each c has one definition)
  std::vector<int32_t> def_a((size_t)nt, -1), def_b((size_t)nt, -1);
  std::vector<uint8_t> first(m, 0);
  rule_c.assign(std::max<size_t>(m, 1), 0);
  for (size_t r = 0; r < m; r++) {
    int32_t a = merges[3 * r], b = merges[3 * r + 1], c = merges[3 * r + 2];
    if (a < 0 || b < 0 || c < 0 || a >= nt || b >= nt || c >= nt)
      return fail(e, BPE_E_INVALID, "merge %zu refers to a token outside the table", r);
    rule_c[r] = (uint16_t)c;
    if (def_a[c] < 0 && a < c && b < c) {
      def_a[c] = a;
      def_b[c] = b;
    } else if (def_a[c] >= 0 && (def_a[c] != a || def_b[c] != b)) {
      return fail(e, BPE_E_INVALID, "token %d is produced by two different merges", c);
    }
    LaneEnt& x = M[pair_key((uint32_t)a, (uint32_t)b)];
    if (x.rk == 0xFFFF) {  // a second rule for the same pair can never fire (the first one removed every occurrence)
      x.rk = (uint16_t)r;
      x.c = (uint16_t)c;
      first[r] = 1;
    }
  }
  for (size_t r = 0; r < m; r++) {
    if (!first[r]) continue;
    int32_t a = merges[3 * r], b = merges[3 * r + 1];
    for (int32_t u = a;;) {  // every token on the right spine of a: anything ending in u may grow into a
      LaneEnt& x = M[pair_key((uint32_t)u, (uint32_t)b)];
      if (x.rs > r) x.rs = (uint16_t)r;
      if (def_a[u] < 0) break;
      u = def_b[u];
    }
    for (int32_t w = b;;) {  // every token on the left spine of b
      LaneEnt& x = M[pair_key((uint32_t)a, (uint32_t)w)];
      if (x.ls > r) x.ls = (uint16_t)r;
      if (def_a[w] < 0) break;
      w = def_a[w];
    }
  }
  return BPE_OK;
}

int ensure_lane_tables(bpe_engine* e) {
  if (!e->lt_dirty && e->d_lt.p) return BPE_OK;
  size_t m = e->h_merges.size() / 3;
  std::unordered_map<uint32_t, LaneEnt> M;
  std::vector<uint16_t> rule_c;
  TRY(build_lane_entries(e, e->h_merges, e->n_tokens, M, rule_c));
  uint32_t cap = pow2_at_least(std::max<size_t>(2 * M.size(), 1024));
  std::vector<uint4> h(cap, make_uint4(EMPTY_KEY, EL_NONE, 0xFFFFFFFFu, 0));
  std::vector<uint2> dense((size_t)EL_DENSE * EL_DENSE, make_uint2(EL_NONE, 0xFFFFFFFFu));
  int shift = 32 - ilog2(cap);
  for (auto& kv : M) {
    uint32_t key = kv.first;
    const LaneEnt& x = kv.second;
    uint32_t y = (uint32_t)x.rk | ((uint32_t)x.c << 16), z = (uint32_t)x.rs | ((uint32_t)x.ls << 16);
    uint32_t a = key >> 16, b = key & 0xFFFFu;
    if (a < (uint32_t)EL_DENSE && b < (uint32_t)EL_DENSE) dense[a * EL_DENSE + b] = make_uint2(y, z);
    uint32_t i = (key * 0x9E3779B1u) >> shift;
    while (h[i].x != EMPTY_KEY) i = (i + 1) & (cap - 1);
    h[i] = make_uint4(key, y, z, 0);
  }
  CK(e->d_lt.reserve(cap));
  CK(cudaMemcpyAsync(e->d_lt.p, h.data(), (size_t)cap * sizeof(uint4), cudaMemcpyHostToDevice, e->stream));
  CK(e->d_lt_dense.reserve(dense.size()));
  CK(cudaMemcpyAsync(e->d_lt_dense.p, dense.data(), dense.size() * sizeof(uint2), cudaMemcpyHostToDevice, e->stream));
  CK(e->d_rule_c.reserve(rule_c.size()));
  CK(cudaMemcpyAsync(e->d_rule_c.p, rule_c.data(), rule_c.size() * sizeof(uint16_t), cudaMemcpyHostToDevice, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  e->lt_cap = cap;
  e->lt_c_affine = m ? (int32_t)rule_c[0] : 0;
  for (size_t r = 0; r < m; r++)
    if ((int64_t)rule_c[r] != (int64_t)rule_c[0] + (int64_t)r) e->lt_c_affine = -1;
  e->lt_dirty = false;
  return BPE_OK;
}

template <int LMAX, int WARPS>
int launch_encode_lanes(bpe_engine* e, const int32_t* dev_ids, const int64_t* dev_doc_off, int64_t n_docs, const uint32_t* range_first,
                        uint32_t n_ranges, const LaneTables& lt, int32_t* out_tmp, uint32_t* out_len, uint32_t* n_long, uint32_t* err,
                        uint32_t* next_range) {
  size_t smem = (size_t)2 * EL_DENSE * EL_DENSE * 4 + (size_t)WARPS * (LMAX * 32 * 2 + LMAX * 16) * 4;
  auto kern = k_encode_lanes<LMAX, WARPS>;
  const uint32_t inst_bit = 1u << (LMAX / 4 - 4);  // LMAX = 16, 20, 24, 32, 48 (one WARPS each): bits 0, 1, 2, 4, 8
  if (!(e->lanes_attr_set & inst_bit)) {
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    e->lanes_attr_set |= inst_bit;
  }
  int per_sm = 1;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, WARPS * 32, smem));
  per_sm = std::max(per_sm, 1);
  int64_t blocks = std::min<int64_t>(((int64_t)n_ranges + WARPS - 1) / WARPS, (int64_t)e->sm_count * per_sm);
  kern<<<(int)std::max<int64_t>(blocks, 1), WARPS * 32, smem, e->stream>>>(dev_ids, dev_doc_off, n_docs, range_first, n_ranges, lt, out_tmp,
                                                                       out_len, n_long, err, next_range);
  CKL();
  return BPE_OK;
}


// streams, events and pinned flag words of the host-buffer encode pipeline (encode_pipeline below)
int ensure_pipe(bpe_engine* e) {
  if (e->h_pipe) return BPE_OK;
  CK(cudaStreamCreateWithFlags(&e->s_in, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&e->s_out, cudaStreamNonBlocking));
  for (cudaEvent_t* ev : {&e->ev_in[0], &e->ev_in[1], &e->ev_in[2], &e->ev_done, &e->ev_res[0], &e->ev_res[1]})
    CK(cudaEventCreateWithFlags(ev, cudaEventDisableTiming));
  if (const char* v = getenv("BPE_ENC_CHUNK"))
    if (atoll(v) > 0) e->enc_chunk = atoll(v);
  CK(cudaHostAlloc((void**)&e->h_pipe, 16 * sizeof(unsigned long long), cudaHostAllocMapped | cudaHostAllocPortable));
  return BPE_OK;
}

// device-resident encode; leaves compacted output in dev_out / dev_out_offsets
int encode_dev(bpe_engine* e, EncodeScratch& sc, const int32_t* dev_ids, const int64_t* dev_doc_off, int64_t n_docs,
               int64_t n_ids, int64_t max_doc_len, const int32_t* dev_tvi, int32_t n_tvi, int32_t* dev_out,
               int64_t* dev_out_offsets, int64_t* dev_first_bad, int64_t* n_out, const std::function<int()>* overlap = nullptr) {
  // `overlap`: host work of the caller that runs while the lane kernel does (the encode pipeline prepares its next chunk there)
  int overlap_rc = BPE_OK;
  if (e->h_merges.size() / 3 > EL_MAX_RANK + 1) return fail(e, BPE_E_DOMAIN, "merge list too long");
  TRY(ensure_lane_tables(e));
  TRY(ensure_pipe(e));
  CK(sc.out_tmp.reserve((size_t)std::max<int64_t>(n_ids, 1)));
  CK(sc.out_len.reserve((size_t)n_docs + 1));
  CK(sc.out_off.reserve((size_t)n_docs + 2));
  CK(sc.flags.reserve(4));
  if (!e->ev0) {
    CK(cudaEventCreate(&e->ev0));
    CK(cudaEventCreate(&e->ev1));
  }
  CK(cudaEventRecord(e->ev0, e->stream));
  bool run_old = e->enc_force_old != 0;
  if (n_docs > 0 && !run_old) {
    // lane path: one warp per batch of whole documents; position ranges of `stride` ids name the batches
    // rows per lane: the smallest batch that still holds the longest document keeps the most warps resident (the kernel is
    // latency bound: 26.4 GB/s with 20 rows / 32 warps per SM vs 22.5 GB/s with 32 rows / 20 warps on the 1 GB text)
    int lmax = e->enc_lmax;
    if (!e->enc_lmax_forced) lmax = max_doc_len <= 512 ? 16 : max_doc_len <= 640 ? 20 : max_doc_len <= 768 ? 24 : max_doc_len <= 1024 ? 32 : 48;
    const uint32_t cap = 32u * (uint32_t)lmax;
    uint32_t stride = 4u * cap;  // a range = the documents starting in `stride` consecutive positions, packed greedily into batches
    uint64_t nr64 = ((uint64_t)n_ids + stride - 1) / stride;
    if (nr64 == 0) nr64 = 1;
    if (nr64 > 0x7FFFFFF0ull || n_docs > 0x7FFFFFF0ll) return fail(e, BPE_E_DOMAIN, "batch too large for one encode call");
    uint32_t n_ranges = (uint32_t)nr64;
    CK(sc.range_first.reserve((size_t)n_ranges + 1));
    CK(cudaMemsetAsync(sc.flags.p, 0, 4 * sizeof(uint32_t), e->stream));
    k_range_starts<<<(int)std::min<uint32_t>((n_ranges + 256) / 256, (uint32_t)e->sm_count * 8), 256, 0, e->stream>>>(dev_doc_off, n_docs, stride, n_ranges,
                                                                                                             sc.range_first.p);
    CKL();
    LaneTables lt{e->d_lt.p, e->lt_cap - 1, (uint32_t)(32 - ilog2(e->lt_cap)), e->d_lt_dense.p, e->d_rule_c.p, e->lt_c_affine};
    e->stats.encode_path = 2;
    if (lmax == 16)
      TRY((launch_encode_lanes<16, 20>(e, dev_ids, dev_doc_off, n_docs, sc.range_first.p, n_ranges, lt, sc.out_tmp.p, sc.out_len.p, sc.flags.p, sc.flags.p + 1, sc.flags.p + 2)));
    else if (lmax == 20)
      TRY((launch_encode_lanes<20, 16>(e, dev_ids, dev_doc_off, n_docs, sc.range_first.p, n_ranges, lt, sc.out_tmp.p, sc.out_len.p, sc.flags.p, sc.flags.p + 1, sc.flags.p + 2)));
    else if (lmax == 24)
      TRY((launch_encode_lanes<24, 13>(e, dev_ids, dev_doc_off, n_docs, sc.range_first.p, n_ranges, lt, sc.out_tmp.p, sc.out_len.p, sc.flags.p, sc.flags.p + 1, sc.flags.p + 2)));
    else if (lmax == 32)
      TRY((launch_encode_lanes<32, 10>(e, dev_ids, dev_doc_off, n_docs, sc.range_first.p, n_ranges, lt, sc.out_tmp.p, sc.out_len.p, sc.flags.p, sc.flags.p + 1, sc.flags.p + 2)));
    else
      TRY((launch_encode_lanes<48, 6>(e, dev_ids, dev_doc_off, n_docs, sc.range_first.p, n_ranges, lt, sc.out_tmp.p, sc.out_len.p, sc.flags.p, sc.flags.p + 1, sc.flags.p + 2)));
    volatile uint32_t* hf = reinterpret_cast<volatile uint32_t*>(e->h_pipe + 12);  // flags[0..1], written by the device (k_copy_u64)
    k_copy_u64<<<1, 32, 0, e->stream>>>(e->h_pipe + 12, reinterpret_cast<const unsigned long long*>(sc.flags.p), 1);
    CKL();
    if (overlap) {
      overlap_rc = (*overlap)();
      overlap = nullptr;
    }
    CK(cudaStreamSynchronize(e->stream));
    if (overlap_rc != BPE_OK) return overlap_rc;
    if (hf[1]) return fail(e, BPE_E_INTERNAL, "encode rounds did not converge");
    run_old = hf[0] != 0;
  }
  if (e->enc_force_old) e->stats.encode_path = 3;
  if (n_docs > 0 && run_old) {
    // per-document kernel: documents longer than a lane batch (marked EL_LONG), or everything when forced
    TRY(ensure_merge_table(e));
    if (max_doc_len > ENC_WARP_MAX) {
      CK(sc.g_tok.reserve((size_t)n_ids));
      CK(sc.g_nxt.reserve((size_t)n_ids));
      CK(sc.g_prv.reserve((size_t)n_ids));
      CK(sc.g_rk.reserve((size_t)n_ids));
      CK(sc.g_sel.reserve((size_t)n_ids));
    }
    EncTables mt{MergeTable{e->d_mt.p, e->mt_cap - 1, (uint32_t)(32 - ilog2(e->mt_cap))}, e->d_minlr.p};
    int64_t blocks = std::min<int64_t>((n_docs + ENC_WARPS - 1) / ENC_WARPS, (int64_t)e->sm_count * 16);
    k_encode<<<(int)blocks, ENC_THREADS, 0, e->stream>>>(dev_ids, dev_doc_off, n_docs, mt, sc.out_tmp.p, sc.out_len.p, sc.g_tok.p, sc.g_nxt.p, sc.g_prv.p,
                                                         sc.g_rk.p, sc.g_sel.p, e->enc_force_old ? 0 : 1);
    CKL();
  }
  if (n_docs <= 65536) {
    k_scan_counts<<<1, 1024, 0, e->stream>>>(sc.out_len.p, sc.out_off.p, (uint32_t)n_docs);
    CKL();
  } else {
    uint32_t n_tiles = (uint32_t)((n_docs + SC_TILE - 1) / SC_TILE);
    CK(sc.tile_sums.reserve(n_tiles));
    CK(sc.tile_off.reserve((size_t)n_tiles + 1));
    k_sum_tiles<<<n_tiles, SC_THREADS, 0, e->stream>>>(sc.out_len.p, (uint32_t)n_docs, sc.tile_sums.p);
    CKL();
    k_scan_counts<<<1, 1024, 0, e->stream>>>(sc.tile_sums.p, sc.tile_off.p, n_tiles);
    CKL();
    k_scan_tiles<<<n_tiles, SC_THREADS, 0, e->stream>>>(sc.out_len.p, (uint32_t)n_docs, sc.tile_off.p, n_tiles, sc.out_off.p);
    CKL();
  }
  {
    int64_t warps = n_docs + 1;
    int64_t blocks = std::min<int64_t>((warps + 3) / 4, (int64_t)e->sm_count * 16);
    k_gather_map<<<(int)blocks, 128, 0, e->stream>>>(sc.out_tmp.p, dev_doc_off, sc.out_off.p, n_docs, dev_tvi, n_tvi, dev_out, dev_out_offsets, dev_first_bad);
    CKL();
  }
  CK(cudaEventRecord(e->ev1, e->stream));
  if (overlap) overlap_rc = (*overlap)();  // the lane kernel did not run
  k_copy_u64<<<1, 32, 0, e->stream>>>(e->h_pipe + 13, reinterpret_cast<const unsigned long long*>(sc.out_off.p + n_docs), 1);
  CKL();
  CK(cudaStreamSynchronize(e->stream));
  if (overlap_rc != BPE_OK) return overlap_rc;
  const uint64_t total = *reinterpret_cast<volatile unsigned long long*>(e->h_pipe + 13);
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, e->ev0, e->ev1));
  e->stats.ms_encode = ms;
  *n_out = (int64_t)total;
  return BPE_OK;
}

int check_offsets(bpe_engine* e, const int64_t* off, int64_t n_docs) {
  if (n_docs < 0 || (!off && n_docs > 0)) return fail(e, BPE_E_INVALID, "bad document offsets");
  for (int64_t d = 0; d < n_docs; d++)
    if (off[d + 1] < off[d]) return fail(e, BPE_E_INVALID, "document offsets must be non-decreasing (doc %lld)", (long long)d);
  return BPE_OK;
}

// append ids (device pointer, already merged or raw) as documents
int append_docs_dev(bpe_engine* e, const int32_t* dev_ids, const int64_t* host_off, int64_t n_docs) {
  int64_t base_in = host_off[0];
  int64_t total = host_off[n_docs] - base_in;
  uint64_t new_n = e->n_slots + (uint64_t)total;
  if (new_n >= 0xFFFFFFF0ull) return fail(e, BPE_E_DOMAIN, "corpus exceeds 2^32 positions per engine");
  CK(e->slots.reserve((size_t)new_n + 4, (size_t)e->n_slots, e->stream, 1.5));
  CK(e->d_st.reserve(1));
  if (total > 0) {
    CK(cudaMemsetAsync(&e->d_st.p->err, 0, sizeof(uint32_t), e->stream));
    int blocks = (int)std::min<int64_t>((total / 4 + 255) / 256 + 1, (int64_t)e->grid(8));
    if (reinterpret_cast<const uint32_t*>(dev_ids + base_in) == e->slots.p + e->n_slots)
      k_validate_ids<<<blocks, 256, 0, e->stream>>>(e->slots.p + e->n_slots, (uint64_t)total, (uint32_t)e->n_tokens, &e->d_st.p->err);
    else
      k_ingest_ids<<<blocks, 256, 0, e->stream>>>(dev_ids + base_in, e->slots.p + e->n_slots, (uint64_t)total, (uint32_t)e->n_tokens, &e->d_st.p->err);
    CKL();
    CK(e->stage_off.reserve((size_t)n_docs + 1, 0, e->stream, 1.5));
    CK(cudaMemcpyAsync(e->stage_off.p, host_off, (size_t)(n_docs + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, e->stream));
    int blocks2 = (int)std::min<int64_t>((n_docs + 255) / 256, (int64_t)e->grid(8));
    k_mark_docstarts<<<blocks2, 256, 0, e->stream>>>(e->slots.p, e->stage_off.p, n_docs, (int64_t)e->n_slots - base_in);
    CKL();
    uint32_t bad = 0;
    CK(cudaMemcpyAsync(&bad, &e->d_st.p->err, sizeof bad, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    if (bad) {
      CK(cudaMemsetAsync(&e->d_st.p->err, 0, sizeof(uint32_t), e->stream));
      return fail(e, BPE_E_INVALID, "document holds a token index >= n_tokens (%d); call bpe_set_tokens first", e->n_tokens);
    }
  }
  for (int64_t d = 0; d < n_docs; d++) e->doc_off.push_back((int64_t)e->n_slots + (host_off[d + 1] - base_in));
  e->n_slots = new_n;
  e->live_tokens += (uint64_t)total;
  e->index_valid = false;
  e->hot_valid = false;
  return BPE_OK;
}


// buffers of k_merge_rounds (round_kernels.cuh): delta cells, slot rows, per-block cell lists, site buffers, partials
int ensure_round_buffers(bpe_engine* e) {
  if (!e->round_blocks) {
    int per_sm = 0;
    CK(cudaFuncSetAttribute(k_merge_rounds, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)R_STAGE_BYTES));  // the staged cells
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_merge_rounds, RD_THREADS, R_STAGE_BYTES));
    if (per_sm < 1) return fail(e, BPE_E_CUDA, "k_merge_rounds does not fit on an SM");
    // (a decision folds RT partial entries per block with one thread each)
    const int most = std::min({e->sm_count * per_sm, (int)(R_QCAP / RT), RD_THREADS / RT});
    e->round_blocks = std::min(e->sm_count, most);
    if (const char* v = getenv("BPE_LOOP_BLOCKS")) e->round_blocks = std::max(1, std::min(atoi(v), most));
  }
  const size_t cells = (size_t)2 * RB * 2 * ND_STRIDE;
  if (!e->r_cells.p) {
    CK(e->r_cells.reserve(cells));
    CK(cudaMemsetAsync(e->r_cells.p, 0, cells * 8, e->stream));  // the kernel keeps the cells zero between launches
    CK(e->r_slotrows.reserve(cells));
    CK(e->r_lists.reserve((size_t)2 * e->round_blocks * R_LISTCAP));
    CK(e->r_bsites.reserve((size_t)2 * RB * R_SMALL));
    CK(e->r_state.reserve(1));
    CK(cudaMemsetAsync(e->r_state.p, 0, sizeof(RoundState), e->stream));
  }
  if (e->mg_world > 1 && !e->r_gcells.p) {
    CK(e->r_gcells.reserve(cells));
    CK(cudaMemsetAsync(e->r_gcells.p, 0, cells * 8, e->stream));
    CK(e->r_glists.reserve((size_t)2 * e->round_blocks * R_LISTCAP));
  }
  CK(e->r_gp.reserve((size_t)RT * e->round_blocks));
  CK(e->r_gk.reserve((size_t)RT * e->round_blocks));
  return BPE_OK;
}

// a merge whose occurrence list is longer than this stages its frequent neighbours' deltas and list cells per block
// (LoopArgs::stage_min, read where each LoopArgs is built)
uint32_t stage_min_knob() {
  if (const char* v = getenv("BPE_BLOCK_CELLS_MIN_SITES")) return (uint32_t)std::max(0ll, std::min(atoll(v), 0xFFFFFFFFll));  // tuning / tests
  return R_STAGE_MIN_DEFAULT;
}

RoundArgs round_args(bpe_engine* e, const LoopArgs& L, int round_k) {
  RoundArgs RA{};
  RA.L = L;
  RA.cells = e->r_cells.p;
  RA.slotrows = e->r_slotrows.p;
  RA.lists = e->r_lists.p;
  RA.bsites = e->r_bsites.p;
  RA.gp = e->r_gp.p;
  RA.gk = e->r_gk.p;
  RA.rs = e->r_state.p;
  RA.kmax = (uint32_t)round_k;
  RA.bar_mode = 1;
  if (const char* v = getenv("BPE_LOOP_BAR")) RA.bar_mode = atoi(v) ? 1 : 0;
  RA.mg_on = 0;
  RA.gcells = e->r_gcells.p;
  RA.glists = e->r_glists.p;
  return RA;
}

void round_stats(bpe_engine* e, const RoundState& hrs) {
  e->stats.loop_rounds = (int64_t)hrs.rounds;
  e->stats.loop_round_merges = (int64_t)hrs.round_merges;
  e->stats.loop_round_tried = (int64_t)hrs.tried;
  e->stats.loop_rounds_cut = (int64_t)hrs.rounds_cut_born;
}

// ---- mergeUntil: persistent cooperative kernels, the host only grows buffers / rebuilds the hot list ----------------------------
// One driver serves one GPU, the batched replay (the winners are given) and every rank of a sharded corpus (mg), where the ranks run
// it in step: their kernels leave at the same merge with the same status.

// the sharded kernels' view of the mailboxes: this rank's place, every peer's flags, inbox and tie mailbox
MgArgs mg_args(bpe_engine* e) {
  MgArgs M{};
  M.rank = e->mg_rank;
  M.world = e->mg_world;
  M.inbox_stride = e->mg_inbox_stride;
  M.tie_cap = e->mg_tie_cap;
  const size_t flags_bytes = (size_t)MG_MAX_WORLD * 128;
  const size_t inbox_bytes = (size_t)2 * e->mg_world * e->mg_inbox_stride * 8;
  for (int q = 0; q < e->mg_world; q++) {
    char* base = static_cast<char*>(e->mg_peer[q]);
    M.flag_data[q] = reinterpret_cast<unsigned long long*>(base);
    M.flag_tie[q] = reinterpret_cast<unsigned long long*>(base + flags_bytes);
    M.inbox[q] = reinterpret_cast<unsigned long long*>(base + 2 * flags_bytes);
    M.tiebox[q] = reinterpret_cast<uint32_t*>(base + 2 * flags_bytes + inbox_bytes);
  }
  M.tie_sorted = e->mg_tie_sorted.p;
  M.newpair = e->mg_newpair.p;
  M.newpair_cap = (uint32_t)e->mg_newpair.cap;
  return M;
}

double ms_since(std::chrono::steady_clock::time_point t) {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t).count();
}

// the arguments of one launch; a sharded engine stages its count deltas (dlt, touched) and lists the pairs born on any rank
LoopArgs loop_args(bpe_engine* e, bool mg, bool use_rounds, uint32_t chunk, uint32_t ml, int64_t mw) {
  LoopArgs L{};
  L.A = apply_args(e);
  if (mg) {
    L.A.newpair = e->mg_newpair.p;
    L.A.newpair_cap = (uint32_t)e->mg_newpair.cap;
    L.A.dlt = e->mg_dlt.p;
    L.A.touched = e->mg_touched.p;
    L.A.touched_cap = (uint32_t)e->mg_touched.cap;
  }
  L.pool_cap = e->pool.cap;
  L.len16_cap = (uint32_t)std::min<size_t>(e->d_len16.cap, 0xFFFFFFF0u);
  L.hot = e->hot.p;
  L.hot_cap = (uint32_t)std::min<size_t>(e->hot.cap, 0xFFFFFFF0u);
  L.hot_limit = e->hot_limit;
  L.cands = e->cands.p;
  L.cand_cap = (uint32_t)std::min<size_t>(e->cands.cap, 0xFFFFFFF0u);
  L.partials = e->partials.p;
  L.partial_keys = e->partial_keys.p;
  L.barrier = e->barrier.p;
  L.log = e->dev_log.p;
  L.log_cap = chunk;
  L.max_length = ml;
  L.min_weight = (uint32_t)std::min<int64_t>(mw, 0xFFFFFFFFll);
  L.max_tokens = BPE_MAX_TOKENS;
  L.tbl_cap = e->tbl_cap;
  L.stage_min = stage_min_knob();
  // warp split of the latency-bound phases, barrier back-off and prefetch depth (tuning knobs, read per launch).
  // measured on cfg3 (profiles/r01i): born pairs / rewrite / old-hot arg-max = 10/2/4 warps beats 8/4/4 by 1 %, 6/x loses 1-2 %;
  // 10..14 site warps and 64..512 ns of back-off are all within noise
  int a = 12, b = 10, c = 2, ns = 256, pf = 0;
  if (!mg) {  // (the sweeps that set these ran on one GPU: the sharded loop keeps the defaults of the rounds)
    if (const char* v = getenv("BPE_LOOP_P1_SITES")) a = atoi(v);
    if (const char* v = getenv("BPE_LOOP_P2_NEW")) b = atoi(v);
    if (const char* v = getenv("BPE_LOOP_P2_RW")) c = atoi(v);
    if (const char* v = getenv("BPE_LOOP_BAR_NS")) ns = atoi(v);
    const char* v = getenv("BPE_LOOP_PREFETCH");
    pf = v ? std::max(0, std::min(atoi(v), 2)) : (use_rounds ? 0 : 1);  // (k_merge_rounds: measured, the helper warps become the tail)
  }
  if (a < 1 || a > 15) a = 12;
  if (b < 1 || c < 1 || b + c > 15) b = 10, c = 2;
  L.p1_sites = (uint32_t)a;
  L.p2_new = (uint32_t)b;
  L.p2_rw = (uint32_t)c;
  L.bar_ns = (uint32_t)std::max(32, std::min(ns, 4096));
  L.prefetch = pf;
  return L;
}

// one launch: k_merge_rounds, or the one-merge kernel (k_merge_loop, k_merge_loop_mg).  `above`: the winner has more sites than the
// packed delta cells of a round can count, so the one-merge kernel takes the merges above R_HUGE -- it stops, "done", at the first
// winner at or below it -- and the rounds continue from there
cudaError_t launch_merge_loop(bpe_engine* e, bool mg, LoopArgs L, bool rounds, bool above, int64_t mw, int round_k) {
  if (!mg || rounds) {  // the second site buffer, which k_merge_loop_mg does not use
    L.sites2 = e->sites2.p;
    L.A.sites_cap = (uint32_t)std::min<size_t>(L.A.sites_cap, e->sites2.cap);
  }
  if (rounds) {
    RoundArgs RA = round_args(e, L, round_k);
    if (mg) {
      RA.mg_on = 1;
      RA.mg = mg_args(e);
    }
    k_rounds_prepare<<<1, 32, 0, e->stream>>>(e->r_state.p);
    e->stats.kernel_launches++;
    void* args[] = {&RA};
    return cudaLaunchCooperativeKernel((void*)k_merge_rounds, dim3(e->round_blocks), dim3(RD_THREADS), args, R_STAGE_BYTES, e->stream);
  }
  if (above) L.min_weight = (uint32_t)std::max<int64_t>(mw, (int64_t)R_HUGE + 1);
  if (mg) {
    LoopArgsMg P{L, mg_args(e)};
    void* args[] = {&P};
    return cudaLaunchCooperativeKernel((void*)k_merge_loop_mg, dim3(e->mg_loop_blocks), dim3(ML_THREADS), args, 0, e->stream);
  }
  void* args[] = {&L};
  return cudaLaunchCooperativeKernel((void*)k_merge_loop, dim3(e->loop_blocks), dim3(ML_THREADS), args, 0, e->stream);
}

// appends the `iters` merges of the last launch to the caller's log and to the host's token lengths and merge list
int read_merge_log(bpe_engine* e, uint32_t iters, bpe_merge* log, int64_t* done, std::vector<MergeRec>& tmp) {
  tmp.resize(iters);
  cudaError_t ce = cudaMemcpyAsync(tmp.data(), e->dev_log.p, (size_t)iters * sizeof(MergeRec), cudaMemcpyDeviceToHost, e->stream);
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(e->stream);
  if (ce != cudaSuccess) return fail(e, BPE_E_CUDA, "merge log read-back: %s", cudaGetErrorString(ce));
  for (const MergeRec& r : tmp) {
    bpe_merge& m = log[(*done)++];
    m.a = r.a;
    m.b = r.b;
    m.c = r.c;
    m.reserved = 0;
    m.weight = r.weight;
    e->h_len16.push_back(e->h_len16[r.a] + e->h_len16[r.b]);
    e->h_merges.push_back(r.a);
    e->h_merges.push_back(r.b);
    e->h_merges.push_back(r.c);
  }
  e->n_tokens += (int32_t)iters;
  e->mt_dirty = e->lt_dirty = true;
  e->stats.merges_applied += iters;
  return BPE_OK;
}

// LOOP_NEED_HOST: grow the pair table, the occurrence pool and the merge buffers for the winner the kernel stopped at.  On a sharded
// corpus every rank is here with the same winner, and each one grows what IT lacks.
int grow_merge_buffers(bpe_engine* e, bool mg, bool use_rounds, bool trace) {
  if (e->n_tokens >= BPE_MAX_TOKENS) return fail(e, BPE_E_DOMAIN, "token table would exceed %d", BPE_MAX_TOKENS);
  const uint64_t w = e->h_st->best_cnt;
  const uint64_t new_keys = std::min<uint64_t>(2 * w + 2, 2 * ((uint64_t)e->n_tokens + 1) + 2);
  const uint64_t keys_after = (uint64_t)e->h_st->n_keys + new_keys;
  if (keys_after * 2 > e->tbl_cap) {
    uint64_t want = std::min<uint64_t>(keys_after * 5 / 2, 0x80000000ull);  // next power of two: load 0.2 .. 0.4
    // a run over a big corpus ends with distinct pairs ~ 5 % of its positions (48 M for the 1 GB Zipf corpus): the first
    // growth goes most of the way instead of doubling eleven times (a relaunch + rehash each).  (A sharded table holds the
    // pairs of every shard.)
    want = std::max<uint64_t>(want, std::min<uint64_t>(e->n_slots * e->mg_world / 16, 1ull << 27));
    if (keys_after * 2 > pow2_at_least(want)) return fail(e, BPE_E_NOMEM, "pair table cannot grow further");
    const auto tt = std::chrono::steady_clock::now();
    TRY(grow_table(e, pow2_at_least(want)));
    if (mg && trace) fprintf(stderr, "[bpe r%d] grow_table -> %u slots: %.1f ms\n", e->mg_rank, e->tbl_cap, ms_since(tt));
  }
  // the in-kernel test is one merge conservative: one GPU reserves 2w cells past the cursor.  A sharded rank reserves 4w, and with
  // rounds one ROUND conservative there: the first merge of a round has at most R_HUGE sites (larger ones take the other kernel),
  // the previous round's batch -- whose allocation the figure in the header does not show yet -- at most as many.
  uint64_t pool_after = (uint64_t)e->h_st->pool_cursor + (mg ? 4 : 2) * w;
  if (use_rounds)  // every block of k_merge_rounds may open a private chunk
    pool_after += mg ? 2ull * R_HUGE + 2ull * std::max(R_HUGE, R_BATCH_SITES) + 2ull * e->round_blocks * R_POOL_CHUNK
                     : (uint64_t)e->round_blocks * R_POOL_CHUNK;
  // (the hot list of a sharded rank takes both the pairs born on its shard and those that only the peers' records bring)
  const auto tp = std::chrono::steady_clock::now();
  cudaError_t ce;
  if ((ce = e->pool.reserve((size_t)pool_after, e->h_st->pool_cursor, e->stream, 1.5)) != cudaSuccess ||
      (ce = e->sites.reserve((size_t)w, 0, e->stream, 1.25)) != cudaSuccess ||
      ((!mg || use_rounds) && (ce = e->sites2.reserve(e->sites.cap, 0, e->stream, 1.0)) != cudaSuccess) ||
      (ce = e->newslots.reserve((size_t)new_keys, 0, e->stream, 1.25)) != cudaSuccess ||
      (ce = e->hot.reserve((size_t)e->h_st->hot_n + (mg ? 2 : 1) * new_keys, e->h_st->hot_n, e->stream, 1.5)) != cudaSuccess ||
      (ce = e->cands.reserve((size_t)e->h_st->best_mult, 0, e->stream, 1.5)) != cudaSuccess)
    return fail(e, BPE_E_NOMEM, "growing merge buffers: %s", cudaGetErrorString(ce));
  if (mg && trace && ms_since(tp) > 1.0) fprintf(stderr, "[bpe r%d] buffer growth (pool %zu cells): %.1f ms\n", e->mg_rank, e->pool.cap, ms_since(tp));
  if (mg && e->h_st->best_mult > e->mg_tie_cap)  // (the ranks settle a tie through the tie mailbox)
    return fail(e, BPE_E_DOMAIN, "%u pairs tie on (weight, index sum): more than the tie mailbox holds (%u)", e->h_st->best_mult, e->mg_tie_cap);
  return BPE_OK;
}

int merge_until(bpe_engine* e, int64_t min_weight, int32_t max_length, int64_t max_iterations, bpe_merge* log, int64_t log_cap,
                int64_t* n_done, const int32_t* dev_replay = nullptr) {
  const bool mg = e->mg_world > 1;
  *n_done = 0;
  e->mg_timed_out = false;  // (a verdict about this call only)
  struct LeaveGate {  // a group member leaves the launch gate on every exit, so that its peers never wait for it there
    LaunchGate* gate;
    ~LeaveGate() {
      if (gate) gate->drop();
    }
  } leave_gate{e->mg_gate};
  CK(cudaSetDevice(e->device));
  if (mg) {  // (no early return on an empty shard: its peers wait for it in every exchange)
    if (!e->mg_connected) return fail(e, BPE_E_INVALID, "sharded engine: call bpe_mg_connect first");
  } else if (e->n_slots == 0) {
    return BPE_OK;
  }
  TRY(ensure_index(e));
  if (mg && !e->mg_counts_global)
    return fail(e, BPE_E_INVALID, "sharded engine: exchange the pair counts first (bpe_mg_export_counts / bpe_mg_import_counts)");
  const uint32_t ml = max_length > 0 ? (uint32_t)max_length : 0;
  const int64_t mw = min_weight > 0 ? min_weight : 2;
  int& loop_blocks = mg ? e->mg_loop_blocks : e->loop_blocks;
  if (!loop_blocks) {
    int per_sm = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mg ? (const void*)k_merge_loop_mg : (const void*)k_merge_loop, ML_THREADS, 0));
    if (per_sm < 1) return fail(e, BPE_E_CUDA, "%s does not fit on an SM", mg ? "k_merge_loop_mg" : "k_merge_loop");
    // one 512-thread block per SM: measured best on cfg3 (1.28 s vs 1.41 s with two per SM, 1.33 s with half an SM count,
    // 1.55 s with 1024-thread blocks) -- a merge is latency bound, fewer arrivals per grid barrier and fewer partials win
    int want = 1;
    if (const char* v = getenv("BPE_LOOP_PER_SM")) want = std::max(1, atoi(v));  // tuning knob: co-resident blocks per SM
    loop_blocks = e->sm_count * std::min(per_sm, want);
    const char* v = getenv("BPE_LOOP_BLOCKS");  // (a single-GPU knob: it has never sized k_merge_loop_mg's grid)
    if (v && !mg) loop_blocks = std::max(1, std::min(atoi(v), e->sm_count * per_sm));
  }
  // several exact merges per barrier round (round_kernels.cuh; on a sharded corpus ONE exchange per round) unless a merge list is
  // replayed; BPE_LOOP_ROUNDS=0 keeps the one-merge kernel
  bool use_rounds = !dev_replay;
  int round_k = RB;
  if (const char* v = getenv("BPE_LOOP_ROUNDS")) use_rounds = use_rounds && atoi(v) != 0;
  if (const char* v = getenv("BPE_LOOP_K")) round_k = std::max(1, std::min(atoi(v), (int)RB));
  if (use_rounds) TRY(ensure_round_buffers(e));
  CK(e->partials.reserve((size_t)std::max(loop_blocks, e->grid(8))));
  CK(e->sites.reserve(1u << 16, 0, e->stream, 1.0));
  if (!mg || use_rounds) CK(e->sites2.reserve(std::max<size_t>(e->sites.cap, 1u << 16), 0, e->stream, 1.0));  // (not read by k_merge_loop_mg)
  CK(e->newslots.reserve(mg ? 1u << 17 : 1u << 16, 0, e->stream, 1.0));
  CK(e->cands.reserve(4096, 0, e->stream, 1.0));
  CK(e->barrier.reserve(64));
  if (mg) {  // the staged deltas' cell list, the sorted tie mailbox, the pairs born on any rank
    CK(e->mg_touched.reserve((size_t)4 * BPE_MAX_TOKENS + 64));
    CK(e->mg_tie_sorted.reserve(e->mg_tie_cap));
    CK(e->mg_newpair.reserve((size_t)2 * BPE_MAX_TOKENS + 64));
  } else {
    CK(e->partial_keys.reserve((size_t)std::max(loop_blocks, e->grid(8))));  // (read by k_merge_loop only)
  }
  static const bool trace = getenv("BPE_TRACE") != nullptr;
  cudaEvent_t t0, t1;
  CK(cudaEventCreate(&t0));
  CK(cudaEventCreate(&t1));
  CK(cudaEventRecord(t0, e->stream));
  int rc = BPE_OK;
  int64_t done = 0;
  bool legacy_above = false;
  std::vector<MergeRec> tmp;
  double host_ms[4] = {0, 0, 0, 0};  // hot rebuilds, growth (NEED_HOST), launch+state fetch, log read-back
  for (;;) {
    int64_t remaining = log_cap - done;
    if (max_iterations > 0) remaining = std::min(remaining, max_iterations - done);  // core.ts:374-377
    if (remaining <= 0) break;
    if (!dev_replay && (!e->hot_valid || e->hot_max_length != ml)) {
      bool any = false;
      const auto th = std::chrono::steady_clock::now();
      rc = rebuild_hot(e, ml, &any);
      host_ms[0] += ms_since(th);
      if (rc != BPE_OK) break;
      if (!any) break;  // nothing countable left, on ANY rank of a sharded corpus: the counts are global (core.ts:312)
    }
    uint32_t chunk = (uint32_t)std::min<int64_t>(remaining, 1 << 16);
    if (e->n_tokens + (int64_t)chunk > BPE_MAX_TOKENS) chunk = (uint32_t)std::max<int64_t>(0, BPE_MAX_TOKENS - e->n_tokens);
    if (chunk == 0) {
      rc = fail(e, BPE_E_DOMAIN, "token table would exceed %d", BPE_MAX_TOKENS);
      break;
    }
    cudaError_t ce;
    if ((ce = e->dev_log.reserve(chunk)) != cudaSuccess ||
        (ce = e->d_len16.reserve((size_t)e->n_tokens + chunk + 1, (size_t)e->n_tokens, e->stream, 1.5)) != cudaSuccess) {
      rc = fail(e, BPE_E_NOMEM, "%s", cudaGetErrorString(ce));
      break;
    }
    LoopArgs L = loop_args(e, mg, use_rounds, chunk, ml, mw);
    L.replay = dev_replay ? dev_replay + 2 * done : nullptr;
    if (dev_replay) e->hot_valid = false;  // replayed merges do not feed the hot list
    const auto tw0 = std::chrono::steady_clock::now();
    if (e->mg_gate) e->mg_gate->arrive();
    k_loop_prepare<<<1, 32, 0, e->stream>>>(e->d_st.p, (uint32_t)e->n_tokens, e->barrier.p);
    e->stats.kernel_launches++;
    ce = launch_merge_loop(e, mg, L, use_rounds && !legacy_above, use_rounds && legacy_above, mw, round_k);
    if (ce != cudaSuccess) {
      rc = fail(e, BPE_E_CUDA, "cooperative launch of the %smergeUntil kernel: %s", mg ? "sharded " : "", cudaGetErrorString(ce));
      break;
    }
    e->stats.kernel_launches++;
    if ((rc = fetch_state(e)) != BPE_OK) break;
    host_ms[2] += ms_since(tw0);
    if (mg) {  // the exchange epochs the next launch continues from
      e->mg_epoch = e->h_st->mg_epoch;
      e->mg_tie_epoch = e->h_st->mg_tie_epoch;
    }
    const uint32_t iters = e->h_st->iters_done;
    if (trace && !mg)
      fprintf(stderr, "[bpe] k_merge_loop: %u merges in %.2f ms, status %u, best_cnt %u, hot_n %u thresh %u, keys %u/%u\n", iters, ms_since(tw0),
              e->h_st->status, e->h_st->best_cnt, e->h_st->hot_n, e->h_st->hot_thresh, e->h_st->n_keys, e->tbl_cap);
    if (trace && mg)
      fprintf(stderr, "[bpe r%d] k_merge_loop_mg: %u merges in %.2f ms, status %u, best_cnt %u, hot_n %u thresh %u, keys %u/%u err 0x%x gerr 0x%x\n",
              e->mg_rank, iters, ms_since(tw0), e->h_st->status, e->h_st->best_cnt, e->h_st->hot_n, e->h_st->hot_thresh, e->h_st->n_keys, e->tbl_cap,
              e->h_st->err, e->h_st->g_vals[0]);
    const auto tl = std::chrono::steady_clock::now();
    if (iters && (rc = read_merge_log(e, iters, log, &done, tmp)) != BPE_OK) break;
    host_ms[3] += ms_since(tl);
    const uint32_t status = e->h_st->status;
    if (use_rounds && legacy_above && status == LOOP_DONE && (int64_t)e->h_st->best_cnt >= mw) {
      legacy_above = false;  // below R_HUGE now: back to the rounds
      continue;
    }
    if (status == LOOP_NEED_LEGACY) {
      legacy_above = true;
      continue;
    }
    if (status == LOOP_DONE || status == LOOP_EMPTY) break;
    if (status == LOOP_LIMIT) continue;
    if (status == LOOP_NEED_REBUILD) {
      e->hot_valid = false;
      continue;
    }
    if (status == LOOP_ERROR) {
      const uint32_t f = e->h_st->err | e->h_st->g_vals[0];
      if (mg && (f & ERR_PEER_TIMEOUT)) {  // (a group reports a member's own error ahead of the timeouts it causes in the others)
        e->mg_timed_out = true;
        rc = fail(e, BPE_E_INTERNAL, "a peer GPU did not answer within %.0f s (flags 0x%x)", MG_TIMEOUT_NS / 1e9, f);
      } else {
        rc = check_dev_err(e);
        if (rc == BPE_OK && mg)
          rc = fail(e, BPE_E_INTERNAL, "sharded merge loop stopped: local flags 0x%x, all ranks 0x%x", e->h_st->err, e->h_st->g_vals[0]);
        if (rc == BPE_OK) rc = fail(e, BPE_E_INTERNAL, "merge loop stopped with an unexplained error (flags 0x%x)", e->h_st->err);
      }
      break;
    }
    if (status == LOOP_NEED_HOST) {
      const auto tg = std::chrono::steady_clock::now();
      if ((rc = grow_merge_buffers(e, mg, use_rounds, trace)) != BPE_OK) break;
      host_ms[1] += ms_since(tg);
      // A rank whose pair table grew must rebuild its hot list (new slot numbers), and the rebuild sets a new hot_thresh.  The
      // ranks decide every merge, and when to leave the kernel (w < hot_thresh), on their own lists and thresholds, so they all
      // rebuild: table sizes follow the shard sizes, and on uneven shards only some ranks grow.
      if (mg) e->hot_valid = false;
      continue;
    }
    rc = fail(e, BPE_E_INTERNAL, "merge loop returned status %u", status);
    break;
  }
  *n_done = done;
  if (rc == BPE_OK) {
    CK(cudaEventRecord(t1, e->stream));
    TRY(fetch_state(e));
    if (!mg) TRY(check_dev_err(e));  // (a sharded run's flags reach every rank at once, through LOOP_ERROR)
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, t0, t1));
    e->stats.ms_last_merge_until = ms;
    e->live_tokens = e->h_st->live_tokens;
    e->stats.sites_merged = (int64_t)e->h_st->sites_total;
    e->stats.tie_breaks = e->h_st->tie_breaks;
    if (use_rounds) {
      RoundState hrs;
      CK(cudaMemcpyAsync(&hrs, e->r_state.p, sizeof(RoundState), cudaMemcpyDeviceToHost, e->stream));
      CK(cudaStreamSynchronize(e->stream));
      round_stats(e, hrs);
      const unsigned long long* f = e->h_st->fine_ns;
      const double ns = std::max(1.0, (double)f[5]), nb = std::max(1.0, (double)f[11]);
      if (trace && !mg) {
        fprintf(stderr, "[bpe] rounds %llu, merges %llu (tried %llu), cut by the born-pair bound %llu, single %llu; batch ends: cap %llu, no-candidate %llu, tie %llu, big %llu, "
                        "token %llu, fresh-token %llu, limits %llu\n", hrs.rounds, hrs.round_merges, hrs.tried, hrs.rounds_cut_born, hrs.rounds_single, hrs.stop_reason[0],
                hrs.stop_reason[1], hrs.stop_reason[2], hrs.stop_reason[3], hrs.stop_reason[4], hrs.stop_reason[5], hrs.stop_reason[6]);
        fprintf(stderr, "[bpe] P1 warp-iterations small %llu big %llu; touched cells small %llu big %llu; sites small %llu big %llu\n", hrs.iters_small, hrs.iters_big,
                hrs.cells_small, hrs.cells_big, hrs.sites_small, hrs.sites_big);
        const unsigned long long* m = e->h_st->mg_prof_ns;
        const double n = std::max(1.0, (double)m[4]);
        fprintf(stderr, "[bpe] P2 of rounds of small merges, block 0, us after the barrier: cells done %.1f, rewrite done %.1f, arg-max done %.1f, partials out %.1f\n",
                m[0] / n * 1e-3, m[1] / n * 1e-3, m[2] / n * 1e-3, m[3] / n * 1e-3);
        fprintf(stderr, "[bpe] block 0, us per round whose first merge has <= 16384 sites (%.0f rounds): decide %.1f, P1 %.1f, wait %.1f, P2 %.1f, wait %.1f; per round whose first merge has more (%.0f): "
                        "decide %.1f, P1 %.1f, wait %.1f, P2 %.1f, wait %.1f\n", (double)f[5], f[0] / ns * 1e-3, f[1] / ns * 1e-3, f[2] / ns * 1e-3, f[3] / ns * 1e-3, f[4] / ns * 1e-3,
                (double)f[11], f[6] / nb * 1e-3, f[7] / nb * 1e-3, f[8] / nb * 1e-3, f[9] / nb * 1e-3, f[10] / nb * 1e-3);
      }
      if (trace && mg && e->mg_rank == 0) {
        fprintf(stderr, "[bpe r0] rounds %llu, merges %llu (tried %llu); block 0, us per round whose first merge has <= 16384 sites (%.0f): decide %.1f, P1 %.1f, wait %.1f, P2 %.1f, wait %.1f; "
                        "whose first merge has more (%.0f): decide %.1f, P1 %.1f, wait %.1f, P2 %.1f, wait %.1f; exchange (emit..summed) ms %.1f\n", hrs.rounds, hrs.round_merges, hrs.tried,
                (double)f[5], f[0] / ns * 1e-3, f[1] / ns * 1e-3, f[2] / ns * 1e-3, f[3] / ns * 1e-3, f[4] / ns * 1e-3, (double)f[11], f[6] / nb * 1e-3, f[7] / nb * 1e-3,
                f[8] / nb * 1e-3, f[9] / nb * 1e-3, f[10] / nb * 1e-3, (double)e->h_st->prof_ns[5] * 1e-6);
        const unsigned long long* m = e->h_st->mg_prof_ns;
        fprintf(stderr, "[bpe r0] exchange, block 0, ms: header + records out + report %.1f, wait + sum as they arrive + fold %.1f, barrier %.1f\n", m[5] * 1e-6, m[6] * 1e-6, m[7] * 1e-6);
      }
    }
    if (trace && mg && e->mg_rank == 0) {
      fprintf(stderr, "[bpe r0] mg phases ms (decide, P1, wait, M1, wait, send+local P2, barrier+peer wait, apply, wait, P3, wait, tie):");
      for (int i = 0; i < 12; i++) fprintf(stderr, " %.1f", (double)e->h_st->mg_prof_ns[i] * 1e-6);
      fprintf(stderr, "  total %.1f ms, %lld merges; host ms: hot rebuild %.1f, growth %.1f, launch..fetch %.1f, log %.1f\n", ms, (long long)done,
              host_ms[0], host_ms[1], host_ms[2], host_ms[3]);
    }
  }
  cudaEventDestroy(t0);
  cudaEventDestroy(t1);
  return rc;
}

// mailbox of rank `rank` in a sharded corpus of `world` engines: the peers store their count deltas into it (mg_kernels.cuh)
int mg_alloc_mailbox(bpe_engine* e, int rank, int world) {
  e->mg_rank = rank;
  e->mg_world = world;
  // records one rank can send per exchange (k_merge_rounds: the cells of up to 16 merges a round; k_merge_loop_mg: of one merge)
  e->mg_inbox_stride = MG_INBOX_STRIDE;
  e->mg_tie_cap = 4096;
  size_t bytes = (size_t)2 * MG_MAX_WORLD * 128 + (size_t)2 * world * e->mg_inbox_stride * 8 + (size_t)2 * world * e->mg_tie_cap * 4;
  CK(cudaMalloc(&e->mg_mailbox, bytes));
  CK(cudaMemset(e->mg_mailbox, 0, bytes));
  e->mg_mailbox_bytes = bytes;
  e->mg_peer[rank] = e->mg_mailbox;
  e->index_valid = false;  // per-slot side arrays are allocated with the table
  return BPE_OK;
}

// a batch of restoreMerge lines (a_i, b_i) -> n_tokens + i: every operand must exist when its merge comes
int check_merge_list(bpe_engine* e, const int32_t* ab, int64_t n) {
  if ((int64_t)e->n_tokens + n > BPE_MAX_TOKENS) return fail(e, BPE_E_DOMAIN, "token table would exceed %d", BPE_MAX_TOKENS);
  for (int64_t i = 0; i < n; i++)
    if (ab[2 * i] < 0 || ab[2 * i + 1] < 0 || ab[2 * i] >= e->n_tokens + i || ab[2 * i + 1] >= e->n_tokens + i)
      return fail(e, BPE_E_INVALID, "merge %lld refers to a token that does not exist yet", (long long)i);
  return BPE_OK;
}

// ---- device groups (bpe_create_group): the GPUs of one process hold one corpus, sharded by document ----------------------------
// Member r is an ordinary engine on devices[r], rank r of the group as bpe_mg_init makes it, so the sharded kernels run unchanged;
// the mailboxes are connected by pointer under peer access (cudaIpcOpenMemHandle cannot open a handle its own process exported).
// Every call that runs device work on several members runs each member on a host thread of its own: the sharded mergeUntil waits
// on the host after every launch, so one thread driving the members in turn would leave member 0's cooperative kernel waiting for
// peers that were never launched.
bool is_group(const bpe_engine* e) { return e && !e->members.empty(); }

#define GROUP_REFUSES(e, what)                                                                                                  \
  do {                                                                                                                          \
    if (is_group(e)) return fail(e, BPE_E_INVALID, "%s is not available on a device group (a corpus sharded over its GPUs)", what); \
  } while (0)

// the group's answer for a call that one member ran on the caller's thread
int member_rc(bpe_engine* g, const bpe_engine* m, int rc) {
  return rc == BPE_OK ? rc : fail(g, rc, "device %d: %s", m->device, m->err.c_str());
}

// Runs fn(r) for every member on its own host thread and joins them all.  A member that fails inside the sharded mergeUntil leaves
// its peers waiting until the peer timeout (MG_TIMEOUT_NS), so the group reports the first member's error that is not such a
// timeout, and the timeout only when there is nothing else.
int run_members(bpe_engine* g, const std::function<int(int)>& fn) {
  const int n = (int)g->members.size();
  std::vector<int> rc((size_t)n, BPE_OK);
  std::vector<std::thread> threads;
  threads.reserve((size_t)n);
  for (bpe_engine* m : g->members) m->mg_timed_out = false;  // (a timeout is a verdict about this call only)
  for (int r = 0; r < n; r++) {
    try {
      threads.emplace_back([&rc, &fn, r] { rc[(size_t)r] = fn(r); });
    } catch (...) {
      rc[(size_t)r] = fail(g->members[(size_t)r], BPE_E_NOMEM, "cannot start a host thread for this member");
      if (g->members[(size_t)r]->mg_gate) g->members[(size_t)r]->mg_gate->drop();  // (the others must not wait for it)
    }
  }
  for (std::thread& t : threads) t.join();
  int pick = -1;
  for (int r = 0; r < n && pick < 0; r++)
    if (rc[(size_t)r] != BPE_OK && !g->members[(size_t)r]->mg_timed_out) pick = r;
  for (int r = 0; r < n && pick < 0; r++)
    if (rc[(size_t)r] != BPE_OK) pick = r;
  return pick < 0 ? BPE_OK : member_rc(g, g->members[(size_t)pick], rc[(size_t)pick]);
}

// Document boundaries of a contiguous partition of documents [0, n_docs) over n parts, balanced by units (ids or bytes): part r owns
// [b[r], b[r+1]), the documents whose first unit lies in [r*T/n, (r+1)*T/n) of the T units; empty trailing documents go to the
// last part.  (bpe_tokenizer_b200/sharded.py, shard_bounds, states the same rule for one process per GPU.)
std::vector<int64_t> shard_bounds(const int64_t* off, int64_t n_docs, int n) {
  std::vector<int64_t> b((size_t)n + 1, 0);
  if (n_docs == 0) return b;
  const int64_t total = off[n_docs] - off[0];
  int64_t d = 0;
  for (int r = 1; r < n; r++) {
    const int64_t cut = (total * r + n - 1) / n;
    while (d < n_docs && off[d] - off[0] < cut) d++;
    b[(size_t)r] = d;
  }
  b[(size_t)n] = n_docs;
  return b;
}

// Where an upload's documents go.  The first upload of a corpus is partitioned; a later one (the reference allows addToCorpus at any
// time, also after merges) goes to the last member whole, so that the global scan order (member, position) stays the document order
// the reference's tie-break needs (core.ts:294-305).
std::vector<int64_t> upload_bounds(const bpe_engine* g, const int64_t* off, int64_t n_docs) {
  const int n = (int)g->members.size();
  if (!g->grp_uploaded) return shard_bounds(off, n_docs, n);
  std::vector<int64_t> b((size_t)n + 1, 0);
  b[(size_t)n] = n_docs;
  return b;
}

// pair counts are global only while no member's corpus changed: an upload anywhere sends every member back to a fresh index
void after_upload(bpe_engine* g) {
  g->grp_uploaded = true;
  for (bpe_engine* m : g->members) {
    m->index_valid = false;
    m->hot_valid = false;
  }
}

uint64_t group_slots(const bpe_engine* g) {
  uint64_t s = 0;
  for (const bpe_engine* m : g->members) s += m->n_slots;
  return s;
}

// The new characters of a text batch split over parts that hold contiguous document ranges in order, in the batch's first-appearance
// order (core.ts:186-199): per part (code points, first positions within the part), the key is (part, first position), and a
// character that several parts report belongs to the first of them.  (sharded.py, order_new_chars, for one process per GPU.)
std::vector<int32_t> order_new_chars(const std::vector<std::vector<int32_t>>& cps, const std::vector<std::vector<int64_t>>& pos) {
  std::unordered_set<int32_t> seen;
  std::vector<int32_t> out;
  for (size_t r = 0; r < cps.size(); r++) {
    std::vector<size_t> order(cps[r].size());
    for (size_t k = 0; k < order.size(); k++) order[k] = k;
    std::stable_sort(order.begin(), order.end(), [&](size_t x, size_t y) { return pos[r][x] < pos[r][y]; });
    for (size_t k : order)
      if (seen.insert(cps[r][k]).second) out.push_back(cps[r][k]);
  }
  return out;
}

int group_add_documents(bpe_engine* g, const int32_t* ids, const int64_t* off, int64_t n_docs, bool restore) {
  TRY(check_offsets(g, off, n_docs));
  if (n_docs == 0) return BPE_OK;
  const std::vector<int64_t> b = upload_bounds(g, off, n_docs);
  // as on one engine, a refused upload adds nothing: the members that appended their range drop it again
  struct Mark {
    uint64_t n_slots, live_tokens;
    size_t n_docs;
  };
  std::vector<Mark> marks;
  for (const bpe_engine* m : g->members) marks.push_back({m->n_slots, m->live_tokens, m->doc_off.size()});
  const int rc = run_members(g, [&](int r) {
    const int64_t nd = b[(size_t)r + 1] - b[(size_t)r];
    if (nd == 0) return BPE_OK;
    bpe_engine* m = g->members[(size_t)r];
    return restore ? bpe_restore_documents(m, ids, off + b[(size_t)r], nd) : bpe_add_documents(m, ids, off + b[(size_t)r], nd);
  });
  if (rc != BPE_OK) {
    for (size_t r = 0; r < g->members.size(); r++) {
      bpe_engine* m = g->members[r];
      if (m->doc_off.size() == marks[r].n_docs) continue;
      m->n_slots = marks[r].n_slots;  // (slots past n_slots are unused storage)
      m->live_tokens = marks[r].live_tokens;
      m->doc_off.resize(marks[r].n_docs);
      m->index_valid = false;
      m->hot_valid = false;
    }
    return rc;
  }
  after_upload(g);
  return BPE_OK;
}

// bpe_add_text: stage on every member, agree on one order of the new characters, commit that list everywhere, sum the counts
int group_add_text(bpe_engine* g, const uint8_t* utf8, const int64_t* off, int64_t n_docs, int32_t* new_code_points, int32_t new_cap,
                   int32_t* n_new, int64_t* counts, int64_t counts_cap) {
  TRY(check_offsets(g, off, n_docs));
  const size_t n = g->members.size();
  const std::vector<int64_t> b = upload_bounds(g, off, n_docs);
  const int32_t list_cap = 1 << 16;  // bpe_add_text_stage reports at most this many
  std::vector<std::vector<int32_t>> cps(n, std::vector<int32_t>((size_t)list_cap));
  std::vector<std::vector<int64_t>> pos(n, std::vector<int64_t>((size_t)list_cap));
  std::vector<int32_t> nn(n, 0);
  auto drop_staged = [&] {
    for (bpe_engine* m : g->members) m->txt_staged = false;
  };
  int rc = run_members(g, [&](int r) {
    return bpe_add_text_stage(g->members[(size_t)r], utf8, off + b[(size_t)r], b[(size_t)r + 1] - b[(size_t)r], cps[(size_t)r].data(),
                              pos[(size_t)r].data(), list_cap, &nn[(size_t)r]);
  });
  if (rc != BPE_OK) {
    drop_staged();
    return rc;
  }
  for (size_t r = 0; r < n; r++) {
    cps[r].resize((size_t)nn[r]);
    pos[r].resize((size_t)nn[r]);
  }
  const std::vector<int32_t> fresh = order_new_chars(cps, pos);
  const int32_t nt = g->members[0]->n_tokens, nf = (int32_t)fresh.size();
  // judged on the global list, before any member changes
  if ((int64_t)nt + nf > BPE_MAX_TOKENS) {
    drop_staged();
    return fail(g, BPE_E_DOMAIN, "token table would exceed %d", BPE_MAX_TOKENS);
  }
  if (nf > new_cap) {
    drop_staged();
    *n_new = nf;
    return fail(g, BPE_E_CAPACITY, "%d new characters, room for %d", nf, new_cap);
  }
  if (counts && counts_cap < (int64_t)nt + nf) {
    drop_staged();
    return fail(g, BPE_E_CAPACITY, "counts holds %lld entries, need %d", (long long)counts_cap, nt + nf);
  }
  std::vector<std::vector<int64_t>> cnt(n, std::vector<int64_t>((size_t)nt + nf + 1));
  rc = run_members(g, [&](int r) { return bpe_add_text_commit(g->members[(size_t)r], fresh.data(), nf, cnt[(size_t)r].data(), (int64_t)nt + nf); });
  if (n_docs) after_upload(g);
  if (rc != BPE_OK) return rc;
  std::copy(fresh.begin(), fresh.end(), new_code_points);
  *n_new = nf;
  if (counts)
    for (int64_t i = 0; i < (int64_t)nt + nf; i++) {
      counts[i] = 0;
      for (size_t r = 0; r < n; r++) counts[i] += cnt[r][(size_t)i];
    }
  return BPE_OK;
}

// Sums the members' pair histograms into every member's table, once per index build: each member exports its (pair, count) list into
// device buffers it owns, then every member imports every peer's list straight from the peer's memory (no host copy).
int group_exchange_counts(bpe_engine* g) {
  bool global = true;
  for (const bpe_engine* m : g->members) global = global && m->index_valid && m->mg_counts_global;
  if (global) return BPE_OK;
  for (bpe_engine* m : g->members) m->index_valid = false;  // (no member may import into counts that are already summed)
  TRY(run_members(g, [&](int r) {
    bpe_engine* e = g->members[(size_t)r];
    int64_t n = 0;
    TRY(bpe_mg_export_counts(e, nullptr, nullptr, 0, &n));  // builds the index; n = its number of pairs
    const size_t cap = (size_t)std::max<int64_t>(n, 1);
    CK(e->grp_keys.reserve(cap));
    CK(e->grp_counts.reserve(cap));
    TRY(bpe_mg_export_counts(e, e->grp_keys.p, e->grp_counts.p, (int64_t)cap, &n));
    e->grp_n = n;
    return BPE_OK;
  }));
  const int n = (int)g->members.size();
  return run_members(g, [&](int r) {
    bpe_engine* e = g->members[(size_t)r];
    const int last = (r == n - 1) ? n - 2 : n - 1;
    for (int q = 0; q < n; q++) {
      if (q == r) continue;
      const bpe_engine* p = g->members[(size_t)q];
      TRY(bpe_mg_import_counts(e, p->grp_keys.p, p->grp_counts.p, p->grp_n, q == last));
    }
    return BPE_OK;
  });
}

int group_merge_until(bpe_engine* g, int64_t min_weight, int32_t max_length, int64_t max_iterations, bpe_merge* log, int64_t log_cap,
                      int64_t* n_done) {
  *n_done = 0;
  if (group_slots(g) == 0) return BPE_OK;  // (as one engine: an empty corpus has no pair)
  TRY(group_exchange_counts(g));
  const size_t n = g->members.size();
  const int64_t cap = std::min<int64_t>(log_cap, BPE_MAX_TOKENS);  // (no run can log more merges than there are free token indices)
  std::vector<std::vector<bpe_merge>> logs(n, std::vector<bpe_merge>((size_t)cap));
  std::vector<int64_t> done(n, 0);
  LaunchGate gate((int)n);
  for (bpe_engine* m : g->members) m->mg_gate = &gate;
  const int rc = run_members(g, [&](int r) {
    return bpe_merge_until(g->members[(size_t)r], min_weight, max_length, max_iterations, logs[(size_t)r].data(), cap, &done[(size_t)r]);
  });
  for (bpe_engine* m : g->members) m->mg_gate = nullptr;
  for (size_t r = 1; r < n; r++)
    if (done[r] != done[0] || (done[0] && memcmp(logs[r].data(), logs[0].data(), (size_t)done[0] * sizeof(bpe_merge)) != 0))
      return rc != BPE_OK ? rc : fail(g, BPE_E_INTERNAL, "device %d and device %d returned different merge logs", g->members[0]->device, g->members[r]->device);
  if (done[0]) memcpy(log, logs[0].data(), (size_t)done[0] * sizeof(bpe_merge));
  *n_done = done[0];
  return rc;
}

// bpe_encode_batch / bpe_encode_text_batch.  The documents are split into contiguous ranges balanced by input units, one per member,
// and the members' pipelines run in parallel, without copying their vectors out: they stay in each member's staging buffer on its
// device, and each member reports its size.  Once every size is known, each member copies its vectors from its device straight to
// their place in the caller's `out`, all members at once.  Cost beside the members' pipelines: the device-to-host copy of the output
// runs after the encode instead of overlapping it.
int group_encode(bpe_engine* g, bool is_text, const int32_t* ids, const uint8_t* utf8, const int64_t* off, int64_t n_docs,
                 const int32_t* to_vector_index, int32_t n_tvi, int32_t* out, int64_t out_cap, int64_t* out_offsets, int64_t* first_bad,
                 int64_t* n_out, int64_t* unknown_pos, int32_t* unknown_code_point) {
  *n_out = 0;
  if (n_docs == 0) {
    out_offsets[0] = 0;
    return BPE_OK;
  }
  TRY(check_offsets(g, off, n_docs));
  const size_t n = g->members.size();
  const std::vector<int64_t> b = shard_bounds(off, n_docs, (int)n);
  std::vector<std::vector<int64_t>> moff(n);
  std::vector<int64_t> k(n, 0), upos(n, -1), cum(n + 1, 0);
  std::vector<int32_t> ucp(n, 0);
  std::vector<int> mrc(n, BPE_OK);
  for (size_t r = 0; r < n; r++) moff[r].assign((size_t)(b[r + 1] - b[r]) + 1, 0);
  const int rc = run_members(g, [&](int r) {
    const size_t i = (size_t)r;
    const int64_t nd = b[i + 1] - b[i];
    if (nd == 0) return BPE_OK;
    bpe_engine* m = g->members[i];
    int64_t* fb = first_bad ? first_bad + b[i] : nullptr;
    const int got = is_text ? bpe_encode_text_batch(m, utf8, off + b[i], nd, to_vector_index, n_tvi, nullptr, 0, moff[i].data(), fb, &k[i], &upos[i], &ucp[i])
                            : bpe_encode_batch(m, ids, off + b[i], nd, to_vector_index, n_tvi, nullptr, 0, moff[i].data(), fb, &k[i]);
    mrc[i] = got == BPE_E_CAPACITY ? BPE_OK : got;  // (no output buffer: the member reports its size, offsets and first_bad complete)
    return mrc[i];
  });
  if (rc != BPE_OK) {
    // the error the first failing member met is the first in batch order; its positions are relative to the member's range
    size_t r = 0;
    while (r < n && mrc[r] == BPE_OK) r++;
    if (r < n && upos[r] >= 0) {  // an unknown character: the members before r held this many code points (lead bytes, as text_kernels.cuh counts)
      int64_t before = 0;
      for (int64_t p = off[0]; p < off[b[r]]; p++) before += (utf8[p] & 0xC0) != 0x80;
      if (unknown_pos) *unknown_pos = before + upos[r];
      if (unknown_code_point) *unknown_code_point = ucp[r];
    }
    if (r < n && !is_text && g->members[r]->enc_bad_id_pos >= 0) {
      const int64_t pos = off[b[r]] - off[0] + g->members[r]->enc_bad_id_pos;
      return fail(g, BPE_E_INVALID, "id %d at %lld outside the token table", ids[off[0] + pos], (long long)pos);
    }
    return rc;
  }
  for (size_t r = 0; r < n; r++) cum[r + 1] = cum[r] + k[r];
  for (size_t r = 0; r < n; r++)
    for (int64_t d = 0; d < b[r + 1] - b[r]; d++) out_offsets[b[r] + d] = moff[r][(size_t)d] + cum[r];
  out_offsets[n_docs] = cum[n];
  *n_out = cum[n];
  if (cum[n] > out_cap || (cum[n] && !out)) return fail(g, BPE_E_CAPACITY, "output buffer holds %lld values, need %lld", (long long)out_cap, (long long)cum[n]);
  return run_members(g, [&](int r) {
    bpe_engine* e = g->members[(size_t)r];
    if (k[(size_t)r] == 0) return BPE_OK;
    CK(cudaSetDevice(e->device));
    int32_t* dst = out + cum[(size_t)r];
    for (size_t c = 0; c + 1 < e->enc_parts.size(); c += 2) {
      const int64_t reg = e->enc_parts[c], len = e->enc_parts[c + 1];
      if (len) CK(cudaMemcpyAsync(dst, e->x_out.p + reg, (size_t)len * sizeof(int32_t), cudaMemcpyDeviceToHost, e->s_out));
      dst += len;
    }
    CK(cudaStreamSynchronize(e->s_out));
    return BPE_OK;
  });
}

// bpe_decode_batch.  Decoded bytes have no bound the caller's buffer must meet, so the members first report their sizes (the values
// and the token bytes go up, the lengths are scanned), then decode straight into the caller's `out` at their place: the upload and
// the length pass run twice, the gather and the copy out once.
int group_decode(bpe_engine* g, const int32_t* values, const int64_t* off, int64_t n_docs, const int32_t* from_vector_index, int32_t n_fvi,
                 const uint8_t* token_bytes, const int64_t* token_byte_offsets, int32_t n_tokens, uint8_t* out, int64_t out_cap,
                 int64_t* out_offsets, int64_t* first_bad, int64_t* n_out) {
  *n_out = 0;
  TRY(check_offsets(g, off, n_docs));
  if (n_docs == 0) {
    bpe_engine* m = g->members[0];
    return member_rc(g, m, bpe_decode_batch(m, values, off, 0, from_vector_index, n_fvi, token_bytes, token_byte_offsets, n_tokens, out, out_cap,
                                            out_offsets, first_bad, n_out));
  }
  const size_t n = g->members.size();
  const std::vector<int64_t> b = shard_bounds(off, n_docs, (int)n);
  std::vector<std::vector<int64_t>> moff(n);
  std::vector<int64_t> k(n, 0), cum(n + 1, 0);
  for (size_t r = 0; r < n; r++) moff[r].assign((size_t)(b[r + 1] - b[r]) + 1, 0);
  auto pass = [&](bool sizes) {
    return run_members(g, [&](int r) {
      const size_t i = (size_t)r;
      const int64_t nd = b[i + 1] - b[i];
      if (nd == 0 || (!sizes && k[i] == 0)) return BPE_OK;
      uint8_t* dst = sizes ? nullptr : out + cum[i];
      const int got = bpe_decode_batch(g->members[i], values, off + b[i], nd, from_vector_index, n_fvi, token_bytes, token_byte_offsets, n_tokens, dst,
                                       sizes ? 0 : k[i], moff[i].data(), first_bad ? first_bad + b[i] : nullptr, &k[i]);
      return (sizes && got == BPE_E_CAPACITY) ? BPE_OK : got;
    });
  };
  TRY(pass(true));
  for (size_t r = 0; r < n; r++) cum[r + 1] = cum[r] + k[r];
  for (size_t r = 0; r < n; r++)
    for (int64_t d = 0; d < b[r + 1] - b[r]; d++) out_offsets[b[r] + d] = moff[r][(size_t)d] + cum[r];
  out_offsets[n_docs] = cum[n];
  *n_out = cum[n];
  if (cum[n] > out_cap || (cum[n] && !out)) return fail(g, BPE_E_CAPACITY, "output buffer holds %lld bytes, need %lld", (long long)out_cap, (long long)cum[n]);
  return pass(false);
}

// bpe_get_corpus: the members' document ranges back to back; sizes first, then every member copies into its place
int group_get_corpus(bpe_engine* g, int64_t doc_begin, int64_t doc_end, int32_t* out, int64_t out_cap, int64_t* out_offsets, int64_t* n_out) {
  const size_t n = g->members.size();
  std::vector<int64_t> lo(n), hi(n), k(n, 0), cum(n + 1, 0);
  int64_t nd = 0;
  for (size_t r = 0; r < n; r++) {
    const int64_t first = nd, count = (int64_t)g->members[r]->doc_off.size() - 1;
    nd += count;
    lo[r] = std::min(std::max<int64_t>(doc_begin - first, 0), count);
    hi[r] = std::min(std::max<int64_t>(doc_end - first, 0), count);
  }
  if (doc_begin < 0 || doc_end < doc_begin || doc_end > nd)
    return fail(g, BPE_E_INVALID, "document range [%lld,%lld) outside [0,%lld)", (long long)doc_begin, (long long)doc_end, (long long)nd);
  std::vector<std::vector<int64_t>> moff(n);
  for (size_t r = 0; r < n; r++) moff[r].assign((size_t)(hi[r] - lo[r]) + 1, 0);
  TRY(run_members(g, [&](int r) {
    const size_t i = (size_t)r;
    if (hi[i] == lo[i]) return BPE_OK;
    const int got = bpe_get_corpus(g->members[i], lo[i], hi[i], nullptr, 0, moff[i].data(), &k[i]);
    return got == BPE_E_CAPACITY ? BPE_OK : got;
  }));
  for (size_t r = 0; r < n; r++) cum[r + 1] = cum[r] + k[r];
  *n_out = cum[n];
  if (cum[n] > out_cap || (!out && cum[n]) || !out_offsets) return fail(g, BPE_E_CAPACITY, "output buffer holds %lld values, need %lld", (long long)out_cap, (long long)cum[n]);
  TRY(run_members(g, [&](int r) {
    const size_t i = (size_t)r;
    if (hi[i] == lo[i]) return BPE_OK;
    int64_t got = 0;
    return bpe_get_corpus(g->members[i], lo[i], hi[i], out ? out + cum[i] : nullptr, k[i], moff[i].data(), &got);
  }));
  int64_t at = 0;
  out_offsets[0] = 0;
  for (size_t r = 0; r < n; r++)
    for (int64_t d = 1; d <= hi[r] - lo[r]; d++) out_offsets[++at] = moff[r][(size_t)d] + cum[r];
  return BPE_OK;
}

int group_get_stats(bpe_engine* g, bpe_stats* out) {
  std::vector<bpe_stats> s(g->members.size());
  TRY(run_members(g, [&](int r) { return bpe_get_stats(g->members[(size_t)r], &s[(size_t)r]); }));
  *out = s[0];
  for (size_t r = 1; r < s.size(); r++) {
    out->kernel_launches += s[r].kernel_launches;
    out->sites_merged += s[r].sites_merged;
    out->corpus_positions += s[r].corpus_positions;
    out->corpus_tokens += s[r].corpus_tokens;
    out->pool_used += s[r].pool_used;
  }
  return BPE_OK;
}

void destroy_group(bpe_engine* g) {
  for (bpe_engine* m : g->members)  // the peers' mailboxes are the other members' allocations, not cudaIpc mappings to close
    for (int q = 0; q < m->mg_world; q++)
      if (q != m->mg_rank) m->mg_peer[q] = nullptr;
  for (bpe_engine* m : g->members) bpe_destroy(m);
  delete g;
}

}  // namespace

// =====================================================================================================
extern "C" {

int bpe_abi_version(void) { return BPE_ABI_VERSION; }

int bpe_create(int device, bpe_engine** out) {
  if (!out) return BPE_E_INVALID;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) return BPE_E_CUDA;
  if (cudaSetDevice(device) != cudaSuccess) return BPE_E_CUDA;
  bpe_engine* e = new bpe_engine();
  e->device = device;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) e->sm_count = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete e;
    return BPE_E_CUDA;
  }
  e->stream = e->own_stream;
  if (getenv("BPE_ENC_OLD")) e->enc_force_old = 1;
  if (getenv("BPE_ENC_LMAX")) e->enc_lmax_forced = 1;
  if (const char* v = getenv("BPE_ENC_LMAX")) e->enc_lmax = (atoi(v) == 48 || atoi(v) == 24 || atoi(v) == 20 || atoi(v) == 16) ? atoi(v) : 32;
  *out = e;
  return BPE_OK;
}

int bpe_create_group(const int* devices, int n, bpe_engine** out) {
  if (!out) return BPE_E_INVALID;
  *out = nullptr;
  if (!devices || n < 1 || n > BPE_MG_MAX_WORLD) return BPE_E_INVALID;
  // BPE_GROUP_SHARE_DEVICE=1 (tests on a host with fewer GPUs than members): members may share a device, each with its share of
  // the SMs, so that the group's cooperative kernels stay co-resident.  It exercises the group, not its speed.
  const char* share_env = getenv("BPE_GROUP_SHARE_DEVICE");
  const bool share = share_env && atoi(share_env) != 0;
  for (int r = 0; r < n; r++)
    for (int q = 0; q < r; q++)
      if (devices[q] == devices[r] && !share) return BPE_E_INVALID;
  if (n == 1) return bpe_create(devices[0], out);
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) return BPE_E_CUDA;
  for (int r = 0; r < n; r++) {
    if (devices[r] < 0 || devices[r] >= count) return BPE_E_CUDA;
    for (int q = 0; q < n; q++) {
      int ok = 0;
      if (devices[q] != devices[r] && (cudaDeviceCanAccessPeer(&ok, devices[r], devices[q]) != cudaSuccess || !ok)) return BPE_E_CUDA;
    }
  }
  bpe_engine* g = new bpe_engine();
  g->device = devices[0];
  int rc = BPE_OK;
  for (int r = 0; r < n && rc == BPE_OK; r++) {
    bpe_engine* m = nullptr;
    rc = bpe_create(devices[r], &m);
    if (rc != BPE_OK) break;
    g->members.push_back(m);
    rc = mg_alloc_mailbox(m, r, n);
  }
  for (int r = 0; r < n && rc == BPE_OK; r++) {
    if (cudaSetDevice(devices[r]) != cudaSuccess) rc = BPE_E_CUDA;
    for (int q = 0; q < n && rc == BPE_OK; q++) {
      if (devices[q] == devices[r]) continue;
      cudaError_t err = cudaDeviceEnablePeerAccess(devices[q], 0);
      if (err == cudaErrorPeerAccessAlreadyEnabled) (void)cudaGetLastError();  // (torch, or an earlier group, enabled it)
      else if (err != cudaSuccess) rc = BPE_E_CUDA;
    }
  }
  if (rc != BPE_OK) {
    destroy_group(g);
    return rc;
  }
  for (bpe_engine* m : g->members) {
    for (int q = 0; q < n; q++) m->mg_peer[q] = g->members[(size_t)q]->mg_mailbox;
    m->mg_connected = true;
    const int sharing = (int)std::count(devices, devices + n, m->device);
    m->sm_count = std::max(1, m->sm_count / sharing);
  }
  *out = g;
  return BPE_OK;
}

void bpe_destroy(bpe_engine* e) {
  if (is_group(e)) {
    destroy_group(e);
    return;
  }
  if (e && e->mg_mailbox) {
    cudaSetDevice(e->device);
    for (int q = 0; q < e->mg_world; q++)
      if (q != e->mg_rank && e->mg_peer[q]) cudaIpcCloseMemHandle(e->mg_peer[q]);
    cudaFree(e->mg_mailbox);
    e->mg_mailbox = nullptr;
  }
  if (!e) return;
  cudaSetDevice(e->device);
  cudaStreamSynchronize(e->stream);
  if (e->h_st) cudaFreeHost(e->h_st);
  if (e->ev0) cudaEventDestroy(e->ev0);
  if (e->ev1) cudaEventDestroy(e->ev1);
  for (cudaEvent_t ev : {e->ev_in[0], e->ev_in[1], e->ev_in[2], e->ev_done, e->ev_res[0], e->ev_res[1]})
    if (ev) cudaEventDestroy(ev);
  if (e->s_in) cudaStreamDestroy(e->s_in);
  if (e->s_out) cudaStreamDestroy(e->s_out);
  if (e->h_pipe) cudaFreeHost(e->h_pipe);
  if (e->own_stream) cudaStreamDestroy(e->own_stream);
  delete e;
}

const char* bpe_last_error(bpe_engine* e) { return e ? e->err.c_str() : "null engine"; }

int bpe_set_stream(bpe_engine* e, void* cuda_stream) {
  if (!e) return BPE_E_INVALID;
  GROUP_REFUSES(e, "bpe_set_stream (a stream belongs to one device)");
  cudaSetDevice(e->device);
  cudaStreamSynchronize(e->stream);
  e->stream = cuda_stream ? (cudaStream_t)cuda_stream : e->own_stream;
  return BPE_OK;
}

int bpe_synchronize(bpe_engine* e) {
  if (!e) return BPE_E_INVALID;
  if (is_group(e)) return run_members(e, [&](int r) { return bpe_synchronize(e->members[(size_t)r]); });
  CK(cudaSetDevice(e->device));
  CK(cudaStreamSynchronize(e->stream));
  return BPE_OK;
}

int bpe_set_profiling(bpe_engine* e, int enabled) {
  if (!e) return BPE_E_INVALID;
  if (is_group(e)) return run_members(e, [&](int r) { return bpe_set_profiling(e->members[(size_t)r], enabled); });
  e->profiling = enabled != 0;
  e->scan_mode = (enabled & 2) ? 1 : 0;  // bit 1: debug full-scan site discovery
  return BPE_OK;
}

int bpe_get_stats(bpe_engine* e, bpe_stats* out) {
  if (!e || !out) return BPE_E_INVALID;
  if (is_group(e)) return group_get_stats(e, out);
  CK(cudaSetDevice(e->device));
  if (e->index_valid && e->d_st.p) {
    TRY(fetch_state(e));
    e->live_tokens = e->h_st->live_tokens;
    e->stats.distinct_pairs = e->h_st->n_keys;
    for (int i = 0; i < 8; i++) e->stats.ms_loop_phase[i] = (double)e->h_st->prof_ns[i] * 1e-6;
#ifdef BPE_FINE_PROF
    fprintf(stderr, "[bpe] phase_sites sub-steps ms (pool, slot+right, left, dec1, new1, right, dec2, new2, record):");
    for (int i = 0; i < 9; i++) fprintf(stderr, " %.1f", (double)e->h_st->fine_ns[i] * 1e-6);
    fprintf(stderr, "\n[bpe] per log2(weight) bucket: merges, P1 us/merge, P2 us/merge, P3 us/merge, P1 ns/site\n");
    for (int b = 0; b < 32; b++) {
      double m = (double)e->h_st->bucket_ns[b][3];
      if (m > 0) fprintf(stderr, "  2^%-2d %8.0f  %8.1f %8.1f %8.1f  %8.2f\n", b, m, e->h_st->bucket_ns[b][0] / m * 1e-3, e->h_st->bucket_ns[b][1] / m * 1e-3,
                         e->h_st->bucket_ns[b][2] / m * 1e-3, e->h_st->bucket_ns[b][0] / m / (1.5 * (double)(1u << b)));
    }
#endif
    e->stats.pool_used = e->h_st->pool_cursor;
  }
  e->stats.corpus_positions = (int64_t)e->n_slots;
  e->stats.corpus_tokens = (int64_t)e->live_tokens;
  *out = e->stats;
  return BPE_OK;
}

int bpe_set_tokens(bpe_engine* e, const int32_t* utf16_len, int32_t n_tokens) {
  if (!e || n_tokens < 0 || (!utf16_len && n_tokens > 0)) return fail(e, BPE_E_INVALID, "bad token table");
  if (n_tokens > BPE_MAX_TOKENS) return fail(e, BPE_E_DOMAIN, "token table of %d exceeds %d", n_tokens, BPE_MAX_TOKENS);
  for (int32_t i = 0; i < n_tokens; i++)
    if (utf16_len[i] < 0) return fail(e, BPE_E_INVALID, "negative token length");
  if (is_group(e)) return run_members(e, [&](int r) { return bpe_set_tokens(e->members[(size_t)r], utf16_len, n_tokens); });
  CK(cudaSetDevice(e->device));
  e->h_len16.assign(utf16_len, utf16_len + n_tokens);
  e->n_tokens = n_tokens;
  e->mt_dirty = e->lt_dirty = true;
  TRY(sync_len16(e));
  e->hot_valid = false;
  return BPE_OK;
}

int bpe_num_tokens(bpe_engine* e, int32_t* n_tokens) {
  if (!e || !n_tokens) return BPE_E_INVALID;
  *n_tokens = is_group(e) ? e->members[0]->n_tokens : e->n_tokens;
  return BPE_OK;
}

int bpe_load_merges(bpe_engine* e, const int32_t* abc, int64_t n_merges) {
  if (!e || n_merges < 0 || (!abc && n_merges > 0)) return fail(e, BPE_E_INVALID, "bad merge list");
  for (int64_t i = 0; i < 3 * n_merges; i++)
    if (abc[i] < 0 || abc[i] >= BPE_MAX_TOKENS) return fail(e, BPE_E_INVALID, "merge %lld holds index %d", (long long)(i / 3), abc[i]);
  if (is_group(e)) return run_members(e, [&](int r) { return bpe_load_merges(e->members[(size_t)r], abc, n_merges); });
  e->h_merges.assign(abc, abc + 3 * n_merges);
  e->mt_dirty = e->lt_dirty = true;
  return BPE_OK;
}

int bpe_add_documents_dev(bpe_engine* e, const int32_t* dev_ids, const int64_t* host_doc_offsets, int64_t n_docs) {
  if (!e) return BPE_E_INVALID;
  GROUP_REFUSES(e, "bpe_add_documents_dev (device pointers belong to one device)");
  TRY(check_offsets(e, host_doc_offsets, n_docs));
  if (n_docs == 0) return BPE_OK;
  if (!dev_ids && host_doc_offsets[n_docs] > host_doc_offsets[0]) return fail(e, BPE_E_INVALID, "null ids");
  CK(cudaSetDevice(e->device));
  return append_docs_dev(e, dev_ids, host_doc_offsets, n_docs);
}

int bpe_add_documents(bpe_engine* e, const int32_t* ids, const int64_t* doc_offsets, int64_t n_docs) {
  if (!e) return BPE_E_INVALID;
  if (is_group(e)) return group_add_documents(e, ids, doc_offsets, n_docs, false);
  TRY(check_offsets(e, doc_offsets, n_docs));
  if (n_docs == 0) return BPE_OK;
  int64_t base = doc_offsets[0], total = doc_offsets[n_docs] - base;
  if (!ids && total > 0) return fail(e, BPE_E_INVALID, "null ids");
  CK(cudaSetDevice(e->device));
  uint64_t new_n = e->n_slots + (uint64_t)total;
  if (new_n >= 0xFFFFFFF0ull) return fail(e, BPE_E_DOMAIN, "corpus exceeds 2^32 positions per engine");
  CK(e->slots.reserve((size_t)new_n + 4, (size_t)e->n_slots, e->stream, 1.5));
  // int32 token ids ARE the slot encoding of single-slot tokens: copy them into place, then validate in place
  if (total > 0)
    CK(cudaMemcpyAsync(e->slots.p + e->n_slots, ids + base, (size_t)total * sizeof(int32_t), cudaMemcpyHostToDevice, e->stream));
  std::vector<int64_t> rel((size_t)n_docs + 1);
  for (int64_t d = 0; d <= n_docs; d++) rel[d] = doc_offsets[d] - base;
  return append_docs_dev(e, reinterpret_cast<const int32_t*>(e->slots.p + e->n_slots), rel.data(), n_docs);
}

int bpe_clear_corpus(bpe_engine* e) {
  if (!e) return BPE_E_INVALID;
  if (is_group(e)) {
    e->grp_uploaded = false;
    return run_members(e, [&](int r) { return bpe_clear_corpus(e->members[(size_t)r]); });
  }
  e->n_slots = 0;
  e->doc_off.assign(1, 0);
  e->live_tokens = 0;
  e->index_valid = false;
  e->hot_valid = false;
  return BPE_OK;
}

int bpe_corpus_size(bpe_engine* e, int64_t* n_docs, int64_t* n_tokens) {
  if (!e) return BPE_E_INVALID;
  if (is_group(e)) {
    std::vector<int64_t> d(e->members.size(), 0), t(e->members.size(), 0);
    TRY(run_members(e, [&](int r) { return bpe_corpus_size(e->members[(size_t)r], &d[(size_t)r], &t[(size_t)r]); }));
    int64_t sd = 0, st = 0;
    for (size_t r = 0; r < d.size(); r++) {
      sd += d[r];
      st += t[r];
    }
    if (n_docs) *n_docs = sd;
    if (n_tokens) *n_tokens = st;
    return BPE_OK;
  }
  CK(cudaSetDevice(e->device));
  if (e->index_valid && e->d_st.p) {
    TRY(fetch_state(e));
    e->live_tokens = e->h_st->live_tokens;
  }
  if (n_docs) *n_docs = (int64_t)e->doc_off.size() - 1;
  if (n_tokens) *n_tokens = (int64_t)e->live_tokens;
  return BPE_OK;
}

int bpe_get_corpus(bpe_engine* e, int64_t doc_begin, int64_t doc_end, int32_t* out, int64_t out_cap, int64_t* out_offsets,
                   int64_t* n_out) {
  if (!e || !n_out) return BPE_E_INVALID;
  if (is_group(e)) return group_get_corpus(e, doc_begin, doc_end, out, out_cap, out_offsets, n_out);
  int64_t nd = (int64_t)e->doc_off.size() - 1;
  if (doc_begin < 0 || doc_end < doc_begin || doc_end > nd) return fail(e, BPE_E_INVALID, "document range [%lld,%lld) outside [0,%lld)", (long long)doc_begin, (long long)doc_end, (long long)nd);
  CK(cudaSetDevice(e->device));
  uint64_t begin = (uint64_t)e->doc_off[doc_begin], end = (uint64_t)e->doc_off[doc_end];
  int64_t n_bounds = doc_end - doc_begin + 1;
  uint64_t span = end - begin;
  uint32_t nblk = (uint32_t)((span + CP_TILE - 1) / CP_TILE);
  DevBuf<uint32_t> bc;
  DevBuf<uint64_t> bo;
  DevBuf<int64_t> dpos, doffs;
  DevBuf<int32_t> dout;
  CK(bc.reserve(nblk + 1));
  CK(bo.reserve(nblk + 2));
  CK(dpos.reserve((size_t)n_bounds));
  CK(doffs.reserve((size_t)n_bounds));
  if (nblk) {
    k_count_ids<<<nblk, CP_THREADS, 0, e->stream>>>(e->slots.p, begin, end, bc.p);
    CKL();
  }
  k_scan_counts<<<1, 1024, 0, e->stream>>>(bc.p, bo.p, nblk);
  CKL();
  uint64_t total = 0;
  CK(cudaMemcpyAsync(&total, bo.p + nblk, sizeof total, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  *n_out = (int64_t)total;
  if ((int64_t)total > out_cap || (!out && total) || !out_offsets) {
    if (!out_offsets || (!out && total)) return fail(e, BPE_E_CAPACITY, "output buffers missing; need %llu values", (unsigned long long)total);
    return fail(e, BPE_E_CAPACITY, "output buffer holds %lld values, need %llu", (long long)out_cap, (unsigned long long)total);
  }
  CK(cudaMemcpyAsync(dpos.p, e->doc_off.data() + doc_begin, (size_t)n_bounds * sizeof(int64_t), cudaMemcpyHostToDevice, e->stream));
  k_doc_ranks<<<(int)std::min<int64_t>((n_bounds * 32 + 255) / 256, (int64_t)e->grid(8)), 256, 0, e->stream>>>(e->slots.p, begin, bo.p, dpos.p, n_bounds, doffs.p);
  CKL();
  CK(cudaMemcpyAsync(out_offsets, doffs.p, (size_t)n_bounds * sizeof(int64_t), cudaMemcpyDeviceToHost, e->stream));
  if (total) {
    CK(dout.reserve((size_t)total));
    k_compact_ids<<<nblk, CP_THREADS, 0, e->stream>>>(e->slots.p, begin, end, bo.p, dout.p);
    CKL();
    CK(cudaMemcpyAsync(out, dout.p, (size_t)total * sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
  }
  CK(cudaStreamSynchronize(e->stream));
  return BPE_OK;
}

int bpe_find_next_merge(bpe_engine* e, int64_t min_weight, int32_t max_length, bpe_merge* out, int* found) {
  if (!e || !out || !found) return BPE_E_INVALID;
  *found = 0;
  // a shard alone would answer with ITS best pair, not the corpus's (core.ts:265-310 counts over all documents)
  GROUP_REFUSES(e, "bpe_find_next_merge (use bpe_merge_until(max_iterations = 1))");
  if (e->mg_world > 1) return fail(e, BPE_E_INVALID, "bpe_find_next_merge is not available on a sharded engine; use bpe_merge_until(max_iterations = 1)");
  CK(cudaSetDevice(e->device));
  if (e->n_slots == 0) return BPE_OK;
  TRY(ensure_index(e));
  uint32_t ml = max_length > 0 ? (uint32_t)max_length : 0;
  int64_t mw = min_weight > 0 ? min_weight : 2;  // core.ts:256
  TRY(run_argmax(e, ml));
  if (!e->h_st->best_primary) return BPE_OK;            // core.ts:312
  if ((int64_t)e->h_st->best_cnt < mw) return BPE_OK;   // core.ts:313
  out->a = (int32_t)e->h_st->best_a;
  out->b = (int32_t)e->h_st->best_b;
  out->c = e->n_tokens;
  out->reserved = 0;
  out->weight = (int64_t)e->h_st->best_cnt;
  *found = 1;
  return BPE_OK;
}

int bpe_apply_merge(bpe_engine* e, int32_t a, int32_t b, int32_t c, int64_t* n_replaced) {
  if (!e) return BPE_E_INVALID;
  if (is_group(e)) {  // on an empty corpus only the vocabulary grows, on every member
    if (group_slots(e)) return fail(e, BPE_E_INVALID, "bpe_apply_merge on a corpus is not available on a device group; use bpe_merge_until");
    if (n_replaced) *n_replaced = 0;
    return run_members(e, [&](int r) { return bpe_apply_merge(e->members[(size_t)r], a, b, c, nullptr); });
  }
  if (a < 0 || b < 0 || a >= e->n_tokens || b >= e->n_tokens) return fail(e, BPE_E_INVALID, "merge operands (%d,%d) outside the token table (%d)", a, b, e->n_tokens);
  if (c != e->n_tokens) return fail(e, BPE_E_INVALID, "new token index must be %d, got %d", e->n_tokens, c);
  if (c >= BPE_MAX_TOKENS) return fail(e, BPE_E_DOMAIN, "token table would exceed %d", BPE_MAX_TOKENS);
  CK(cudaSetDevice(e->device));
  if (n_replaced) *n_replaced = 0;
  if (e->n_slots == 0) {  // no corpus: only the vocabulary grows (example/import-merge-log-to-ram.ts:22-31)
    e->h_len16.push_back(e->h_len16[a] + e->h_len16[b]);
    e->h_merges.push_back(a);
    e->h_merges.push_back(b);
    e->h_merges.push_back(c);
    e->mt_dirty = e->lt_dirty = true;
    e->n_tokens++;
    e->index_valid = false;
    return BPE_OK;
  }
  // a single step would update this shard's counts with its local deltas only (the sharded loop exchanges them)
  if (e->mg_world > 1) return fail(e, BPE_E_INVALID, "bpe_apply_merge on a corpus is not available on a sharded engine; use bpe_merge_until");
  TRY(ensure_index(e));
  k_lookup_pair<<<1, 32, 0, e->stream>>>(e->table(), (uint32_t)a, (uint32_t)b, e->d_st.p);
  CKL();
  TRY(fetch_state(e));
  TRY(run_apply(e, (uint32_t)a, (uint32_t)b, (uint32_t)c, e->h_st->list_len));
  TRY(fetch_state(e));
  TRY(check_dev_err(e));
  e->stats.sites_merged += e->h_st->n_sites[0];
  if (n_replaced) *n_replaced = e->h_st->n_sites[0];
  return BPE_OK;
}


// Batched restoreMerge (core.ts:477-494; example/import-merge-log-to-ram.ts:24-31 replays one line per call): applies
// merges (a_i, b_i) -> n_tokens + i in order inside the persistent loop kernel, no arg-max, no host round trip per merge.
int bpe_apply_merges(bpe_engine* e, const int32_t* ab, int64_t n, int64_t* n_replaced) {
  if (!e || n < 0 || (n > 0 && !ab)) return fail(e, BPE_E_INVALID, "bad merge list");
  if (n == 0) return BPE_OK;
  if (is_group(e)) {  // on an empty corpus only the vocabulary grows, on every member (one bpe_apply_merge per line: no device work)
    if (group_slots(e)) return fail(e, BPE_E_INVALID, "bpe_apply_merges on a corpus is not available on a device group; use bpe_merge_until");
    bpe_engine* m0 = e->members[0];
    TRY(member_rc(e, m0, check_merge_list(m0, ab, n)));
    if (n_replaced) std::fill(n_replaced, n_replaced + n, (int64_t)0);
    return run_members(e, [&](int r) {
      bpe_engine* m = e->members[(size_t)r];
      for (int64_t i = 0; i < n; i++) TRY(bpe_apply_merge(m, ab[2 * i], ab[2 * i + 1], m->n_tokens, nullptr));
      return BPE_OK;
    });
  }
  CK(cudaSetDevice(e->device));
  if (e->mg_world > 1) return fail(e, BPE_E_INVALID, "bpe_apply_merges is not available on a sharded engine");
  TRY(check_merge_list(e, ab, n));
  if (e->n_slots == 0) {  // no corpus: only the vocabulary / merge list grow (import-merge-log-to-ram.ts:22 empties the corpus first)
    for (int64_t i = 0; i < n; i++) {
      e->h_len16.push_back(e->h_len16[ab[2 * i]] + e->h_len16[ab[2 * i + 1]]);
      e->h_merges.push_back(ab[2 * i]);
      e->h_merges.push_back(ab[2 * i + 1]);
      e->h_merges.push_back(e->n_tokens);
      e->n_tokens++;
      if (n_replaced) n_replaced[i] = 0;
    }
    e->mt_dirty = e->lt_dirty = true;
    TRY(sync_len16(e));
    return BPE_OK;
  }
  DevBuf<int32_t> d_ab;
  CK(d_ab.reserve((size_t)2 * n));
  CK(cudaMemcpyAsync(d_ab.p, ab, (size_t)2 * n * 4, cudaMemcpyHostToDevice, e->stream));
  std::vector<bpe_merge> log((size_t)n);
  int64_t done = 0;
  TRY(merge_until(e, 1, 0, n, log.data(), n, &done, d_ab.p));
  if (done != n) return fail(e, BPE_E_INTERNAL, "replayed %lld of %lld merges", (long long)done, (long long)n);
  if (n_replaced)
    for (int64_t i = 0; i < n; i++) n_replaced[i] = log[(size_t)i].weight;
  return BPE_OK;
}

int bpe_merge_until(bpe_engine* e, int64_t min_weight, int32_t max_length, int64_t max_iterations, bpe_merge* log,
                    int64_t log_cap, int64_t* n_done) {
  if (!e || !n_done || (log_cap > 0 && !log) || log_cap < 0) return BPE_E_INVALID;
  if (is_group(e)) return group_merge_until(e, min_weight, max_length, max_iterations, log, log_cap, n_done);
  return merge_until(e, min_weight, max_length, max_iterations, log, log_cap, n_done);
}


// ---- sharded training: mailbox set-up and the initial pair-count exchange ------------------------------------------
int bpe_mg_init(bpe_engine* e, int rank, int world, void* handle_out64) {
  if (!e || !handle_out64 || world < 1 || world > MG_MAX_WORLD || rank < 0 || rank >= world) return fail(e, BPE_E_INVALID, "bad rank/world");
  GROUP_REFUSES(e, "bpe_mg_init (the group's members are connected already)");
  CK(cudaSetDevice(e->device));
  if (e->mg_mailbox) return fail(e, BPE_E_INVALID, "bpe_mg_init called twice");
  TRY(mg_alloc_mailbox(e, rank, world));
  cudaIpcMemHandle_t h;
  static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
  CK(cudaIpcGetMemHandle(&h, e->mg_mailbox));
  memcpy(handle_out64, &h, sizeof h);
  e->mg_connected = (world == 1);
  return BPE_OK;
}

int bpe_mg_connect(bpe_engine* e, const char* handles /* world x 64 bytes, by rank */) {
  GROUP_REFUSES(e, "bpe_mg_connect (the group's members are connected already)");
  if (!e || !handles || !e->mg_mailbox) return fail(e, BPE_E_INVALID, "call bpe_mg_init first");
  CK(cudaSetDevice(e->device));
  for (int q = 0; q < e->mg_world; q++) {
    if (q == e->mg_rank || e->mg_peer[q]) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, handles + (size_t)q * 64, sizeof h);
    CK(cudaIpcOpenMemHandle(&e->mg_peer[q], h, cudaIpcMemLazyEnablePeerAccess));
  }
  e->mg_connected = true;
  return BPE_OK;
}

int bpe_mg_state(bpe_engine* e, int* counts_global) {
  if (!e || !counts_global) return BPE_E_INVALID;
  GROUP_REFUSES(e, "bpe_mg_state (the group exchanges its pair counts itself)");
  *counts_global = (e->index_valid && e->mg_counts_global) ? 1 : 0;
  return BPE_OK;
}

int bpe_mg_export_counts(bpe_engine* e, uint32_t* dev_keys, uint32_t* dev_counts, int64_t cap, int64_t* n) {
  if (!e || !n || cap < 0 || (cap > 0 && (!dev_keys || !dev_counts))) return fail(e, BPE_E_INVALID, "bad export arguments");
  GROUP_REFUSES(e, "bpe_mg_export_counts (the group exchanges its pair counts itself)");
  CK(cudaSetDevice(e->device));
  TRY(ensure_index(e));
  if (e->mg_counts_global) return fail(e, BPE_E_INVALID, "pair counts of this index were already exchanged");
  TRY(fetch_state(e));
  *n = e->h_st->n_keys;
  if (cap == 0) return BPE_OK;  // size query
  CK(e->mg_export_n.reserve(1));
  CK(cudaMemsetAsync(e->mg_export_n.p, 0, 4, e->stream));
  k_mg_export_counts<<<e->grid(4), 256, 0, e->stream>>>(e->table(), dev_keys, dev_counts, (uint32_t)std::min<int64_t>(cap, 0xFFFFFFFFll), e->mg_export_n.p);
  CKL();
  uint32_t got = 0;
  CK(cudaMemcpyAsync(&got, e->mg_export_n.p, 4, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  *n = got;
  if ((int64_t)got > cap) return fail(e, BPE_E_CAPACITY, "export buffers hold %lld pairs, need %u", (long long)cap, got);
  return BPE_OK;
}

int bpe_mg_import_counts(bpe_engine* e, const uint32_t* dev_keys, const uint32_t* dev_counts, int64_t n, int last) {
  if (!e || n < 0 || (n > 0 && (!dev_keys || !dev_counts))) return fail(e, BPE_E_INVALID, "bad import arguments");
  GROUP_REFUSES(e, "bpe_mg_import_counts (the group exchanges its pair counts itself)");
  CK(cudaSetDevice(e->device));
  if (!e->index_valid) return fail(e, BPE_E_INVALID, "no pair index to import into");
  TRY(fetch_state(e));
  uint64_t keys_after = (uint64_t)e->h_st->n_keys + (uint64_t)n;
  if (keys_after * 2 > e->tbl_cap) {
    uint64_t want = std::min<uint64_t>(keys_after * 5 / 2, 0x80000000ull);
    if (keys_after * 2 > pow2_at_least(want)) return fail(e, BPE_E_NOMEM, "pair table cannot grow further");
    TRY(grow_table(e, pow2_at_least(want)));
  }
  if (n) {
    k_mg_import_counts<<<e->grid(4), 256, 0, e->stream>>>(e->table(), dev_keys, dev_counts, (uint32_t)n, e->d_st.p);
    CKL();
  }
  TRY(fetch_state(e));
  TRY(check_dev_err(e));
  e->hot_valid = false;
  if (last) e->mg_counts_global = true;
  return BPE_OK;
}

int bpe_pair_counts(bpe_engine* e, int32_t* a, int32_t* b, int64_t* count, int64_t cap, int64_t* n) {
  if (!e || !n || cap < 0) return BPE_E_INVALID;
  *n = 0;
  if (is_group(e)) {  // after the exchange every member's table holds the corpus-wide counts: read one that has a corpus
    for (bpe_engine* m : e->members) {
      if (m->n_slots == 0) continue;
      TRY(group_exchange_counts(e));
      return member_rc(e, m, bpe_pair_counts(m, a, b, count, cap, n));
    }
    return BPE_OK;
  }
  CK(cudaSetDevice(e->device));
  if (e->n_slots == 0) return BPE_OK;
  TRY(ensure_index(e));
  DevBuf<int32_t> da, db;
  DevBuf<int64_t> dc;
  DevBuf<uint32_t> dn;
  size_t c = (size_t)std::max<int64_t>(cap, 1);
  CK(da.reserve(c));
  CK(db.reserve(c));
  CK(dc.reserve(c));
  CK(dn.reserve(1));
  CK(cudaMemsetAsync(dn.p, 0, 4, e->stream));
  k_dump_pairs<<<e->grid(4), 256, 0, e->stream>>>(e->table(), da.p, db.p, dc.p, (uint32_t)std::min<int64_t>(cap, 0x7FFFFFFF), dn.p);
  CKL();
  uint32_t cnt = 0;
  CK(cudaMemcpyAsync(&cnt, dn.p, 4, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  *n = cnt;
  if ((int64_t)cnt > cap) return fail(e, BPE_E_CAPACITY, "need room for %u pairs", cnt);
  if (cnt) {
    CK(cudaMemcpy(a, da.p, cnt * sizeof(int32_t), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(b, db.p, cnt * sizeof(int32_t), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(count, dc.p, cnt * sizeof(int64_t), cudaMemcpyDeviceToHost));
  }
  return BPE_OK;
}

int bpe_encode_batch_dev(bpe_engine* e, const int32_t* dev_ids, const int64_t* dev_doc_offsets, int64_t n_docs, int64_t n_ids,
                         int64_t max_doc_len, const int32_t* dev_to_vector_index, int32_t n_tvi, int32_t* dev_out,
                         int64_t* dev_out_offsets, int64_t* dev_first_bad, int64_t* n_out) {
  if (!e || !n_out || n_docs < 0 || n_ids < 0 || !dev_doc_offsets || !dev_out_offsets || (n_ids > 0 && (!dev_ids || !dev_out)))
    return fail(e, BPE_E_INVALID, "bad encode arguments");
  GROUP_REFUSES(e, "bpe_encode_batch_dev (device pointers belong to one device)");
  CK(cudaSetDevice(e->device));
  // scratch owned by the engine (freed by bpe_destroy, on the engine's device): reused across calls so that steady-state
  // encode does not allocate
  return encode_dev(e, e->dev_scratch, dev_ids, dev_doc_offsets, n_docs, n_ids, max_doc_len, dev_to_vector_index, n_tvi, dev_out,
                    dev_out_offsets, dev_first_bad, n_out);
}

// host buffers in, host buffers out: stage through grow-only device buffers owned by the engine
int stage_encode_inputs(bpe_engine* e, const int32_t* ids, const int64_t* doc_offsets, int64_t n_docs, int64_t* total_out, int64_t* max_len_out) {
  e->txt_staged = false;  // x_ids / h_rel are about to be reused
  int64_t base = n_docs ? doc_offsets[0] : 0, total = n_docs ? doc_offsets[n_docs] - base : 0;
  if (total > 0 && !ids) return fail(e, BPE_E_INVALID, "null ids");
  int64_t max_len = 0;
  e->h_rel.resize((size_t)n_docs + 1);
  e->h_rel[0] = 0;
  for (int64_t d = 0; d < n_docs; d++) {
    e->h_rel[d + 1] = doc_offsets[d + 1] - base;
    max_len = std::max(max_len, doc_offsets[d + 1] - doc_offsets[d]);
  }
  CK(e->x_ids.reserve((size_t)std::max<int64_t>(total, 1)));
  CK(e->x_out.reserve((size_t)std::max<int64_t>(total, 1)));
  CK(e->x_off.reserve((size_t)n_docs + 1));
  CK(e->x_ooff.reserve((size_t)n_docs + 1));
  CK(e->x_flag.reserve(1));
  if (total) CK(cudaMemcpyAsync(e->x_ids.p, ids + base, (size_t)total * 4, cudaMemcpyHostToDevice, e->stream));
  CK(cudaMemcpyAsync(e->x_off.p, e->h_rel.data(), (size_t)(n_docs + 1) * 8, cudaMemcpyHostToDevice, e->stream));
  if (total) {  // ids must name existing tokens; report the first offender like the reference's left-to-right scan would
    CK(cudaMemsetAsync(e->x_flag.p, 0xFF, 8, e->stream));
    k_first_bad_id<<<e->grid(8), 256, 0, e->stream>>>(e->x_ids.p, (uint64_t)total, (uint32_t)e->n_tokens, e->x_flag.p);
    CKL();
    unsigned long long fb = ~0ull;
    CK(cudaMemcpyAsync(&fb, e->x_flag.p, 8, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    if (fb != ~0ull) return fail(e, BPE_E_INVALID, "id %d at %lld outside the token table", ids[base + (int64_t)fb], (long long)fb);
  }
  *total_out = total;
  *max_len_out = max_len;
  return BPE_OK;
}

int encode_host(bpe_engine* e, bool is_text, const int32_t* ids, const uint8_t* utf8, const int64_t* off, int64_t n_docs, const int32_t* to_vector_index,
                int32_t n_tvi, int32_t* out, int64_t out_cap, int64_t* out_offsets, int64_t* first_bad, int64_t* n_out, int64_t* unknown_pos,
                int32_t* unknown_code_point);

int bpe_encode_batch(bpe_engine* e, const int32_t* ids, const int64_t* doc_offsets, int64_t n_docs, const int32_t* to_vector_index,
                     int32_t n_tvi, int32_t* out, int64_t out_cap, int64_t* out_offsets, int64_t* first_bad, int64_t* n_out) {
  if (!e || !n_out || !out_offsets) return fail(e, BPE_E_INVALID, "bad encode arguments");
  if (n_docs < 0 || (!doc_offsets && n_docs > 0)) return fail(e, BPE_E_INVALID, "bad document offsets");
  if (n_docs > 0 && doc_offsets[n_docs] > doc_offsets[0] && !ids) return fail(e, BPE_E_INVALID, "null ids");
  if (is_group(e))
    return group_encode(e, false, ids, nullptr, doc_offsets, n_docs, to_vector_index, n_tvi, out, out_cap, out_offsets, first_bad, n_out, nullptr, nullptr);
  CK(cudaSetDevice(e->device));
  return encode_host(e, false, ids, nullptr, doc_offsets, n_docs, to_vector_index, n_tvi, out, out_cap, out_offsets, first_bad, n_out, nullptr, nullptr);
}


// exclusive scan u32 -> u64 (n + 1 outputs) with the tiled kernels of encode_kernels.cuh
int scan_u32(bpe_engine* e, EncodeScratch& sc, const uint32_t* in, uint64_t* out, uint32_t n) {
  if (n <= 65536) {
    k_scan_counts<<<1, 1024, 0, e->stream>>>(in, out, n);
    CKL();
    return BPE_OK;
  }
  uint32_t n_tiles = (n + SC_TILE - 1) / SC_TILE;
  CK(sc.tile_sums.reserve(n_tiles));
  CK(sc.tile_off.reserve((size_t)n_tiles + 1));
  k_sum_tiles<<<n_tiles, SC_THREADS, 0, e->stream>>>(in, n, sc.tile_sums.p);
  CKL();
  k_scan_counts<<<1, 1024, 0, e->stream>>>(sc.tile_sums.p, sc.tile_off.p, n_tiles);
  CKL();
  k_scan_tiles<<<n_tiles, SC_THREADS, 0, e->stream>>>(in, n, sc.tile_off.p, n_tiles, out);
  CKL();
  return BPE_OK;
}


// ---- text front end: UTF-8 documents -> token indices on the device ----------------------------------------------
int ensure_cpmap(bpe_engine* e) {
  if (e->d_cpmap.p) return BPE_OK;
  CK(e->d_cpmap.reserve(CP_LIMIT));
  CK(e->d_firstpos.reserve(CP_LIMIT));
  CK(cudaMemsetAsync(e->d_cpmap.p, 0xFF, (size_t)CP_LIMIT * 4, e->stream));
  CK(cudaMemsetAsync(e->d_firstpos.p, 0xFF, (size_t)CP_LIMIT * 4, e->stream));
  return BPE_OK;
}

// launches only, no synchronisation: the UTF-8 bytes of whole documents (d_text, boundaries d_byte_off relative to it) become
// ids (placeholders -(cp+1) for unknown code points) and document boundaries in code points (d_char_off, n_docs + 1).
// track_new: keep the first positions of unknown code points (addToCorpus); otherwise d_flags[0] receives
// (pos << 32 | cp) of the first unknown code point or ~0.  d_flags[1] = code points of the longest document,
// d_flags[2] = code points in total.
int text_decode_dev(bpe_engine* e, const uint8_t* d_text, int64_t nbytes, const int64_t* d_byte_off, int64_t n_docs, int32_t* d_ids,
                    int64_t* d_char_off, bool track_new, unsigned long long* d_flags) {
  if ((uint64_t)nbytes >= 0xFFFFFFF0ull) return fail(e, BPE_E_DOMAIN, "text batch too large for one call");
  uint32_t n_tiles = (uint32_t)((nbytes + TX_TILE - 1) / TX_TILE);
  CK(e->x_tilecnt.reserve((size_t)n_tiles + 1));
  CK(e->x_tileoff.reserve((size_t)n_tiles + 2));
  CK(e->x_doccnt.reserve((size_t)n_docs + 1));
  CK(e->x_docoff.reserve((size_t)n_docs + 2));
  CK(cudaMemsetAsync(d_flags, 0xFF, 8, e->stream));
  CK(cudaMemsetAsync(d_flags + 1, 0, 8, e->stream));
  if (n_tiles) {
    k_utf8_count<<<n_tiles, TX_THREADS, 0, e->stream>>>(d_text, (uint64_t)nbytes, e->x_tilecnt.p);
    CKL();
  }
  TRY(scan_u32(e, e->x_scratch, e->x_tilecnt.p, e->x_tileoff.p, n_tiles));
  if (n_tiles) {
    k_utf8_decode<<<n_tiles, TX_THREADS, 0, e->stream>>>(d_text, (uint64_t)nbytes, e->x_tileoff.p, e->d_cpmap.p, d_ids,
                                                         track_new ? e->d_firstpos.p : nullptr, track_new ? nullptr : d_flags);
    CKL();
  }
  // document boundaries in code points: per-document counts, then a scan
  if (n_docs) {
    k_utf8_doc_counts<<<(int)std::min<int64_t>((n_docs + 7) / 8, (int64_t)e->grid(16)), 256, 0, e->stream>>>(d_text, d_byte_off, n_docs, e->x_doccnt.p);
    CKL();
    k_max_u32<<<(int)std::min<int64_t>((n_docs + 255) / 256, (int64_t)e->grid(4)), 256, 0, e->stream>>>(e->x_doccnt.p, n_docs, d_flags + 1);
    CKL();
  }
  TRY(scan_u32(e, e->x_scratch, e->x_doccnt.p, e->x_docoff.p, (uint32_t)n_docs));
  k_u64_to_i64<<<(int)std::min<int64_t>((n_docs + 256) / 256, (int64_t)e->grid(8)), 256, 0, e->stream>>>(e->x_docoff.p, d_char_off, n_docs + 1);
  CKL();
  CK(cudaMemcpyAsync(d_flags + 2, e->x_docoff.p + n_docs, 8, cudaMemcpyDeviceToDevice, e->stream));
  return BPE_OK;
}

// one un-pipelined batch (bpe_add_text): decodes into e->x_ids, document boundaries in code points into e->x_off (device)
// and e->h_rel (host)
int text_to_ids(bpe_engine* e, const uint8_t* utf8, const int64_t* doc_byte_offsets, int64_t n_docs, bool track_new, int64_t* n_chars,
                unsigned long long* unknown) {
  e->txt_staged = false;
  TRY(check_offsets(e, doc_byte_offsets, n_docs));
  TRY(ensure_cpmap(e));
  int64_t base = n_docs ? doc_byte_offsets[0] : 0, nbytes = n_docs ? doc_byte_offsets[n_docs] - base : 0;
  if (nbytes > 0 && !utf8) return fail(e, BPE_E_INVALID, "null text");
  if ((uint64_t)nbytes >= 0xFFFFFFF0ull) return fail(e, BPE_E_DOMAIN, "text batch too large for one call");
  std::vector<int64_t> rel((size_t)n_docs + 1, 0);
  for (int64_t d = 0; d < n_docs; d++) rel[d + 1] = doc_byte_offsets[d + 1] - base;
  CK(e->x_text.reserve((size_t)std::max<int64_t>(nbytes, 1)));
  CK(e->x_ids.reserve((size_t)std::max<int64_t>(nbytes, 1)));  // at most one code point per byte
  CK(e->x_off.reserve((size_t)n_docs + 1));
  CK(e->x_ooff.reserve((size_t)n_docs + 1));
  CK(e->x_flag.reserve(8));
  if (nbytes) CK(cudaMemcpyAsync(e->x_text.p, utf8 + base, (size_t)nbytes, cudaMemcpyHostToDevice, e->stream));
  CK(cudaMemcpyAsync(e->x_ooff.p, rel.data(), (size_t)(n_docs + 1) * 8, cudaMemcpyHostToDevice, e->stream));  // byte offsets
  TRY(text_decode_dev(e, e->x_text.p, nbytes, e->x_ooff.p, n_docs, e->x_ids.p, e->x_off.p, track_new, e->x_flag.p));
  e->h_rel.resize((size_t)n_docs + 1);
  CK(cudaMemcpyAsync(e->h_rel.data(), e->x_off.p, (size_t)(n_docs + 1) * 8, cudaMemcpyDeviceToHost, e->stream));
  unsigned long long unk = ~0ull;
  CK(cudaMemcpyAsync(&unk, e->x_flag.p, 8, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  *n_chars = n_docs ? e->h_rel[(size_t)n_docs] : 0;
  if (unknown) *unknown = unk;
  return BPE_OK;
}

// ---- host buffers in, host buffers out: chunks of whole documents flow through three streams ----------------------------
// copy in (s_in) | front end + encode (e->stream) | copy out (s_out).  Chunk c+1 is uploaded while chunk c is encoded and the
// vectors of chunk c-1 travel back; every chunk owns its own region of the staging buffers, so no stage waits for a buffer.
// With pinned host buffers the call costs max(PCIe in, encode, PCIe out) instead of their sum; with pageable buffers the
// copies are synchronous and the call degrades to the serial order.
struct PipeChunk {
  int64_t d0 = 0, d1 = 0;    // documents [d0, d1)
  int64_t in0 = 0, in1 = 0;  // input units (ids or bytes) relative to the first document of the batch
  int64_t max_len = 0;       // longest document in input units
  int64_t reg = 0, oreg = 0; // where the chunk lives in the unit staging buffers / the offset staging buffers
};

// the next chunk starting at document d0: about `target` input units, at least one document.  The offsets are checked on the
// way (nothing is read through an offset that was not) and written, relative to the chunk, to `rel` (d1 - d0 + 1 values).
int next_chunk(bpe_engine* e, const int64_t* off, int64_t n_docs, int64_t d0, int64_t target, int64_t* rel, PipeChunk* c) {
  const int64_t first = off[d0], limit = first + target;
  int64_t d = d0, max_len = 0;
  rel[0] = 0;
  while (d < n_docs && (d == d0 || off[d + 1] <= limit)) {
    int64_t len = off[d + 1] - off[d];
    if (len < 0) return fail(e, BPE_E_INVALID, "document offsets must be non-decreasing (doc %lld)", (long long)d);
    max_len = std::max(max_len, len);
    d++;
    rel[d - d0] = off[d] - first;
  }
  c->d0 = d0;
  c->d1 = d;
  c->in0 = first - off[0];
  c->in1 = off[d] - off[0];
  c->max_len = max_len;
  return BPE_OK;
}

// Sizes of the pipeline for a batch of `total` input units in n_docs documents.  The first chunks are small and double up to
// `target` (the first copy in is exposed), the last ones halve again (so are the last encode and the last copy out).  A chunk
// closes when the next document would pass its target, so two consecutive chunks always hold more than the smallest target
// -- which bounds their number and with it the staging buffers (tests/test_abi_symbols.py checks the bound through
// bpe_debug_plan_chunks).
struct PipePlan {
  int64_t target, min_target, max_chunks, pad;
  size_t unit_cap, off_cap;
};

PipePlan pipe_plan(int64_t total, int64_t n_docs, int64_t chunk_units) {
  PipePlan P;
  P.target = std::min<int64_t>(std::max<int64_t>(chunk_units, 1), 1ll << 40);
  P.min_target = std::max<int64_t>(P.target / 8, 1);
  P.max_chunks = std::min<int64_t>(2 * (total / P.min_target) + 8, n_docs + 1);
  P.pad = 256;  // every chunk's region of the unit buffers starts on a multiple of this
  P.unit_cap = (size_t)(total + P.pad * P.max_chunks);
  P.off_cap = (size_t)(n_docs + P.max_chunks + 1);
  return P;
}

// target of chunk number `index` when `remaining` units are left
int64_t pipe_want(const PipePlan& P, int64_t index, int64_t remaining) {
  int64_t want = P.target >> std::max<int64_t>(0, 3 - index);          // ramp up: 1/8, 1/4, 1/2, 1
  want = std::min(want, std::max(remaining / 2, P.min_target));        // ramp down
  return std::max(want, P.min_target);
}

int encode_pipeline(bpe_engine* e, const bool is_text, const int32_t* ids, const uint8_t* utf8, const int64_t* off, int64_t n_docs,
                    const int32_t* to_vector_index, int32_t n_tvi, int32_t* out, int64_t out_cap, int64_t* out_offsets, int64_t* first_bad,
                    int64_t* n_out, int64_t* unknown_pos, int32_t* unknown_code_point) {
  e->txt_staged = false;
  e->enc_parts.clear();
  e->enc_bad_id_pos = -1;
  const int64_t base = off[0];
  if (off[n_docs] < base) return fail(e, BPE_E_INVALID, "document offsets must be non-decreasing");
  const int64_t total = off[n_docs] - base;
  const PipePlan P = pipe_plan(total, n_docs, e->enc_chunk);
  const int64_t pad = P.pad;
  const size_t unit_cap = P.unit_cap, off_cap = P.off_cap;
  // everything a chunk in flight may touch is allocated before the first copy starts
  if (is_text) {
    TRY(ensure_cpmap(e));
    CK(e->x_text.reserve(unit_cap));
    CK(e->x_ooff2.reserve(off_cap));
  }
  CK(e->x_ids.reserve(unit_cap));  // text: at most one code point per byte
  CK(e->x_out.reserve(unit_cap));
  CK(e->x_off.reserve(off_cap));
  CK(e->x_ooff.reserve(off_cap));
  CK(e->x_flag.reserve(12));
  CK(e->h_in_off.reserve(off_cap));
  CK(e->h_out_off.reserve((size_t)n_docs + 1));
  if (first_bad) {
    CK(e->x_bad.reserve((size_t)n_docs));
    CK(e->h_bad.reserve((size_t)n_docs));
  }
  const int32_t* d_tvi = nullptr;
  if (to_vector_index && n_tvi > 0) {
    CK(e->x_tvi.reserve((size_t)n_tvi));
    CK(cudaMemcpyAsync(e->x_tvi.p, to_vector_index, (size_t)n_tvi * 4, cudaMemcpyHostToDevice, e->stream));
  }
  if (to_vector_index) d_tvi = e->x_tvi.p;
  int64_t* d_in_off = is_text ? e->x_ooff.p : e->x_off.p;  // the caller's offsets relative to the chunk (text: in bytes)
  int64_t* d_out_off = is_text ? e->x_ooff2.p : e->x_ooff.p;

  int64_t n_up = 0;  // chunks sent so far
  // s_in: the chunk after `prev` goes to the device (units, offsets; ids are checked against the token table there)
  auto upload_next = [&](const PipeChunk& prev, int slot, PipeChunk* c) -> int {
    const int64_t reg = (prev.reg + (prev.in1 - prev.in0) + pad - 1) / pad * pad, oreg = prev.oreg + (prev.d1 - prev.d0) + (prev.d1 ? 1 : 0);
    TRY(next_chunk(e, off, n_docs, prev.d1, pipe_want(P, n_up, total - prev.in1), e->h_in_off.p + oreg, c));
    c->reg = reg;
    c->oreg = oreg;
    const int64_t len = c->in1 - c->in0, nd = c->d1 - c->d0;
    CK(cudaMemcpyAsync(d_in_off + oreg, e->h_in_off.p + oreg, (size_t)(nd + 1) * 8, cudaMemcpyHostToDevice, e->s_in));
    if (len && is_text) CK(cudaMemcpyAsync(e->x_text.p + reg, utf8 + base + c->in0, (size_t)len, cudaMemcpyHostToDevice, e->s_in));
    if (len && !is_text) CK(cudaMemcpyAsync(e->x_ids.p + reg, ids + base + c->in0, (size_t)len * 4, cudaMemcpyHostToDevice, e->s_in));
    if (!is_text) {  // ids must name existing tokens; the first offender is reported like the reference's left-to-right scan would
      CK(cudaMemsetAsync(e->x_flag.p + slot * 4, 0xFF, 8, e->s_in));
      if (len) {
        k_first_bad_id<<<e->grid(8), 256, 0, e->s_in>>>(e->x_ids.p + reg, (uint64_t)len, (uint32_t)e->n_tokens, e->x_flag.p + slot * 4);
        CKL();
      }
      k_copy_u64<<<1, 32, 0, e->s_in>>>(e->h_pipe + slot * 4, e->x_flag.p + slot * 4, 1);
      CKL();
    }
    CK(cudaEventRecord(e->ev_in[slot], e->s_in));
    return BPE_OK;
  };
  // the per-document results of a finished chunk leave the pinned staging for the caller's arrays
  auto deliver = [&](const PipeChunk& c, int res_slot, bool last) -> int {
    CK(cudaEventSynchronize(e->ev_res[res_slot]));
    const int64_t nd = c.d1 - c.d0;
    memcpy(out_offsets + c.d0, e->h_out_off.p + c.d0, (size_t)(nd + (last ? 1 : 0)) * 8);
    if (first_bad) memcpy(first_bad + c.d0, e->h_bad.p + c.d0, (size_t)nd * 8);
    return BPE_OK;
  };

  PipeChunk chunks[3], done;  // chunks[c % 3]: current, next, the one after
  int64_t cum = 0, char_cum = 0;
  bool overflow = false, have_done = false;
  float ms_sum = 0;
  TRY(upload_next(PipeChunk(), 0, &chunks[0]));
  n_up = 1;
  if (chunks[0].d1 < n_docs) {
    TRY(upload_next(chunks[0], 1, &chunks[1]));
    n_up = 2;
  }
  for (int64_t c = 0;; c++) {
    const PipeChunk cur = chunks[c % 3];
    const int slot = (int)(c % 3);
    const int64_t nd = cur.d1 - cur.d0, len = cur.in1 - cur.in0;
    const bool last = cur.d1 >= n_docs;
    int64_t n_units = len, max_len = cur.max_len;
    if (!is_text) {
      CK(cudaEventSynchronize(e->ev_in[slot]));
      unsigned long long fb = *static_cast<volatile unsigned long long*>(e->h_pipe + slot * 4);
      if (fb != ~0ull) {
        e->enc_bad_id_pos = cur.in0 + (int64_t)fb;
        return fail(e, BPE_E_INVALID, "id %d at %lld outside the token table", ids[base + e->enc_bad_id_pos], (long long)e->enc_bad_id_pos);
      }
    } else {
      CK(cudaStreamWaitEvent(e->stream, e->ev_in[slot], 0));
      TRY(text_decode_dev(e, e->x_text.p + cur.reg, len, d_in_off + cur.oreg, nd, e->x_ids.p + cur.reg, e->x_off.p + cur.oreg, false,
                          e->x_flag.p + slot * 4));
      k_copy_u64<<<1, 32, 0, e->stream>>>(e->h_pipe + slot * 4, e->x_flag.p + slot * 4, 3);
      CKL();
      CK(cudaStreamSynchronize(e->stream));
      const volatile unsigned long long* hp = e->h_pipe;
      unsigned long long unk = hp[slot * 4];
      if (unk != ~0ull) {  // encodeToCode throws at the first unknown character (core.ts:398-400)
        int64_t pos = char_cum + (int64_t)(unk >> 32);
        if (unknown_pos) *unknown_pos = pos;
        if (unknown_code_point) *unknown_code_point = (int32_t)(unk & 0xFFFFFFFFu);
        return fail(e, BPE_E_INVALID, "unknown token, char: U+%04X at code point %lld", (unsigned)(unk & 0xFFFFFFFFu), (long long)pos);
      }
      max_len = (int64_t)hp[slot * 4 + 1];
      n_units = (int64_t)hp[slot * 4 + 2];
    }
    // host work hidden under the encode kernel: the chunk after the next one starts its way in, the previous one is handed over
    const std::function<int()> overlap = [&]() -> int {
      if (n_up == c + 2 && chunks[(c + 1) % 3].d1 < n_docs) {
        TRY(upload_next(chunks[(c + 1) % 3], (int)((c + 2) % 3), &chunks[(c + 2) % 3]));
        n_up++;
      }
      if (have_done) TRY(deliver(done, (int)((c - 1) & 1), false));
      have_done = false;
      return BPE_OK;
    };
    int64_t k = 0;
    TRY(encode_dev(e, e->x_scratch, e->x_ids.p + cur.reg, e->x_off.p + cur.oreg, nd, n_units, max_len, d_tvi, n_tvi, e->x_out.p + cur.reg,
                   d_out_off + cur.oreg, first_bad ? e->x_bad.p + cur.d0 : nullptr, &k, &overlap));
    ms_sum += e->stats.ms_encode;
    if (cum) {  // the chunk's output offsets take their place in the batch
      k_shift_i64<<<(int)std::min<int64_t>((nd + 256) / 256, (int64_t)e->grid(4)), 256, 0, e->stream>>>(d_out_off + cur.oreg, nd + 1, cum);
      CKL();
    }
    CK(cudaEventRecord(e->ev_done, e->stream));
    CK(cudaStreamWaitEvent(e->s_out, e->ev_done, 0));
    CK(cudaMemcpyAsync(e->h_out_off.p + cur.d0, d_out_off + cur.oreg, (size_t)(nd + (last ? 1 : 0)) * 8, cudaMemcpyDeviceToHost, e->s_out));
    if (first_bad && nd) CK(cudaMemcpyAsync(e->h_bad.p + cur.d0, e->x_bad.p + cur.d0, (size_t)nd * 8, cudaMemcpyDeviceToHost, e->s_out));
    CK(cudaEventRecord(e->ev_res[c & 1], e->s_out));
    if (cum + k > out_cap || (k && !out)) overflow = true;  // keep going: the caller learns the size it needs
    if (!overflow && k) CK(cudaMemcpyAsync(out + cum, e->x_out.p + cur.reg, (size_t)k * 4, cudaMemcpyDeviceToHost, e->s_out));
    e->enc_parts.push_back(cur.reg);
    e->enc_parts.push_back(k);
    cum += k;
    char_cum += n_units;
    done = cur;
    have_done = true;
    if (last) {
      TRY(deliver(done, (int)(c & 1), true));
      break;
    }
  }
  *n_out = cum;
  e->stats.ms_encode = ms_sum;
  if (overflow) return fail(e, BPE_E_CAPACITY, "output buffer holds %lld values, need %lld", (long long)out_cap, (long long)cum);
  return BPE_OK;
}

int encode_host(bpe_engine* e, bool is_text, const int32_t* ids, const uint8_t* utf8, const int64_t* off, int64_t n_docs, const int32_t* to_vector_index,
                int32_t n_tvi, int32_t* out, int64_t out_cap, int64_t* out_offsets, int64_t* first_bad, int64_t* n_out, int64_t* unknown_pos,
                int32_t* unknown_code_point) {
  *n_out = 0;
  if (n_docs == 0) {
    out_offsets[0] = 0;
    return BPE_OK;
  }
  TRY(ensure_pipe(e));
  int rc = encode_pipeline(e, is_text, ids, utf8, off, n_docs, to_vector_index, n_tvi, out, out_cap, out_offsets, first_bad, n_out, unknown_pos, unknown_code_point);
  // whatever happened, nothing may still read or write the caller's buffers when the call returns
  cudaError_t c0 = cudaStreamSynchronize(e->s_in), c1 = cudaStreamSynchronize(e->stream), c2 = cudaStreamSynchronize(e->s_out);
  if (rc == BPE_OK && (c0 != cudaSuccess || c1 != cudaSuccess || c2 != cudaSuccess))
    rc = fail(e, BPE_E_CUDA, "encode pipeline: %s", cudaGetErrorString(c0 != cudaSuccess ? c0 : c1 != cudaSuccess ? c1 : c2));
  return rc;
}

int bpe_decode_batch(bpe_engine* e, const int32_t* values, const int64_t* doc_offsets, int64_t n_docs, const int32_t* from_vector_index,
                     int32_t n_fvi, const uint8_t* token_bytes, const int64_t* token_byte_offsets, int32_t n_tokens, uint8_t* out,
                     int64_t out_cap, int64_t* out_offsets, int64_t* first_bad, int64_t* n_out) {
  if (!e || !n_out || !out_offsets || n_tokens < 0 || (n_tokens > 0 && (!token_byte_offsets))) return fail(e, BPE_E_INVALID, "bad decode arguments");
  if (is_group(e))
    return group_decode(e, values, doc_offsets, n_docs, from_vector_index, n_fvi, token_bytes, token_byte_offsets, n_tokens, out, out_cap, out_offsets,
                        first_bad, n_out);
  e->txt_staged = false;
  TRY(check_offsets(e, doc_offsets, n_docs));
  CK(cudaSetDevice(e->device));
  int64_t base = n_docs ? doc_offsets[0] : 0, total = n_docs ? doc_offsets[n_docs] - base : 0;
  if (total > 0 && !values) return fail(e, BPE_E_INVALID, "null values");
  if ((uint64_t)total >= 0xFFFFFFF0ull) return fail(e, BPE_E_DOMAIN, "batch too large for one decode call");
  const int64_t arena = n_tokens ? token_byte_offsets[n_tokens] : 0;
  if (arena > 0 && !token_bytes) return fail(e, BPE_E_INVALID, "null token bytes");
  e->h_rel.resize((size_t)n_docs + 1);
  e->h_rel[0] = 0;
  for (int64_t d = 0; d < n_docs; d++) e->h_rel[d + 1] = doc_offsets[d + 1] - base;
  DevBuf<uint8_t> d_arena, d_out;
  DevBuf<int64_t> d_tokoff;
  DevBuf<uint32_t> d_lens;
  DevBuf<uint64_t> d_boff;
  DevBuf<unsigned long long> d_bad;
  CK(e->x_ids.reserve((size_t)std::max<int64_t>(total, 1)));
  CK(e->x_off.reserve((size_t)n_docs + 1));
  CK(e->x_ooff.reserve((size_t)n_docs + 1));
  CK(d_arena.reserve((size_t)std::max<int64_t>(arena, 1)));
  CK(d_tokoff.reserve((size_t)n_tokens + 1));
  CK(d_lens.reserve((size_t)std::max<int64_t>(total, 1)));
  CK(d_boff.reserve((size_t)total + 1));
  if (total) CK(cudaMemcpyAsync(e->x_ids.p, values + base, (size_t)total * 4, cudaMemcpyHostToDevice, e->stream));
  CK(cudaMemcpyAsync(e->x_off.p, e->h_rel.data(), (size_t)(n_docs + 1) * 8, cudaMemcpyHostToDevice, e->stream));
  if (arena) CK(cudaMemcpyAsync(d_arena.p, token_bytes, (size_t)arena, cudaMemcpyHostToDevice, e->stream));
  if (n_tokens) CK(cudaMemcpyAsync(d_tokoff.p, token_byte_offsets, (size_t)(n_tokens + 1) * 8, cudaMemcpyHostToDevice, e->stream));
  else CK(cudaMemsetAsync(d_tokoff.p, 0, 8, e->stream));
  if (from_vector_index && n_fvi > 0) {
    CK(e->x_tvi.reserve((size_t)n_fvi));
    CK(cudaMemcpyAsync(e->x_tvi.p, from_vector_index, (size_t)n_fvi * 4, cudaMemcpyHostToDevice, e->stream));
  }
  if (first_bad) {
    CK(d_bad.reserve((size_t)std::max<int64_t>(n_docs, 1)));
    CK(cudaMemsetAsync(d_bad.p, 0xFF, (size_t)std::max<int64_t>(n_docs, 1) * 8, e->stream));
  }
  const int32_t* fvi = from_vector_index ? e->x_tvi.p : nullptr;
  int blocks = (int)std::min<int64_t>((total + 255) / 256 + 1, (int64_t)e->grid(8));
  k_decode_lens<<<blocks, 256, 0, e->stream>>>(e->x_ids.p, (uint64_t)total, fvi, from_vector_index ? n_fvi : 0, d_tokoff.p, n_tokens, e->x_off.p, n_docs, d_lens.p,
                                            first_bad ? d_bad.p : nullptr);
  CKL();
  TRY(scan_u32(e, e->x_scratch, d_lens.p, d_boff.p, (uint32_t)total));
  uint64_t nbytes = 0;
  CK(cudaMemcpyAsync(&nbytes, d_boff.p + total, 8, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  *n_out = (int64_t)nbytes;
  k_decode_doc_offsets<<<(int)std::min<int64_t>((n_docs + 256) / 256, (int64_t)e->grid(8)), 256, 0, e->stream>>>(e->x_off.p, n_docs, d_boff.p, e->x_ooff.p);
  CKL();
  CK(cudaMemcpyAsync(out_offsets, e->x_ooff.p, (size_t)(n_docs + 1) * 8, cudaMemcpyDeviceToHost, e->stream));
  if (first_bad && n_docs) {
    CK(cudaMemcpyAsync(first_bad, d_bad.p, (size_t)n_docs * 8, cudaMemcpyDeviceToHost, e->stream));  // ~0 (== -1) = no offender
  }
  if ((int64_t)nbytes > out_cap || (nbytes && !out)) {
    CK(cudaStreamSynchronize(e->stream));
    return fail(e, BPE_E_CAPACITY, "output buffer holds %lld bytes, need %llu", (long long)out_cap, (unsigned long long)nbytes);
  }
  if (nbytes) {
    CK(d_out.reserve((size_t)nbytes));
    k_decode_gather<<<blocks, 256, 0, e->stream>>>(e->x_ids.p, (uint64_t)total, fvi, from_vector_index ? n_fvi : 0, d_arena.p, d_tokoff.p, n_tokens, d_boff.p, d_out.p);
    CKL();
    CK(cudaMemcpyAsync(out, d_out.p, (size_t)nbytes, cudaMemcpyDeviceToHost, e->stream));
  }
  CK(cudaStreamSynchronize(e->stream));
  return BPE_OK;
}


// ---- text in, tokens out ---------------------------------------------------------------------------------------------
int bpe_set_chars(bpe_engine* e, const int32_t* code_points, const int32_t* indices, int32_t n) {
  if (!e || n < 0 || (n > 0 && (!code_points || !indices))) return fail(e, BPE_E_INVALID, "bad character table");
  if (is_group(e)) return run_members(e, [&](int r) { return bpe_set_chars(e->members[(size_t)r], code_points, indices, n); });
  e->txt_staged = false;  // its ids were resolved against the table being replaced
  CK(cudaSetDevice(e->device));
  TRY(ensure_cpmap(e));
  CK(cudaMemsetAsync(e->d_cpmap.p, 0xFF, (size_t)CP_LIMIT * 4, e->stream));
  if (n) {
    DevBuf<int32_t> a, b;
    CK(a.reserve((size_t)n));
    CK(b.reserve((size_t)n));
    CK(cudaMemcpyAsync(a.p, code_points, (size_t)n * 4, cudaMemcpyHostToDevice, e->stream));
    CK(cudaMemcpyAsync(b.p, indices, (size_t)n * 4, cudaMemcpyHostToDevice, e->stream));
    k_set_cpmap<<<(n + 255) / 256, 256, 0, e->stream>>>(e->d_cpmap.p, a.p, b.p, (uint32_t)n);
    CKL();
    CK(cudaStreamSynchronize(e->stream));
  }
  return BPE_OK;
}

int bpe_add_text_stage(bpe_engine* e, const uint8_t* utf8, const int64_t* doc_byte_offsets, int64_t n_docs, int32_t* new_code_points,
                       int64_t* first_pos, int32_t new_cap, int32_t* n_new) {
  if (!e || !n_new || new_cap < 0 || (new_cap > 0 && (!new_code_points || !first_pos))) return fail(e, BPE_E_INVALID, "bad arguments");
  GROUP_REFUSES(e, "bpe_add_text_stage (bpe_add_text orders the new characters over the group itself)");
  *n_new = 0;
  CK(cudaSetDevice(e->device));
  int64_t n_chars = 0;
  TRY(text_to_ids(e, utf8, doc_byte_offsets, n_docs, true, &n_chars, nullptr));
  // the unknown code points with their first positions; k_collect_new_cps resets d_firstpos as it reads it
  DevBuf<uint32_t> d_cp, d_pos, d_n;
  const uint32_t cap = 1u << 16;
  CK(d_cp.reserve(cap));
  CK(d_pos.reserve(cap));
  CK(d_n.reserve(1));
  CK(cudaMemsetAsync(d_n.p, 0, 4, e->stream));
  k_collect_new_cps<<<e->grid(4), 256, 0, e->stream>>>(e->d_firstpos.p, d_cp.p, d_pos.p, cap, d_n.p);
  CKL();
  uint32_t nn = 0;
  CK(cudaMemcpyAsync(&nn, d_n.p, 4, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  if (nn > cap || (int64_t)e->n_tokens + nn > BPE_MAX_TOKENS) return fail(e, BPE_E_DOMAIN, "token table would exceed %d", BPE_MAX_TOKENS);
  if ((int32_t)nn > new_cap) {
    *n_new = (int32_t)nn;
    return fail(e, BPE_E_CAPACITY, "%u new characters, room for %d", nn, new_cap);
  }
  std::vector<uint32_t> cps(nn), pos(nn), order(nn);
  if (nn) {
    CK(cudaMemcpy(cps.data(), d_cp.p, (size_t)nn * 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(pos.data(), d_pos.p, (size_t)nn * 4, cudaMemcpyDeviceToHost));
  }
  // reported in first-appearance order (the collection order is arbitrary)
  for (uint32_t i = 0; i < nn; i++) order[i] = i;
  std::sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) { return pos[x] < pos[y]; });
  e->txt_new.resize(nn);
  for (uint32_t k = 0; k < nn; k++) {
    new_code_points[k] = (int32_t)cps[order[k]];
    first_pos[k] = (int64_t)pos[order[k]];
    e->txt_new[k] = (int32_t)cps[k];
  }
  std::sort(e->txt_new.begin(), e->txt_new.end());
  *n_new = (int32_t)nn;
  e->txt_chars = n_chars;
  e->txt_docs = n_docs;
  e->txt_staged = true;
  return BPE_OK;
}

int bpe_add_text_commit(bpe_engine* e, const int32_t* code_points, int32_t n, int64_t* counts, int64_t counts_cap) {
  if (!e) return BPE_E_INVALID;
  GROUP_REFUSES(e, "bpe_add_text_commit (bpe_add_text orders the new characters over the group itself)");
  if (!e->txt_staged) return fail(e, BPE_E_INVALID, "no staged text batch: bpe_add_text_stage first (another call since then reused its buffers)");
  if (n < 0 || (n > 0 && !code_points)) return fail(e, BPE_E_INVALID, "bad code point list");
  CK(cudaSetDevice(e->device));
  // the list comes from outside the library (another rank's exchange): check it before anything changes
  std::vector<int32_t> sorted(code_points, code_points + n);
  std::sort(sorted.begin(), sorted.end());
  for (int32_t i = 0; i < n; i++) {
    if ((uint32_t)sorted[i] >= CP_LIMIT) return fail(e, BPE_E_INVALID, "code point %d is not a Unicode code point", sorted[i]);
    if (i && sorted[i] == sorted[i - 1]) return fail(e, BPE_E_INVALID, "code point U+%04X is listed twice", sorted[i]);
  }
  for (int32_t cp : e->txt_new)
    if (!std::binary_search(sorted.begin(), sorted.end(), cp)) return fail(e, BPE_E_INVALID, "the list misses U+%04X, a new character of the staged batch", cp);
  DevBuf<int32_t> a, b;
  if (n) {
    std::vector<int32_t> known((size_t)n);
    CK(a.reserve((size_t)n));
    CK(b.reserve((size_t)n));
    CK(cudaMemcpyAsync(a.p, code_points, (size_t)n * 4, cudaMemcpyHostToDevice, e->stream));
    k_get_cpmap<<<(n + 255) / 256, 256, 0, e->stream>>>(e->d_cpmap.p, a.p, b.p, (uint32_t)n);
    CKL();
    CK(cudaMemcpyAsync(known.data(), b.p, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    for (int32_t k = 0; k < n; k++)
      if (known[k] >= 0) return fail(e, BPE_E_INVALID, "code point U+%04X already is token %d", code_points[k], known[k]);
  }
  if ((int64_t)e->n_tokens + n > BPE_MAX_TOKENS) return fail(e, BPE_E_DOMAIN, "token table would exceed %d", BPE_MAX_TOKENS);
  if (counts && counts_cap < (int64_t)e->n_tokens + n)
    return fail(e, BPE_E_CAPACITY, "counts holds %lld entries, need %d", (long long)counts_cap, e->n_tokens + n);
  e->txt_staged = false;
  if (n) {
    // code_points[k] becomes token n_tokens + k (core.ts:186-199)
    std::vector<int32_t> h_idx((size_t)n);
    for (int32_t k = 0; k < n; k++) {
      h_idx[k] = e->n_tokens + k;
      e->h_len16.push_back(code_points[k] >= 0x10000 ? 2 : 1);  // `chars.length` in UTF-16 units (core.ts:272)
    }
    e->n_tokens += n;
    e->mt_dirty = e->lt_dirty = true;
    TRY(sync_len16(e));
    CK(cudaMemcpyAsync(b.p, h_idx.data(), (size_t)n * 4, cudaMemcpyHostToDevice, e->stream));
    k_set_cpmap<<<(n + 255) / 256, 256, 0, e->stream>>>(e->d_cpmap.p, a.p, b.p, (uint32_t)n);
    CKL();
    CK(cudaStreamSynchronize(e->stream));
  }
  CK(e->x_counts.reserve((size_t)std::max(e->n_tokens, 1)));
  CK(cudaMemsetAsync(e->x_counts.p, 0, (size_t)std::max(e->n_tokens, 1) * 8, e->stream));
  if (e->txt_chars) {
    k_fix_and_count<<<e->grid(8), 256, 0, e->stream>>>(e->x_ids.p, (uint64_t)e->txt_chars, e->d_cpmap.p, e->x_counts.p, (uint32_t)e->n_tokens);
    CKL();
  }
  if (counts) CK(cudaMemcpyAsync(counts, e->x_counts.p, (size_t)e->n_tokens * 8, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  return append_docs_dev(e, e->x_ids.p, e->h_rel.data(), e->txt_docs);
}

int bpe_add_text(bpe_engine* e, const uint8_t* utf8, const int64_t* doc_byte_offsets, int64_t n_docs, int32_t* new_code_points, int32_t new_cap,
                 int32_t* n_new, int64_t* counts, int64_t counts_cap) {
  if (!e || !n_new) return fail(e, BPE_E_INVALID, "bad arguments");
  *n_new = 0;
  if (is_group(e)) return group_add_text(e, utf8, doc_byte_offsets, n_docs, new_code_points, new_cap, n_new, counts, counts_cap);
  const bool trace_t = getenv("BPE_TRACE") != nullptr;
  auto clk = [] { return std::chrono::steady_clock::now(); };
  auto since = [&](std::chrono::steady_clock::time_point t) { return std::chrono::duration<double, std::milli>(clk() - t).count(); };
  auto tt0 = clk();
  // one engine holds the whole batch: its own first-appearance order is the global one
  std::vector<int32_t> cps(1u << 16);
  std::vector<int64_t> pos(1u << 16);
  int32_t nn = 0;
  TRY(bpe_add_text_stage(e, utf8, doc_byte_offsets, n_docs, cps.data(), pos.data(), (int32_t)cps.size(), &nn));
  const double ms_stage = since(tt0);
  if (nn > new_cap) {
    e->txt_staged = false;
    *n_new = nn;
    return fail(e, BPE_E_CAPACITY, "%d new characters, room for %d", nn, new_cap);
  }
  std::copy(cps.begin(), cps.begin() + nn, new_code_points);  // (stage reports them in first-appearance order)
  const int64_t n_chars = e->txt_chars;
  int rc = bpe_add_text_commit(e, cps.data(), nn, counts, counts_cap);
  if (rc == BPE_OK) *n_new = nn;
  if (trace_t) {
    cudaStreamSynchronize(e->stream);
    fprintf(stderr, "[bpe] add_text: %lld chars: copy in + decode + new characters %.1f ms, commit (table, counts, append) %.1f ms\n", (long long)n_chars,
            ms_stage, since(tt0) - ms_stage);
  }
  return rc;
}

int bpe_encode_text_batch(bpe_engine* e, const uint8_t* utf8, const int64_t* doc_byte_offsets, int64_t n_docs, const int32_t* to_vector_index,
                          int32_t n_tvi, int32_t* out, int64_t out_cap, int64_t* out_offsets, int64_t* first_bad, int64_t* n_out,
                          int64_t* unknown_pos, int32_t* unknown_code_point) {
  if (!e || !n_out || !out_offsets) return fail(e, BPE_E_INVALID, "bad encode arguments");
  if (n_docs < 0 || (!doc_byte_offsets && n_docs > 0)) return fail(e, BPE_E_INVALID, "bad document offsets");
  if (unknown_pos) *unknown_pos = -1;
  if (!utf8 && n_docs > 0 && doc_byte_offsets[n_docs] > doc_byte_offsets[0]) return fail(e, BPE_E_INVALID, "null text");
  if (is_group(e))
    return group_encode(e, true, nullptr, utf8, doc_byte_offsets, n_docs, to_vector_index, n_tvi, out, out_cap, out_offsets, first_bad, n_out, unknown_pos,
                        unknown_code_point);
  CK(cudaSetDevice(e->device));
  return encode_host(e, true, nullptr, utf8, doc_byte_offsets, n_docs, to_vector_index, n_tvi, out, out_cap, out_offsets, first_bad, n_out, unknown_pos,
                     unknown_code_point);
}

int bpe_encode_text_batch_dev(bpe_engine* e, const uint8_t* dev_utf8, int64_t n_bytes, const int64_t* dev_doc_byte_offsets, int64_t n_docs,
                              const int32_t* dev_to_vector_index, int32_t n_tvi, int32_t* dev_out, int64_t* dev_out_offsets, int64_t* dev_first_bad,
                              int64_t* n_out, int64_t* unknown_pos, int32_t* unknown_code_point) {
  if (!e || !n_out || n_docs < 0 || n_bytes < 0 || !dev_doc_byte_offsets || !dev_out_offsets || (n_bytes > 0 && (!dev_utf8 || !dev_out)) ||
      (dev_to_vector_index && n_tvi < 0))
    return fail(e, BPE_E_INVALID, "bad encode arguments");
  *n_out = 0;
  if (unknown_pos) *unknown_pos = -1;
  GROUP_REFUSES(e, "bpe_encode_text_batch_dev (device pointers belong to one device)");
  CK(cudaSetDevice(e->device));
  e->txt_staged = false;  // x_ids is about to be reused
  TRY(ensure_cpmap(e));
  CK(e->x_flag.reserve(8));
  // the offsets live in the caller's device memory: check them there, before any kernel reads the text through them
  unsigned long long chk[3] = {0, 0, 0};
  CK(cudaMemsetAsync(e->x_flag.p + 6, 0, 8, e->stream));
  k_check_byte_offsets<<<(int)std::min<int64_t>((n_docs + 256) / 256, (int64_t)e->grid(4)), 256, 0, e->stream>>>(dev_doc_byte_offsets, n_docs, n_bytes,
                                                                                                                 e->x_flag.p + 4);
  CKL();
  CK(cudaMemcpyAsync(chk, e->x_flag.p + 4, sizeof chk, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  if (chk[2]) return fail(e, BPE_E_INVALID, "document offsets must be non-decreasing and lie inside the text (0 .. %lld)", (long long)n_bytes);
  const int64_t base = (int64_t)chk[0], nbytes = (int64_t)chk[1] - base;
  if ((uint64_t)nbytes >= 0xFFFFFFF0ull) return fail(e, BPE_E_DOMAIN, "text batch too large for one call");
  if (n_docs == 0) {
    CK(cudaMemsetAsync(dev_out_offsets, 0, 8, e->stream));
    return BPE_OK;
  }
  const int64_t* d_byte_off = dev_doc_byte_offsets;  // text_decode_dev wants offsets relative to the first document
  if (base) {
    CK(e->x_ooff.reserve((size_t)n_docs + 1));
    CK(cudaMemcpyAsync(e->x_ooff.p, dev_doc_byte_offsets, (size_t)(n_docs + 1) * 8, cudaMemcpyDeviceToDevice, e->stream));
    k_shift_i64<<<(int)std::min<int64_t>((n_docs + 256) / 256, (int64_t)e->grid(4)), 256, 0, e->stream>>>(e->x_ooff.p, n_docs + 1, -base);
    CKL();
    d_byte_off = e->x_ooff.p;
  }
  CK(e->x_ids.reserve((size_t)std::max<int64_t>(nbytes, 1)));  // at most one code point per byte
  CK(e->x_off.reserve((size_t)n_docs + 1));
  TRY(text_decode_dev(e, dev_utf8 + base, nbytes, d_byte_off, n_docs, e->x_ids.p, e->x_off.p, false, e->x_flag.p));
  // the lane width of encode_dev depends on the longest document, so the decode's flags come back before the encode starts
  unsigned long long fl[3];
  CK(cudaMemcpyAsync(fl, e->x_flag.p, sizeof fl, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  if (fl[0] != ~0ull) {  // encodeToCode throws at the first unknown character (core.ts:398-400)
    const int64_t pos = (int64_t)(fl[0] >> 32);
    if (unknown_pos) *unknown_pos = pos;
    if (unknown_code_point) *unknown_code_point = (int32_t)(fl[0] & 0xFFFFFFFFu);
    return fail(e, BPE_E_INVALID, "unknown token, char: U+%04X at code point %lld", (unsigned)(fl[0] & 0xFFFFFFFFu), (long long)pos);
  }
  return encode_dev(e, e->x_scratch, e->x_ids.p, e->x_off.p, n_docs, (int64_t)fl[2], (int64_t)fl[1], dev_to_vector_index, n_tvi, dev_out, dev_out_offsets,
                    dev_first_bad, n_out);
}

int bpe_pad_batch_dev(bpe_engine* e, const int32_t* dev_values, const int64_t* dev_offsets, int64_t n_docs, int64_t width, int32_t pad_value,
                      int32_t* dev_out, int64_t* dev_lengths) {
  if (!e || n_docs < 0 || width < 0 || (n_docs > 0 && (!dev_offsets || (width > 0 && (!dev_values || !dev_out)))))
    return fail(e, BPE_E_INVALID, "bad pad arguments");
  if (n_docs > 0 && width > INT64_MAX / n_docs) return fail(e, BPE_E_DOMAIN, "%lld rows of %lld values overflow", (long long)n_docs, (long long)width);
  GROUP_REFUSES(e, "bpe_pad_batch_dev (device pointers belong to one device)");
  CK(cudaSetDevice(e->device));
  if (n_docs == 0) return BPE_OK;
  k_pad_rows<<<(int)std::min<int64_t>((n_docs + 7) / 8, (int64_t)e->grid(16)), 256, 0, e->stream>>>(dev_values, dev_offsets, n_docs, width, pad_value, dev_out,
                                                                                                      dev_lengths);
  CKL();
  return BPE_OK;
}

int bpe_debug_lane_table(const int32_t* abc, int64_t n_merges, int32_t n_tokens, int32_t* a, int32_t* b, int32_t* rank, int32_t* c,
                         int32_t* right_spine_bound, int32_t* left_spine_bound, int64_t cap, int64_t* n) {
  if (n_merges < 0 || (n_merges > 0 && !abc) || !n) return BPE_E_INVALID;
  std::vector<int32_t> merges(abc, abc + 3 * n_merges);
  std::unordered_map<uint32_t, LaneEnt> M;
  std::vector<uint16_t> rule_c;
  TRY(build_lane_entries(nullptr, merges, n_tokens, M, rule_c));
  *n = (int64_t)M.size();
  if ((int64_t)M.size() > cap) return BPE_E_CAPACITY;
  int64_t i = 0;
  for (const auto& kv : M) {
    a[i] = (int32_t)(kv.first >> 16);
    b[i] = (int32_t)(kv.first & 0xFFFFu);
    rank[i] = kv.second.rk == 0xFFFF ? -1 : (int32_t)kv.second.rk;
    c[i] = kv.second.rk == 0xFFFF ? -1 : (int32_t)kv.second.c;
    right_spine_bound[i] = kv.second.rs == 0xFFFF ? -1 : (int32_t)kv.second.rs;
    left_spine_bound[i] = kv.second.ls == 0xFFFF ? -1 : (int32_t)kv.second.ls;
    i++;
  }
  return BPE_OK;
}

int bpe_debug_plan_chunks(const int64_t* doc_offsets, int64_t n_docs, int64_t chunk_units, int64_t* first_doc, int64_t cap, int64_t* n_chunks,
                          int64_t* bounds) {
  if (!doc_offsets || n_docs <= 0 || !n_chunks || !bounds) return BPE_E_INVALID;
  if (doc_offsets[n_docs] < doc_offsets[0]) return BPE_E_INVALID;
  const int64_t total = doc_offsets[n_docs] - doc_offsets[0];
  const PipePlan P = pipe_plan(total, n_docs, chunk_units);
  std::vector<int64_t> rel((size_t)n_docs + 2);
  PipeChunk prev, c;
  int64_t n = 0, reg = 0, oreg = 0;
  while (prev.d1 < n_docs) {
    reg = (prev.reg + (prev.in1 - prev.in0) + P.pad - 1) / P.pad * P.pad;
    oreg = prev.oreg + (prev.d1 - prev.d0) + (prev.d1 ? 1 : 0);
    TRY(next_chunk(nullptr, doc_offsets, n_docs, prev.d1, pipe_want(P, n, total - prev.in1), rel.data(), &c));
    c.reg = reg;
    c.oreg = oreg;
    if (first_doc && n < cap) first_doc[n] = c.d0;
    n++;
    prev = c;
  }
  *n_chunks = n;
  bounds[0] = P.max_chunks;
  bounds[1] = (int64_t)P.unit_cap;
  bounds[2] = prev.reg + (prev.in1 - prev.in0);       // units of the staging buffers the last chunk reaches
  bounds[3] = (int64_t)P.off_cap;
  bounds[4] = prev.oreg + (prev.d1 - prev.d0) + 1;    // offset entries the last chunk reaches
  return BPE_OK;
}

int bpe_restore_documents(bpe_engine* e, const int32_t* ids, const int64_t* doc_offsets, int64_t n_docs) {
  if (!e) return BPE_E_INVALID;
  if (is_group(e)) return group_add_documents(e, ids, doc_offsets, n_docs, true);
  TRY(check_offsets(e, doc_offsets, n_docs));
  if (n_docs == 0) return BPE_OK;
  CK(cudaSetDevice(e->device));
  int64_t total = 0, max_len = 0;
  TRY(stage_encode_inputs(e, ids, doc_offsets, n_docs, &total, &max_len));
  int64_t n_out = 0;
  TRY(encode_dev(e, e->x_scratch, e->x_ids.p, e->x_off.p, n_docs, total, max_len, nullptr, 0, e->x_out.p, e->x_ooff.p, nullptr, &n_out));
  std::vector<int64_t> ooff((size_t)n_docs + 1);
  CK(cudaMemcpyAsync(ooff.data(), e->x_ooff.p, (size_t)(n_docs + 1) * 8, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  return append_docs_dev(e, e->x_out.p, ooff.data(), n_docs);
}

}  // extern "C"
