/*
 * bpe_b200.h -- C ABI of the B200-native BPE engine (libbpe_b200.so).
 *
 * This is the drop-in boundary for the hot path of beenotung/bpe-tokenizer's in-memory
 * `class BPETokenizer` (reference core.ts:77-495).  The reference has no FFI of its own
 * (it is pure TypeScript); a Node-API addon, the Python ctypes host in
 * bpe_tokenizer_b200/tokenizer.py, or any other host binds exactly these entry points and keeps
 * the dictionary / Token / JSON work on its side (INTEGRATION.md shows the N-API stub).
 *
 * Vocabulary (the reference's):
 *   token index  = position in `token_table` (core.ts:85); the reference's `code` is
 *                  String.fromCodePoint(index + 1) (core.ts:149,189) -- the ABI passes indices.
 *   document     = one `addToCorpus` call = one merge-isolation unit (core.ts:206, :265-267).
 *   merge        = (a, b) -> c with weight = counted occurrences (core.ts:315-325).
 *
 * Conventions:
 *   - Every function returns BPE_OK (0) or a negative BPE_E_* code; none throws or aborts.
 *     bpe_last_error() gives the text for the last failure on that engine.
 *   - The caller owns all buffers.  Host-pointer entry points copy during the call and retain
 *     nothing.  `_dev` entry points take CUDA device pointers valid on the engine's device and
 *     are ordered on the engine's stream (bpe_set_stream).
 *   - Output buffers carry an explicit capacity; when it is too small the call returns
 *     BPE_E_CAPACITY and stores the required size in the corresponding count output.
 *   - One engine per tokenizer instance; an engine is not thread-safe (like a JS object).
 *   - There is no CPU fallback: without a usable CUDA device bpe_create fails with BPE_E_CUDA.
 *   - Valid domain: token indices < BPE_MAX_TOKENS (the reference's codes stop being single
 *     UTF-16 units past 0xDBFF, SURVEY.md Appendix B); a corpus of < 2^32 - 2 positions per engine.
 */
#ifndef BPE_B200_H_
#define BPE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BPE_OK 0
#define BPE_E_INVALID -1   /* bad argument (null pointer, negative size, id out of range)      */
#define BPE_E_CUDA -2      /* CUDA runtime / kernel failure, text in bpe_last_error             */
#define BPE_E_CAPACITY -3  /* caller's output buffer too small; required size was stored        */
#define BPE_E_DOMAIN -4    /* token table would exceed BPE_MAX_TOKENS, or corpus too large      */
#define BPE_E_NOMEM -5     /* device or host allocation failed                                  */
#define BPE_E_INTERNAL -6  /* internal consistency check failed (a bug: please report)          */

#define BPE_MAX_TOKENS 56319 /* reference is well-defined only for token_table.length <= 56319 */

#define BPE_ABI_VERSION 2

typedef struct bpe_engine bpe_engine;

/* One learned merge, as findNextMerge returns it (core.ts:315-325): c = a + b, weight = count. */
typedef struct bpe_merge {
  int32_t a;
  int32_t b;
  int32_t c;
  int32_t reserved;
  int64_t weight;
} bpe_merge;

/* Cumulative device-time counters of the engine's kernels (CUDA events on the engine's stream). */
typedef struct bpe_stats {
  int64_t kernel_launches;     /* kernels of this library launched so far                         */
  int64_t merges_applied;      /* merges applied to the device corpus                             */
  int64_t index_builds;        /* full pair-index builds (K1)                                     */
  int64_t hot_rebuilds;        /* arg-max candidate-list rebuilds                                 */
  int64_t tie_breaks;          /* iterations that needed the last-position tie-break              */
  int64_t sites_merged;        /* pair occurrences rewritten                                      */
  int64_t corpus_positions;    /* slots of the device corpus (= characters ingested)              */
  int64_t corpus_tokens;       /* live tokens in the device corpus                                */
  int64_t distinct_pairs;      /* keys in the pair table                                          */
  int64_t pool_used;           /* occurrence-list cells in use                                    */
  double ms_index_build;       /* K1 histogram + occurrence lists                                 */
  double ms_argmax;            /* K2 (only when timing is enabled)                                */
  double ms_apply;             /* K3                                                              */
  double ms_encode;            /* K4 + K5, last bpe_encode_batch* call (summed over its chunks)   */
  double ms_last_merge_until;  /* device time of the last bpe_merge_until call                    */
  double ms_loop_phase[8];     /* the mergeUntil kernel as seen by block 0, cumulative since the last index build:
                                  decide, P1 sites, P1 barrier wait, P2, P2 barrier wait, (unused), (unused), tie path */
  /* bpe_merge_until commits several exact merges per pair of grid barriers (csrc/round_kernels.cuh); cumulative: */
  int64_t loop_rounds;         /* barrier rounds                                                  */
  int64_t loop_round_merges;   /* merges those rounds committed (/ loop_rounds = merges per round) */
  int64_t loop_round_tried;    /* merges whose site pass ran (committed + dropped by the born-pair bound) */
  int64_t loop_rounds_cut;     /* rounds that dropped a tail of their batch                       */
  int64_t encode_path;         /* kernel the last encode call ran: 2 lane rounds (csrc/encode_lanes.cuh), 3 per-document
                                  kernel only; 1 (a forward pass per document, since removed) is no longer produced */
} bpe_stats;

int bpe_abi_version(void);

/* ---- lifetime ---------------------------------------------------------------------------- */
/* Replaces `new BPETokenizer()` (core.ts:77) for the device-side state. */
int bpe_create(int device, bpe_engine** out);
void bpe_destroy(bpe_engine* e);
const char* bpe_last_error(bpe_engine* e);
/* Run the engine's kernels on `cuda_stream` (a cudaStream_t; NULL = the engine's own stream). */
int bpe_set_stream(bpe_engine* e, void* cuda_stream);
int bpe_synchronize(bpe_engine* e);
int bpe_get_stats(bpe_engine* e, bpe_stats* out);
/* Enable per-phase CUDA-event timing inside bpe_merge_until (adds host syncs; default off).  Bit 1 (debug): site discovery
 * scans every slot instead of the occurrence lists.  Other bits are ignored. */
int bpe_set_profiling(bpe_engine* e, int enabled);

/* ---- vocabulary --------------------------------------------------------------------------- */
/* UTF-16 length of every token's `chars` (core.ts:272 uses chars.length in the max_length test).
 * Replaces the device's view of token_table; must cover every index present in the corpus. */
int bpe_set_tokens(bpe_engine* e, const int32_t* utf16_len, int32_t n_tokens);
int bpe_num_tokens(bpe_engine* e, int32_t* n_tokens);
/* Merge list in training order, abc[3*i..] = (a, b, c) indices: what fromJSON rebuilds from
 * json.merge_codes (core.ts:163-169).  Used by encode / restore. */
int bpe_load_merges(bpe_engine* e, const int32_t* abc, int64_t n_merges);

/* ---- corpus (core.ts:106 corpus_in_code) -------------------------------------------------- */
/* addToCorpus (core.ts:182-207) for n_docs documents at once: ids = single-character token
 * indices (the char -> index dictionary stays on the host), doc_offsets[n_docs+1] delimit them.
 * Empty documents are kept (core.ts:206 pushes a sample even for ''). */
int bpe_add_documents(bpe_engine* e, const int32_t* ids, const int64_t* doc_offsets, int64_t n_docs);
int bpe_add_documents_dev(bpe_engine* e, const int32_t* dev_ids, const int64_t* host_doc_offsets, int64_t n_docs);
/* restoreToCorpus (core.ts:213-216): encodes the documents with the loaded merge list on the
 * device and appends the result; token weights are the host's business and stay untouched. */
int bpe_restore_documents(bpe_engine* e, const int32_t* ids, const int64_t* doc_offsets, int64_t n_docs);
/* `tokenizer.corpus_in_code = []` (example/import-merge-log-to-ram.ts:22) and fromJSON's reset. */
int bpe_clear_corpus(bpe_engine* e);
int bpe_corpus_size(bpe_engine* e, int64_t* n_docs, int64_t* n_tokens);
/* Getter for corpus_in_code: current token indices of documents [doc_begin, doc_end).
 * out_offsets[doc_end-doc_begin+1] are offsets into `out`. */
int bpe_get_corpus(bpe_engine* e, int64_t doc_begin, int64_t doc_end, int32_t* out, int64_t out_cap,
                   int64_t* out_offsets, int64_t* n_out);

/* ---- training ----------------------------------------------------------------------------- */
/* findNextMerge (core.ts:247-326).  min_weight <= 0 means the default 2 (core.ts:256, falsy),
 * max_length <= 0 means unlimited (core.ts:272).  *found = 0 stands for `null`.  Pure: does not
 * change the corpus.  out->c is the index the new token would get (= number of tokens). */
int bpe_find_next_merge(bpe_engine* e, int64_t min_weight, int32_t max_length, bpe_merge* out, int* found);
/* applyMerge's corpus part (core.ts:350-359): appends token c = n_tokens with
 * utf16_len[c] = utf16_len[a] + utf16_len[b], records the merge, rewrites every document
 * left to right, non-overlapping.  The weight bookkeeping of core.ts:345-346 stays on the host,
 * which is what makes restoreMerge (core.ts:477-494) the same call.  *n_replaced (optional)
 * receives the number of replacements performed. */
int bpe_apply_merge(bpe_engine* e, int32_t a, int32_t b, int32_t c, int64_t* n_replaced);
/* mergeUntil (core.ts:365-383), device-resident loop.  max_iterations <= 0 means unlimited.
 * log[0..*n_done) receives the merges in order; stops early (BPE_OK) when log_cap is reached. */
int bpe_merge_until(bpe_engine* e, int64_t min_weight, int32_t max_length, int64_t max_iterations,
                    bpe_merge* log, int64_t log_cap, int64_t* n_done);
/* Batched restoreMerge (core.ts:477-494): merge i rewrites (ab[2i], ab[2i+1]) -> token n_tokens + i, in order, inside
 * the device-resident loop (the reference's resume script replays its merge log one call per line,
 * example/import-merge-log-to-ram.ts:24-31).  A pair that does not occur still appends its token (core.ts:350-354).
 * n_replaced (optional, [n]) receives the replacements each merge performed.  Weights stay with the host. */
int bpe_apply_merges(bpe_engine* e, const int32_t* ab, int64_t n, int64_t* n_replaced);
/* Debug / parity: dump the pair histogram (pairs with count > 0, unspecified order). */
int bpe_pair_counts(bpe_engine* e, int32_t* a, int32_t* b, int64_t* count, int64_t cap, int64_t* n);

/* ---- sharded training: one engine (process) per GPU of an NVLink domain --------------------------
 * The reference has ONE corpus in one process (core.ts:106; findNextMerge counts over all documents,
 * core.ts:265-310, applyMerge rewrites all of them, core.ts:356-359) and no device boundary.  A sharded
 * deployment keeps that contract: rank r adds a contiguous range of the documents (ranks in document
 * order), pair counts are global, and bpe_merge_until returns the same merge log on every rank as a
 * single engine holding the whole corpus would (csrc/mg_kernels.cuh).  Call order on every rank:
 *   bpe_create -> bpe_mg_init -> (exchange the 64-byte handles, e.g. torch.distributed all_gather)
 *   -> bpe_mg_connect -> bpe_set_tokens / bpe_add_documents* (this rank's shard)
 *   -> bpe_mg_export_counts -> (all-gather the (pair,count) lists) -> bpe_mg_import_counts per peer
 *   -> bpe_merge_until (collective: all ranks, same arguments).
 * Single-step bpe_find_next_merge / bpe_apply_merge (on a non-empty corpus) / bpe_apply_merges return BPE_E_INVALID on
 * an engine initialised with world > 1: a shard alone cannot answer for the whole corpus; bpe_merge_until(max_iterations
 * = 1) is the exact single step. */
#define BPE_MG_MAX_WORLD 8
/* One engine over the GPUs devices[0..n) of this process: a corpus sharded by document, as bpe_mg_* does across processes.
 * n == 1 gives a plain engine.  Fails with BPE_E_INVALID on n < 1, n > BPE_MG_MAX_WORLD, or a repeated device;
 * with BPE_E_CUDA when a pair of the devices has no peer access.
 * The handle is an ordinary bpe_engine* that every entry point accepts.  It holds one member engine per device, member r on
 * devices[r] as rank r of n; their mailboxes are connected by pointer (peer access is enabled for every ordered pair, and stays
 * enabled after bpe_destroy).  A call that runs device work on several members runs each on a host thread of its own and joins
 * them all before it returns; when a member fails, the call returns the first member's error that is not a peer timeout, else the
 * timeout, and bpe_last_error names the device.
 *   - bpe_set_tokens, bpe_load_merges, bpe_set_chars, bpe_clear_corpus, bpe_set_profiling, bpe_synchronize: every member.
 *   - bpe_add_documents, bpe_restore_documents, bpe_add_text: the first upload after creation or bpe_clear_corpus is split into
 *     contiguous ranges of documents balanced by ids (bytes for text), one per member; a later upload goes to the last member
 *     whole, so that (member, position) stays the document order.  A document upload that any member refuses adds nothing on
 *     any member, as on one engine.  bpe_add_text gives the new characters one first-appearance order over the whole batch and
 *     returns the counts summed over the members; its checks all come before any member changes, so only a CUDA or memory
 *     failure in the final step can leave some members with the batch.
 *   - bpe_merge_until sums the members' pair histograms first when an upload made them stale (device to device, no host
 *     copy), then runs on every member; all of them return the same log (BPE_E_INTERNAL otherwise).  The members meet on the
 *     host before every launch of the loop kernel, so that none waits in a kernel for a peer still doing host work.
 *   - bpe_encode_batch, bpe_encode_text_batch, bpe_decode_batch: contiguous ranges of documents balanced by input units, one
 *     per member, encoded in parallel; the results are exactly one engine's, BPE_E_CAPACITY, the sizes and the positions in
 *     error messages included.  Encode copies each member's vectors from its device to their place in `out` once every
 *     member's size is known (that copy follows the encode instead of overlapping it); decode sizes first, then decodes into
 *     place (the values go up twice).
 *   - bpe_get_corpus, bpe_corpus_size, bpe_pair_counts: the whole corpus (members' ranges in order; corpus-wide counts).
 *   - bpe_get_stats: kernel_launches, sites_merged, corpus_positions, corpus_tokens and pool_used summed over the members;
 *     every other field (the times included) is member 0's.
 *   - BPE_E_INVALID, as on a sharded engine: bpe_find_next_merge, bpe_apply_merge and bpe_apply_merges on a non-empty corpus
 *     (on an empty one they grow the vocabulary of every member), bpe_set_stream, bpe_add_documents_dev,
 *     bpe_encode_batch_dev, bpe_encode_text_batch_dev, bpe_pad_batch_dev, bpe_add_text_stage / _commit and bpe_mg_*.
 * With BPE_GROUP_SHARE_DEVICE=1 in the environment, devices may repeat: the members on one device share its SMs.  It lets the
 * group run on a host with fewer GPUs than members (tests); it gives no speed-up. */
int bpe_create_group(const int* devices, int n, bpe_engine** out);
/* Allocates this rank's mailbox (peers store count deltas into it over NVLink) and writes its
 * cudaIpcMemHandle_t (64 bytes) to handle_out. */
int bpe_mg_init(bpe_engine* e, int rank, int world, void* handle_out);
/* handles: world x 64 bytes, ordered by rank (the entry of this rank is ignored). */
int bpe_mg_connect(bpe_engine* e, const char* handles);
/* *counts_global = 1 when the pair index holds counts summed over all ranks. */
int bpe_mg_state(bpe_engine* e, int* counts_global);
/* This shard's pair histogram as device arrays: dev_keys[i] = (a << 16) | b, dev_counts[i].
 * cap = 0 only reports an upper bound of the number of pairs in *n. */
int bpe_mg_export_counts(bpe_engine* e, uint32_t* dev_keys, uint32_t* dev_counts, int64_t cap, int64_t* n);
/* Adds a peer's histogram (device arrays) to this engine's counts; last != 0 on the final peer. */
int bpe_mg_import_counts(bpe_engine* e, const uint32_t* dev_keys, const uint32_t* dev_counts, int64_t n, int last);

/* ---- encode / decode ---------------------------------------------------------------------- */
/* encodeToCode + encodeToVector (core.ts:392-409, :424-445) for a batch of documents.
 *   ids/doc_offsets      single-character token indices per document (as bpe_add_documents)
 *   to_vector_index      n_tvi entries, -1 = hole (token has zero weight, core.ts:235,437-441);
 *                        NULL = emit raw token indices (encodeToTokens semantics, core.ts:411-422)
 *   out/out_cap          encoded values, documents back to back
 *   out_offsets          [n_docs+1] offsets into out
 *   first_bad            optional [n_docs]: -1, or the offset WITHIN the document's output of the
 *                        first token whose to_vector_index is a hole (the reference throws
 *                        `unknown token index: ${index}` there); out holds -(index+1) at holes.
 *   n_out                total values written (or required when BPE_E_CAPACITY; out_offsets and
 *                        first_bad are complete in that case as well)
 * The call is a three-stream pipeline over chunks of whole documents (copy in | encode | copy out;
 * BPE_ENC_CHUNK = input units per full-size chunk, default 128 Mi;
 * the first and last chunks are smaller): with page-locked `ids` / `out` buffers it costs
 * max(PCIe in, encode, PCIe out); pageable buffers are correct but their copies serialise.  The small
 * per-document arrays are staged through pinned memory of the engine either way. */
int bpe_encode_batch(bpe_engine* e, const int32_t* ids, const int64_t* doc_offsets, int64_t n_docs,
                     const int32_t* to_vector_index, int32_t n_tvi, int32_t* out, int64_t out_cap,
                     int64_t* out_offsets, int64_t* first_bad, int64_t* n_out);
/* Same with every buffer resident on the device (dev_doc_offsets int64[n_docs+1], max_doc_len = the
 * longest document).  dev_out must hold at least as many values as there are input ids;
 * dev_out_offsets int64[n_docs+1]; dev_first_bad may be NULL.  *n_out is read back (one sync). */
int bpe_encode_batch_dev(bpe_engine* e, const int32_t* dev_ids, const int64_t* dev_doc_offsets, int64_t n_docs,
                         int64_t n_ids, int64_t max_doc_len, const int32_t* dev_to_vector_index, int32_t n_tvi,
                         int32_t* dev_out, int64_t* dev_out_offsets, int64_t* dev_first_bad, int64_t* n_out);

/* decodeVector / decodeTokens (core.ts:447-471) for a batch of documents.
 *   values/doc_offsets          vector indices (from_vector_index != NULL) or raw token indices per document
 *   from_vector_index           n_fvi entries, -1 = hole: `unknown vector index: ${v}` (core.ts:466-468)
 *   token_bytes/token_byte_offsets  UTF-8 of every token's chars back to back, [n_tokens+1] offsets
 *   out/out_cap                 decoded UTF-8 bytes, documents back to back (unknown values contribute nothing)
 *   out_offsets                 [n_docs+1] byte offsets into out
 *   first_bad                   optional [n_docs]: -1, or the position within the document of the first unknown value
 *   n_out                       total bytes written (or required when BPE_E_CAPACITY) */
int bpe_decode_batch(bpe_engine* e, const int32_t* values, const int64_t* doc_offsets, int64_t n_docs,
                     const int32_t* from_vector_index, int32_t n_fvi, const uint8_t* token_bytes,
                     const int64_t* token_byte_offsets, int32_t n_tokens, uint8_t* out, int64_t out_cap,
                     int64_t* out_offsets, int64_t* first_bad, int64_t* n_out);

/* Debug / test: the pair table the encode kernel works from (csrc/encode_lanes.cuh), built from a merge list abc[3*i..] =
 * (a, b, c) without touching a device: for every pair that is a rule or lies on a spine of one, its rank and token (-1: no
 * rule) and the lowest rank of any rule that can consume its right / left half through a spine (-1: none).
 * *n = number of pairs (BPE_E_CAPACITY when cap is smaller); unspecified order. */
int bpe_debug_lane_table(const int32_t* abc, int64_t n_merges, int32_t n_tokens, int32_t* a, int32_t* b, int32_t* rank, int32_t* c,
                         int32_t* right_spine_bound, int32_t* left_spine_bound, int64_t cap, int64_t* n);
/* Debug / test: how the host-buffer encode calls above would cut a batch into chunks of whole documents
 * (chunk_units = full-size chunk; no device work, no engine).  first_doc[0..min(*n_chunks, cap)) receives the first
 * document of every chunk; bounds[5] = {chunk-count bound, unit capacity of the staging buffers, units reached by the
 * last chunk, offset-entry capacity, offset entries reached}: the reached values must not exceed the capacities. */
int bpe_debug_plan_chunks(const int64_t* doc_offsets, int64_t n_docs, int64_t chunk_units, int64_t* first_doc, int64_t cap,
                          int64_t* n_chunks, int64_t* bounds);

/* ---- text front end on the device (core.ts:185-205 ingest, :396-402 encode front end) --------------
 * Documents arrive as UTF-8 bytes (lone surrogates in their generalised 3-byte form); one token per CODE POINT, as
 * the reference's `for (let char of content)` yields them.  The engine keeps a code point -> token index table. */
/* Replaces the engine's character table (after fromJSON, or when the host created character tokens itself). */
int bpe_set_chars(bpe_engine* e, const int32_t* code_points, const int32_t* indices, int32_t n);
/* addToCorpus for a batch of documents given as text: unknown code points become tokens n_tokens, n_tokens+1, ...
 * in first-appearance order (core.ts:186-199); new_code_points[0..*n_new) lists them so the host can append the
 * same tokens.  counts[i] (optional, counts_cap >= the new token count) = occurrences of token i in this batch
 * (the `weight++ / original_weight++` of core.ts:201-202). */
int bpe_add_text(bpe_engine* e, const uint8_t* utf8, const int64_t* doc_byte_offsets, int64_t n_docs,
                 int32_t* new_code_points, int32_t new_cap, int32_t* n_new, int64_t* counts, int64_t counts_cap);
/* bpe_add_text in two steps, for a corpus sharded over engines whose ranks must agree on ONE first-appearance order
 * (bpe_add_text is exactly stage, then commit of the list stage reported).
 * Step 1 on one rank: decode the batch into the engine's staging buffers and report the code points the character
 * table does not know, each with its first position (code-point index within the batch), in first-appearance order.
 * Nothing is added to the corpus or the vocabulary yet.  BPE_E_CAPACITY stores the required new_cap in *n_new;
 * BPE_E_DOMAIN when the new characters alone would take the table past BPE_MAX_TOKENS. */
int bpe_add_text_stage(bpe_engine* e, const uint8_t* utf8, const int64_t* doc_byte_offsets, int64_t n_docs,
                       int32_t* new_code_points, int64_t* first_pos, int32_t new_cap, int32_t* n_new);
/* Step 2: code_points[i] becomes token n_tokens + i.  The list must hold every code point the staged batch reported and
 * may hold others (those only other ranks saw).  Appends the staged documents; counts as in bpe_add_text (this batch only,
 * counts_cap >= n_tokens + n).  Changes nothing and returns BPE_E_INVALID when no batch is staged, or when the list misses a
 * code point the batch reported, repeats one, or names one the table already knows; BPE_E_DOMAIN when n_tokens + n would
 * exceed BPE_MAX_TOKENS.  Every other call that reuses the staging buffers (encode, decode, restore, another stage) or
 * replaces the character table (bpe_set_chars) discards the staged batch. */
int bpe_add_text_commit(bpe_engine* e, const int32_t* code_points, int32_t n, int64_t* counts, int64_t counts_cap);
/* bpe_encode_batch with the char -> index step on the device.  An unknown character fails the call with
 * BPE_E_INVALID (the reference throws `unknown token, char: ...`, core.ts:398-400); *unknown_pos / *unknown_code_point
 * (optional) identify the first one (code-point index within the batch). */
int bpe_encode_text_batch(bpe_engine* e, const uint8_t* utf8, const int64_t* doc_byte_offsets, int64_t n_docs,
                          const int32_t* to_vector_index, int32_t n_tvi, int32_t* out, int64_t out_cap,
                          int64_t* out_offsets, int64_t* first_bad, int64_t* n_out, int64_t* unknown_pos,
                          int32_t* unknown_code_point);
/* bpe_encode_text_batch with every buffer on the engine's device, ordered on the engine's stream: text that is already on
 * the GPU (a dataloader's output, another kernel's result) is encoded without a trip through the host.
 *   dev_utf8[0..n_bytes)         the text; dev_doc_byte_offsets[n_docs+1] index into it.  They are checked on the device:
 *                                non-decreasing and inside [0, n_bytes].  Otherwise BPE_E_INVALID, and nothing is written.
 *                                offsets[0] need not be 0; bytes after offsets[n_docs] are not read.
 *   dev_to_vector_index / n_tvi  device, as bpe_encode_batch_dev (NULL: raw token indices)
 *   dev_out                      room for at least as many values as the batch has code points (n_bytes always suffices)
 *   dev_out_offsets[n_docs+1]    from 0; dev_first_bad[n_docs] optional, as bpe_encode_batch_dev
 *   n_out, unknown_pos, unknown_code_point   host, as bpe_encode_text_batch (same BPE_E_INVALID, same position)
 * A batch of 2^32 - 16 bytes or more: BPE_E_DOMAIN.  Discards a staged text batch, as every encode does.
 * Staging: the engine's grow-only buffers hold the decoded characters (4 B per byte of the batch) and the encode's scratch
 * (4 B per code point), as bpe_encode_text_batch's do.  The call waits for the stream a fixed number of times (offsets check,
 * decode flags, encode), whatever the batch size; when it returns BPE_OK, dev_out and dev_out_offsets are complete. */
int bpe_encode_text_batch_dev(bpe_engine* e, const uint8_t* dev_utf8, int64_t n_bytes, const int64_t* dev_doc_byte_offsets,
                              int64_t n_docs, const int32_t* dev_to_vector_index, int32_t n_tvi, int32_t* dev_out,
                              int64_t* dev_out_offsets, int64_t* dev_first_bad, int64_t* n_out, int64_t* unknown_pos,
                              int32_t* unknown_code_point);
/* Ragged -> dense on the device, ordered on the engine's stream (no wait).  Row d of dev_out[n_docs x width] holds the first
 * min(len_d, width) values of document d (dev_values[dev_offsets[d] .. dev_offsets[d+1])), then pad_value.
 * dev_lengths[d] (optional) = min(len_d, width).  Works on the output of either _dev encode; dev_offsets must be
 * non-decreasing and index dev_values (they are not checked). */
int bpe_pad_batch_dev(bpe_engine* e, const int32_t* dev_values, const int64_t* dev_offsets, int64_t n_docs, int64_t width,
                      int32_t pad_value, int32_t* dev_out, int64_t* dev_lengths);

/* ---- synthetic corpus (bench / tests; SURVEY.md section 8(d), spec in synth.py) ------------ */
/* Fills `text` (may be NULL to size) with documents until target_bytes is reached. */
int bpe_synth_corpus(int64_t target_bytes, uint64_t seed, int32_t vocab, uint64_t word_seed, uint8_t* text,
                     int64_t text_cap, int64_t* doc_offsets, int64_t offsets_cap, int64_t* n_bytes, int64_t* n_docs);

#ifdef __cplusplus
}
#endif
#endif /* BPE_B200_H_ */
