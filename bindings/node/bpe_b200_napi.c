/*
 * bpe_b200_napi.c -- Node-API addon over the C ABI of include/bpe_b200.h.
 *
 * This is the binding a maintainer of beenotung/bpe-tokenizer adds so that `class BPETokenizer`
 * (reference core.ts:77-495) keeps its TypeScript surface while the corpus lives on a B200:
 * bindings/node/bpe_tokenizer.ts is the class, this file is the only native code it needs.
 *
 * STATUS: Node.js, node_api.h and tsc are absent from the authoring image, so this file has never been
 * loaded by Node.  It is compiled (syntax + types, -Wall -Werror) against the declarations in
 * tests/mock_node_api/node_api.h by tests/test_node_binding_sources.py, which also checks that every
 * bpe_* call matches include/bpe_b200.h.  The same ABI calls, in the same order, are exercised on the GPU by
 * the Python ctypes host (bpe_tokenizer_b200/tokenizer.py).
 *
 * Build (on a machine with Node >= 18 headers):
 *   cc -O2 -shared -fPIC -I$(node -p "process.execPath+'/../../include/node'") -I../../include \
 *      bpe_b200_napi.c -L../../bpe_tokenizer_b200 -lbpe_b200 -Wl,-rpath,'$ORIGIN' -o bpe_b200.node
 *
 * Conventions: every exported function is synchronous (the reference's methods are, core.ts has no Promise);
 * the first argument is the engine (a napi external created by `create`); bulk data crosses as typed arrays
 * without copies (Int32Array ids / values, BigInt64Array offsets, Uint8Array text); failures throw
 * `Error(bpe_last_error())` with `.code` = the BPE_E_* name, except data errors whose message the reference
 * fixes -- those are returned as values so that the TypeScript class throws the reference's exact text.
 */
#include <node_api.h>
#include <stddef.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "bpe_b200.h"

#define MAX_ARGS 10

typedef struct {
  napi_env env;
  size_t argc;
  napi_value argv[MAX_ARGS];
  bpe_engine* e;
  int ok;
} call_t;

static const char* code_name(int rc) {
  switch (rc) {
    case BPE_E_INVALID: return "BPE_E_INVALID";
    case BPE_E_CUDA: return "BPE_E_CUDA";
    case BPE_E_CAPACITY: return "BPE_E_CAPACITY";
    case BPE_E_DOMAIN: return "BPE_E_DOMAIN";
    case BPE_E_NOMEM: return "BPE_E_NOMEM";
    case BPE_E_INTERNAL: return "BPE_E_INTERNAL";
    default: return "BPE_E_UNKNOWN";
  }
}

static napi_value throw_rc(napi_env env, bpe_engine* e, int rc) {
  napi_throw_error(env, code_name(rc), e ? bpe_last_error(e) : "no CUDA device (there is no CPU fallback)");
  return NULL;
}

static napi_value throw_type(napi_env env, const char* what) {
  napi_throw_type_error(env, "ERR_INVALID_ARG_TYPE", what);
  return NULL;
}

/* argument 0 is always the engine */
static call_t begin(napi_env env, napi_callback_info info, size_t want) {
  call_t c;
  memset(&c, 0, sizeof c);
  c.env = env;
  c.argc = MAX_ARGS;
  void* p = NULL;
  if (napi_get_cb_info(env, info, &c.argc, c.argv, NULL, NULL) != napi_ok || c.argc < want ||
      napi_get_value_external(env, c.argv[0], &p) != napi_ok || !p) {
    throw_type(env, "expected (engine, ...)");
    return c;
  }
  c.e = (bpe_engine*)p;
  c.ok = 1;
  return c;
}

/* typed-array views; `null` / `undefined` give a NULL pointer of length 0 */
static int view(call_t* c, size_t i, napi_typedarray_type want, void** data, size_t* len) {
  *data = NULL;
  *len = 0;
  napi_valuetype vt;
  if (i >= c->argc || napi_typeof(c->env, c->argv[i], &vt) != napi_ok) return 0;
  if (vt == napi_null || vt == napi_undefined) return 1;
  napi_typedarray_type t;
  if (napi_get_typedarray_info(c->env, c->argv[i], &t, len, data, NULL, NULL) != napi_ok || t != want) {
    throw_type(c->env, "typed array of the wrong element type");
    return 0;
  }
  return 1;
}
static int arg_i64(call_t* c, size_t i, int64_t* v) {
  double d;
  if (i >= c->argc || napi_get_value_double(c->env, c->argv[i], &d) != napi_ok) {
    throw_type(c->env, "expected a number");
    return 0;
  }
  *v = (int64_t)d; /* JS numbers on this path are exact integers < 2^53 (SURVEY.md section 8) */
  return 1;
}
static int arg_i32(call_t* c, size_t i, int32_t* v) {
  int64_t w;
  if (!arg_i64(c, i, &w)) return 0;
  *v = (int32_t)w;
  return 1;
}
static int arg_bool(call_t* c, size_t i) {
  bool b = false;
  if (i < c->argc) napi_get_value_bool(c->env, c->argv[i], &b);
  return b ? 1 : 0;
}

static napi_value num(napi_env env, int64_t v) {
  napi_value r;
  napi_create_double(env, (double)v, &r);
  return r;
}
static napi_value undefined(napi_env env) {
  napi_value r;
  napi_get_undefined(env, &r);
  return r;
}
static void set_num(napi_env env, napi_value obj, const char* key, int64_t v) { napi_set_named_property(env, obj, key, num(env, v)); }

/* ---- lifetime: `new BPETokenizer()` core.ts:77 ------------------------------------------------------------------ */
static void finalize_engine(napi_env env, void* data, void* hint) {
  (void)env;
  (void)hint;
  bpe_destroy((bpe_engine*)data);
}

static napi_value Create(napi_env env, napi_callback_info info) { /* create(device = 0) -> engine */
  size_t argc = 1;
  napi_value argv[1], out;
  int32_t device = 0;
  if (napi_get_cb_info(env, info, &argc, argv, NULL, NULL) == napi_ok && argc >= 1) napi_get_value_int32(env, argv[0], &device);
  bpe_engine* e = NULL;
  int rc = bpe_create(device, &e);
  if (rc != BPE_OK) return throw_rc(env, NULL, rc);
  if (napi_create_external(env, e, finalize_engine, NULL, &out) != napi_ok) {
    bpe_destroy(e);
    return NULL;
  }
  return out;
}

static napi_value CreateGroup(napi_env env, napi_callback_info info) { /* createGroup(Int32Array devices) -> engine over those GPUs */
  size_t argc = 1;
  napi_value argv[1], out;
  napi_typedarray_type t;
  size_t n = 0;
  void* p = NULL;
  if (napi_get_cb_info(env, info, &argc, argv, NULL, NULL) != napi_ok || argc < 1 ||
      napi_get_typedarray_info(env, argv[0], &t, &n, &p, NULL, NULL) != napi_ok || t != napi_int32_array)
    return throw_type(env, "expected (Int32Array devices)");
  bpe_engine* e = NULL;
  int rc = bpe_create_group((const int*)p, (int)n, &e);
  if (rc == BPE_E_INVALID) {
    char msg[64];
    snprintf(msg, sizeof msg, "devices must list 1 to %d distinct GPUs", BPE_MG_MAX_WORLD);
    napi_throw_error(env, code_name(rc), msg);
    return NULL;
  }
  if (rc != BPE_OK) return throw_rc(env, NULL, rc);
  if (napi_create_external(env, e, finalize_engine, NULL, &out) != napi_ok) {
    bpe_destroy(e);
    return NULL;
  }
  return out;
}

/* ---- vocabulary ----------------------------------------------------------------------------------------------------- */
static napi_value SetTokens(napi_env env, napi_callback_info info) { /* (e, Int32Array utf16_len) */
  call_t c = begin(env, info, 2);
  void* p;
  size_t n;
  if (!c.ok || !view(&c, 1, napi_int32_array, &p, &n)) return NULL;
  int rc = bpe_set_tokens(c.e, (const int32_t*)p, (int32_t)n);
  return rc == BPE_OK ? undefined(env) : throw_rc(env, c.e, rc);
}

static napi_value NumTokens(napi_env env, napi_callback_info info) { /* (e) -> number */
  call_t c = begin(env, info, 1);
  if (!c.ok) return NULL;
  int32_t n = 0;
  int rc = bpe_num_tokens(c.e, &n);
  return rc == BPE_OK ? num(env, n) : throw_rc(env, c.e, rc);
}

static napi_value LoadMerges(napi_env env, napi_callback_info info) { /* (e, Int32Array abc) : fromJSON, core.ts:163-169 */
  call_t c = begin(env, info, 2);
  void* p;
  size_t n;
  if (!c.ok || !view(&c, 1, napi_int32_array, &p, &n)) return NULL;
  int rc = bpe_load_merges(c.e, (const int32_t*)p, (int64_t)(n / 3));
  return rc == BPE_OK ? undefined(env) : throw_rc(env, c.e, rc);
}

static napi_value SetChars(napi_env env, napi_callback_info info) { /* (e, Int32Array code_points, Int32Array indices) */
  call_t c = begin(env, info, 3);
  void *cp, *ix;
  size_t n, m;
  if (!c.ok || !view(&c, 1, napi_int32_array, &cp, &n) || !view(&c, 2, napi_int32_array, &ix, &m)) return NULL;
  if (n != m) return throw_type(env, "code_points and indices differ in length");
  int rc = bpe_set_chars(c.e, (const int32_t*)cp, (const int32_t*)ix, (int32_t)n);
  return rc == BPE_OK ? undefined(env) : throw_rc(env, c.e, rc);
}

/* ---- corpus: addToCorpus core.ts:182-207, restoreToCorpus :213-216, corpus_in_code :106 --------------------------- */
static napi_value docs_call(napi_env env, napi_callback_info info, int restore) { /* (e, Int32Array ids, BigInt64Array offsets) */
  call_t c = begin(env, info, 3);
  void *ids, *off;
  size_t n_ids, n_off;
  if (!c.ok || !view(&c, 1, napi_int32_array, &ids, &n_ids) || !view(&c, 2, napi_bigint64_array, &off, &n_off)) return NULL;
  if (n_off == 0) return throw_type(env, "offsets need n_docs + 1 entries");
  int rc = restore ? bpe_restore_documents(c.e, (const int32_t*)ids, (const int64_t*)off, (int64_t)n_off - 1)
                   : bpe_add_documents(c.e, (const int32_t*)ids, (const int64_t*)off, (int64_t)n_off - 1);
  return rc == BPE_OK ? undefined(env) : throw_rc(env, c.e, rc);
}
static napi_value AddDocuments(napi_env env, napi_callback_info info) { return docs_call(env, info, 0); }
static napi_value RestoreDocuments(napi_env env, napi_callback_info info) { return docs_call(env, info, 1); }

/* (e, Uint8Array utf8, BigInt64Array byte_offsets, Int32Array new_code_points, BigInt64Array counts) -> n_new
 * (a value above new_code_points.length asks the caller to retry with more room) */
static napi_value AddText(napi_env env, napi_callback_info info) {
  call_t c = begin(env, info, 5);
  void *txt, *off, *ncp, *cnt;
  size_t n_txt, n_off, n_ncp, n_cnt;
  if (!c.ok || !view(&c, 1, napi_uint8_array, &txt, &n_txt) || !view(&c, 2, napi_bigint64_array, &off, &n_off) ||
      !view(&c, 3, napi_int32_array, &ncp, &n_ncp) || !view(&c, 4, napi_bigint64_array, &cnt, &n_cnt))
    return NULL;
  if (n_off == 0) return throw_type(env, "offsets need n_docs + 1 entries");
  int32_t n_new = 0;
  int rc = bpe_add_text(c.e, (const uint8_t*)txt, (const int64_t*)off, (int64_t)n_off - 1, (int32_t*)ncp, (int32_t)n_ncp, &n_new, (int64_t*)cnt,
                        (int64_t)n_cnt);
  if (rc != BPE_OK && rc != BPE_E_CAPACITY) return throw_rc(env, c.e, rc);
  return num(env, n_new);
}

static napi_value ClearCorpus(napi_env env, napi_callback_info info) { /* (e) : `corpus_in_code = []`, fromJSON */
  call_t c = begin(env, info, 1);
  if (!c.ok) return NULL;
  int rc = bpe_clear_corpus(c.e);
  return rc == BPE_OK ? undefined(env) : throw_rc(env, c.e, rc);
}

static napi_value CorpusSize(napi_env env, napi_callback_info info) { /* (e) -> {docs, tokens} */
  call_t c = begin(env, info, 1);
  if (!c.ok) return NULL;
  int64_t nd = 0, nt = 0;
  int rc = bpe_corpus_size(c.e, &nd, &nt);
  if (rc != BPE_OK) return throw_rc(env, c.e, rc);
  napi_value o;
  napi_create_object(env, &o);
  set_num(env, o, "docs", nd);
  set_num(env, o, "tokens", nt);
  return o;
}

/* (e, doc_begin, doc_end, Int32Array out, BigInt64Array out_offsets) -> n_out */
static napi_value GetCorpus(napi_env env, napi_callback_info info) {
  call_t c = begin(env, info, 5);
  int64_t d0, d1;
  void *out, *off;
  size_t n_out, n_off;
  if (!c.ok || !arg_i64(&c, 1, &d0) || !arg_i64(&c, 2, &d1) || !view(&c, 3, napi_int32_array, &out, &n_out) ||
      !view(&c, 4, napi_bigint64_array, &off, &n_off))
    return NULL;
  if ((int64_t)n_off < d1 - d0 + 1) return throw_type(env, "out_offsets too short");
  int64_t n = 0;
  int rc = bpe_get_corpus(c.e, d0, d1, (int32_t*)out, (int64_t)n_out, (int64_t*)off, &n);
  if (rc != BPE_OK && rc != BPE_E_CAPACITY) return throw_rc(env, c.e, rc);
  return num(env, n); /* > out.length: retry with that much room */
}

/* ---- training ----------------------------------------------------------------------------------------------------- */
/* (e, min_weight, max_length) -> null | {a, b, c, weight} : findNextMerge core.ts:247-326 */
static napi_value FindNextMerge(napi_env env, napi_callback_info info) {
  call_t c = begin(env, info, 3);
  int64_t min_weight;
  int32_t max_length;
  if (!c.ok || !arg_i64(&c, 1, &min_weight) || !arg_i32(&c, 2, &max_length)) return NULL;
  bpe_merge m;
  int found = 0;
  int rc = bpe_find_next_merge(c.e, min_weight, max_length, &m, &found);
  if (rc != BPE_OK) return throw_rc(env, c.e, rc);
  napi_value o;
  if (!found) {
    napi_get_null(env, &o);
    return o;
  }
  napi_create_object(env, &o);
  set_num(env, o, "a", m.a);
  set_num(env, o, "b", m.b);
  set_num(env, o, "c", m.c);
  set_num(env, o, "weight", m.weight);
  return o;
}

/* (e, a, b, c) -> replacements : the corpus part of applyMerge core.ts:350-359 (also restoreMerge :477-494) */
static napi_value ApplyMerge(napi_env env, napi_callback_info info) {
  call_t c = begin(env, info, 4);
  int32_t a, b, t;
  if (!c.ok || !arg_i32(&c, 1, &a) || !arg_i32(&c, 2, &b) || !arg_i32(&c, 3, &t)) return NULL;
  int64_t n = 0;
  int rc = bpe_apply_merge(c.e, a, b, t, &n);
  return rc == BPE_OK ? num(env, n) : throw_rc(env, c.e, rc);
}

/* (e, Int32Array ab [2 per merge]) : a whole merge log in one call (example/import-merge-log-to-ram.ts:24-31) */
static napi_value ApplyMerges(napi_env env, napi_callback_info info) {
  call_t c = begin(env, info, 2);
  void* ab;
  size_t n;
  if (!c.ok || !view(&c, 1, napi_int32_array, &ab, &n)) return NULL;
  int rc = bpe_apply_merges(c.e, (const int32_t*)ab, (int64_t)(n / 2), NULL);
  return rc == BPE_OK ? undefined(env) : throw_rc(env, c.e, rc);
}

/* (e, min_weight, max_length, max_iterations, Int32Array abc [3 per merge], Float64Array weights) -> n_done
 * mergeUntil core.ts:365-383 as ONE device-resident loop; the class replays abc/weights into token_table. */
static napi_value MergeUntil(napi_env env, napi_callback_info info) {
  call_t c = begin(env, info, 6);
  int64_t min_weight, max_iterations;
  int32_t max_length;
  void *abc, *w;
  size_t n_abc, n_w;
  if (!c.ok || !arg_i64(&c, 1, &min_weight) || !arg_i32(&c, 2, &max_length) || !arg_i64(&c, 3, &max_iterations) ||
      !view(&c, 4, napi_int32_array, &abc, &n_abc) || !view(&c, 5, napi_float64_array, &w, &n_w))
    return NULL;
  size_t cap = n_abc / 3 < n_w ? n_abc / 3 : n_w;
  /* the ABI logs bpe_merge records; they are unpacked into the two typed arrays in chunks */
  enum { CHUNK = 4096 };
  bpe_merge log[CHUNK];
  size_t done = 0;
  int rc = BPE_OK;
  while (done < cap) {
    int64_t room = (int64_t)(cap - done < CHUNK ? cap - done : CHUNK), n = 0;
    int64_t left = max_iterations > 0 ? max_iterations - (int64_t)done : 0;
    if (max_iterations > 0 && left <= 0) break;
    rc = bpe_merge_until(c.e, min_weight, max_length, max_iterations > 0 ? (left < room ? left : room) : room, log, room, &n);
    for (int64_t i = 0; i < n; i++) {
      ((int32_t*)abc)[3 * (done + (size_t)i) + 0] = log[i].a;
      ((int32_t*)abc)[3 * (done + (size_t)i) + 1] = log[i].b;
      ((int32_t*)abc)[3 * (done + (size_t)i) + 2] = log[i].c;
      ((double*)w)[done + (size_t)i] = (double)log[i].weight;
    }
    done += (size_t)n;
    if (rc != BPE_OK || n < room) break; /* no further pair reaches min_weight (core.ts:377-379), or an error */
  }
  if (rc != BPE_OK) return throw_rc(env, c.e, rc); /* the merges already applied stay applied: call numTokens() to resync */
  return num(env, (int64_t)done);
}

/* ---- encode / decode: core.ts:392-445, :447-471 ---------------------------------------------------------------------- */
/* (e, Int32Array ids | Uint8Array utf8, BigInt64Array offsets, Int32Array|null to_vector_index, Int32Array out,
 *  BigInt64Array out_offsets, BigInt64Array|null first_bad, is_text)
 *  -> {n, unknown_pos, unknown_code_point}   (n > out.length: retry with that much room; unknown_pos >= 0: the class throws
 *  `unknown token, char: ...` core.ts:399) */
static napi_value EncodeBatch(napi_env env, napi_callback_info info) {
  call_t c = begin(env, info, 8);
  if (!c.ok) return NULL;
  int is_text = arg_bool(&c, 7);
  void *in, *off, *tvi, *out, *ooff, *bad;
  size_t n_in, n_off, n_tvi, n_out, n_ooff, n_bad;
  if (!view(&c, 1, is_text ? napi_uint8_array : napi_int32_array, &in, &n_in) || !view(&c, 2, napi_bigint64_array, &off, &n_off) ||
      !view(&c, 3, napi_int32_array, &tvi, &n_tvi) || !view(&c, 4, napi_int32_array, &out, &n_out) ||
      !view(&c, 5, napi_bigint64_array, &ooff, &n_ooff) || !view(&c, 6, napi_bigint64_array, &bad, &n_bad))
    return NULL;
  if (n_off == 0 || n_ooff < n_off || (bad && n_bad + 1 < n_off)) return throw_type(env, "offset arrays need n_docs + 1 entries");
  int64_t n = 0, upos = -1;
  int32_t ucp = 0;
  int rc = is_text ? bpe_encode_text_batch(c.e, (const uint8_t*)in, (const int64_t*)off, (int64_t)n_off - 1, (const int32_t*)tvi, (int32_t)n_tvi,
                                           (int32_t*)out, (int64_t)n_out, (int64_t*)ooff, (int64_t*)bad, &n, &upos, &ucp)
                   : bpe_encode_batch(c.e, (const int32_t*)in, (const int64_t*)off, (int64_t)n_off - 1, (const int32_t*)tvi, (int32_t)n_tvi,
                                      (int32_t*)out, (int64_t)n_out, (int64_t*)ooff, (int64_t*)bad, &n);
  if (rc != BPE_OK && rc != BPE_E_CAPACITY && !(rc == BPE_E_INVALID && upos >= 0)) return throw_rc(env, c.e, rc);
  napi_value o;
  napi_create_object(env, &o);
  set_num(env, o, "n", n);
  set_num(env, o, "unknown_pos", upos);
  set_num(env, o, "unknown_code_point", ucp);
  return o;
}

/* (e, Int32Array values, BigInt64Array offsets, Int32Array|null from_vector_index, Uint8Array token_bytes,
 *  BigInt64Array token_byte_offsets, Uint8Array out, BigInt64Array out_offsets, BigInt64Array|null first_bad) -> n_bytes */
static napi_value DecodeBatch(napi_env env, napi_callback_info info) {
  call_t c = begin(env, info, 8);
  void *val, *off, *fvi, *tb, *tbo, *out, *ooff, *bad = NULL;
  size_t n_val, n_off, n_fvi, n_tb, n_tbo, n_out, n_ooff, n_bad = 0;
  if (!c.ok || !view(&c, 1, napi_int32_array, &val, &n_val) || !view(&c, 2, napi_bigint64_array, &off, &n_off) ||
      !view(&c, 3, napi_int32_array, &fvi, &n_fvi) || !view(&c, 4, napi_uint8_array, &tb, &n_tb) ||
      !view(&c, 5, napi_bigint64_array, &tbo, &n_tbo) || !view(&c, 6, napi_uint8_array, &out, &n_out) ||
      !view(&c, 7, napi_bigint64_array, &ooff, &n_ooff))
    return NULL;
  if (c.argc > 8 && !view(&c, 8, napi_bigint64_array, &bad, &n_bad)) return NULL;
  if (n_off == 0 || n_tbo == 0 || n_ooff < n_off || (bad && n_bad + 1 < n_off)) return throw_type(env, "offset arrays need n + 1 entries");
  int64_t n = 0;
  int rc = bpe_decode_batch(c.e, (const int32_t*)val, (const int64_t*)off, (int64_t)n_off - 1, (const int32_t*)fvi, (int32_t)n_fvi,
                            (const uint8_t*)tb, (const int64_t*)tbo, (int32_t)(n_tbo - 1), (uint8_t*)out, (int64_t)n_out, (int64_t*)ooff,
                            (int64_t*)bad, &n);
  if (rc != BPE_OK && rc != BPE_E_CAPACITY) return throw_rc(env, c.e, rc);
  return num(env, n);
}

/* ---- module ---------------------------------------------------------------------------------------------------------- */
static napi_value Init(napi_env env, napi_value exports) {
  static const struct {
    const char* name;
    napi_callback fn;
  } table[] = {
      {"create", Create},           {"createGroup", CreateGroup},   {"setTokens", SetTokens},       {"numTokens", NumTokens},       {"loadMerges", LoadMerges},
      {"setChars", SetChars},       {"addDocuments", AddDocuments}, {"restoreDocuments", RestoreDocuments},
      {"addText", AddText},         {"clearCorpus", ClearCorpus},   {"corpusSize", CorpusSize},     {"getCorpus", GetCorpus},
      {"findNextMerge", FindNextMerge}, {"applyMerge", ApplyMerge}, {"applyMerges", ApplyMerges},   {"mergeUntil", MergeUntil},
      {"encodeBatch", EncodeBatch}, {"decodeBatch", DecodeBatch},
  };
  for (size_t i = 0; i < sizeof table / sizeof table[0]; i++) {
    napi_value fn;
    if (napi_create_function(env, table[i].name, NAPI_AUTO_LENGTH, table[i].fn, NULL, &fn) != napi_ok) return NULL;
    napi_set_named_property(env, exports, table[i].name, fn);
  }
  napi_value v;
  napi_create_int32(env, BPE_MAX_TOKENS, &v);
  napi_set_named_property(env, exports, "MAX_TOKENS", v);
  napi_create_int32(env, bpe_abi_version(), &v);
  napi_set_named_property(env, exports, "ABI_VERSION", v);
  return exports;
}

NAPI_MODULE(NODE_GYP_MODULE_NAME, Init)
