/**
 * bpe_tokenizer.ts -- the TypeScript host of the B200 engine: same exports and members as the reference's `core.ts`
 * (beenotung/bpe-tokenizer 2.2.0), so `import { BPETokenizer } from './bpe_tokenizer'` replaces
 * `import { BPETokenizer } from 'bpe-tokenizer'`.
 *
 * Division of labour (INTEGRATION.md): the dictionaries, `Token` objects, the JSON snapshot and every error message live
 * here; whatever walks the corpus -- pair counting, arg-max with the reference's tie-break, in-place merging, encoding --
 * is one call into `bpe_b200.node` (bindings/node/bpe_b200_napi.c) and from there into libbpe_b200.so.  There is no
 * JavaScript fallback: constructing a tokenizer without the addon and a CUDA device throws.
 *
 * STATUS: written against the C ABI and the addon's exports, NOT executed -- Node and tsc are absent from the authoring
 * image.  The executable twin of this file is bpe_tokenizer_b200/tokenizer.py (same structure, same ABI calls), which the
 * GPU parity tests drive; tests/test_node_binding_sources.py checks that this file covers the reference's public surface
 * and only calls functions the addon exports.
 *
 * Reference lines are cited as core.ts:N.
 */

// eslint-disable-next-line @typescript-eslint/no-var-requires
const native = require('./bpe_b200.node') as Native

type Engine = unknown
interface Native {
  MAX_TOKENS: number
  ABI_VERSION: number
  create(device?: number): Engine
  createGroup(devices: Int32Array): Engine
  setTokens(e: Engine, utf16_len: Int32Array): void
  numTokens(e: Engine): number
  loadMerges(e: Engine, abc: Int32Array): void
  setChars(e: Engine, code_points: Int32Array, indices: Int32Array): void
  addDocuments(e: Engine, ids: Int32Array, offsets: BigInt64Array): void
  restoreDocuments(e: Engine, ids: Int32Array, offsets: BigInt64Array): void
  addText(e: Engine, utf8: Uint8Array, offsets: BigInt64Array, new_code_points: Int32Array, counts: BigInt64Array): number
  clearCorpus(e: Engine): void
  corpusSize(e: Engine): { docs: number; tokens: number }
  getCorpus(e: Engine, doc_begin: number, doc_end: number, out: Int32Array, out_offsets: BigInt64Array): number
  findNextMerge(e: Engine, min_weight: number, max_length: number): null | { a: number; b: number; c: number; weight: number }
  applyMerge(e: Engine, a: number, b: number, c: number): number
  applyMerges(e: Engine, ab: Int32Array): void
  mergeUntil(e: Engine, min_weight: number, max_length: number, max_iterations: number, abc: Int32Array, weights: Float64Array): number
  encodeBatch(
    e: Engine, input: Int32Array | Uint8Array, offsets: BigInt64Array, to_vector_index: Int32Array | null, out: Int32Array,
    out_offsets: BigInt64Array, first_bad: BigInt64Array | null, is_text: boolean,
  ): { n: number; unknown_pos: number; unknown_code_point: number }
  decodeBatch(
    e: Engine, values: Int32Array, offsets: BigInt64Array, from_vector_index: Int32Array | null, token_bytes: Uint8Array,
    token_byte_offsets: BigInt64Array, out: Uint8Array, out_offsets: BigInt64Array, first_bad?: BigInt64Array | null,
  ): number
}

/** core.ts:1-10 */
export type Token = {
  chars: string
  weight: number
  original_weight: number
  code: string
  index: number
}
/** [a, b, c] core.ts:15 */
export type MergeToken = [a: Token, b: Token, c: Token]
/** [a_code, b_code, c_weight] core.ts:20 */
export type CompactMerge = [a_code: string, b_code: string, c_weight: number]
/** [from_code, to_code] core.ts:25 */
export type MergeCode = [from_code: string, to_code: string]
/** core.ts:28-33 */
export type BPETokenizerJSON = {
  version: 2
  char_count: number
  token_table: [chars: string, weight: number, original_weight: number][]
  merge_codes: [a_code: string, b_code: string, c_code: string][]
}

/** core.ts:36-45 */
export const FS = String.fromCharCode(28)
export const EOF = String.fromCharCode(4)
export const LF = '\n'
export const CR = '\r'

/** core.ts:55-58 */
export function fileContentToCorpus(content: Buffer | string): string {
  return FS + content.toString() + EOF
}
/** core.ts:61-64 (trims every line) */
export function linesToCorpus(text: string): string[] {
  return text.split('\n').map(line => CR + line.trim() + LF)
}
/** core.ts:67-75 (strips one trailing '\r' only) */
export function linesTrimmedToCorpus(text: string): string[] {
  return text.split('\n').map(line => CR + (line.endsWith('\r') ? line.slice(0, -1) : line) + LF)
}

/** core.ts:500-503 */
export function compactMerge(merge: MergeToken): CompactMerge {
  return [merge[0].code, merge[1].code, merge[2].weight]
}

export type MergeOptions = { min_weight?: number; max_length?: number }
export type MergeUntilOptions = MergeOptions & { max_iterations?: number }

const utf8 = new TextEncoder()

function offsetsOf(lengths: number[]): BigInt64Array {
  const off = new BigInt64Array(lengths.length + 1)
  let sum = 0
  lengths.forEach((n, i) => {
    sum += n
    off[i + 1] = BigInt(sum)
  })
  return off
}

export class BPETokenizer {
  /** core.ts:79 */ char_to_token: Record<string, Token> = {}
  /** core.ts:82 */ code_to_token: Record<string, Token> = {}
  /** core.ts:85 */ token_table: Token[] = []
  /** core.ts:88 */ merge_tokens: MergeToken[] = []
  /** core.ts:91 */ merge_codes: MergeCode[] = []
  /** core.ts:97 */ to_vector_index: number[] | null = null
  /** core.ts:103 */ from_vector_index: number[] | null = null

  private engine: Engine
  /** documents added on the host since the last device call: uploaded together (one bpe_add_documents) */
  private pending: Int32Array[] = []
  private tvi: Int32Array | null = null
  private chars_synced = -1

  /** `devices`: one engine over those GPUs of this process (bpe_create_group), the corpus sharded by document across them */
  constructor(options?: { device?: number; devices?: number[] }) {
    this.engine = options?.devices ? native.createGroup(Int32Array.from(options.devices)) : native.create(options?.device ?? 0)
  }

  // ---- plumbing ---------------------------------------------------------------------------------------------------
  private syncTokens(): void {
    if (native.numTokens(this.engine) !== this.token_table.length) {
      // `chars.length` is the UTF-16 length the max_length test uses (core.ts:272)
      native.setTokens(this.engine, Int32Array.from(this.token_table, t => t.chars.length))
    }
  }
  private flush(): void {
    this.syncTokens()
    if (this.pending.length === 0) return
    const docs = this.pending
    this.pending = []
    const off = offsetsOf(docs.map(d => d.length))
    const ids = new Int32Array(Number(off[docs.length]))
    docs.forEach((d, i) => ids.set(d, Number(off[i])))
    native.addDocuments(this.engine, ids, off)
  }
  private newToken(chars: string, weight: number): Token {
    const index = this.token_table.length
    if (index >= native.MAX_TOKENS) {
      // past this index `code` stops being one UTF-16 unit and the reference's own replaceAll goes wrong (SURVEY.md Appendix B)
      throw new RangeError(`token table exceeds ${native.MAX_TOKENS} entries`)
    }
    return { chars, weight, original_weight: weight, code: String.fromCodePoint(index + 1), index }
  }
  /** core.ts:185-204 / :396-402: one token per code point, created in first-appearance order when `create` */
  private charIds(content: string, create: boolean): Int32Array {
    const ids: number[] = []
    for (const char of content) {
      let token = this.char_to_token[char]
      if (!token) {
        if (!create) throw new Error('unknown token, char: ' + JSON.stringify(char)) // core.ts:399
        token = this.newToken(char, 1)
        this.char_to_token[char] = token
        this.code_to_token[token.code] = token
        this.token_table.push(token)
      } else if (create) {
        token.weight++
        token.original_weight++
      }
      ids.push(token.index)
    }
    return Int32Array.from(ids)
  }
  private invalidateVectorIndex(): void {
    // core.ts:173-176
    this.to_vector_index = null
    this.from_vector_index = null
    this.tvi = null
  }

  // ---- snapshot: core.ts:112-171 ------------------------------------------------------------------------------------
  toJSON(): BPETokenizerJSON {
    return {
      version: 2,
      char_count: Object.keys(this.char_to_token).length,
      token_table: this.token_table.map(t => [t.chars, t.weight, t.original_weight]),
      merge_codes: this.merge_tokens.map(([a, b, c]) => [a.code, b.code, c.code]),
    }
  }
  fromJSON(json: BPETokenizerJSON): void {
    if (!json || json.version !== 2 || !Array.isArray(json.token_table) || !Array.isArray(json.merge_codes)) {
      throw new Error('invalid format') // core.ts:136
    }
    // every field is replaced, the corpus included (core.ts:138-146)
    this.char_to_token = {}
    this.code_to_token = {}
    this.token_table = []
    this.merge_tokens = []
    this.merge_codes = []
    this.pending = []
    this.chars_synced = -1
    this.invalidateVectorIndex()
    native.clearCorpus(this.engine)
    for (const [chars, weight, original_weight] of json.token_table) {
      const token = this.newToken(chars, weight)
      token.original_weight = original_weight
      if (token.index < json.char_count) this.char_to_token[chars] = token
      this.code_to_token[token.code] = token
      this.token_table.push(token)
    }
    const abc = new Int32Array(json.merge_codes.length * 3)
    json.merge_codes.forEach(([a_code, b_code, c_code], i) => {
      const a = this.code_to_token[a_code]
      const b = this.code_to_token[b_code]
      const c = this.code_to_token[c_code]
      this.merge_tokens.push([a, b, c])
      this.merge_codes.push([a.code + b.code, c.code])
      abc.set([a.index, b.index, c.index], 3 * i)
    })
    native.setTokens(this.engine, Int32Array.from(this.token_table, t => t.chars.length))
    native.loadMerges(this.engine, abc)
    this.compactVectorIndex() // core.ts:170
  }

  // ---- corpus -----------------------------------------------------------------------------------------------------------
  /** core.ts:182-207 */
  addToCorpus(content: string): void {
    this.pending.push(this.charIds(content, true))
  }
  /** core.ts:213-216 */
  restoreToCorpus(content: string): void {
    const ids = this.charIds(content, false)
    this.flush()
    native.restoreDocuments(this.engine, ids, offsetsOf([ids.length]))
  }
  /** core.ts:106: materialised from the device on demand; assignable (example/import-merge-log-to-ram.ts:22) */
  get corpus_in_code(): string[] {
    this.flush()
    const { docs, tokens } = native.corpusSize(this.engine)
    const out = new Int32Array(Math.max(tokens, 1))
    const off = new BigInt64Array(docs + 1)
    native.getCorpus(this.engine, 0, docs, out, off)
    const result: string[] = []
    for (let d = 0; d < docs; d++) {
      let s = ''
      for (let i = Number(off[d]); i < Number(off[d + 1]); i++) s += String.fromCodePoint(out[i] + 1)
      result.push(s)
    }
    return result
  }
  set corpus_in_code(value: string[]) {
    this.pending = []
    native.clearCorpus(this.engine)
    this.syncTokens()
    if (value.length === 0) return
    const docs = value.map(s => Int32Array.from(Array.from(s), ch => ch.codePointAt(0)! - 1))
    const off = offsetsOf(docs.map(d => d.length))
    const ids = new Int32Array(Number(off[docs.length]))
    docs.forEach((d, i) => ids.set(d, Number(off[i])))
    native.addDocuments(this.engine, ids, off)
  }

  // ---- bulk text in: the code-point loop, first-appearance token creation and weights run on the device --------------------
  private syncChars(): void {
    const keys = Object.keys(this.char_to_token)
    if (this.chars_synced === keys.length) return
    const single = keys.filter(k => Array.from(k).length === 1) // multi-character keys can never match a character
    native.setChars(
      this.engine,
      Int32Array.from(single, k => k.codePointAt(0)!),
      Int32Array.from(single, k => this.char_to_token[k].index),
    )
    this.chars_synced = keys.length
  }
  /** `for (doc of docs) addToCorpus(doc)` (core.ts:182-207) in one device call */
  addTextBatch(docs: string[]): void {
    this.flush()
    this.syncChars()
    const parts = docs.map(d => utf8.encode(d))
    const off = offsetsOf(parts.map(p => p.length))
    const text = new Uint8Array(Math.max(Number(off[parts.length]), 1))
    parts.forEach((p, i) => text.set(p, Number(off[i])))
    const new_cps = new Int32Array(1 << 16)
    const counts = new BigInt64Array(this.token_table.length + (1 << 16))
    const n_new = native.addText(this.engine, text, off, new_cps, counts)
    for (let k = 0; k < n_new; k++) {
      // the same tokens the engine just appended (core.ts:188-199)
      const token = this.newToken(String.fromCodePoint(new_cps[k]), 0)
      this.char_to_token[token.chars] = token
      this.code_to_token[token.code] = token
      this.token_table.push(token)
    }
    this.chars_synced = Object.keys(this.char_to_token).length
    this.token_table.forEach((t, i) => {
      const n = Number(counts[i])
      t.weight += n
      t.original_weight += n
    })
    // like addToCorpus (core.ts:182-207), no vector-index invalidation: a stale index throws `unknown token index`
  }

  // ---- vector index: core.ts:222-241 ---------------------------------------------------------------------------------------
  compactVectorIndex(): void {
    if (this.token_table.length === 0) {
      throw new Error('token table is empty, have you called tokenizer.addToCorpus()?')
    }
    const to_vector_index: number[] = []
    const from_vector_index: number[] = []
    let vector_index = 0
    this.token_table.forEach((token, index) => {
      if (token.weight <= 0) return // a hole: `index in to_vector_index` is false (core.ts:437)
      to_vector_index[index] = vector_index
      from_vector_index[vector_index] = index
      vector_index++
    })
    this.to_vector_index = to_vector_index
    this.from_vector_index = from_vector_index
    this.tvi = null
  }
  private tviArray(): Int32Array {
    if (!this.to_vector_index) this.compactVectorIndex()
    if (!this.tvi) {
      this.tvi = new Int32Array(this.token_table.length).fill(-1)
      this.to_vector_index!.forEach((v, index) => (this.tvi![index] = v)) // forEach skips the holes of a sparse array
    }
    return this.tvi
  }

  // ---- training ---------------------------------------------------------------------------------------------------------------
  /** core.ts:247-326; falsy options mean the defaults (core.ts:255-256) */
  findNextMerge(options?: MergeOptions): MergeToken | null {
    this.flush()
    const max_length = options?.max_length || 0
    if (max_length && max_length < 2) return null
    const m = native.findNextMerge(this.engine, Math.max(1, Math.ceil(options?.min_weight || 2)), max_length)
    if (!m) return null
    // the SAME Token objects that sit in token_table: callers mutate them through applyMerge (core.ts:345-346)
    const a = this.token_table[m.a]
    const b = this.token_table[m.b]
    return [a, b, this.newToken(a.chars + b.chars, m.weight)] // core.ts:315-325
  }
  private recordMerge(a: Token, b: Token, c: Token): void {
    // core.ts:345-354
    a.weight -= c.weight
    b.weight -= c.weight
    this.code_to_token[c.code] = c
    this.token_table.push(c)
    this.merge_tokens.push([a, b, c])
    this.merge_codes.push([a.code + b.code, c.code])
  }
  /** core.ts:332-360 */
  applyMerge(merge: MergeToken): void {
    const [a, b, c] = merge
    this.flush()
    if (c.index !== this.token_table.length) {
      throw new Error(`merge is stale: its token index ${c.index} is not the next free index ${this.token_table.length}`)
    }
    native.applyMerge(this.engine, a.index, b.index, c.index)
    this.recordMerge(a, b, c)
    this.invalidateVectorIndex()
  }
  /** core.ts:365-383: the whole loop runs on the device; the log is replayed here exactly as core.ts:315-325,345-354 */
  mergeUntil(options?: MergeUntilOptions): void {
    this.flush()
    const max_length = options?.max_length || 0
    const max_iterations = options?.max_iterations || 0
    if ((max_length && max_length < 2) || (max_iterations && max_iterations < 1)) return
    const room = native.MAX_TOKENS - this.token_table.length
    const cap = max_iterations ? Math.min(room, Math.floor(max_iterations)) : room
    if (room <= 0) throw new RangeError(`token table exceeds ${native.MAX_TOKENS} entries`)
    const abc = new Int32Array(3 * cap)
    const weights = new Float64Array(cap)
    const n = native.mergeUntil(this.engine, Math.max(1, Math.ceil(options?.min_weight || 2)), max_length, cap, abc, weights)
    for (let i = 0; i < n; i++) {
      const a = this.token_table[abc[3 * i]]
      const b = this.token_table[abc[3 * i + 1]]
      this.recordMerge(a, b, this.newToken(a.chars + b.chars, weights[i]))
    }
    if (n) this.invalidateVectorIndex()
  }
  /** core.ts:477-494 */
  restoreMerge(compact: CompactMerge): void {
    const [a_code, b_code, c_weight] = compact
    const a = this.code_to_token[a_code]
    if (!a) throw new Error(`unknown token, a_code: ${JSON.stringify(a_code)}`)
    const b = this.code_to_token[b_code]
    if (!b) throw new Error(`unknown token, b_code: ${JSON.stringify(b_code)}`)
    this.applyMerge([a, b, this.newToken(a.chars + b.chars, c_weight)])
  }
  /** a whole merge log (lines written by compactMerge, example/scan-to-merge-log.ts:38-40) in ONE device call;
   *  equivalent to restoreMerge per line (example/import-merge-log-to-ram.ts:24-31), including its throws */
  restoreMerges(lines: CompactMerge[]): void {
    this.flush()
    const base = this.token_table.length
    const fresh: Record<string, Token> = {}
    const ab = new Int32Array(2 * lines.length)
    const merges: MergeToken[] = lines.map(([a_code, b_code, c_weight], i) => {
      const a = this.code_to_token[a_code] || fresh[a_code]
      if (!a) throw new Error(`unknown token, a_code: ${JSON.stringify(a_code)}`)
      const b = this.code_to_token[b_code] || fresh[b_code]
      if (!b) throw new Error(`unknown token, b_code: ${JSON.stringify(b_code)}`)
      const index = base + i
      if (index >= native.MAX_TOKENS) throw new RangeError(`token table exceeds ${native.MAX_TOKENS} entries`)
      const c: Token = { chars: a.chars + b.chars, weight: c_weight, original_weight: c_weight, code: String.fromCodePoint(index + 1), index }
      fresh[c.code] = c
      ab.set([a.index, b.index], 2 * i)
      return [a, b, c]
    })
    if (merges.length === 0) return
    native.applyMerges(this.engine, ab)
    merges.forEach(([a, b, c]) => this.recordMerge(a, b, c))
    this.invalidateVectorIndex()
  }

  // ---- encode / decode ------------------------------------------------------------------------------------------------------------
  /** many documents in one device call; `vector: false` gives token indices (encodeToTokens semantics) */
  encodeBatch(docs: string[], vector = true): { values: Int32Array; offsets: BigInt64Array; first_bad: BigInt64Array } {
    this.flush()
    this.syncChars()
    const parts = docs.map(d => utf8.encode(d))
    const off = offsetsOf(parts.map(p => p.length))
    const text = new Uint8Array(Math.max(Number(off[parts.length]), 1))
    parts.forEach((p, i) => text.set(p, Number(off[i])))
    const out = new Int32Array(text.length) // never more tokens than bytes
    const out_offsets = new BigInt64Array(docs.length + 1)
    const first_bad = new BigInt64Array(Math.max(docs.length, 1)).fill(-1n)
    const r = native.encodeBatch(this.engine, text, off, vector ? this.tviArray() : null, out, out_offsets, first_bad, true)
    if (r.unknown_pos >= 0) {
      throw new Error('unknown token, char: ' + JSON.stringify(String.fromCodePoint(r.unknown_code_point))) // core.ts:399
    }
    return { values: out.subarray(0, r.n), offsets: out_offsets, first_bad }
  }
  private encodeIds(content: string, vector: boolean): { values: Int32Array; first_bad: number } {
    const ids = this.charIds(content, false) // core.ts:396-402
    this.flush()
    const out = new Int32Array(Math.max(ids.length, 1))
    const out_offsets = new BigInt64Array(2)
    const first_bad = new BigInt64Array(1).fill(-1n)
    const r = native.encodeBatch(this.engine, ids, offsetsOf([ids.length]), vector ? this.tviArray() : null, out, out_offsets, first_bad, false)
    return { values: out.subarray(0, r.n), first_bad: Number(first_bad[0]) }
  }
  /** core.ts:392-409 */
  encodeToCode(content: string): string {
    let code = ''
    for (const index of this.encodeIds(content, false).values) code += String.fromCodePoint(index + 1)
    return code
  }
  /** core.ts:411-422 */
  encodeToTokens(content: string): Token[] {
    return Array.from(this.encodeIds(content, false).values, index => this.token_table[index])
  }
  /** core.ts:424-445 */
  encodeToVector(content: string): number[] {
    const { values, first_bad } = this.encodeIds(content, true)
    if (first_bad >= 0) throw new Error(`unknown token index: ${-values[first_bad] - 1}`) // core.ts:440
    return Array.from(values) // a plain Array<number>: the reference's tests deep-equal against array literals
  }
  /** core.ts:447-453 */
  decodeTokens(tokens: Token[]): string {
    let content = ''
    for (const token of tokens) content += token.chars
    return content
  }
  /** core.ts:455-471 */
  decodeVector(vector: number[]): string {
    if (!this.from_vector_index) this.compactVectorIndex()
    let content = ''
    for (const vector_index of vector) {
      if (!(vector_index in this.from_vector_index!)) throw new Error(`unknown vector index: ${vector_index}`) // core.ts:467
      content += this.token_table[this.from_vector_index![vector_index]].chars
    }
    return content
  }
  /** decodeVector for many documents in one device call; first_bad[d] >= 0 is where the reference would throw */
  decodeBatch(values: Int32Array, offsets: BigInt64Array, vector = true): { text: Uint8Array; offsets: BigInt64Array; first_bad: BigInt64Array } {
    this.flush()
    if (vector && !this.from_vector_index) this.compactVectorIndex()
    const parts = this.token_table.map(t => utf8.encode(t.chars))
    const tok_off = offsetsOf(parts.map(p => p.length))
    const tok_bytes = new Uint8Array(Math.max(Number(tok_off[parts.length]), 1))
    parts.forEach((p, i) => tok_bytes.set(p, Number(tok_off[i])))
    const fvi = vector ? Int32Array.from(this.from_vector_index!) : null // dense by construction (core.ts:233-240)
    const n_docs = offsets.length - 1
    const out_offsets = new BigInt64Array(n_docs + 1)
    const first_bad = new BigInt64Array(Math.max(n_docs, 1)).fill(-1n)
    let out = new Uint8Array(Math.max(values.length * 4, 1))
    let n = native.decodeBatch(this.engine, values, offsets, fvi, tok_bytes, tok_off, out, out_offsets, first_bad)
    if (n > out.length) {
      out = new Uint8Array(n)
      n = native.decodeBatch(this.engine, values, offsets, fvi, tok_bytes, tok_off, out, out_offsets, first_bad)
    }
    return { text: out.subarray(0, n), offsets: out_offsets, first_bad }
  }
}
