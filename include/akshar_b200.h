/* akshar_b200 -- C ABI of the B200-native batch path for Akshar's hot path.
 *
 * The reference (Bhasha-Open/Akshar) has no FFI: its boundary is the Python API in src/akshar.  Each entry point
 * below replaces, for a whole BATCH of sentences resident in HBM, the per-string Python call cited next to it.
 * INTEGRATION.md shows the ctypes binding a maintainer adds on the reference side.
 *
 * Conventions
 *   - plain pointers and sizes only; every `d_` pointer is DEVICE memory owned by the caller.
 *   - text layout: concatenated UTF-8 `d_text`, `d_row_offsets[n_rows + 1]` (int64, absolute byte indices into
 *     d_text, non-decreasing); the host passes the first and last offset (`text_begin`, `text_end`) by value.
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); nothing synchronises.
 *   - ragged outputs: values + `row_splits[n_rows + 1]` (int64).  Capacities are in elements; writes beyond a
 *     capacity are dropped, totals stay exact and AKSHAR_ST_OVERFLOW is raised in the result block.
 *   - `d_result` is 4 x int64 in device memory: [0] primary total, [1] secondary total, [2] status bits, [3] 0 (encoders
 *     that raise AKSHAR_ST_OVERFLOW for want of event slots: the slots per 960 text bytes that were needed; the id
 *     total of akshar_tokenizer_encode_batch is then 0, as it is when its normalize stage overflowed).
 *   - return value: 0 on success, negative AKSHAR_E_* for host-side errors (bad argument, CUDA launch failure).
 *   - one context per device; a context is not thread-safe.
 */
#ifndef AKSHAR_B200_H
#define AKSHAR_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct akshar_ctx akshar_ctx;

enum {
    AKSHAR_OK = 0,
    AKSHAR_E_ARG = -1,
    AKSHAR_E_CUDA = -2,
    AKSHAR_E_MODEL = -3,      /* model file could not be parsed / unsupported configuration */
    AKSHAR_E_NOMODEL = -4,    /* encode called before the matching akshar_load_* */
    AKSHAR_E_WORKSPACE = -5,
};

/* one call takes at most this much: positions inside a call are 32-bit.  Larger inputs go in as several calls over row
 * ranges of the same buffers (text_begin / text_end are absolute, nothing is rebased) */
#define AKSHAR_MAX_CALL_BYTES ((int64_t)4294901760)        /* 4 GiB - 64 KiB */
#define AKSHAR_MAX_CALL_ROWS ((int64_t)536870911)          /* 2^29 - 1 */

/* status bits in d_result[2] */
enum {
    AKSHAR_ST_OVERFLOW = 1,      /* an output capacity was too small: re-run with capacity >= total */
    AKSHAR_ST_NFC_SEGMENT = 2,   /* an NFC segment that needs work exceeds 256 decomposed code points: a starter followed by
                                    that many combining marks, or that many letters in a row that NFC itself decomposes
                                    (U+0958-095F, compatibility ideographs ...) with no other character between them */
    AKSHAR_ST_PATHOLOGICAL = 4,  /* bounded look-back gave up: re-run the same call with AKSHAR_MODE_ROWS */
    AKSHAR_ST_ALPHABET = 8,      /* reserved: until round 2 the BPE encoder refused a batch that held an added token ('<s>' ...)
                                  * or a code point HF's NFKC changes; such rows are now encoded exactly by the row kernel
                                  * (HF's added-token split + NFKC on the device), no entry point raises this bit */
    AKSHAR_ST_SPIN = 16,
    AKSHAR_ST_WORD = 32,         /* the pool for long words / rows encoded by the exact row kernel ran out: call again with a
                                    larger workspace -- half of what exceeds akshar_workspace_bytes() goes to the pools */
    AKSHAR_ST_INTERNAL = 64,     /* an internal consistency check failed (never expected): the result is not to be used */
    AKSHAR_ST_BAD_ID = 128,      /* decode: a token id outside the vocabulary of a SentencePiece model (DecodeIds raises
                                    IndexError "piece id is out of range."); HF's decode skips such ids */
    AKSHAR_ST_TEMPLATE = 256,    /* windows: a row does not begin with the template's bos / end with its eos (ids that the
                                    encoder of this model did not produce) */
    AKSHAR_ST_PAIR_TRUNC = 512,  /* pair windows: a pair cannot be truncated as asked (result[3] names it) */
    AKSHAR_ST_PACK_LONG = 1024,  /* packed batches: the stream of the call holds 2^31 ids or more */
};

/* normalize flags: normalize_text(text, normalize_roman, clean_hinglish) (normalize.py:117) is
 * (normalize_roman ? ROMAN : 0) | (clean_hinglish ? CLEAN : 0); the single stages map to the stand-alone functions:
 * ROMAN|NO_NFC = semantic_normalize (:21), FILTER|NO_NFC = filter_garbage (:92), COLLAPSE|NO_NFC =
 * remove_elongations (:48), CLEAN|NO_NFC = normalize_hinglish (:110), 0 = normalize_unicode (:13). */
#define AKSHAR_NORM_ROMAN 1u
#define AKSHAR_NORM_FILTER 2u
#define AKSHAR_NORM_COLLAPSE 4u
#define AKSHAR_NORM_CLEAN 6u
#define AKSHAR_NORM_NO_NFC 8u
/* segment flags */
#define AKSHAR_SEG_CLUSTERS 1u   /* segment_akshars(text)               (segment.py:40-78)  */
#define AKSHAR_SEG_MATRAS 2u     /* segment_akshars(text, matras=True)  (segment.py:80-125) */
#define AKSHAR_SEG_RUNS 4u       /* detect_code_switches(text)          (segment.py:150-201) */
#define AKSHAR_SEG_MASK 8u       /* the same boundaries as bit masks (tile mode only), see akshar_segment_batch */
/* mode */
#define AKSHAR_MODE_TILES 0      /* fixed-size byte spans, one thread per span (fast path) */
#define AKSHAR_MODE_ROWS 1       /* one span per row (exact for any input, slow for very long rows) */

int akshar_version(void);
const char* akshar_status_str(int code);
int akshar_ctx_create(int device, akshar_ctx** out);
void akshar_ctx_destroy(akshar_ctx* ctx);
const char* akshar_last_error(akshar_ctx* ctx);

/* bytes of device workspace the batch calls need for a buffer of n_bytes / n_rows */
size_t akshar_workspace_bytes(int64_t n_bytes, int64_t n_rows);

/* normalize_text over a batch (normalize.py:13-56, 92-148).  d_out_text capacity in bytes;
 * d_out_row_offsets[n_rows + 1] always written.  result[0] = output bytes. */
int akshar_normalize_batch(akshar_ctx* ctx, const uint8_t* d_text, const int64_t* d_row_offsets, int64_t n_rows,
                           int64_t text_begin, int64_t text_end, uint32_t flags, int mode, uint8_t* d_out_text,
                           int64_t out_capacity, int64_t* d_out_row_offsets, int64_t* d_result, void* d_workspace,
                           size_t workspace_bytes, void* stream);

/* segment_akshars / detect_code_switches over a batch (segment.py:40-201).
 * cluster_ends / run_ends: int32 byte offset of each cluster / run END relative to its row start;
 * run_tags: 0 devanagari 1 roman 2 digit 3 punct 4 other 255 None (identify_script, segment.py:128-147).
 * Outputs not selected by `flags` may be NULL.  result[0] = clusters, result[1] = runs.
 * With AKSHAR_SEG_MASK the boundaries come as one bit per text byte instead (1/8 byte per text byte and stream rather than
 * 4 bytes per boundary): d_cluster_ends / d_run_ends receive W = (text_end - text_begin + 32) / 32 uint32 words each
 * (capacities are counted in words), bit (p - text_begin) set when a cluster / run ENDS at byte p (the end of a non-empty
 * row included); d_run_tags receives 2 W words: the planes t0 then t1 of the tag of the run that ends at a bit,
 * (t1 t0) = 00 devanagari, 01 roman, 10 other, 11 none.  The split arrays are not written (may be NULL). */
int akshar_segment_batch(akshar_ctx* ctx, const uint8_t* d_text, const int64_t* d_row_offsets, int64_t n_rows,
                         int64_t text_begin, int64_t text_end, uint32_t flags, int mode, int32_t* d_cluster_ends,
                         int64_t cluster_capacity, int64_t* d_cluster_splits, int32_t* d_run_ends, uint8_t* d_run_tags,
                         int64_t run_capacity, int64_t* d_run_splits, int64_t* d_result, void* d_workspace,
                         size_t workspace_bytes, void* stream);

/* word_tokenize_hindi / word_tokenize_sanskrit / word_tokenize over a batch (segment.py:239-401).
 * rule AKSHAR_WORDS_HINDI: the loop of segment.py:270-297 (= :335-362) over text that normalize_text has already been
 *   applied to (segment.py:258): str.isspace() separates, U+0964 / U+0965 are tokens of their own, .,!?;:()[]{}"' separate
 *   and are dropped.  rule AKSHAR_WORDS_SPLIT: text.split() (segment.py:391-393, 400-401) -- only str.isspace() separates.
 * word_begin / word_end: int32 byte offsets of each token (end exclusive) relative to its row start; word_splits[r] =
 * tokens in rows before r (n_rows + 1 entries).  row_flags (optional, n_rows bytes): bit 0 = the row holds a code point of
 * U+0900-097F, the test `word_tokenize(language='auto')` routes on (segment.py:384-388).  result[0] = tokens (exact also
 * when AKSHAR_ST_OVERFLOW says word_capacity was too small). */
#define AKSHAR_WORDS_HINDI 0
#define AKSHAR_WORDS_SPLIT 1
int akshar_word_tokenize_batch(akshar_ctx* ctx, const uint8_t* d_text, const int64_t* d_row_offsets, int64_t n_rows,
                               int64_t text_begin, int64_t text_end, int rule, int32_t* d_word_begin, int32_t* d_word_end,
                               int64_t word_capacity, int64_t* d_word_splits, uint8_t* d_row_flags, int64_t* d_result,
                               void* d_workspace, size_t workspace_bytes, void* stream);

/* aksharTokenizer.decode / detokenize over a batch of id rows (tokenizer.py:195-246); kind 0 BPE, 1 Unigram.
 * form AKSHAR_FORM_DECODE: SentencePiece DecodeIds (control pieces dropped, <unk> -> " \u2047 ", runs of byte pieces
 *   reassembled as UTF-8 with U+FFFD for every byte that is not part of a well-formed sequence, U+2581 -> ' ', the dummy
 *   prefix consumed) / HF Tokenizer.decode with `decoder: null` (the tokens of the non-special ids joined by ' ').
 * form AKSHAR_FORM_DETOKENIZE: `detokenize(tokenize pieces)` -- the piece strings of the ids joined the way
 *   tokenizer.py:236-246 joins them (SentencePiece: ''.join, U+2581 -> ' ', strip; BPE: ' '.join, ' ##' removed,
 *   U+0120 -> ' ', strip).
 * d_ids: int32 (or uint16 with ids_u16 != 0: the compact output of akshar_tokenizer_encode_batch_ex), n_ids of them;
 * d_row_splits: int64 [n_rows + 1] positions in d_ids.  Output: UTF-8 bytes + int64 [n_rows + 1] row offsets.
 * result[0] = output bytes (exact also when AKSHAR_ST_OVERFLOW says out_capacity was too small). */
#define AKSHAR_FORM_DECODE 0
#define AKSHAR_FORM_DETOKENIZE 1
size_t akshar_decode_workspace_bytes(int64_t n_ids, int64_t n_rows);
int akshar_decode_batch(akshar_ctx* ctx, int kind, int form, const void* d_ids, int ids_u16, int64_t n_ids, const int64_t* d_row_splits,
                        int64_t n_rows, uint8_t* d_out_text, int64_t out_capacity, int64_t* d_out_row_offsets, int64_t* d_result,
                        void* d_workspace, size_t workspace_bytes, void* stream);

/* analyze_text_composition over a batch (segment.py:210-236), from the outputs of akshar_segment_batch (clusters + runs of
 * the same text): d_stats[5 r ..] = akshars, script runs, code points, code points in devanagari runs, in roman runs.
 * (script_switches = runs - 1; the two ratios are the last two counts over the third.) */
int akshar_composition_batch(akshar_ctx* ctx, const uint8_t* d_text, const int64_t* d_row_offsets, int64_t n_rows,
                             const int64_t* d_cluster_splits, const int32_t* d_run_ends, const uint8_t* d_run_tags,
                             const int64_t* d_run_splits, int32_t* d_stats, void* stream);

/* the feature wrappers that are functions of the cluster boundaries: akshara_level_tokenization (features.py:28-55,
 * AKSHAR_MERGE_AKSHARA: consecutive clusters that hold U+094D are one akshara) and preserve_nukta (features.py:173-206,
 * AKSHAR_MERGE_NUKTA: a cluster that holds U+093C takes the next cluster with it).  In: the clusters of
 * akshar_segment_batch(matras = 0); out: the merged clusters in the same form.  result[0] = merged clusters. */
#define AKSHAR_MERGE_AKSHARA 0
#define AKSHAR_MERGE_NUKTA 1
size_t akshar_merge_workspace_bytes(int64_t n_clusters);
int akshar_merge_clusters_batch(akshar_ctx* ctx, const uint8_t* d_text, const int64_t* d_row_offsets, int64_t n_rows,
                                const int32_t* d_cluster_ends, const int64_t* d_cluster_splits, int64_t n_clusters, int rule,
                                int32_t* d_out_ends, int64_t out_capacity, int64_t* d_out_splits, int64_t* d_result,
                                void* d_workspace, size_t workspace_bytes, void* stream);

/* The lines of a text file as rows (cli.py:165-190 = scripts/train_bpe.py:16-35 = train_spm.py:18-44: `readlines()` of a
 * universal-newlines text file, `strip()`, empty lines skipped).  d_file: the file's bytes (valid UTF-8; Python would raise
 * on anything else) on the device.  Output: the rows packed next to each other + int64 [rows + 1] row offsets -- the form
 * every other entry point takes.  result[0] = rows (exact also when AKSHAR_ST_OVERFLOW says row_capacity or out_capacity
 * was too small), result[1] = packed bytes. */
size_t akshar_lines_workspace_bytes(int64_t n_bytes, int64_t row_capacity);
int akshar_lines_batch(akshar_ctx* ctx, const uint8_t* d_file, int64_t n_bytes, uint8_t* d_out_text, int64_t out_capacity,
                       int64_t* d_out_row_offsets, int64_t row_capacity, int64_t* d_result, void* d_workspace, size_t workspace_bytes,
                       void* stream);

/* rows -> one byte stream, every row followed by the byte `sep`: the file preprocess_corpus writes (cli.py:185-187).
 * d_out holds (row_offsets[n_rows] - row_offsets[0]) + n_rows bytes. */
int akshar_join_rows(akshar_ctx* ctx, const uint8_t* d_text, const int64_t* d_row_offsets, int64_t n_rows, int sep, uint8_t* d_out,
                     void* stream);

/* normalize_text -> akshars / script runs in one call, nothing read back in between (BASELINE config 4: "normalize +
 * grapheme + code-switch pipeline"): the normalized rows as akshar_normalize_batch writes them, and the boundaries of the
 * NORMALIZED text as AKSHAR_SEG_MASK bit masks (mask_words >= (norm_capacity + 32) / 32 words per mask; the tag planes
 * t0 / t1 are mask_words apart).  result[0] = clusters, result[1] = runs, result[3] = normalized bytes.
 * AKSHAR_ST_PATHOLOGICAL / AKSHAR_ST_OVERFLOW as in akshar_normalize_batch (call the two stages separately then). */
int akshar_normalize_segment_batch(akshar_ctx* ctx, const uint8_t* d_text, const int64_t* d_row_offsets, int64_t n_rows,
                                   int64_t text_begin, int64_t text_end, uint32_t norm_flags, uint32_t seg_flags, uint8_t* d_norm_text,
                                   int64_t norm_capacity, int64_t* d_norm_row_offsets, uint32_t* d_cluster_mask, uint32_t* d_run_mask,
                                   uint32_t* d_run_tag_planes, int64_t mask_words, int64_t* d_result, void* d_workspace,
                                   size_t workspace_bytes, void* stream);

/* roman_phonetic_signature over a batch of words (normalize.py:59-89); one word per row. result[0] = out bytes */
int akshar_signature_batch(akshar_ctx* ctx, const uint8_t* d_text, const int64_t* d_row_offsets, int64_t n_rows,
                           int64_t text_begin, int64_t text_end, uint8_t* d_out_text, int64_t out_capacity,
                           int64_t* d_out_row_offsets, int64_t* d_result, void* d_workspace, size_t workspace_bytes,
                           void* stream);

/* model loading (host buffers): the HF tokenizers JSON written by scripts/train_bpe.py:68-98 and the SentencePiece
 * ModelProto written by scripts/train_spm.py:80-108 -- replaces Tokenizer.from_file / SentencePieceProcessor.Load
 * (tokenizer.py:88-98). */
int akshar_load_bpe_json(akshar_ctx* ctx, const char* json, size_t len);
int akshar_load_spm_model(akshar_ctx* ctx, const void* proto, size_t len);
/* vocabulary access for host-side decode / vocab_size (tokenizer.py:195-219, 278-288); kind 0 = BPE, 1 = Unigram */
int akshar_vocab_size(akshar_ctx* ctx, int kind);
/* returns the UTF-8 bytes of token `id` (not NUL-terminated) and its type:
 * BPE: 0 normal, 1 special; Unigram: SentencePiece type (1 NORMAL 2 UNKNOWN 3 CONTROL 4 USER_DEFINED 5 UNUSED 6 BYTE) */
int akshar_vocab_token(akshar_ctx* ctx, int kind, int id, const char** bytes, int* len, int* type);

/* Tokenizer.encode(norm).ids over a batch of ALREADY NORMALIZED rows (tokenizer.py:193): ids include <s> / </s>
 * from the template post-processor.  result[0] = ids. */
int akshar_encode_bpe_batch(akshar_ctx* ctx, const uint8_t* d_text, const int64_t* d_row_offsets, int64_t n_rows,
                            int64_t text_begin, int64_t text_end, int mode, int32_t* d_ids, int64_t id_capacity,
                            int64_t* d_id_splits, int64_t* d_result, void* d_workspace, size_t workspace_bytes,
                            void* stream);

/* SentencePieceProcessor.EncodeAsIds(norm) over a batch of ALREADY NORMALIZED rows (tokenizer.py:191). */
int akshar_encode_unigram_batch(akshar_ctx* ctx, const uint8_t* d_text, const int64_t* d_row_offsets, int64_t n_rows,
                                int64_t text_begin, int64_t text_end, int mode, int32_t* d_ids, int64_t id_capacity,
                                int64_t* d_id_splits, int64_t* d_result, void* d_workspace, size_t workspace_bytes,
                                void* stream);

/* aksharTokenizer.encode(text) over a batch of RAW rows (tokenizer.py:167-193): preprocess (= normalize_text with
 * `norm_flags`) then the model selected by `kind` (0 BPE, 1 Unigram), enqueued back to back with no host
 * synchronisation in between (the normalized length stays on the device).  The normalized rows are returned too
 * (d_norm_text / d_norm_row_offsets) because token offsets refer to them.  The workspace must be sized for
 * max(text_end - text_begin, norm_capacity) bytes.  result[0] = ids, result[1] = normalized bytes. */
int akshar_tokenizer_encode_batch(akshar_ctx* ctx, const uint8_t* d_text, const int64_t* d_row_offsets, int64_t n_rows,
                                  int64_t text_begin, int64_t text_end, uint32_t norm_flags, int kind, int mode,
                                  uint8_t* d_norm_text, int64_t norm_capacity, int64_t* d_norm_row_offsets, int32_t* d_ids,
                                  int64_t id_capacity, int64_t* d_id_splits, int64_t* d_result, void* d_workspace,
                                  size_t workspace_bytes, void* stream);

/* The same call with compact outputs for callers that ship the result over a host link (the ids of a 24k vocabulary
 * need 16 bits, the splits of a chunk 32): out_flags = AKSHAR_OUT_IDS_U16 -> d_ids is uint16_t[id_capacity] (refused when
 * the vocabulary has more than 65536 entries), AKSHAR_OUT_SPLITS_I32 -> d_id_splits is int32_t[n_rows + 1].
 * Needs AKSHAR_MODE_TILES. */
#define AKSHAR_OUT_IDS_U16 1u
#define AKSHAR_OUT_SPLITS_I32 2u
int akshar_tokenizer_encode_batch_ex(akshar_ctx* ctx, const uint8_t* d_text, const int64_t* d_row_offsets, int64_t n_rows,
                                     int64_t text_begin, int64_t text_end, uint32_t norm_flags, int kind, int mode,
                                     uint8_t* d_norm_text, int64_t norm_capacity, int64_t* d_norm_row_offsets, void* d_ids,
                                     int64_t id_capacity, void* d_id_splits, uint32_t out_flags, int64_t* d_result,
                                     void* d_workspace, size_t workspace_bytes, void* stream);

/* Model-ready windows of encoder output, bit-exact with HF tokenizers' Tokenizer.enable_truncation(max_length, stride,
 * direction) + enable_padding(direction, pad_id, length, pad_to_multiple_of) + encode_batch, flattened row by row as
 * transformers flattens `[enc] + enc.overflowing` (return_overflowing_tokens=True).
 * In: the ragged ids of one encoder call of model `kind` (0 BPE, 1 Unigram): d_ids int32 (or uint16 with ids_u16 != 0,
 * the compact output of akshar_tokenizer_encode_batch_ex; may be NULL when the rows hold no ids), d_row_splits int64
 * [n_rows + 1] positions in d_ids; fewer than 2^31 ids in one call.  The template ids s (2 for a BPE model whose post-processor is `<s> $A </s>`, 0 without one and
 * for Unigram) come from the context's model; a row's content c is the row without them, m = max_length - s.
 * Truncation (AKSHAR_WIN_TRUNCATE): a row with |c| <= m is one window; otherwise step = m - stride and window k is
 * c[k step : min(k step + m, |c|)] (right) or c[max(|c| - k step - m, 0) : |c| - k step] (AKSHAR_WIN_TRUNC_LEFT) until a
 * window reaches the end (start) of c: 1 + ceil((|c| - m) / step) windows; without AKSHAR_WIN_OVERFLOW only window 0.
 * Every window is re-wrapped in the template ids.  Illegal values are refused with AKSHAR_E_ARG where HF misbehaves:
 * max_length <= s, stride < 0 or >= m with truncation; stride != 0 or AKSHAR_WIN_OVERFLOW without it.
 * Two calls:
 *   akshar_windows_count: d_window_splits int64 [n_rows + 1] (window n belongs to row r for splits[r] <= n < splits[r + 1]);
 *     result[0] = N windows, result[1] = longest window (template ids included), result[2] |= AKSHAR_ST_TEMPLATE when a
 *     row is not framed by the template ids.
 *   akshar_windows_write: for a width L >= the longest window (the caller picks it: the longest, or max_length, rounded up
 *     to a multiple), d_input_ids / d_attention_mask int64 [n_windows, L] and d_sample int64 [n_windows] (the row of each
 *     window: overflow_to_sample_mapping).  Pad positions hold pad_id and mask 0, on the right or on the left
 *     (AKSHAR_WIN_PAD_LEFT); the other positions hold the window and mask 1.  n_windows, max_length, stride and flags are
 *     those of the count call. */
#define AKSHAR_WIN_TRUNCATE 1u
#define AKSHAR_WIN_OVERFLOW 2u
#define AKSHAR_WIN_TRUNC_LEFT 4u
#define AKSHAR_WIN_PAD_LEFT 8u
size_t akshar_windows_workspace_bytes(int64_t n_rows);
int akshar_windows_count(akshar_ctx* ctx, int kind, const void* d_ids, int ids_u16, const int64_t* d_row_splits, int64_t n_rows,
                         int64_t max_length, int64_t stride, uint32_t flags, int64_t* d_window_splits, int64_t* d_result,
                         void* d_workspace, size_t workspace_bytes, void* stream);
int akshar_windows_write(akshar_ctx* ctx, int kind, const void* d_ids, int ids_u16, const int64_t* d_row_splits,
                         const int64_t* d_window_splits, int64_t n_rows, int64_t n_windows, int64_t max_length, int64_t stride,
                         uint32_t flags, int64_t width, int64_t pad_id, int64_t* d_input_ids, int64_t* d_attention_mask,
                         int64_t* d_sample, void* stream);

/* Model-ready windows of sentence pairs, bit-exact with HF tokenizers' Tokenizer.enable_truncation(max_length, stride,
 * strategy, direction) + enable_padding(...) + encode_batch of (a, b) pairs through the model's TemplateProcessing
 * pair template, flattened as transformers flattens `[enc] + enc.overflowing` (tokenizer(texts, text_pair, ...)).
 * In: two ragged id sets of the encoder of model `kind`, one row per pair on each side: d_ids_a / d_splits_a [n_pairs + 1]
 * and d_ids_b / d_splits_b [n_pairs + 1], int32 ids (uint16 with ids_u16 != 0, both sides); the two sides may share one
 * ids buffer (texts and pairs encoded in one call: d_splits_b = d_splits_a + n_pairs).  Every row is framed by the
 * single template as the encoder writes it; A and B are the rows without those ids, of ca and cb ids.
 * The pair template is `pre $A mid $B post` (at most 4 ids per slot; the `<s> $A </s> <s> $B </s>` of a BPE model
 * has P = |pre| + |mid| + |post| = 4; no post-processor and Unigram: P = 0); m = max_length - P.
 * Truncation (AKSHAR_WIN_TRUNCATE; longest_first unless AKSHAR_WIN_ONLY_FIRST or AKSHAR_WIN_ONLY_SECOND):
 *   1. ca + cb <= m: nothing is cut, one window.
 *   2. else the lengths na, nb that A and B are cut to: longest_first: n1 = min(ca, cb); n2 = n1 if n1 > m, else
 *      max(n1, m - n1); if n1 + n2 > m then n1 = m / 2 and n2 = n1 + m % 2; the larger goes to the longer sequence,
 *      to B on a tie.  only_first / only_second: rem = ca + cb - m; the target sequence is cut to its length - rem.
 *   3. a sequence that is cut (n < its length) has the windows of akshar_windows_count with m = n and the same
 *      direction (AKSHAR_WIN_TRUNC_LEFT), wa windows for A and wb for B; a sequence not cut is one window.
 *   4. with AKSHAR_WIN_OVERFLOW the pair gives wa * wb windows in the order (0, 0); (i, 0 .. wb - 1) for
 *      i = 1 .. wa - 1; (0, j) for j = 1 .. wb - 1; without it only (0, 0).  Window (i, j) is pre + A_i + mid + B_j + post.
 * Refused where HF misbehaves or raises: with AKSHAR_E_ARG for the call: m <= 0, stride < 0, stride > max_length - s
 * with truncation (s: the single template's ids; HF's enable_truncation raises there, pairs or not), stride != 0 or
 * AKSHAR_WIN_OVERFLOW without truncation, both ONLY flags, a model whose pair template is not of the form above
 * ("unsupported pair template"); per pair, in result[2] |= AKSHAR_ST_PAIR_TRUNC and result[3] = the lowest
 * pair * 8 + reason (1: longest_first would cut a sequence to 0 ids, 2: stride >= the length a sequence is cut to,
 * 3: only_first / only_second and the target has no more than rem ids, 4: more than 2^31 - 1 windows); and for the
 * whole call, when no pair is refused but the pairs give more than 2^31 - 1 windows in all, result[2] |=
 * AKSHAR_ST_PAIR_TRUNC and result[3] = n_pairs * 8 + 5 (result[0] and d_window_splits are then not to be used).
 * Two calls, as the single windows (workspace: akshar_windows_workspace_bytes(n_pairs)):
 *   akshar_pair_windows_count: d_window_splits int64 [n_pairs + 1]; result[0] = N windows, result[1] = longest window
 *     (always window (0, 0) of its pair), result[2] |= AKSHAR_ST_TEMPLATE when a row is not framed by the template ids.
 *   akshar_pair_windows_write: d_input_ids / d_attention_mask int64 [n_windows, L] for a width L >= the longest window,
 *     d_sample int64 [n_windows] (the pair of each window); pads as akshar_windows_write.  n_windows, max_length,
 *     stride and flags are those of the count call. */
#define AKSHAR_WIN_ONLY_FIRST 16u
#define AKSHAR_WIN_ONLY_SECOND 32u
int akshar_pair_windows_count(akshar_ctx* ctx, int kind, const void* d_ids_a, const int64_t* d_splits_a, const void* d_ids_b,
                              const int64_t* d_splits_b, int ids_u16, int64_t n_pairs, int64_t max_length, int64_t stride,
                              uint32_t flags, int64_t* d_window_splits, int64_t* d_result, void* d_workspace,
                              size_t workspace_bytes, void* stream);
int akshar_pair_windows_write(akshar_ctx* ctx, int kind, const void* d_ids_a, const int64_t* d_splits_a, const void* d_ids_b,
                              const int64_t* d_splits_b, int ids_u16, const int64_t* d_window_splits, int64_t n_pairs,
                              int64_t n_windows, int64_t max_length, int64_t stride, uint32_t flags, int64_t width,
                              int64_t pad_id, int64_t* d_input_ids, int64_t* d_attention_mask, int64_t* d_sample, void* stream);

/* Packed language-model batches: the rows of one call concatenated into one stream and cut into blocks of L ids, as
 * transformers' run_clm.py `group_texts` does, with what a padding-free model needs to keep the documents apart, as
 * transformers' DataCollatorWithFlattening(return_flash_attn_kwargs=True, return_seq_idx=True) returns it.
 * In: ragged rows of ids, one per document (d_ids int32, or uint16 with ids_u16 != 0; d_row_splits int64 [n_rows + 1]),
 * block_size L >= 1, eos_id in [0, 2^31) or -1 for none, and a carry: the rest of the previous call (d_carry int32 ids,
 * d_carry_splits int64 [n_carry + 1]; n_carry = 0 and NULL pointers for none).
 *   1. Stream S: the carry's fragments verbatim, then every row's ids, each followed by eos_id when one is given.  A
 *      document start is the start of a non-empty fragment or row (an empty row adds nothing without eos_id, and the
 *      document [eos] with it).  Unit u (fragment u, then row u - n_carry) starts at s_u = carry_splits[u] -
 *      carry_splits[0], or C + (splits[r] - splits[0]) + (eos ? r : 0) for row r, C the carry's ids.
 *   2. T = |S| < 2^31, N = T / L; block b is S[b L : (b + 1) L].  The rest S[N L : T] (< L ids) is returned in the carry's
 *      form, its fragments split at document starts; passed as the next call's carry, packing in chunks equals packing
 *      in one call.
 *   3. Pieces start at every block start and every document start below N L.  Position p < N L of the document that
 *      starts at s: position_ids = p - max(s, (p / L) L); labels = separator_id where position_ids = 0, else S[p];
 *      seq_idx = the index of p's piece; cu_seq_lens = the piece starts, then N L; the longest piece is max_length.
 * Refused with AKSHAR_E_ARG: L < 1, eos_id outside [0, 2^31) and not -1, more than 2^29 - 1 rows or fragments; and on
 * the device with result[2] |= AKSHAR_ST_PACK_LONG: a stream of 2^31 ids or more (cu_seq_lens and seq_idx are int32).
 * Two calls (workspace: akshar_pack_workspace_bytes(n_rows + n_carry), the same for both and kept between them):
 *   akshar_pack_count: d_result int64 [8]: [0] N, [1] P pieces, [2] status, [3] longest piece, [4] T, [5] F fragments of
 *     the rest, [6..7] 0.  Read back once; every size below follows from it.
 *   akshar_pack_write, with T, P and F of the count call: d_input_ids and d_labels int64 [N L]; d_position_ids int64
 *     [N L], d_seq_idx int32 [N L] and d_cu_seq_lens int32 [P + 1], each NULL when not wanted; d_rest_ids int32
 *     [T - N L] and d_rest_splits int64 [F + 1] (always).  The other arguments are those of the count call. */
size_t akshar_pack_workspace_bytes(int64_t n_units);
int akshar_pack_count(akshar_ctx* ctx, const void* d_ids, int ids_u16, const int64_t* d_row_splits, int64_t n_rows,
                      const int32_t* d_carry, const int64_t* d_carry_splits, int64_t n_carry, int64_t block_size, int64_t eos_id,
                      int64_t* d_result, void* d_workspace, size_t workspace_bytes, void* stream);
int akshar_pack_write(akshar_ctx* ctx, const void* d_ids, int ids_u16, const int64_t* d_row_splits, int64_t n_rows,
                      const int32_t* d_carry, const int64_t* d_carry_splits, int64_t n_carry, int64_t block_size, int64_t eos_id,
                      int64_t separator_id, int64_t total, int64_t n_pieces, int64_t n_rest_fragments, int64_t* d_input_ids,
                      int64_t* d_labels, int64_t* d_position_ids, int32_t* d_seq_idx, int32_t* d_cu_seq_lens,
                      int32_t* d_rest_ids, int64_t* d_rest_splits, void* d_workspace, size_t workspace_bytes, void* stream);

/* Masked language-model batches: transformers' DataCollatorForLanguageModeling(mlm=True) `torch_mask_tokens` over a dense
 * batch, with its draws keyed by (seed, epoch, row, position), so that the masks do not depend on how a corpus is cut
 * into calls, padded or spread over GPUs.
 * In: d_input_ids int64 [n_rows, width] (as akshar_windows_write / akshar_pair_windows_write / akshar_pack_write write
 * it), model `kind`, seed in [0, 2^64), epoch in [0, 2^32), row_base >= 0, the thresholds t1 t2 t3 (each <= 2^32), mask_id
 * in [0, V), pad_id (-1: none).  V = the model's vocabulary size (akshar_vocab_size).
 *   1. Special ids: the model's own (BPE: the added tokens marked "special": true; SentencePiece: the UNKNOWN and CONTROL
 *      pieces) and pad_id: the collator's get_special_tokens_mask(already_has_special_tokens=True).  Other ids, those
 *      outside [0, V) included, are not special.
 *   2. Draws: one Philox4x32-10 block (Random123 / cuRAND Philox) per position: key (seed mod 2^32, seed >> 32),
 *      counter (j, R mod 2^32, R >> 32, epoch) with R = row_base + n the row and j the position; its words are
 *      (u_select, u_mask, u_random, r_id).
 *   3. Thresholds, computed by the caller from the collator's probabilities p, m, r: t(q) = min(2^32, ceil(fl32(q) 2^32)),
 *      fl32 = rounding to float32 (the collator's probability matrices are float32); t1 = t(p), t2 = t(m), t3 =
 *      t(r / (1 - m)) with the ratio in double, and t3 = 0 when m = 1 or r = 0 (the collator returns before its third
 *      draw).  u < t means drawn: u / 2^32 < fl32(q), what torch.bernoulli decides from a uniform u / 2^32.
 *   4. Per position: selected = not special and u_select < t1; replaced = selected and u_mask < t2; random = selected,
 *      not replaced and u_random < t3.
 *   5. d_labels int64 [n_rows, width] = the original id where selected, else -100; d_input_ids, in place: mask_id where
 *      replaced, floor(r_id V / 2^32) where random.  The random id is a multiply-high, not torch.randint's exactly
 *      uniform draw: its relative bias is at most V / 2^32 (5.6e-6 for V = 24000).
 * Refused with AKSHAR_E_ARG: a threshold above 2^32, width >= 2^32, mask_id outside [0, V), pad_id < -1, row_base +
 * n_rows > 2^64; AKSHAR_E_NOMODEL when `kind` is not loaded.  n_rows = 0 or width = 0 launches nothing.  One kernel,
 * no workspace, no synchronisation. */
int akshar_mlm_mask(akshar_ctx* ctx, int kind, int64_t* d_input_ids, int64_t n_rows, int64_t width, uint64_t seed, uint32_t epoch,
                    uint64_t row_base, const uint64_t thresholds[3], int64_t mask_id, int64_t pad_id, int64_t* d_labels,
                    void* stream);

/* Optional device-side timing of the dominant kernel of each stage, for roofline reporting: when enabled, the
 * library brackets that one launch with CUDA events on the caller's stream; akshar_timing_read waits for the
 * kernel and returns its duration of the most recent call. */
enum {
    AKSHAR_TIMER_NORMALIZE_CLASSIFY = 0,   /* ak_nf3_classify_kernel */
    AKSHAR_TIMER_NORMALIZE_WRITE = 1,      /* ak_nf_write_kernel */
    AKSHAR_TIMER_BPE_ENCODE = 2,           /* ak_resolve_kernel<0> (word events -> BPE ids through the word cache) */
    AKSHAR_TIMER_SEGMENT = 3,              /* ak_seg_off_kernel<emit> / ak_seg_mask_kernel */
    AKSHAR_TIMER_UNIGRAM = 4,              /* ak_resolve_kernel<1> (word events -> Unigram ids), or ak_unigram_kernel in row mode */
    AKSHAR_TIMER_WORDS = 5,                /* ak_words_kernel (text -> word / row events) */
    AKSHAR_TIMER_EMIT = 6,                 /* ak_emit_kernel (ids to their final place) */
    AKSHAR_TIMER_WORDTOK = 7,              /* ak_wtok_kernel<emit> (word tokenizers) */
    AKSHAR_TIMER_DECODE = 8,               /* ak_dec_kernel<write> (ids -> text) */
    AKSHAR_TIMER_LINES = 9,                /* ak_lines_kernel<emit> (file bytes -> rows) */
    AKSHAR_TIMER_COUNT = 10
};
int akshar_timing_enable(akshar_ctx* ctx, int enable);

/* Word caches of the encoders (pre-tokenized word -> ids; HF tokenizers keeps the same kind of cache for the lifetime of
 * its Tokenizer, reference tokenizer.py:96-98 -> tokenizers BPE `cache`).  A cache lives as long as its model: words
 * met in one call serve the next ones; results never depend on its contents.  It has no eviction: when the words learned
 * since the last restore fill a quarter of the table, the image built at model load is copied back at the start of the
 * next call (decided on the device).  hold = 1 switches that restore off, hold = 0 (default) on again, hold < 0
 * restores the image at the next encode call whatever the fill. */
int akshar_word_cache_hold(akshar_ctx* ctx, int hold);
/* Read-only state of the word cache of model `kind` (0 BPE, 1 Unigram), for tests and monitoring: out[0] = slots of the
 * table, out[1] = entries of the image built at load, out[2] = entries learned since the last restore (read on `stream`,
 * which is then synchronised), out[3] = the context's hold flag.  Only a restore empties a slot, so out[1] + out[2] slots
 * are occupied.  AKSHAR_E_NOMODEL when the model is not loaded or has no word cache (a Unigram model without the
 * word-wise shape). */
int akshar_word_cache_stats(akshar_ctx* ctx, int kind, int64_t* out, void* stream);
int akshar_timing_read(akshar_ctx* ctx, int timer, float* ms);

/* number of kernels this library has launched on this context since creation (bench.py's gpu_launches) */
int64_t akshar_launch_count(akshar_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif
