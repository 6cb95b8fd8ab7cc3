/* wordpiece_b200 — C ABI of the B200-native fast WordPiece encoder.
 *
 * This is the drop-in boundary for ONE path of gleb-kov/wordpiece: the Fast
 * greedy longest-match encoder (reference src/fast.cpp).  The reference has no
 * FFI of its own — its public surface is seven C++ free functions in
 * src/word_piece.hpp:10-36 — so the boundary is two-layered:
 *
 *   include/word_piece.hpp   the reference's own C++ signatures (namespace
 *                            word_piece::fast), implemented by a host shim that
 *   include/wordpiece_b200.h calls THIS C ABI, which launches the sm_100a kernels.
 *
 * Each entry point below names the reference interface it replaces.  Plain
 * pointers and sizes only; no C++ or torch types; nothing throws across the
 * boundary (status codes + wp_last_error()).  There is NO CPU fallback: every
 * encode call runs the CUDA kernels or fails with WP_ERR_CUDA / WP_ERR_NO_DEVICE.
 *
 * Threading: a wp_vocab handle owns one CUDA stream and scratch buffers on one
 * device; use a handle from one host thread at a time, and let every encode call on
 * it finish being ENQUEUED before the next (the device work of consecutive calls is
 * serialised by the library, whatever streams they use) (the reference is not
 * re-entrant either: one process-global pool, utils.cpp:25-28).  Several handles
 * (e.g. one per GPU) may be used concurrently.
 */
#ifndef WORDPIECE_B200_H_
#define WORDPIECE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct wp_vocab wp_vocab;

typedef enum wp_status {
  WP_OK = 0,
  WP_ERR_INVALID_ARG = 1,
  WP_ERR_EMPTY_VOCAB_WORD = 2, /* reference: throw runtime_error("Vocab word is empty"), utils.cpp:99-101 */
  WP_ERR_CUDA = 3,
  WP_ERR_NO_DEVICE = 4,
  WP_ERR_CAPACITY = 5, /* caller's id buffer too small; *n_ids still holds the exact count */
  WP_ERR_IO = 6,
  WP_ERR_NOMEM = 7,
  WP_ERR_ID_RANGE = 8 /* wp_decode: id == vocab size (reference: .at() throws out_of_range, fast.cpp:175) */
} wp_status;

/* Counters of the last encode call on a handle (diagnostics; tests use them to
 * prove that the slow lanes were exercised). */
typedef struct wp_stats {
  uint64_t n_bytes;        /* text bytes encoded */
  uint64_t n_ids;          /* ids produced */
  uint64_t n_tiles;        /* text tiles processed */
  uint64_t dirty_tiles;    /* tiles that held invalid UTF-8 (bytes dropped, utf8.cpp:130-147) */
  uint64_t long_segments;  /* segments longer than 256 bytes / a tile's window (matched from the raw text) */
  uint64_t kernel_launches;/* kernels launched by this call */
  uint64_t memo_hits;      /* segments settled by a word recorded earlier in the call (repeats of a word K2 matched) */
} wp_stats;

/* Message for the last non-OK status returned on the calling thread. */
const char *wp_last_error(void);

/* Number of CUDA kernels this library has launched in this process. */
uint64_t wp_kernel_launch_count(void);

/* Text bytes one thread block owns (the tile size of the encode kernel). */
uint32_t wp_tile_bytes(void);

/* ---- vocabulary ---------------------------------------------------------
 * Replaces utils::parseVocab (utils.cpp:108-121) + the WordPieceToken
 * constructor (utils.cpp:81-106) + the two-map build (fast.cpp:21-36), done
 * ONCE per vocabulary instead of once per encode call: id = index; "[UNK]"
 * (last such line) gives the UNK id, else -1; "##" prefix => continuation
 * token; "[...]" tokens and all-punctuation tokens of length > 1 are never
 * matched; duplicate tokens: the last index wins.  The table is uploaded to
 * `device` (CUDA ordinal).  device == -1 builds a HOST-ONLY handle (vocabulary
 * queries and wp_decode work; every encode call returns WP_ERR_NO_DEVICE). */
wp_status wp_vocab_create(const char *const *tokens, const size_t *token_lens, size_t n_tokens, int device,
                          wp_vocab **out);

/* Replaces utils::readVocabFromFile (utils.cpp:123-137): one token per line
 * ('\n' separated, a trailing '\r' stays in the token, an empty line is
 * WP_ERR_EMPTY_VOCAB_WORD). */
wp_status wp_vocab_create_from_file(const char *vocab_file, int device, wp_vocab **out);

void wp_vocab_destroy(wp_vocab *v);

size_t wp_vocab_size(const wp_vocab *v);        /* number of lines/tokens */
int32_t wp_vocab_unk_id(const wp_vocab *v);     /* WordPieceVocabulary::unk_token_id, utils.hpp:33 */
size_t wp_vocab_max_len(const wp_vocab *v);     /* max code points over matchable tokens, fast.cpp:31 */
int wp_vocab_device(const wp_vocab *v);
/* bit0 is_prefix, bit1 is_special, bit2 is_malformed (utils.hpp:23-25); bit3: token held invalid UTF-8 */
int wp_vocab_token_flags(const wp_vocab *v, size_t index);
/* Size in bytes of the device-resident tables (edge trie + static word table). */
size_t wp_vocab_device_bytes(const wp_vocab *v);

/* ---- encode -------------------------------------------------------------
 * All three replace encodeFastWordPiece (fast.cpp:143-150), i.e. parseText
 * (utils.cpp:37-79) + encodeFastWordPieceImpl (fast.cpp:19-141): UTF-8 text in,
 * int32 token ids out, bit-identical to the reference.  n_bytes == 0 => 0 ids. */

/* Host text -> host ids.  *ids_out is malloc'd by the library (wp_free). */
wp_status wp_encode(wp_vocab *v, const char *text, size_t n_bytes, int32_t **ids_out, size_t *n_ids);

/* Host text -> the ids as decimal text, every id followed by one space ("id id id "): the wire format that
 * encodeExternal appends to its output file (fast.cpp:214-216) and utils::writeToFile writes
 * (utils.cpp:30-35).  Formatted on the device.  *out is malloc'd by the library (wp_free), NUL-terminated,
 * *out_len excludes the NUL. */
wp_status wp_encode_text(wp_vocab *v, const char *text, size_t n_bytes, char **out, size_t *out_len, size_t *n_ids);

/* Host text -> caller's host buffer of `capacity` ids. */
wp_status wp_encode_into(wp_vocab *v, const char *text, size_t n_bytes, int32_t *ids, size_t capacity,
                         size_t *n_ids);

/* Device text -> device ids, both resident on the handle's device.  Enqueues
 * the kernels on `stream` (a cudaStream_t; NULL = the CUDA default stream),
 * then synchronises that stream to return the count.  At most `capacity` ids
 * are written; if more were produced the status is WP_ERR_CAPACITY and *n_ids
 * is the count needed (n_bytes ids always suffice). */
wp_status wp_encode_device(wp_vocab *v, const void *d_text, size_t n_bytes, int32_t *d_ids, size_t capacity,
                           size_t *n_ids, void *stream);

/* As above but fully asynchronous: the id count is written to the device
 * word *d_n_ids (uint64) and nothing is synchronised.  The internal scratch is sized for every text whose
 * segments longer than 256 bytes add up to at most the text size of one 64 MiB range; if a call outgrows it
 * *d_n_ids is UINT64_MAX and d_ids is incomplete — repeat the call through wp_encode_device, which retries
 * with a larger scratch.  Calls on one handle share its scratch: the library orders them with an event, so
 * they may be enqueued on different streams, but they never overlap. */
wp_status wp_encode_device_async(wp_vocab *v, const void *d_text, size_t n_bytes, int32_t *d_ids, size_t capacity,
                                 uint64_t *d_n_ids, void *stream);

/* ---- several GPUs ---------------------------------------------------------
 * The path shards with no exchange step: the reference itself cuts the code points into ranges at is_space
 * chars, encodes them on its pool threads and concatenates (fast.cpp:101-138).  Here the ranges are byte
 * ranges of the UTF-8 text, one per GPU, with a replicated vocabulary (one handle per device). */

/* Cuts of [0, n_bytes) into n_shards contiguous ranges of near-equal size: cuts[0] = 0, cuts[i] = the first
 * safe cut at or after n_bytes * i / n_shards, cuts[n_shards] = n_bytes (n_shards + 1 values; returns that
 * number).  Safe cuts: right after an is_space char (fast.cpp:113-115), and — for space-free CJK text — at a
 * punctuation char, right after one, or at a Han char (SURVEY A.2).  Pure host code. */
size_t wp_plan_shards(const char *text, size_t n_bytes, size_t n_shards, size_t *cuts);
/* The first safe cut at or after pos (n_bytes if there is none): what wp_plan_shards applies to every
 * nominal boundary.  Lets a rank that holds only its part of a corpus find its own shard borders. */
size_t wp_next_safe_cut(const char *text, size_t n_bytes, size_t pos);

typedef struct wp_shard {
  size_t begin, end;    /* byte range of the text */
  uint64_t n_ids;       /* ids of this shard */
  uint64_t id_offset;   /* exclusive scan of n_ids: where this shard's ids start in the global array */
  int device;           /* CUDA ordinal that encoded it */
  float encode_ms;      /* host wall clock of this shard's copy-in + kernels */
} wp_shard;

/* Host text -> host ids over n_handles GPUs (one handle per device, same vocabulary): wp_plan_shards, one
 * host thread per device (H2D + kernels, ids stay on the device), host exclusive scan of the counts, then
 * every device copies its ids to ids[id_offset ...).  `shards` (optional) receives n_handles entries.
 * The result is the id array of the whole text (fast.cpp:125-137). */
wp_status wp_encode_sharded(wp_vocab *const *handles, size_t n_handles, const char *text, size_t n_bytes, int32_t *ids,
                            size_t capacity, size_t *n_ids, wp_shard *shards);

/* Same, but the ids are gathered in DEVICE memory of handles[gather_index]'s GPU (d_ids, capacity ids): each
 * shard's ids travel peer to peer (NVLink) to d_ids + id_offset.  *gather_ms (optional): wall clock of the
 * gather alone. */
wp_status wp_encode_sharded_gather(wp_vocab *const *handles, size_t n_handles, const char *text, size_t n_bytes,
                                   size_t gather_index, int32_t *d_ids, size_t capacity, size_t *n_ids, wp_shard *shards,
                                   float *gather_ms);

/* Many texts in ONE call (SURVEY 8(f): the batch entry the reference lacks — it rebuilds its maps per call,
 * fast.cpp:154-157, :21-35).  Text i (texts[i], lens[i] bytes; may be empty) is encoded exactly as
 * fast::encode(texts[i], vocab) would encode it; its ids are ids[offsets[i] .. offsets[i + 1]), offsets has
 * n_texts + 1 entries and *n_ids = offsets[n_texts].  The texts are packed into one buffer and encoded by one
 * pass of the kernels; a large batch is cut into parts of whole texts that are packed, copied in, encoded and
 * copied back in a pipeline.  WP_ERR_CAPACITY (with *n_ids and offsets set) if capacity is short. */
wp_status wp_encode_batch(wp_vocab *v, const char *const *texts, const size_t *lens, size_t n_texts, int32_t *ids,
                          size_t capacity, size_t *offsets, size_t *n_ids);

/* Device string column -> device ids.  Text i is d_chars[d_offsets[i] .. d_offsets[i + 1]) (Arrow layout: n_texts + 1
 * uint64 offsets into a buffer of n_chars bytes; d_offsets[0] need not be 0).  Every text is encoded exactly as
 * fast::encode(text_i, vocab) would encode it.  Its ids are d_ids[d_id_offsets[i] .. d_id_offsets[i + 1]), and
 * d_id_offsets[n_texts] is the total.  Both offset arrays are in device memory of the handle's device.  The column
 * is packed on the device as wp_encode_batch packs host texts (n_chars + n_texts bytes) and encoded by one call of
 * the kernels on `stream` (NULL = the CUDA default stream), which is then synchronised.  WP_ERR_CAPACITY (with
 * *n_ids and d_id_offsets set) if capacity is short (n_chars ids always suffice); WP_ERR_INVALID_ARG if the offsets
 * do not ascend or end past n_chars.  n_texts == 0: d_id_offsets[0] = 0 and no kernel runs. */
wp_status wp_encode_batch_device(wp_vocab *v, const void *d_chars, size_t n_chars, const uint64_t *d_offsets,
                                 size_t n_texts, int32_t *d_ids, size_t capacity, uint64_t *d_id_offsets, size_t *n_ids,
                                 void *stream);

/* As above but fully asynchronous, with the contract of wp_encode_device_async: if the call outgrows its scratch,
 * or the column is malformed, d_id_offsets[n_texts] is UINT64_MAX and the ids are incomplete — repeat the call
 * through wp_encode_batch_device.  Host-side argument errors are reported at once. */
wp_status wp_encode_batch_device_async(wp_vocab *v, const void *d_chars, size_t n_chars, const uint64_t *d_offsets,
                                       size_t n_texts, int32_t *d_ids, size_t capacity, uint64_t *d_id_offsets,
                                       void *stream);

/* Counters of the last completed encode call on the handle (every encode entry point sets them; for a pipelined
 * call they are summed over its parts).  Decode calls (wp_decode, wp_decode_device[_async]) and row calls
 * (wp_rows_device[_async]) leave them as they are. */
wp_status wp_last_stats(wp_vocab *v, wp_stats *out);

/* Per-kernel device time (diagnostics for bench.py's roofline): when enabled, every following encode call
 * on the handle records CUDA events around its three kernels — K1 split + word-table lookup, K2 match,
 * K3 scan + scatter — on the stream the kernels are launched on.  wp_last_kernel_ms waits for the last
 * call and returns the summed milliseconds of each kernel over the call's ranges. */
wp_status wp_set_kernel_timing(wp_vocab *v, int enabled);
wp_status wp_last_kernel_ms(wp_vocab *v, float ms[3], uint32_t *n_ranges);

/* ---- decode -------------------------------------------------------------
 * Replaces word_piece::fast::decode (fast.cpp:165-187): id -> token text with
 * "##" re-added for continuation tokens.  The texts are concatenated into one
 * malloc'd buffer *out; token i is (*out)[(*offsets_out)[i] .. (*offsets_out)[i+1])
 * with *n_tokens + 1 offsets (both buffers: wp_free).  ids < 0 or > size and
 * malformed tokens are skipped (the reference prints a warning and skips them);
 * id == size is WP_ERR_ID_RANGE.  *n_skipped (optional) counts skipped ids. */
wp_status wp_decode(const wp_vocab *v, const int32_t *ids, size_t n_ids, char **out, size_t **offsets_out,
                    size_t *n_tokens, size_t *n_skipped);

/* Device ids -> device token strings (Arrow layout).  Entry i is the text fast::decode gives ids[i]
 * ("##" re-added for continuation tokens), or EMPTY where the reference skips the id (id < 0, id > size,
 * malformed token).  Entry i is d_chars[d_char_offsets[i] .. d_char_offsets[i + 1]); d_char_offsets has
 * n_ids + 1 uint64 entries, d_char_offsets[0] = 0.  No kept token decodes to zero bytes, so an empty entry means
 * exactly "skipped".  Because there is one entry per id, the d_id_offsets of wp_encode_batch_device index this
 * column directly: text t's tokens are entries d_id_offsets[t] .. d_id_offsets[t + 1].
 * Layout differs from wp_decode on purpose: wp_decode drops the skipped ids, this keeps one (empty) entry for
 * each, so the column stays aligned with the ids; dropping the empty entries gives wp_decode's output exactly.
 * The device decode table (every token's decoded bytes) is built and uploaded on a handle's first device decode
 * call and freed with the handle; it is not counted in wp_vocab_device_bytes.  It uses 32-bit offsets: a
 * vocabulary whose decoded tokens exceed 4 GiB in all gets WP_ERR_INVALID_ARG.
 * Synchronises `stream` (NULL = the default stream).  WP_ERR_ID_RANGE if any id == size (as wp_decode).
 * WP_ERR_CAPACITY if capacity < the bytes needed; then *n_chars holds that number and nothing is written
 * (d_chars may be NULL with capacity 0: a size query).  *n_skipped (optional) counts the empty entries.
 * Host-only handle: WP_ERR_NO_DEVICE.  n_ids == 0: d_char_offsets[0] = 0 and no kernel runs.
 * Calls on one handle are ordered with its encode calls (they share its scratch), on whatever streams. */
wp_status wp_decode_device(wp_vocab *v, const int32_t *d_ids, size_t n_ids, char *d_chars, size_t capacity,
                           uint64_t *d_char_offsets, size_t *n_chars, size_t *n_skipped, void *stream);

/* Fully asynchronous form, with the contract of wp_encode_device_async: d_char_offsets[n_ids] is the total byte
 * count, or UINT64_MAX if an id == size or the capacity is short.  In the UINT64_MAX case nothing is written past
 * `capacity` and the column is incomplete; repeat the call through wp_decode_device to get the status. */
wp_status wp_decode_device_async(wp_vocab *v, const int32_t *d_ids, size_t n_ids, char *d_chars, size_t capacity,
                                 uint64_t *d_char_offsets, void *stream);

/* ---- model-input rows ---------------------------------------------------
 * Per-text ids in device memory (e.g. the d_ids / d_id_offsets of wp_encode_batch_device) -> the fixed-length rows a
 * BERT-family model takes, in device memory.  Each row is max_len (L) int32 ids:
 *     [CLS]? content [SEP]? pad ... pad
 * SEP follows the content directly (not the end of the row); the mask row is 1 on the CLS, content and SEP positions
 * and 0 on the padding.  The content width is W = L - [CLS present] - [SEP present] and must be at least 1.
 *   stride == 0       truncate: one row per text, holding its first min(n_t, W) ids.
 *   1 <= stride <= W  overflow windows: a text of n_t ids has 1 row if n_t <= W, else 1 + ceil((n_t - W) / stride);
 *                     row k holds the text's ids [k * stride, min(k * stride + W, n_t)), so the last row ends at n_t.
 *                     `stride` is the distance between the STARTS of consecutive windows (cuDF subword_tokenize's
 *                     meaning); HuggingFace's `stride` is the overlap, W - stride here.
 * An empty text gives one row with no content.  Ids are copied verbatim, never interpreted (-1 stays -1). */
#define WP_ROWS_CLS 1u
#define WP_ROWS_SEP 2u
typedef struct wp_rows_spec {
  uint32_t max_len; /* L, special tokens included */
  uint32_t stride;  /* 0: truncate; else window starts `stride` content ids apart, 1 <= stride <= W */
  int32_t pad_id, cls_id, sep_id;
  uint32_t flags;   /* WP_ROWS_CLS | WP_ROWS_SEP: which of cls_id / sep_id the rows carry */
} wp_rows_spec;

/* Text t's ids are d_ids[d_id_offsets[t] .. d_id_offsets[t + 1]) (n_texts + 1 uint64 offsets that ascend and end at
 * most at n_ids; d_id_offsets[0] need not be 0).  Writes n_texts + 1 uint64 d_row_offsets: text t's rows are rows
 * d_row_offsets[t] .. d_row_offsets[t + 1] (d_row_offsets[0] = 0), which with the rule above describes every row.
 * Rows are row-major: row r is d_rows[r * L .. (r + 1) * L), mask row r is d_mask[r * L .. (r + 1) * L).  d_rows
 * holds row_capacity rows and may be any 4-byte-aligned pointer; d_mask (optional, NULL = no mask) holds as many
 * rows of L bytes at any alignment.
 * Synchronises `stream` (NULL = the default stream).  WP_ERR_INVALID_ARG for a null argument, a spec with W < 1, a
 * stride > W or unknown flags, a misaligned d_rows, row_capacity * L * 4 overflowing, or id offsets that descend
 * or end past n_ids (found on the device).  WP_ERR_CAPACITY if row_capacity < the rows needed: then *n_rows and
 * d_row_offsets are still exact and nothing is written to d_rows / d_mask (d_rows may be NULL with row_capacity 0:
 * a size query).  Host-only handle: WP_ERR_NO_DEVICE.  n_texts == 0: d_row_offsets[0] = 0, *n_rows = 0 and no
 * kernel runs.  Calls on one handle are ordered with its encode and decode calls (they share its scratch). */
wp_status wp_rows_device(wp_vocab *v, const int32_t *d_ids, size_t n_ids, const uint64_t *d_id_offsets, size_t n_texts,
                         const wp_rows_spec *spec, int32_t *d_rows, uint8_t *d_mask, size_t row_capacity,
                         uint64_t *d_row_offsets, size_t *n_rows, void *stream);

/* Fully asynchronous form, with the contract of wp_encode_device_async: d_row_offsets[n_texts] is the row total, or
 * UINT64_MAX if the id offsets are malformed or row_capacity is short.  In the UINT64_MAX case nothing is written to
 * d_rows / d_mask and the other offsets are unspecified; repeat the call through wp_rows_device for the status. */
wp_status wp_rows_device_async(wp_vocab *v, const int32_t *d_ids, size_t n_ids, const uint64_t *d_id_offsets,
                               size_t n_texts, const wp_rows_spec *spec, int32_t *d_rows, uint8_t *d_mask,
                               size_t row_capacity, uint64_t *d_row_offsets, void *stream);

void wp_free(void *p);

/* ---- test hooks (not part of the drop-in surface) -------------------------
 * Host mirror of the device longest-match query over the table image, and table
 * statistics; used by the CPU unit tests of the vocabulary builder. */
wp_status wp_debug_longest_match(const wp_vocab *v, const char *text, size_t window_bytes, int kind,
                                 uint32_t *len_out, int32_t *id_out);
size_t wp_debug_table_slots(const wp_vocab *v);
size_t wp_debug_table_nodes(const wp_vocab *v);
size_t wp_debug_long_tokens(const wp_vocab *v);
/* chunk plan of the host-buffer pipeline (cut offsets, first 0, last n); 0 if the text cannot be cut */
size_t wp_debug_plan_chunks(const char *text, size_t n, size_t chunk, size_t *cuts, size_t cap);
/* host-only run of the staging copies: mode 0/1 = the batch packer (ordinary / streaming stores), 2/3 = the
 * pooled copy of texts[0]; returns the bytes written to out */
size_t wp_debug_stage(const char *const *texts, const size_t *lens, size_t n, char *out, size_t out_cap, int mode);
/* code points of single-char word-initial tokens whose word-table slot lies at least min_displacement slots
 * from its home slot; returns their number */
size_t wp_debug_displaced_singles(const wp_vocab *v, uint32_t min_displacement, uint32_t *out, size_t cap);
/* word table: slots, static words, and the host mirror of K1's whole-segment lookup in the static image
 * (returns the id count, 0 = absent; ids_out takes up to 11 ids) */
size_t wp_debug_word_slots(const wp_vocab *v);
size_t wp_debug_static_words(const wp_vocab *v);
uint32_t wp_debug_word_lookup(const wp_vocab *v, const char *text, size_t len, int32_t *ids_out, uint32_t *displacement);
/* the limits the kernels were compiled with, in this order: tile bytes, LONG segment bytes, K1 segments per tile,
 * K3 segments per block, K3 staged ids per block, ids of a segment K3 copies warp-wise (more than this), K3 mixed-path
 * limit of such segments per block, K2L bytes per round, word-key bytes, ids of a word slot, the 5-bit id count
 * of a slow segment (at this value the count is in the slow entry), ids a slow entry holds inline.  Writes at most
 * `cap` of them to `out`; returns their number (no device needed) */
size_t wp_debug_kernel_geometry(uint32_t *out, size_t cap);

#ifdef __cplusplus
}
#endif
#endif /* WORDPIECE_B200_H_ */
