// Launch interface of the three encode kernels (wp_encode.cu).
//
//   K1 wp_split_kernel   word split + whole-window probe, one text tile per CTA
//   K2 wp_match_kernel   greedy longest-match chains of the segments K1 could
//                        not settle with one probe, load-balanced over the GPU
//   K2L wp_long_kernel   the same for the rare very long segments (URLs, blobs, texts without a space),
//                        one CTA per segment, matched from the raw text
//   K3 wp_scatter_kernel scan of per-segment id counts + scatter of the ids
//
// They run back to back on one stream over one RANGE of tiles of a text
// (a whole text, or a block of it when the host bounds the scratch memory);
// nothing is synchronised in between — K2 and K3 read their work sizes from
// device memory.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "wp_table.h"

namespace wp {

// One segment that K1's word-table lookup did not settle (16 bytes).
// K1 writes the WORK form below; K2 overwrites the entry with the RESULT form: word 0 = id count
// (| SLOW_RESULT_INLINE if at most three ids, which then sit in words 1..3), else word 1 = arena offset of the ids.
struct SlowEntry {
  uint32_t off;      // arena offset (in words) of the segment's area: `len` words for its ids, then its clean
                     // bytes in (len + 3) / 4 words (the last one zero padded).  LONG entries: id spill, set by K2.
  uint32_t meta;     // bits 0..15 byte length (0 for LONG), 16..17 char class of the first char,
                     // bit 18 LONG (leaves the tile window or longer than LONG_SEGMENT_BYTES: matched from the raw
                     // text in global memory), bits 24..31 raw text position bits 32..39 (LONG only)
  uint32_t pos_lo;   // raw text position of the segment start, low 32 bits (LONG only)
  uint32_t seg;      // the segment's number within the range: K2 puts the id count into seg_result[seg]
};
static_assert(sizeof(SlowEntry) == 16, "slow entries are read as one 16-byte load");

constexpr uint32_t SLOW_META_LONG = 1u << 18;
constexpr uint32_t SLOW_RESULT_INLINE = 0x80000000u;  // result form of an entry (after K2): word 0 = id count | this
// seg_result, one word per segment: settled by K1 with one id = id + 1 (< 2^30); slow = SEG_RESULT_SLOW |
// id count << 26 (31 = 31 or more: the count is in the slow entry; filled in by K2) | slow index; word-table
// hit with several ids = SEG_RESULT_WORD | id count << 26 | word slot.  K3 so knows every segment's id count
// without a dependent load.
constexpr uint32_t SEG_RESULT_SLOW = 0x80000000u;
constexpr uint32_t SEG_RESULT_WORD = 0x40000000u;
constexpr uint32_t SEG_SLOW_INDEX_BITS = 26;
constexpr uint32_t SEG_SLOW_INDEX_MASK = (1u << SEG_SLOW_INDEX_BITS) - 1u;
constexpr uint32_t SEG_SLOW_COUNT_MAX = 31;
constexpr uint32_t SEG_WORD_SLOT_BITS = 26;
constexpr uint32_t SEG_WORD_SLOT_MASK = (1u << SEG_WORD_SLOT_BITS) - 1u;

// Segments longer than this are matched from the raw text by the long-segment lane (one K2 lane would walk
// them byte by byte while its warp waits); it is also the halo a tile reads past its end.
constexpr uint32_t LONG_SEGMENT_BYTES = 256;

// The dynamic part of the word table pays only if words repeat (natural-language text); on text whose
// unsettled words never repeat (random strings, long CJK runs) K2 stops recording once enough lookups of
// the ranges >= 1 have shown that the recorded words settle less than 1/3 of the segments the static part
// leaves over (an atomic insert per miss and a dependent read in K3 per hit cost about that much).
// Judged once per range, by K2, for the ranges after it.  The first verdict (after range 1) sees a table
// that was warmed by 2 MiB only — English and Russian text hit 37 % there and 65-75 % later, Japanese 5 %,
// random strings 1 % — so it only asks for 1/6.  A heuristic on speed only: ids never depend on it.
__host__ __device__ inline bool memo_worthwhile(unsigned long long lookups, unsigned long long hits, bool early) {
  return !(lookups > 20000ull && hits * (early ? 6ull : 3ull) < lookups);
}

// Counters in device memory, zeroed before every range.
struct RangeCounters {
  unsigned int split_ticket;         // tile dispenser of K1
  unsigned int scatter_ticket;       // block dispenser of K3
  unsigned int n_slow;               // slow entries appended by K1
  unsigned int arena_reserved;       // arena words reserved by K1 (ids + clean bytes of the plain entries)
  unsigned int arena_spill;          // arena words reserved by K2L past the K1 part (ids of LONG entries)
  unsigned int n_long;               // LONG entries appended to long_list by K1
  unsigned int long_ticket;          // entry dispenser of K2L
  unsigned int pad;
  unsigned long long n_segs;         // segments of the range (K1, last tile)
};

// Counters in device memory, zeroed once per encode call.
struct CallCounters {
  unsigned long long ids_total[2];   // running id count; range r reads [r & 1] and writes [(r + 1) & 1]
  unsigned long long dirty_tiles;
  unsigned long long long_segments;
  unsigned int overflow;             // set if a scratch capacity was exceeded (the host retries with more)
  unsigned int stalled;              // set if a K1 look-back gave up waiting (the host retries in ticket mode)
  unsigned long long memo_hits;      // segments settled in K1 by a word that K2 recorded during this call
  unsigned long long memo_lookups;   // those + the segments K1 left to K2, in ranges >= 1 (range 0 cannot hit)
  unsigned int dense;                // set if a K1 tile held more segments than its lists (the host retries with the full-capacity K1)
  unsigned int pad2[17];             // (the counters above are hit by atomics from every tile)
  unsigned int memo_off;             // set by K2 once recording has shown not to pay (memo_worthwhile)
  unsigned int pad3[31];
};
static_assert(offsetof(CallCounters, memo_off) % 128 == 0, "memo_off sits in a cache line of its own");

struct EncodeParams {
  DeviceVocab vocab;
  const uint8_t *text;              // device, the whole text (tiles read their halo from it)
  size_t n_bytes;                   // size of the whole text
  uint32_t first_tile;              // range = tiles [first_tile, first_tile + n_tiles)
  uint32_t n_tiles;
  // outputs
  int32_t *ids;                     // device, capacity entries
  unsigned long long capacity;
  CallCounters *call;               // K3 appends at call->ids_total[range_parity]
  uint32_t range_parity;
  // scratch
  RangeCounters *counters;
  unsigned long long *tile_state;   // n_tiles look-back words (K1), zeroed
  unsigned long long *block_state;  // look-back words of K3, zeroed
  uint32_t *seg_result;             // seg_capacity entries
  uint32_t seg_capacity;
  SlowEntry *slow;                  // slow_capacity entries
  uint32_t slow_capacity;
  uint32_t *long_list;              // long_capacity slow-list indices of the LONG entries (K2L's work list)
  uint32_t long_capacity;
  uint32_t *arena;                  // arena_capacity words: per slow segment its id scratch and its clean bytes
  uint32_t arena_capacity;
  uint32_t n_scatter_blocks;        // size of block_state
  WordSlot *words;                  // the word table of this call: the static image (small calls), or a larger
                                    // working table seeded from it that K2 records into
  uint32_t word_mask;               // its slots - 1
  uint32_t word_shift;              // 32 - log2(slots)
  uint32_t record_words;            // K2 records the words it matches (working table only)
  uint32_t range_index;             // 0, 1, 2, ... within the call
  uint32_t use_ticket;              // K1 takes its tiles from RangeCounters::split_ticket instead of blockIdx.x
  uint32_t dense_tiles;             // K1 with full-capacity segment lists (seven tiles per SM instead of eight)
  // batch of texts in one buffer (wp_encode_batch), else bounds = nullptr: bounds[i] = byte offset at which
  // text i starts (ascending, each preceded by a space); tile_bound[t] = index of the first text that starts in
  // absolute tile t or later (n_tiles_total + 1 entries); K1 writes bound_seg[i] = the number, within the
  // range, of the first segment that starts at or after bounds[i]; K5 turns that into id_offsets[i]
  const unsigned long long *bounds;
  const uint32_t *tile_bound;
  uint32_t *bound_seg;
  unsigned long long *id_offsets;
  // L2 residency hint (0 bytes = none): K1 and K3 keep the word table, K2 the edge table
  size_t persist_words_bytes, persist_edges_bytes;
  float persist_words_ratio, persist_edges_ratio;
};

// Zero-filled working table <- every word of the static image (re-hashed for the working table's size).
cudaError_t launch_seed_words(const WordSlot *image, uint32_t image_slots, WordSlot *work, uint32_t work_slots_log2,
                              cudaStream_t stream, uint64_t *launches);

// *d_out <- the id count of the call whose counters are `call` (UINT64_MAX if its scratch overflowed, or if
// `invalid` is given and *invalid is set).
cudaError_t launch_publish_count(const CallCounters *call, uint32_t parity, unsigned long long *d_out, cudaStream_t stream,
                                 uint64_t *launches, const unsigned int *invalid = nullptr);

// K5 (batch calls): id_offsets[i] = index of the first id of text i, for the texts [i0, i1) that start in the
// range whose K3 has just run on `stream` (same EncodeParams).
cudaError_t launch_text_offsets(const EncodeParams &P, uint32_t i0, uint32_t i1, cudaStream_t stream, uint64_t *launches);
// The same for the texts [tile_bound[first_tile], tile_bound[first_tile + n_tiles]), read on the device.
cudaError_t launch_text_offsets_device(const EncodeParams &P, int sm_count, cudaStream_t stream, uint64_t *launches);

// A string column in device memory (wp_encode_batch_device) and the packed text it becomes.
struct ColumnArgs {
  const uint8_t *chars;              // the column's chars, any alignment
  unsigned long long n_chars;
  const unsigned long long *offsets; // n_texts + 1 entries: text i = chars[offsets[i] .. offsets[i + 1])
  uint32_t n_texts;
  uint32_t n_tiles;                  // tiles of the packed text
  unsigned int *bad;                 // zeroed; set by the check if the offsets do not ascend within [0, n_chars]
  uint8_t *text;                     // n_tiles whole tiles, 16-byte aligned: the packed texts, then spaces
  unsigned long long *bounds;        // n_texts: where text i starts in `text` (EncodeParams::bounds)
  uint32_t *tile_bound;              // n_tiles + 1 (EncodeParams::tile_bound)
};
// The column check (one thread per text) and the packer (one CTA per tile of the packed text).
cudaError_t launch_column_pack(const ColumnArgs &A, cudaStream_t stream, uint64_t *launches);

uint32_t encode_tile_bytes();
uint32_t scatter_block_segments();
// The compiled limits of the kernels, in the order of wp_debug_kernel_geometry (wordpiece_b200.h); returns their
// number and writes at most `cap` of them.
size_t kernel_geometry(uint32_t *out, size_t cap);
// Enqueue the kernels of one range (K1, K2 + K2L, K3).  *launches is incremented per kernel launched.
// `timing` (optional): 4 events recorded around the launches (before K1, K1|K2, K2+K2L|K3, after K3).
cudaError_t launch_encode_range(const EncodeParams &P, int sm_count, cudaStream_t stream, uint64_t *launches,
                                cudaEvent_t *timing = nullptr);

// ids -> "id id id " (decimal, one space after every id).  launch_format_total adds the text length to *total
// (zeroed by the caller); launch_format writes it to `out` (block_state: one zeroed word per
// format_block_ids() ids, ticket: one zeroed word).
uint32_t format_block_ids();
cudaError_t launch_format_total(const int32_t *ids, size_t n, unsigned long long *total, int sm_count, cudaStream_t stream,
                                uint64_t *launches);
cudaError_t launch_format(const int32_t *ids, size_t n, char *out, unsigned long long *block_state, unsigned int *ticket,
                          int sm_count, cudaStream_t stream, uint64_t *launches);

}  // namespace wp
