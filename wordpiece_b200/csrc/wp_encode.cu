// WordPiece encode kernels for sm_100a: word split -> longest match -> scan +
// scatter.  Text is read from HBM once (plus the bytes of the ~20 % of words
// that need more than one probe); ids are written once; the intermediates are a
// 4-byte result per segment and a 16-byte entry per unsettled segment.
//
// What they reproduce (gleb-kov/wordpiece, see SURVEY.md Appendix A):
//   utils.cpp:37-79 / utf8.cpp:130-147   strict UTF-8 decode, invalid bytes dropped
//   utf8.cpp:10-29                       space / punctuation / Han classes
//   fast.cpp:38-41                       word-initial positions
//   fast.cpp:43-99                       the greedy longest-match worker with
//                                        whole-word UNK roll-back
//   fast.cpp:101-138                     chunk + concat (here: tiles + decoupled
//                                        look-back scans)
//
// K1 wp_split_kernel (one 4 KB tile per CTA)
//   S1 split : the tile + halo is staged in shared memory with 16-byte loads;
//              each thread classifies a 32-byte chunk into bit masks (valid lead
//              / space / punct / Han) with SWAR arithmetic; tiles holding invalid
//              UTF-8 are compacted in shared memory; segment starts and ends
//              ("safe starts", SURVEY A.2) fall out of mask operations and are
//              compacted into lists in text order.
//   S2 lookup: one lookup per segment (<= 16 bytes) in the WORD TABLE
//              (wp_table.h): whole segment bytes -> ids.  Its static part holds
//              every word-initial token (a segment that is a token is that token,
//              ~80 % of English words), its dynamic part the words K2 matched
//              earlier in this call.  Uniform work for every lane.  The rest go
//              to the global slow list together with their clean bytes.
// K2 wp_match_kernel (whole GPU, no tiles, no barriers)
//   S2b match: every lane owns many slow segments and runs the greedy matcher as
//              a FLATTENED state machine over the EDGE TRIE — one trie step (one
//              char, a 16-byte load) per loop iteration — so a warp stays converged on
//              the step and chains of very different length average out over a
//              lane's share.  Segments that left their tile's window or are very
//              long are matched from the raw text in global memory.
// K3 wp_scatter_kernel
//   S3 scatter: per-segment id counts -> block scan -> decoupled look-back ->
//              ids staged in shared memory and written out coalesced.
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "wp_encode.h"
#include "wp_table.h"

// Debug build (make variant NAME=bounds DEFS=-DWP_DEBUG_BOUNDS): every index into the scratch arrays, the lists in
// shared memory and the output is checked where it is used; a violation prints its place and traps.  The
// parity suites and the fuzz sweep are run under this build once per round (tools/gpu_bounds.sh).
#ifdef WP_DEBUG_BOUNDS
#include <cstdio>
#define WP_CHECK(cond)                                                                                              \
  do {                                                                                                              \
    if (!(cond)) {                                                                                                  \
      printf("WP_CHECK failed: %s (wp_encode.cu:%d, block %d, thread %d)\n", #cond, __LINE__, static_cast<int>(blockIdx.x), \
             static_cast<int>(threadIdx.x));                                                                        \
      __trap();                                                                                                     \
    }                                                                                                               \
  } while (0)
#else
#define WP_CHECK(cond) \
  do {                 \
  } while (0)
#endif

namespace wp {

// ------------------------------------------------------------------ geometry
constexpr int TILE = 4096;                       // text bytes owned by one CTA of K1
constexpr int CHUNK = 32;                        // bytes classified by one thread
constexpr int THREADS = 160;                     // K1: 5 warps
constexpr int HALO = 256;                        // classified bytes past the tile (segment completion)
constexpr int LOOKAHEAD = 32;                    // loaded, not classified (UTF-8 validation look-ahead)
constexpr int LEFT = 16;                         // bytes before the tile (ownership of leading continuation bytes)
constexpr int WINDOW = TILE + HALO;              // classified window
constexpr int NCHUNK = WINDOW / CHUNK;           // 136
constexpr int OWNED_CHUNKS = TILE / CHUNK;       // 128
constexpr int RAW_BYTES = LEFT + WINDOW + LOOKAHEAD;  // 4400
constexpr int WARPS = THREADS / 32;
constexpr int MAX_TILE_SLOW = TILE / 2 + 8;      // slow segments have >= 2 bytes
constexpr int PREFETCH_TILES = 2 * 6 * 148;      // K1 pulls the text of the tile this far ahead into L2
constexpr uint32_t FULL = 0xFFFFFFFFu;
constexpr uint32_t POS_MASK = 0x3FFFu;           // window positions fit 14 bits
constexpr uint32_t SLOW_LONG = 0x8000u;          // tile slow-list flag: matched from the raw text (leaves the window / very long)

// tuning knobs (make variant DEFS=...)
#ifndef WP_K2_BLOCKS
#define WP_K2_BLOCKS 5                           // K2 CTAs per SM (launch bound and grid); 5 x 8 warps x 48 registers fill the register file (4: +3 %, 6 spills: +5 %)
#endif
#ifndef WP_K2_THREADS
#define WP_K2_THREADS 256
#endif
#ifndef WP_K1_PER_TURN
#define WP_K1_PER_TURN 2                         // word-table lookups in flight per lane
#endif
#ifndef WP_K3_BLOCKS
#define WP_K3_BLOCKS 4
#endif
#ifndef WP_K1_SEG_CAP
#define WP_K1_SEG_CAP 3072                       // segments per tile the lists of the regular K1 hold (see TileSmemT)
#endif
constexpr int MATCH_THREADS = WP_K2_THREADS;     // K2
constexpr int SCATTER_THREADS = 256;             // K3
constexpr int SCATTER_ITEMS = 8;                 // segments per thread and block iteration
constexpr int SCATTER_SEGS = SCATTER_THREADS * SCATTER_ITEMS;  // 2048
constexpr int SCATTER_STAGE = 6144;              // ids staged in shared memory per block iteration
#ifndef WP_SCATTER_BIG
#define WP_SCATTER_BIG 8
#endif
constexpr int SCATTER_BIG = WP_SCATTER_BIG;      // a segment with more ids (a long word, a URL, a blob) is copied by a whole warp

static_assert(RAW_BYTES % 16 == 0, "raw buffer is loaded in 16-byte units");
static_assert(WORD_KEY_BYTES + 4 <= LOOKAHEAD, "key window reads stay inside the loaded bytes");
static_assert(LONG_SEGMENT_BYTES <= HALO, "a segment that starts in the tile and is not LONG ends inside the window");
static_assert(NCHUNK + 1 <= THREADS, "one thread per chunk in the classification and compaction passes");
static_assert(WINDOW <= static_cast<int>(POS_MASK), "positions must fit the packed list entries");
static_assert(TILE <= 4096, "segment ordinals must fit 12 bits of the tile slow list");
static_assert(NCHUNK < 256, "chunk indices are kept in bytes (hi_list)");

// The segment lists are sized for SEG_CAP owned segments.  A tile CAN hold TILE of them (every byte a
// punctuation char), but text does not: with 3 072 a tile's shared memory shrinks enough for EIGHT tiles per
// SM instead of seven (K1 -4.4 %, profiles/r2g_variants.txt).  A tile that holds more flags the call as
// "dense"; the call is void and the host repeats it with the full-capacity instantiation (sticky per handle).
template <int SEG_CAP>
struct __align__(16) TileSmemT {
  uint8_t raw[RAW_BYTES];              // [0,LEFT) left halo, then the window, then look-ahead
  uint16_t seg_s[SEG_CAP];             // owned segment k (text order): start position | class << 14
  uint16_t seg_e[SEG_CAP + HALO + 64]; // j-th segment end in the window
  uint16_t slow[MAX_TILE_SLOW];        // segments the whole-window probe did not settle: ordinal | flags
  uint32_t dyn_hits;                   // segments settled by a word K2 recorded during this call
  uint32_t n_eligible;                 // slow segments short enough for the word table (recording statistics)
  uint32_t any_single;                 // some single-char segment is still to be settled (see S2)
  uint32_t m_lead[NCHUNK + 1];         // valid lead bytes
  uint32_t m_space[NCHUNK + 1];
  uint32_t m_punct[NCHUNK + 1];
  uint32_t m_han[NCHUNK + 1];
  uint32_t m_cover[NCHUNK + 1];        // bytes covered by a valid sequence that starts in this chunk
  uint32_t m_kept[NCHUNK + 1];         // bytes of the RAW window that survive the strict decoder (dirty tiles)
  uint32_t kept_scan[NCHUNK + 2];      // exclusive scan of kept bytes per chunk (dirty tiles)
  uint8_t spill[NCHUNK + 1];           // bytes by which the chunk's last sequence runs into the next chunk
  uint8_t hi_list[NCHUNK + 8];         // chunks that hold a byte >= 0x80 (classification pass 2)
  uint32_t n_hi;
  uint32_t tile_ticket;                // ticket mode: the tile this CTA took
  uint4 key_mask[WORD_KEY_BYTES + 1];  // row k: byte masks of the four key words for a k-byte key
  uint32_t warp_sums[WARPS];
  uint32_t prev_class;                 // class of the last valid char before the tile
  uint32_t left_spill;                 // bytes of the tile start covered by a sequence that began before it
  uint32_t n_segs;                     // owned segments in this tile
  uint32_t n_ends;                     // segment ends found in the window
  uint32_t n_slow;                     // entries of slow[]
  uint32_t slow_base;                  // first global slow index of this tile
  uint32_t arena_base;                 // first arena word reserved for this tile
  unsigned long long seg_base;         // segments of all earlier tiles of the range
};

static_assert(sizeof(TileSmemT<TILE>) + 1024 <= 233472 / 7, "seven full-capacity K1 tiles must fit one SM's shared memory");
static_assert(sizeof(TileSmemT<WP_K1_SEG_CAP>) + 1024 <= 233472 / 8, "eight regular K1 tiles must fit one SM's shared memory");
static_assert(WP_K1_SEG_CAP <= TILE && WP_K1_SEG_CAP % 8 == 0, "list capacity");

// ------------------------------------------------------------------- helpers

// Streaming 16-byte load of text: not kept in L1 (and through the coherent path: the buffers the text lives in are
// rewritten between calls).
__device__ __forceinline__ uint4 ldg_stream(const uint4 *p) {
  uint4 r;
  asm volatile("ld.global.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

__device__ __forceinline__ uint32_t ld_u32(const uint8_t *p) { return *reinterpret_cast<const uint32_t *>(p); }

// Shared-memory add by ONE lane that already speaks for its warp (ballot + popc done by the caller).  Plain
// atomicAdd() here makes the compiler wrap its own warp aggregation (vote, flo, popc, shfl: 16 instructions)
// around the single active lane.
__device__ __forceinline__ uint32_t smem_add(uint32_t *p, uint32_t v) {
  uint32_t old;
  asm volatile("atom.shared.add.u32 %0, [%1], %2;"
               : "=r"(old)
               : "r"(static_cast<uint32_t>(__cvta_generic_to_shared(p))), "r"(v)
               : "memory");
  return old;
}
__device__ __forceinline__ void smem_add_noret(uint32_t *p, uint32_t v) {
  asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(static_cast<uint32_t>(__cvta_generic_to_shared(p))), "r"(v) : "memory");
}

__device__ __forceinline__ void prefetch_l1(const void *p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// The first 32 bytes of a word-table slot (key, meta, ids 0..2) with ONE 256-bit load (sm_100: LDG.E.256)
// through the read-only path.  Writers (K2) and readers (K1, K3) of a slot run in different kernels.
__device__ __forceinline__ void ld_word_slot(const WordSlot *tab, uint32_t idx, uint4 *a, uint4 *b) {
  asm volatile("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(a->x), "=r"(a->y), "=r"(a->z), "=r"(a->w), "=r"(b->x), "=r"(b->y), "=r"(b->z), "=r"(b->w)
               : "l"(tab + idx));
}

// 0x80 in every byte lane whose (7-bit) value lies in [lo, hi]; lanes must be < 0x80.
__device__ __forceinline__ uint32_t swar_range(uint32_t w, uint32_t lo, uint32_t hi) {
  const uint32_t ge_lo = w + (0x80808080u - lo * 0x01010101u);
  const uint32_t gt_hi = w + (0x80808080u - (hi + 1u) * 0x01010101u);
  return ge_lo & ~gt_hi & 0x80808080u;
}

// gather the four 0x80 flags of a word into a nibble (lane 0 -> bit 0)
__device__ __forceinline__ uint32_t swar_nibble(uint32_t flags) { return (((flags >> 7) * 0x01020408u) >> 24) & 0xFu; }

// Class of a decoded char from its UTF-8 bytes (valid sequence of length len).
__device__ __forceinline__ uint32_t class_of(uint32_t cp) { return cp_class(cp); }

// ------------------------------------------------------------------ trie step

// One descent step: the edge (node, char), or false.  e = {parent, char, child | flags, term_id}.
__device__ __forceinline__ bool trie_step(const DeviceVocab &V, uint32_t node, uint32_t ch, uint4 *e) {
  const uint4 *tab = reinterpret_cast<const uint4 *>(V.edges);
  uint32_t idx = edge_hash(node, ch, V.edge_shift);
  uint4 v = __ldg(tab + idx);
  while (!(v.x == node && v.y == ch) && v.x != EDGE_EMPTY) {  // linear probing, load factor <= 0.25
    idx = (idx + 1) & V.edge_mask;
    v = __ldg(tab + idx);
  }
  *e = v;
  return v.x == node;  // (a node number is never EDGE_EMPTY)
}
__device__ __forceinline__ uint32_t edge_child(const uint4 &e) { return e.z & EDGE_CHILD_MASK; }
__device__ __forceinline__ bool edge_extends(const uint4 &e) { return (e.z & EDGE_HAS_CHILDREN) != 0; }
__device__ __forceinline__ int32_t edge_term(const uint4 &e) { return static_cast<int32_t>(e.w); }

// ------------------------------------------- raw-text lane (long segments, K2L)
// Decoding and matching straight from the text in global memory, dropping invalid
// bytes on the fly: for segments that leave their tile's window or are very long.

struct TextView {
  const uint8_t *t;
  size_t n;
};

// Decode the char at pos; returns its length (0 = invalid byte) and class.
__device__ uint32_t gdecode(const TextView &tv, size_t pos, uint32_t *cls) {
  const size_t rem = tv.n - pos;
  const uint32_t b0 = tv.t[pos];
  if (b0 < 0x80u) {
    *cls = cp_class(b0);
    return 1;
  }
  const uint32_t b1 = rem > 1 ? tv.t[pos + 1] : 0u;
  const uint32_t b2 = rem > 2 ? tv.t[pos + 2] : 0u;
  const uint32_t b3 = rem > 3 ? tv.t[pos + 3] : 0u;
  uint32_t cp = 0;
  const uint32_t len = utf8_decode(b0, b1, b2, b3, rem > 4 ? 4u : static_cast<uint32_t>(rem), &cp);
  if (len) *cls = cp_class(cp);
  return len;
}

// First valid lead at or after pos (n if none); returns its length and class.
__device__ size_t gnext(const TextView &tv, size_t pos, uint32_t *len, uint32_t *cls) {
  while (pos < tv.n) {
    const uint32_t l = gdecode(tv, pos, cls);
    if (l) {
      *len = l;
      return pos;
    }
    pos++;
  }
  *len = 0;
  *cls = CLS_SPACE;
  return tv.n;
}

// Class of the last valid char that starts before pos (SPACE at the text start).
__device__ uint32_t gprev_class(const TextView &tv, size_t pos) {
  size_t p = pos;
  while (p > 0) {
    size_t q = p - 1;
    while (q > 0 && is_cont_byte(tv.t[q])) q--;
    if (!is_cont_byte(tv.t[q])) {
      uint32_t cls;
      if (gdecode(tv, q, &cls)) return cls;
    }
    p = q;
  }
  return CLS_SPACE;
}

// Longest match for the window that starts at the valid lead `p` (first char of
// any non-space class, then ordinary chars only).  Returns the raw text position
// right behind the match (p itself: no match) and the token id.
__device__ size_t longest_match_global(const DeviceVocab &V, const TextView &tv, size_t p, uint32_t kind, int32_t *id) {
  uint32_t node = kind;
  size_t q = p, best = p;
  bool first = true;
  while (q < tv.n) {
    uint32_t len, cls;
    q = gnext(tv, q, &len, &cls);
    if (q >= tv.n || (!first && cls != CLS_OTHER)) break;
    uint4 e;
    uint32_t ch = 0;
    for (uint32_t i = 0; i < len; i++) ch |= static_cast<uint32_t>(tv.t[q + i]) << (8 * i);
    if (!trie_step(V, node, ch, &e)) break;
    node = edge_child(e);
    q += len;
    if (edge_term(e) != WP_NO_ID) {
      best = q;
      *id = edge_term(e);
    }
    if (!edge_extends(e) || (first && cls == CLS_PUNCT)) break;
    first = false;
  }
  return best;
}

// The char at pos as its packed UTF-8 bytes (the edge trie's key); returns its length, 0 = invalid byte.  No class
// is computed: for text whose chars are known to be ordinary (inside a long segment, whose end has been found).
__device__ __forceinline__ uint32_t gchar(const TextView &tv, size_t pos, uint32_t *ch) {
  const uint32_t b0 = tv.t[pos];
  if (b0 < 0x80u) {
    *ch = b0;
    return 1;
  }
  const size_t rem = tv.n - pos;
  const uint32_t b1 = rem > 1 ? tv.t[pos + 1] : 0u;
  const uint32_t b2 = rem > 2 ? tv.t[pos + 2] : 0u;
  const uint32_t b3 = rem > 3 ? tv.t[pos + 3] : 0u;
  uint32_t cp = 0;
  const uint32_t len = utf8_decode(b0, b1, b2, b3, rem > 4 ? 4u : static_cast<uint32_t>(rem), &cp);
  *ch = edge_char(b0 | (b1 << 8) | (b2 << 16) | (b3 << 24), len);
  return len;
}

// longest_match_global for a window inside a long segment: every valid char before tv.n (the segment's end) is an
// ordinary char, so the walk only skips invalid bytes and never looks at classes.
__device__ size_t longest_match_inside(const DeviceVocab &V, const TextView &tv, size_t p, uint32_t kind, int32_t *id) {
  uint32_t node = kind;
  size_t q = p, best = p;
  while (q < tv.n) {
    uint32_t ch;
    const uint32_t len = gchar(tv, q, &ch);
    if (len == 0) {  // dropped by the strict decoder (utf8.cpp:130-147)
      q++;
      continue;
    }
    uint4 e;
    if (!trie_step(V, node, ch, &e)) break;
    node = edge_child(e);
    q += len;
    if (edge_term(e) != WP_NO_ID) {
      best = q;
      *id = edge_term(e);
    }
    if (!edge_extends(e)) break;
  }
  return best;
}

// ------------------------------------------------------------- classification

// exact: 0x80 in every byte lane whose byte is zero
__device__ __forceinline__ uint32_t swar_zero(uint32_t x) {
  return ~(((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x | 0x7F7F7F7Fu);
}

// flags of the byte lane d (1..3) positions earlier: lane j gets cur/prev lane j-d
__device__ __forceinline__ uint32_t lanes_back(uint32_t prev, uint32_t cur, int d) {
  return __funnelshift_l(prev, cur, 8 * d);
}

struct WordFlags {
  uint32_t cont;     // 10xxxxxx
  uint32_t m1;       // 11xxxxxx  (any multi-byte lead)
  uint32_t m2;       // 111xxxxx
  uint32_t m3;       // 1111xxxx
  uint32_t suspect;  // leads whose validity depends on their value: C0 C1 E0 ED F0..FF
};

__device__ __forceinline__ WordFlags word_flags(uint32_t w) {
  WordFlags f;
  const uint32_t hi = w & 0x80808080u;
  const uint32_t t1 = w << 1, t2 = w << 2, t3 = w << 3;
  f.cont = hi & ~t1;
  f.m1 = hi & t1;
  f.m2 = f.m1 & t2;
  f.m3 = f.m2 & t3;
  const uint32_t lead2 = f.m1 & ~t2;
  const uint32_t lead3 = f.m2 & ~t3;
  const uint32_t low = w & 0x0F0F0F0Fu;
  f.suspect = f.m3 | (lead2 & swar_zero(w & 0x1E1E1E1Eu)) | (lead3 & (swar_zero(low) | swar_zero(low ^ 0x0D0D0D0Du)));
  return f;
}

// Classification of the window into the mask arrays, in two passes.  `limit` is the number of meaningful
// bytes in buf (positions >= limit are ignored).
//
// Pass 1, every chunk: the ASCII classes by SWAR range tests, and whether the chunk holds any byte >= 0x80.
// Pass 2, only the chunks that do, COMPACTED into a list so that all lanes of a warp are busy (in
// English-like text one chunk in eight holds a non-ASCII byte; run in place, those few lanes made their
// whole warp execute the pass): multi-byte text is validated STRUCTURALLY (every lead followed by exactly its
// continuation bytes) with byte-lane shifts; only leads that can be space / punctuation / Han (C2, E2..E9,
// EF) are decoded.  Chunks holding a lead whose validity depends on its value (overlong / surrogate /
// 4-byte forms) or any structural error take the exact per-byte lane.
__device__ __forceinline__ uint32_t limit_mask(int c, int limit) {
  const int left = limit - c * CHUNK;
  return left >= CHUNK ? 0xFFFFFFFFu : (left <= 0 ? 0u : ((1u << left) - 1u));
}

template <class TileSmem>
__device__ __forceinline__ bool classify_ascii(TileSmem &sm, const uint8_t *buf, int c, int limit) {
  const uint8_t *cb = buf + c * CHUNK;
  uint32_t sp = 0, pu = 0, any_high = 0;
  // (the loops over the chunk's eight words are deliberately NOT fully unrolled: K1's executed code must fit
  // the SM's 32 KB instruction cache — the tiles resident on an SM are in different phases — and these loops
  // alone were a sixth of it; the words are re-read from shared memory where they are needed)
#pragma unroll 2
  for (int i = 0; i < 8; i++) {
    const uint32_t wi = ld_u32(cb + 4 * i);
    const uint32_t w7 = wi & 0x7F7F7F7Fu;
    const uint32_t asc = ~wi & 0x80808080u;
    const uint32_t s = (swar_range(w7, 0x09, 0x0D) | swar_range(w7, 0x20, 0x20)) & asc;
    const uint32_t q = (swar_range(w7, 0x21, 0x2F) | swar_range(w7, 0x3A, 0x40) | swar_range(w7, 0x5B, 0x60) |
                        swar_range(w7, 0x7B, 0x7E)) & asc;
    sp |= swar_nibble(s) << (4 * i);
    pu |= swar_nibble(q) << (4 * i);
    any_high |= wi;
  }
  const uint32_t in = limit_mask(c, limit);
  sm.m_space[c] = sp & in;
  sm.m_punct[c] = pu & in;
  const bool high = (any_high & 0x80808080u) != 0;
  if (!high) {
    sm.m_lead[c] = in;
    sm.m_han[c] = 0;
    sm.m_cover[c] = 0xFFFFFFFFu;
    sm.spill[c] = 0;
  }
  return high;
}

template <class TileSmem>
__device__ __forceinline__ void classify_multibyte(TileSmem &sm, const uint8_t *buf, int c, int limit) {
  const uint8_t *cb = buf + c * CHUNK;
  uint32_t lead = 0xFFFFFFFFu, sp = sm.m_space[c], pu = sm.m_punct[c], ha = 0, cover = 0xFFFFFFFFu, spill = 0;
  // ---- structural validation in the byte-lane domain
  WordFlags prev = word_flags(ld_u32(cb - 4));
  // (a lead in the four bytes before the chunk that already misses a continuation byte THERE is invalid, and
  // the continuation bytes it would have owned at the start of this chunk are strays: the per-position
  // expectation below cannot see that, e.g. E2 's' | 80)
  uint32_t bad = prev.suspect | (((prev.m1 << 8) | (prev.m2 << 16) | (prev.m3 << 24)) & ~prev.cont & 0x80808080u);
  uint32_t contm = 0, cand = 0;
#pragma unroll 1
  for (int i = 0; i < 8; i++) {
    const uint32_t wi = ld_u32(cb + 4 * i);
    const WordFlags f = word_flags(wi);
    const uint32_t expect = lanes_back(prev.m1, f.m1, 1) | lanes_back(prev.m2, f.m2, 2) | lanes_back(prev.m3, f.m3, 3);
    bad |= (expect ^ f.cont) | f.suspect;
    contm |= swar_nibble(f.cont) << (4 * i);
    // leads that may be a spacing char: C2 (Latin-1 punctuation), E2 (U+2010.., U+2581), E3..E9, EF (Han)
    const uint32_t low = wi & 0x0F0F0F0Fu;
    const uint32_t lead3 = f.m2 & ~(wi << 3);
    const uint32_t cf = swar_zero(wi ^ 0xC2C2C2C2u) | (lead3 & (swar_range(low, 2, 9) | swar_zero(low ^ 0x0F0F0F0Fu)));
    cand |= swar_nibble(cf) << (4 * i);
    prev = f;
  }
  {
    // sequences that run past the chunk must find their continuation bytes in the next word
    const WordFlags nx = word_flags(ld_u32(cb + CHUNK));
    const uint32_t expect = lanes_back(prev.m1, 0u, 1) | lanes_back(prev.m2, 0u, 2) | lanes_back(prev.m3, 0u, 3);
    bad |= expect & ~nx.cont;
    spill = __popc(expect);
  }
  if (bad == 0) {
    lead = ~contm;
    while (cand) {
      const int j = __ffs(cand) - 1;
      cand &= cand - 1;
      const uint32_t b0 = cb[j], b1 = cb[j + 1], b2 = cb[j + 2];
      const uint32_t cp = b0 < 0xE0u ? (((b0 & 0x1Fu) << 6) | (b1 & 0x3Fu))
                                     : (((b0 & 0x0Fu) << 12) | ((b1 & 0x3Fu) << 6) | (b2 & 0x3Fu));
      const uint32_t cls = cp_class(cp);
      sp |= (cls == CLS_SPACE ? 1u : 0u) << j;
      pu |= (cls == CLS_PUNCT ? 1u : 0u) << j;
      ha |= (cls == CLS_HAN ? 1u : 0u) << j;
    }
  } else {
    // ---- exact per-byte lane (utf8.cpp:54-90): overlongs, surrogates, 4-byte forms, stray bytes
    lead = 0;
    cover = 0;
    spill = 0;
    sp = 0;
    pu = 0;
    for (int j = 0; j < CHUNK; j++) {
      const uint32_t b0 = cb[j];
      if (is_cont_byte(b0)) continue;
      uint32_t cp = 0;
      const uint32_t len = b0 < 0x80u ? (cp = b0, 1u) : utf8_decode(b0, cb[j + 1], cb[j + 2], cb[j + 3], 4u, &cp);
      if (len == 0) continue;
      lead |= 1u << j;
      cover |= ((1u << len) - 1u) << j;
      if (j + static_cast<int>(len) > CHUNK) spill = j + len - CHUNK;
      const uint32_t cls = cp_class(cp);
      sp |= (cls == CLS_SPACE ? 1u : 0u) << j;
      pu |= (cls == CLS_PUNCT ? 1u : 0u) << j;
      ha |= (cls == CLS_HAN ? 1u : 0u) << j;
    }
  }
  // ignore everything at or past `limit`
  const uint32_t in = limit_mask(c, limit);
  sm.m_lead[c] = lead & in;
  sm.m_space[c] = sp & in;
  sm.m_punct[c] = pu & in;
  sm.m_han[c] = ha & in;
  sm.m_cover[c] = cover;
  sm.spill[c] = static_cast<uint8_t>(spill);
}

// Both passes over the whole window (block-wide; sm.n_hi must be zero on entry; the caller synchronises
// before it reads the masks).  Out of line: K1 calls it from two places.
template <class TileSmem>
__device__ __noinline__ void classify_window(TileSmem &sm, const uint8_t *buf, int limit) {
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const bool high = tid < NCHUNK && classify_ascii(sm, buf, tid, limit);
  const uint32_t hm = __ballot_sync(FULL, high);
  if (hm) {
    uint32_t at = 0;
    const int leader = __ffs(hm) - 1;
    if (lane == leader) at = smem_add(&sm.n_hi, static_cast<uint32_t>(__popc(hm)));
    at = __shfl_sync(FULL, at, leader);
    WP_CHECK(!high || at + __popc(hm & ((1u << lane) - 1u)) < NCHUNK + 8);
    if (high) sm.hi_list[at + __popc(hm & ((1u << lane) - 1u))] = static_cast<uint8_t>(tid);
  }
  __syncthreads();
  const uint32_t n_hi = sm.n_hi;
  for (uint32_t i = tid; i < n_hi; i += THREADS) classify_multibyte(sm, buf, sm.hi_list[i], limit);
}

// block-wide exclusive scan of one value per thread; returns the exclusive prefix, *total = sum
template <int NWARPS, class T = uint32_t>
__device__ __forceinline__ T block_exclusive_scan(T *warp_sums, T v, T *total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  T incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const T y = __shfl_up_sync(FULL, incl, o);
    if (lane >= o) incl += y;
  }
  __syncthreads();  // warp_sums may still be in use by an earlier scan
  if (lane == 31) warp_sums[warp] = incl;
  __syncthreads();
  T wbase = 0, tot = 0;
#pragma unroll
  for (int wi = 0; wi < NWARPS; wi++) {
    const T ws = warp_sums[wi];
    if (wi < warp) wbase += ws;
    tot += ws;
  }
  *total = tot;
  return wbase + incl - v;
}

// K1 calls the scan from three places; one out-of-line copy keeps its executed code inside the instruction
// cache (see classify_ascii).  Returns the exclusive prefix in the low and the total in the high 32 bits.
__device__ __noinline__ unsigned long long tile_exclusive_scan(uint32_t *warp_sums, uint32_t v) {
  uint32_t total;
  const uint32_t at = block_exclusive_scan<WARPS>(warp_sums, v, &total);
  return (static_cast<unsigned long long>(total) << 32) | at;
}

// Decoupled look-back over a chain of units (tiles of K1, blocks of K3).  state[i] = flag << 62 | value;
// flag 1 = the unit's own total, 2 = inclusive prefix.  Units are handed out in launch order by a
// ticket, so every predecessor is already running: the spin always ends.
//
// lookback_publish (one thread) makes the unit's total visible as early as possible; lookback_walk (one
// full warp) later returns the sum over all earlier units and publishes the inclusive prefix.  Work that
// does not need the prefix goes in between: by then the predecessors have published theirs and the
// walk is short (when every unit walked right away, it crossed hundreds of concurrent units).
__device__ __forceinline__ void lookback_publish(volatile unsigned long long *state, uint32_t index,
                                                 unsigned long long total) {
  state[index] = ((index == 0 ? 2ull : 1ull) << 62) | total;
}

// A walk that has spun this long on one predecessor has lost its forward-progress guarantee (see K1 about the
// order in which tiles are taken): it gives up, reports it, and the host repeats the call in ticket mode.
constexpr uint32_t LOOKBACK_SPIN_LIMIT = 1u << 24;  // (a spin is an L2 round trip, ~1 us: many seconds)

__device__ __forceinline__ unsigned long long lookback_walk(volatile unsigned long long *state, uint32_t index,
                                                            unsigned long long total, int lane,
                                                            unsigned int *stalled = nullptr, unsigned int *void_call = nullptr) {
  constexpr unsigned long long VALUE_MASK = (1ull << 62) - 1;
  unsigned long long base = 0;
  if (index == 0) return 0;
  long long pred = static_cast<long long>(index) - 1 - lane;  // lane i looks at unit index-1-i
  for (;;) {
    unsigned long long sv = 2ull << 62;  // units before 0 count as a zero prefix
    if (pred >= 0) {
      uint32_t spins = 0;
      do {
        sv = state[pred];
        if (++spins > LOOKBACK_SPIN_LIMIT && stalled != nullptr) {
          *stalled = 1u;
          if (void_call != nullptr) *void_call = 1u;  // (the kernels behind this one do nothing)
          sv = 2ull << 62;  // give up: the result is wrong and the call is void
        }
      } while ((sv >> 62) == 0);
    }
    const uint32_t is_prefix = __ballot_sync(FULL, (sv >> 62) == 2);
    // add the totals of the lanes before the first inclusive prefix, and that prefix
    const int stop = is_prefix ? __ffs(is_prefix) - 1 : 31;
    unsigned long long v = lane <= stop ? (sv & VALUE_MASK) : 0ull;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    base += v;
    if (is_prefix) break;
    pred -= 32;
  }
  if (lane == 0) state[index] = (2ull << 62) | (base + total);
  return base;
}

// 16 window bytes starting at p (any alignment) as four little-endian words
__device__ __forceinline__ void load_window(const uint8_t *buf, int p, uint32_t r[4]) {
  const int a = p & ~3;
  const uint32_t sh = (p & 3) * 8;
  uint32_t x[5];
#pragma unroll
  for (int i = 0; i < 5; i++) x[i] = ld_u32(buf + a + 4 * i);
#pragma unroll
  for (int i = 0; i < 4; i++) r[i] = __funnelshift_r(x[i], x[i + 1], sh);
}

// Row k (0..16) of the key-mask table: byte masks of the four key words of a k-byte key.  Rows are 16 bytes
// apart and lanes read the row of their own length: rows 1..8 — nearly all segments — lie in eight different
// groups of four banks, so a quarter warp's 16-byte loads do not collide.
__device__ __forceinline__ void init_key_mask(uint4 *key_mask, int tid) {
  if (tid <= static_cast<int>(WORD_KEY_BYTES)) {
    uint32_t m[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int nb = tid - 4 * i;
      m[i] = nb >= 4 ? 0xFFFFFFFFu : (nb <= 0 ? 0u : ((1u << (8 * nb)) - 1u));
    }
    key_mask[tid] = make_uint4(m[0], m[1], m[2], m[3]);
  }
}

// ================================================================ K1: split

// A single-char segment whose lookup ran past WORD_PROBES slots: follow the probe sequence to the word or to
// an empty slot (the static part is complete, so absence means no such token).  Rare, so kept out of line;
// returns the id or SINGLE_WALK_MISS.
constexpr int32_t SINGLE_WALK_MISS = WP_NO_ID - 1;
constexpr uint16_t PARK_PENDING = 0xFFFFu;  // parked high half of a result is < 0x8000
// (a template only so that each instantiation of K1 has a copy of its own: ptxas 12.9 crashes on one
// out-of-line function shared by the two)
template <int SEG_CAP>
__device__ __noinline__ int32_t single_char_walk(const WordSlot *tab, uint32_t mask, uint32_t idx, uint32_t k0,
                                                 uint32_t len) {
  for (uint32_t n = 0; n <= mask; n++) {  // (a working table that K2 has filled to the last slot has no empty one)
    uint4 a, b;
    ld_word_slot(tab, idx, &a, &b);
    if (b.x == 0) break;
    if ((b.x & WORD_READY) && word_meta_len(b.x) == len && a.x == k0) return static_cast<int32_t>(b.y);
    idx = (idx + 1) & mask;
  }
  return SINGLE_WALK_MISS;
}

template <int SEG_CAP>
__global__ void __launch_bounds__(THREADS) wp_split_kernel(EncodeParams P) {
  using TileSmem = TileSmemT<SEG_CAP>;
  extern __shared__ __align__(16) uint8_t smem_raw[];
  TileSmem &sm = *reinterpret_cast<TileSmem *>(smem_raw);
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  const DeviceVocab &V = P.vocab;

  // tile = block index: blocks of a 1-D grid are dispatched in index order on every GPU so far, so a tile's
  // predecessors are always already running (decoupled look-back needs that forward progress) and no ticket
  // round trip sits in front of the tile's loads.  CUDA does not PROMISE the order (time slicing, debuggers),
  // so the look-back spin is bounded: a walk that gives up voids the call (CALL_STALLED), and the host repeats
  // it with P.use_ticket, where tiles are handed out by an atomic counter and the guarantee holds by construction.
  if (tid == 0) {
    if (P.use_ticket) sm.tile_ticket = atomicAdd(&P.counters->split_ticket, 1u);
    sm.left_spill = 0;
    sm.n_slow = 0;
    sm.dyn_hits = 0;
    sm.n_eligible = 0;
    sm.any_single = 0;
    sm.n_hi = 0;
  }
  init_key_mask(sm.key_mask, tid);
  __syncthreads();
  const uint32_t rel_tile = P.use_ticket ? sm.tile_ticket : blockIdx.x;  // within the range
  const size_t t0 = (static_cast<size_t>(P.first_tile) + rel_tile) * TILE;
  const size_t n = P.n_bytes;
  const size_t avail = n - t0;  // > 0
  const bool more_text = avail > static_cast<size_t>(WINDOW);
  const TextView tv{P.text, n};
  {
    // tiles run in index order, about 6 x 148 at a time: pull the tile two such waves ahead into L2 so that
    // its own loads do not wait on DRAM
    const size_t pf = t0 + static_cast<size_t>(PREFETCH_TILES) * TILE + static_cast<size_t>(tid) * 128u;
    if (tid < TILE / 128 && pf < n) prefetch_l2(P.text + pf);
  }

  // ---- S1a: stage raw bytes [t0-LEFT, t0+WINDOW+LOOKAHEAD) in shared memory
  {
    const bool aligned = (reinterpret_cast<uintptr_t>(P.text) & 15u) == 0;
#pragma unroll 1
    for (int u = tid; u < RAW_BYTES / 16; u += THREADS) {
      const long long g = static_cast<long long>(t0) - LEFT + 16ll * u;  // text offset of this unit
      uint4 v;
      if (aligned && g >= 0 && static_cast<size_t>(g) + 16 <= n) {
        v = ldg_stream(reinterpret_cast<const uint4 *>(P.text + g));
      } else {
        uint32_t q[4] = {0x20202020u, 0x20202020u, 0x20202020u, 0x20202020u};
        for (int i = 0; i < 16; i++) {
          const long long gi = g + i;
          if (gi >= 0 && static_cast<size_t>(gi) < n) {
            q[i >> 2] = (q[i >> 2] & ~(0xFFu << (8 * (i & 3)))) | (uint32_t(P.text[gi]) << (8 * (i & 3)));
          }
        }
        v = make_uint4(q[0], q[1], q[2], q[3]);
      }
      *reinterpret_cast<uint4 *>(sm.raw + 16 * u) = v;
    }
  }
  __syncthreads();
  if (tid == THREADS - 1) {
    // class of the last valid char before the tile: from the left halo in shared memory when it holds one
    // (always, for valid UTF-8), else by walking back through the text in global memory
    uint32_t pc = CLS_SPACE;
    bool found = t0 == 0;
    if (!found) {
      const uint8_t *h = sm.raw + LEFT;  // h[-1] is the byte before the tile
      for (int j = -1; j >= -4 && !found; j--) {
        const uint32_t b0 = h[j];
        if (is_cont_byte(b0)) continue;
        uint32_t cp = 0;
        const uint32_t len = b0 < 0x80u ? (cp = b0, 1u) : utf8_decode(b0, h[j + 1], h[j + 2], h[j + 3], 4u, &cp);
        if (len != 0) {
          pc = cp_class(cp);
          found = true;
        }
        break;  // an invalid lead: the exact answer needs the walk below
      }
      if (!found) pc = gprev_class(tv, t0);
    }
    sm.prev_class = pc;
  }

  // ---- S1b: classify the window; find bytes that the strict decoder drops
  uint8_t *const buf = sm.raw + LEFT;
  int limit = WINDOW;
  classify_window(sm, buf, WINDOW);
  if (tid == THREADS - 2) {
    // a sequence that starts in the last 3 bytes before the tile may own its first bytes
    uint32_t ls = 0;
    for (int j = -3; j < 0; j++) {
      const uint32_t b0 = buf[j];
      if (is_cont_byte(b0) || b0 < 0x80u) continue;
      uint32_t cp;
      const uint32_t len = utf8_decode(b0, buf[j + 1], buf[j + 2], buf[j + 3], 4u, &cp);
      if (len && j + static_cast<int>(len) > 0) ls = j + len;
    }
    sm.left_spill = ls;
  }
  __syncthreads();
  uint32_t kept = 0xFFFFFFFFu;  // surviving bytes of chunk `tid` (chunk NCHUNK = look-ahead: only a spilled tail)
  if (tid <= NCHUNK) {
    const uint32_t sp_in = tid == 0 ? sm.left_spill : sm.spill[tid - 1];
    kept = (tid < NCHUNK ? sm.m_cover[tid] : 0u) | ((1u << sp_in) - 1u);
  }
  const bool dirty = __syncthreads_or(tid < NCHUNK && kept != 0xFFFFFFFFu);

  if (dirty) {
    // ---- S1c (rare): drop the invalid bytes by compacting the window IN PLACE
    // (every thread first pulls its chunk into registers), then classify again.
    // utf8.cpp:130-147.
    uint32_t w[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    uint32_t my_cnt = 0;
    if (tid == 0) sm.n_hi = 0;  // for the second classification below (barriers lie on both sides)
    if (tid <= NCHUNK) {
      const uint4 a = *reinterpret_cast<const uint4 *>(buf + tid * CHUNK);
      const uint4 b = *reinterpret_cast<const uint4 *>(buf + tid * CHUNK + 16);
      w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w;
      w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
      my_cnt = __popc(kept);
      sm.m_kept[tid] = kept;
    }
    uint32_t packed_len;
    const unsigned long long sc0 = tile_exclusive_scan(sm.warp_sums, my_cnt);  // syncs: chunks are in registers
    const uint32_t dst0 = static_cast<uint32_t>(sc0);
    packed_len = static_cast<uint32_t>(sc0 >> 32);
    if (tid <= NCHUNK) {
      sm.kept_scan[tid] = dst0;
      if (tid == NCHUNK) sm.kept_scan[NCHUNK + 1] = packed_len;
      uint32_t dst = dst0, m = kept;
      while (m) {
        const int j = __ffs(m) - 1;
        m &= m - 1;
        buf[dst++] = static_cast<uint8_t>(w[j >> 2] >> (8 * (j & 3)));
      }
    }
    __syncthreads();
    for (int i = static_cast<int>(packed_len) + tid; i < WINDOW + LOOKAHEAD; i += THREADS) buf[i] = 0x20;
    __syncthreads();
    limit = static_cast<int>(packed_len) < WINDOW ? static_cast<int>(packed_len) : WINDOW;
    classify_window(sm, buf, limit);
    __syncthreads();
  }
  // owned range in buffer coordinates: segments that start in [0, own_end)
  const int own_end = dirty ? static_cast<int>(sm.kept_scan[OWNED_CHUNKS]) : TILE;

  // ---- S1d: segment starts (SURVEY A.2 safe starts) and segment ends, by mask
  // arithmetic, compacted in text order into seg_s[] / seg_e[].  A segment ends
  // at a lead p whose previous char is not a space and (is punctuation, or p
  // itself is a spacing char).  Starts and ends alternate, so owned segment k
  // pairs with end k + skip, skip = 1 iff a segment of the previous tile is
  // still open at the tile border.
  {
    uint32_t starts = 0, ends = 0, pu = 0, ha = 0;
    const int c = tid;
    if (c < NCHUNK) {
      const uint32_t lead = sm.m_lead[c];
      pu = sm.m_punct[c];
      ha = sm.m_han[c];
      const uint32_t sp = sm.m_space[c];
      uint32_t carry_s, carry_p;
      if (c == 0) {
        carry_s = sm.prev_class == CLS_SPACE;
        carry_p = sm.prev_class == CLS_PUNCT;
      } else {
        const uint32_t pl = sm.m_lead[c - 1];
        uint32_t xs = sm.m_space[c - 1], xp = sm.m_punct[c - 1];
#pragma unroll
        for (int i = 0; i < 3; i++) {
          xs |= (xs << 1) & ~pl;
          xp |= (xp << 1) & ~pl;
        }
        carry_s = xs >> 31;
        carry_p = xp >> 31;
      }
      uint32_t xs = sp | (carry_s & ~lead & 1u), xp = pu | (carry_p & ~lead & 1u);
#pragma unroll
      for (int i = 0; i < 3; i++) {
        xs |= (xs << 1) & ~lead;
        xp |= (xp << 1) & ~lead;
      }
      const uint32_t prev_s = (xs << 1) | carry_s;
      const uint32_t prev_p = (xp << 1) | carry_p;
      ends = lead & ~prev_s & (prev_p | sp | pu | ha);
      starts = lead & ~sp & (pu | ha | prev_s | prev_p);
      const int left = own_end - c * CHUNK;
      starts &= left >= CHUNK ? 0xFFFFFFFFu : (left <= 0 ? 0u : ((1u << left) - 1u));
    }
    uint32_t totals;
    const unsigned long long sc1 = tile_exclusive_scan(sm.warp_sums, __popc(starts) | (__popc(ends) << 16));
    const uint32_t at = static_cast<uint32_t>(sc1);
    totals = static_cast<uint32_t>(sc1 >> 32);
    uint32_t at_s = at & 0xFFFFu, at_e = at >> 16;
    if (SEG_CAP < TILE && ((totals & 0xFFFFu) > SEG_CAP || (totals >> 16) > SEG_CAP + HALO + 63)) {  // uniform
      // a dense tile (more segments than the lists of this instantiation hold): the call is void, the host
      // repeats it with the full-capacity kernel.  The tile still publishes a count: nobody may wait for it.
      if (tid == 0) {
        P.call->dense = 1u;
        P.call->overflow = 1u;
        lookback_publish(P.tile_state, rel_tile, totals & 0xFFFFu);
      }
      return;
    }
    if (P.bounds != nullptr && c < NCHUNK) {
      // batch call: the text starts of this tile are numbered after the look-back walk from the chunk's start
      // bits and their prefix (the class masks are not needed any more; the scan above was a barrier)
      sm.m_space[c] = starts;
      sm.m_punct[c] = at_s;
    }
    while (starts) {
      const int j = __ffs(starts) - 1;
      starts &= starts - 1;
      const uint32_t bit = 1u << j;
      const uint32_t cls = (pu & bit) ? CLS_PUNCT : ((ha & bit) ? CLS_HAN : CLS_OTHER);
      WP_CHECK(at_s < SEG_CAP);
      sm.seg_s[at_s++] = static_cast<uint16_t>((c * CHUNK + j) | (cls << 14));
    }
    while (ends) {
      const int j = __ffs(ends) - 1;
      ends &= ends - 1;
      WP_CHECK(at_e < SEG_CAP + HALO + 64);
      sm.seg_e[at_e++] = static_cast<uint16_t>(c * CHUNK + j);
    }
    if (tid == 0) {
      sm.n_segs = totals & 0xFFFFu;
      sm.n_ends = totals >> 16;
      // The last owned segment may have no end inside the window (it leaves the window, or the compacted text
      // of a dirty tile ends with it): its end entry, seg_e[n_ends], is read below like any other and must not
      // look like a parked PARK_PENDING.  (Left to whatever an earlier kernel had in this shared memory, it made
      // the pass for undecided single-char segments overwrite the START of a long segment with a token id: wrong
      // ids that depended on the kernels that had run before — found by the randomised sweep, see DESIGN 7.)
      sm.seg_e[totals >> 16] = 0;
    }
  }
  __syncthreads();
  const uint32_t n_segs = sm.n_segs;
  const uint32_t n_ends = sm.n_ends;
  const uint32_t skip = sm.prev_class != CLS_SPACE ? 1u : 0u;

  // ---- segment numbering across tiles: publish this tile's segment count now, walk back after S2a
  if (tid == 0) {
    lookback_publish(P.tile_state, rel_tile, n_segs);
    if (dirty) atomicAdd(&P.call->dirty_tiles, 1ull);
  }
  const WordSlot *wtab = P.words;

  // ---- S2: one word-table lookup per segment of at most 16 bytes, statically assigned (uniform work: every
  // lane does the same thing; two segments per lane and turn so that two table loads are in flight).  A hit
  // settles the segment — with the token it is (static part, fast.cpp:66-72: the longest candidate is the
  // whole window) or with the ids K2 recorded for these bytes earlier in this call.  A single-char segment
  // that is absent is UNK.  The rest go to the slow list.
  //
  // Straight-line on purpose: every lane — also one past the last segment, or with a segment too long for the
  // table — loads a window, hashes it and loads a slot (clamped to something harmless), and the outcome is
  // applied with predicates; only the further probes behind an occupied slot are a loop.
  constexpr int PER_TURN = WP_K1_PER_TURN;
  uint32_t my_dyn = 0, my_elig = 0;
  const uint32_t word_mask = P.word_mask;
#pragma unroll 1
  for (uint32_t base = 0; base < n_segs; base += PER_TURN * THREADS) {
    uint32_t state[PER_TURN], wlen[PER_TURN], idx[PER_TURN], key[PER_TURN][4];
    uint4 sa[PER_TURN], sb[PER_TURN];
#pragma unroll
    for (int u = 0; u < PER_TURN; u++) {
      const uint32_t k = base + u * THREADS + tid;
      const bool valid = k < n_segs;
      const uint32_t kc = min(k, n_segs - 1u);  // (a lane past the last segment reads that one's entries: they may
      const uint32_t j = kc + skip;             //  already hold a parked result, so what it reads is replaced below)
      const bool has_end = j < n_ends;
      const int s0 = static_cast<int>(sm.seg_s[kc] & POS_MASK);
      const int e0 = sm.seg_e[j];  // (in bounds either way: j <= TILE)
      const int s = valid ? s0 : 0;
      const int e = valid ? (has_end ? e0 : limit) : 1;
      const uint32_t len = static_cast<uint32_t>(e - s);
      const bool is_long = (!has_end && more_text) || len > LONG_SEGMENT_BYTES;  // no end inside the window / very long
      // 0 = no segment, 1 = looked up, 2 = slow, 3 = slow and LONG
      state[u] = !valid ? 0u : (is_long ? 3u : (len > WORD_KEY_BYTES ? 2u : 1u));
      wlen[u] = len;
      const uint32_t lc = min(len, WORD_KEY_BYTES);
      uint32_t r[4];
      WP_CHECK(s >= 0 && s + 20 <= WINDOW + LOOKAHEAD);
      WP_CHECK(e > s);
      WP_CHECK(j <= TILE);
      load_window(buf, s, r);
      const uint4 km = sm.key_mask[lc];
      key[u][0] = r[0] & km.x;
      key[u][1] = r[1] & km.y;
      key[u][2] = r[2] & km.z;
      key[u][3] = r[3] & km.w;
      idx[u] = word_hash(key[u][0], key[u][1], key[u][2], key[u][3], lc, P.word_shift);
      WP_CHECK(idx[u] <= P.word_mask);
      ld_word_slot(wtab, idx[u], &sa[u], &sb[u]);
    }
#pragma unroll
    for (int u = 0; u < PER_TURN; u++) {
      const bool look = state[u] == 1u;
      auto slot_hit = [&](const uint4 &a, const uint4 &m) {
        return (m.x & WORD_READY) && word_meta_len(m.x) == wlen[u] && a.x == key[u][0] && a.y == key[u][1] &&
               a.z == key[u][2] && a.w == key[u][3];
      };
      bool hit = slot_hit(sa[u], sb[u]);
      bool absent = sb[u].x == 0u;         // an empty slot ends the probe sequence: no such word
      bool more = look && !hit && !absent;  // the slot holds another word: look at the next ones
      if (__any_sync(FULL, more)) {
#pragma unroll 1
        for (uint32_t t = 1; t < WORD_PROBES; t++) {
          if (more) {
            idx[u] = (idx[u] + 1u) & word_mask;
            ld_word_slot(wtab, idx[u], &sa[u], &sb[u]);
            hit = slot_hit(sa[u], sb[u]);
            absent = sb[u].x == 0u;
            more = !hit && !absent;
          }
          if (!__any_sync(FULL, more)) break;
        }
      }
      // hit / absent / (neither:) not decided within WORD_PROBES slots
      const bool single = wlen[u] == utf8_lead_len(key[u][0] & 0xFFu);
      const bool settled = look && (hit || single);
      if (settled) {
        // park the result in the two list entries of the segment, which are no longer needed, until the tile
        // knows its first global segment number
        const uint32_t cnt = word_meta_count(sb[u].x);
        uint32_t res = cnt == 1u ? sb[u].y + 1u : (SEG_RESULT_WORD | (cnt << SEG_WORD_SLOT_BITS) | idx[u]);
        if (!hit) res = absent ? static_cast<uint32_t>(V.unk_id + 1) : (static_cast<uint32_t>(PARK_PENDING) << 16);
        if (!hit && !absent) sm.any_single = 1u;  // (seg_s keeps the position for the pass below)
        else sm.seg_s[base + u * THREADS + tid] = static_cast<uint16_t>(res);
        sm.seg_e[base + u * THREADS + tid + skip] = static_cast<uint16_t>(res >> 16);
        my_dyn += (hit && (sb[u].x & WORD_DYNAMIC)) ? 1u : 0u;
      } else if (look) {
        state[u] = 2u;
        my_elig++;
      }
      const uint32_t slowm = __ballot_sync(FULL, state[u] >= 2u);
      if (slowm) {
        uint32_t at = 0;
        const int leader = __ffs(slowm) - 1;
        if (lane == leader) at = smem_add(&sm.n_slow, static_cast<uint32_t>(__popc(slowm)));
        at = __shfl_sync(FULL, at, leader);
        WP_CHECK(state[u] < 2u || at + __popc(slowm & ((1u << lane) - 1u)) < MAX_TILE_SLOW);
        if (state[u] >= 2u)
          sm.slow[at + __popc(slowm & ((1u << lane) - 1u))] =
              static_cast<uint16_t>((base + u * THREADS + tid) | (state[u] == 3u ? SLOW_LONG : 0u));
      }
    }
  }
  if (P.record_words) {
    // statistics for K2's decision whether recording words still pays (memo_worthwhile)
    my_dyn = __reduce_add_sync(FULL, my_dyn);
    my_elig = __reduce_add_sync(FULL, my_elig);
    if (lane == 0 && (my_dyn | my_elig)) {
      smem_add_noret(&sm.dyn_hits, my_dyn);
      smem_add_noret(&sm.n_eligible, my_elig);
    }
  }
  __syncthreads();

  // ---- (rare) single-char segments whose lookup was not decided within WORD_PROBES slots
  if (sm.any_single) {  // uniform
#pragma unroll 1
    for (uint32_t k = tid; k < n_segs; k += THREADS) {
      if (sm.seg_e[k + skip] != PARK_PENDING) continue;  // (an end position and a parked high half are smaller; the
                                                         //  entry of a segment without an end was zeroed in S1d)
      uint32_t r[4];
      load_window(buf, static_cast<int>(sm.seg_s[k] & POS_MASK), r);
      const uint32_t len = utf8_lead_len(r[0] & 0xFFu);
      const uint32_t k0 = r[0] & sm.key_mask[len].x;
      const int32_t id = single_char_walk<SEG_CAP>(wtab, P.word_mask, word_hash(k0, 0u, 0u, 0u, len, P.word_shift), k0, len);
      const uint32_t res = static_cast<uint32_t>((id != SINGLE_WALK_MISS ? id : V.unk_id) + 1);
      sm.seg_s[k] = static_cast<uint16_t>(res);
      sm.seg_e[k + skip] = static_cast<uint16_t>(res >> 16);
    }
  }

  // ---- the walk back over earlier tiles (short by now), then the settled results go out coalesced
  if (warp == 0) {
    const unsigned long long base = lookback_walk(P.tile_state, rel_tile, n_segs, lane, &P.call->stalled, &P.call->overflow);
    if (lane == 0) {
      sm.seg_base = base;
      if (rel_tile == P.n_tiles - 1) P.counters->n_segs = base + n_segs;
    }
  }
  __syncthreads();
  const unsigned long long seg_base = sm.seg_base;
  if (seg_base + n_segs > P.seg_capacity) {
    if (tid == 0) P.call->overflow = 1u;
    return;  // uniform
  }
  if (P.bounds != nullptr) {
    // batch call: for every text that starts in this tile, the number of the first segment at or after its start
    const size_t abs_tile = static_cast<size_t>(P.first_tile) + rel_tile;
    const uint32_t b0 = P.tile_bound[abs_tile], b1 = P.tile_bound[abs_tile + 1];
#pragma unroll 1
    for (uint32_t i = b0 + tid; i < b1; i += THREADS) {
      uint32_t q = static_cast<uint32_t>(P.bounds[i] - t0);  // < TILE, raw window position
      WP_CHECK(P.bounds[i] >= t0 && q < TILE);
      if (dirty) q = sm.kept_scan[q >> 5] + __popc(sm.m_kept[q >> 5] & ((1u << (q & 31u)) - 1u));  // -> compacted
      P.bound_seg[i] = static_cast<uint32_t>(seg_base) + sm.m_punct[q >> 5] + __popc(sm.m_space[q >> 5] & ((1u << (q & 31u)) - 1u));
    }
  }
  // (every segment is written: the words of the unsettled ones are garbage here and are overwritten below,
  // behind a barrier, when their slow entries exist)
#pragma unroll 1
  WP_CHECK(seg_base + n_segs <= P.seg_capacity);
  for (uint32_t k = tid; k < n_segs; k += THREADS)
    P.seg_result[seg_base + k] = static_cast<uint32_t>(sm.seg_s[k]) | (static_cast<uint32_t>(sm.seg_e[k + skip]) << 16);
  if (tid == 0 && P.record_words && P.range_index >= 1) {
    const uint32_t h = sm.dyn_hits, l = sm.dyn_hits + sm.n_eligible;
    if (h) atomicAdd(&P.call->memo_hits, static_cast<unsigned long long>(h));
    if (l) atomicAdd(&P.call->memo_lookups, static_cast<unsigned long long>(l));
  }

  // ---- hand the unsettled segments to K2: 16-byte entries in the global slow list and, per entry, an area
  // of the arena (one reservation per tile): `len` words for its ids (a segment never has more ids than
  // bytes), then its clean bytes, so that K2 never goes back to the text
  const uint32_t n_slow = sm.n_slow;
  if (n_slow == 0) return;  // uniform
  {
    const uint32_t per = (n_slow + THREADS - 1) / THREADS;
    const uint32_t lo = min(n_slow, static_cast<uint32_t>(tid) * per);
    const uint32_t hi = min(n_slow, lo + per);
    uint32_t my_words = 0, n_long = 0;
#pragma unroll 1
    for (uint32_t i = lo; i < hi; i++) {
      const uint32_t ent = sm.slow[i];
      const uint32_t k = ent & 0xFFFu;
      if (ent & SLOW_LONG) {
        n_long++;
        continue;
      }
      const int e = k + skip < n_ends ? static_cast<int>(sm.seg_e[k + skip]) : limit;
      const uint32_t len = static_cast<uint32_t>(e - static_cast<int>(sm.seg_s[k] & POS_MASK));
      my_words += len + ((len + 3u) >> 2);
    }
    const unsigned long long sc2 = tile_exclusive_scan(sm.warp_sums, my_words);
    uint32_t run = static_cast<uint32_t>(sc2);
    const uint32_t total_words = static_cast<uint32_t>(sc2 >> 32);
    if (tid == 0) {
      // n_slow and arena_reserved sit side by side: one 64-bit atomic reserves both (one round trip to L2)
      static_assert(offsetof(RangeCounters, arena_reserved) == offsetof(RangeCounters, n_slow) + 4 &&
                        offsetof(RangeCounters, n_slow) % 8 == 0,
                    "n_slow / arena_reserved must form one aligned 64-bit word");
      const unsigned long long old = atomicAdd(reinterpret_cast<unsigned long long *>(&P.counters->n_slow),
                                               (static_cast<unsigned long long>(total_words) << 32) | n_slow);
      sm.slow_base = static_cast<uint32_t>(old);
      sm.arena_base = static_cast<uint32_t>(old >> 32);
    }
    uint32_t long_at = 0;
    if (n_long) {
      atomicAdd(&P.call->long_segments, static_cast<unsigned long long>(n_long));
      long_at = atomicAdd(&P.counters->n_long, n_long);
    }
    __syncthreads();
    const uint32_t slow_base = sm.slow_base;
    const uint32_t arena_base = sm.arena_base;
    if (static_cast<unsigned long long>(slow_base) + n_slow > P.slow_capacity ||
        static_cast<unsigned long long>(arena_base) + total_words > P.arena_capacity) {
      if (tid == 0) P.call->overflow = 1u;
      return;  // uniform
    }
#pragma unroll 1
    for (uint32_t i = lo; i < hi; i++) {
      const uint32_t ent = sm.slow[i];
      const uint32_t k = ent & 0xFFFu;
      const uint32_t sv = sm.seg_s[k];
      int wpos = static_cast<int>(sv & POS_MASK);
      SlowEntry out;
      out.seg = static_cast<uint32_t>(seg_base + k);
      if (ent & SLOW_LONG) {
        if (dirty) {
          // window position -> raw window position: undo the compaction
          int a = 0, b = NCHUNK;  // last chunk whose first surviving byte is at or before wpos
          while (a < b) {
            const int m = (a + b + 1) >> 1;
            if (sm.kept_scan[m] <= static_cast<uint32_t>(wpos)) a = m; else b = m - 1;
          }
          const uint32_t kk = static_cast<uint32_t>(wpos) - sm.kept_scan[a];
          wpos = a * CHUNK + static_cast<int>(__fns(sm.m_kept[a], 0, static_cast<int>(kk) + 1));
        }
        const size_t pos = t0 + static_cast<size_t>(wpos);
        out.off = 0;
        out.meta = ((sv >> 14) << 16) | SLOW_META_LONG | (static_cast<uint32_t>((pos >> 32) & 0xFFu) << 24);
        out.pos_lo = static_cast<uint32_t>(pos);
        if (long_at < P.long_capacity) P.long_list[long_at] = slow_base + i;  // K2L's work list
        long_at++;
      } else {
        const int e = k + skip < n_ends ? static_cast<int>(sm.seg_e[k + skip]) : limit;
        const uint32_t len = static_cast<uint32_t>(e - wpos);
        out.off = arena_base + run;
        WP_CHECK(static_cast<unsigned long long>(out.off) + len + ((len + 3u) >> 2) <= P.arena_capacity && len >= 1 && len <= LONG_SEGMENT_BYTES);
        out.meta = len | ((sv >> 14) << 16);
        out.pos_lo = 0;
        uint32_t *dst = P.arena + out.off + len;
        const uint32_t nw = (len + 3u) >> 2;
        const uint8_t *src = buf + (wpos & ~3);
        const uint32_t sh = (wpos & 3) * 8;
        uint32_t x0 = ld_u32(src);
#pragma unroll 1
        for (uint32_t q = 0; q < nw; q++) {
          const uint32_t x1 = ld_u32(src + 4 * q + 4);
          uint32_t w = __funnelshift_r(x0, x1, sh);
          if (q == nw - 1 && (len & 3u)) w &= (1u << (8 * (len & 3u))) - 1u;
          dst[q] = w;
          x0 = x1;
        }
        run += len + nw;
      }
      WP_CHECK(slow_base + i < P.slow_capacity && out.seg < P.seg_capacity);
      *reinterpret_cast<uint4 *>(&P.slow[slow_base + i]) = *reinterpret_cast<const uint4 *>(&out);
      P.seg_result[seg_base + k] = SEG_RESULT_SLOW | (slow_base + i);
    }
  }
}

// ================================================================ K2: match

constexpr uint32_t SEG_HAN_FIRST = 1u;   // about to match the first piece of a Han-led segment

// Every lane owns a long run of slow-list entries (its warp's share / 32), so chains of very different
// length average out.  One loop iteration = one trie step for every lane that holds a segment, whatever the
// lane is doing: a step that succeeds moves one byte down the trie and remembers the last terminal seen; a
// step that fails, reaches a leaf or the end of the segment closes the piece (fast.cpp:66-91: emit the
// longest match, continue behind it in the "##" map, or roll the whole word back to UNK).  Lanes without a
// segment take the next entries of their warp's share at the top of the loop.
__global__ void __launch_bounds__(MATCH_THREADS, WP_K2_BLOCKS) wp_match_kernel(EncodeParams P) {
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const DeviceVocab &V = P.vocab;

  if (P.call->overflow) return;  // a K1 tile gave up (scratch too small): its entries are unwritten, the host retries
  const uint32_t n_slow = min(P.counters->n_slow, P.slow_capacity);
  // Fixed shares: every warp owns one contiguous run of entries.  (Handing the entries out in chunks from an
  // atomic counter was measured: with 32 per warp and fetch it is no faster than the shares — English +5 %,
  // Japanese -5 % — and with 64 or 128 it is 1.6x / 2.8x SLOWER, profiles/r2g_variants.txt.)
  const uint32_t n_warps = gridDim.x * (MATCH_THREADS / 32);
  const uint32_t gw = blockIdx.x * (MATCH_THREADS / 32) + (tid >> 5);
  const uint32_t per = ((n_slow + n_warps - 1) / n_warps + 31u) & ~31u;
  uint32_t cursor = min(n_slow, gw * per);             // warp-uniform: next unassigned entry of this warp
  const uint32_t cursor_end = min(n_slow, cursor + per);

  // K1 of this range is done, so the counters are final: every lane reads the same verdict
  const bool worth = memo_worthwhile(P.call->memo_lookups, P.call->memo_hits, P.range_index <= 1);
  if (blockIdx.x == 0 && tid == 0 && !worth) P.call->memo_off = 1u;
  bool record = P.record_words != 0 && (P.range_index < 2 || worth);

  bool have = false;       // this lane holds an unfinished segment
  bool ext = false;        // the current node has children
  const uint8_t *txt = nullptr;  // the segment's clean bytes (arena)
  int32_t *out = nullptr;        // the segment's id scratch (arena)
  uint32_t ent_index = 0, area = 0, seg = 0, seg_len = 0, first_len = 0;
  uint32_t p = 0, d = 0, node = 0, last_d = 0;          // piece start, depth, trie node, depth of the last terminal
  uint32_t nid = 0, word_first = 0, kind = WP_KIND_PREFIX, flags = 0;
  int32_t last_id = WP_NO_ID, t0 = 0, t1 = 0, t2 = 0;   // the first three ids of the segment stay in registers
  // The text runs one char ahead of the trie: raw_cur = the four bytes at p + d, loaded while the table lookup
  // of the char before it was in flight; raw_term = the four bytes behind the last terminal, i.e. the start of
  // the next piece if that terminal stays the longest match.  The walk so depends on one load per char (the
  // edge) instead of two in a row (text word, then edge).
  uint32_t raw_cur = 0, raw_term = 0;
  // four clean bytes at offset `at` of the segment (word-aligned in the arena; the word behind the text is in bounds)
  auto text_at = [&](uint32_t at) {
    const uint32_t *tw = reinterpret_cast<const uint32_t *>(txt) + (at >> 2);
    return __funnelshift_r(tw[0], tw[1], (at & 3u) * 8u);
  };

  for (;;) {
    // -- refill: lanes without a segment take the next entries of this warp's share
    const uint32_t needm = __ballot_sync(FULL, !have);
    if (needm && cursor < cursor_end) {
      const uint32_t i = cursor + __popc(needm & ((1u << lane) - 1u));
      cursor += __popc(needm);  // may pass cursor_end; entries beyond it are simply not taken
      if (cursor + lane < cursor_end) prefetch_l2(&P.slow[cursor + lane]);  // the next 32 entries of this share
      if (!have && i < cursor_end) {
        // (L2, coherent: K2 itself rewrites entries of this array — results are stored in place — so the
        // non-coherent path, which PTX allows only for data that is read-only during the whole kernel, is out)
        const uint4 raw = __ldcg(reinterpret_cast<const uint4 *>(&P.slow[i]));
        const uint32_t meta = raw.y;
        if (!(meta & SLOW_META_LONG)) {  // LONG entries are matched by K2L
          ent_index = i;
          area = raw.x;
          seg = raw.w;
          seg_len = meta & 0xFFFFu;
          WP_CHECK(static_cast<unsigned long long>(area) + seg_len + ((seg_len + 3u) >> 2) <= P.arena_capacity && seg_len >= 1 &&
                   seg < P.seg_capacity);
          out = reinterpret_cast<int32_t *>(P.arena + area);
          txt = reinterpret_cast<const uint8_t *>(P.arena + area + seg_len);
          raw_cur = text_at(0);
          first_len = utf8_lead_len(raw_cur & 0xFFu);
          have = true;
          ext = true;
          p = 0;
          d = 0;
          last_d = 0;
          nid = 0;
          word_first = 0;
          kind = WP_KIND_PREFIX;
          node = WP_KIND_PREFIX;
          flags = ((meta >> 16) & 3u) == CLS_HAN ? SEG_HAN_FIRST : 0u;
        }
      }
    }
    if (!__any_sync(FULL, have)) {
      if (cursor >= cursor_end) break;
      continue;
    }
    if (!have) continue;

    // -- one trie step
    bool closed = true;
    if (ext && p + d < seg_len) {
      const uint32_t cl = utf8_lead_len(raw_cur & 0xFFu);
      const uint32_t raw_next = text_at(p + d + cl);  // (independent of the lookup below: both loads are in flight together)
      uint4 e;
      if (trie_step(V, node, edge_char(raw_cur, cl), &e)) {
        node = edge_child(e);
        d += cl;
        raw_cur = raw_next;
        if (edge_term(e) != WP_NO_ID) {
          last_d = d;
          last_id = edge_term(e);
          raw_term = raw_next;
        }
        ext = edge_extends(e);
        closed = !ext || p + d >= seg_len;
      }
    }
    if (!closed) continue;

    // -- the piece is closed: its longest match is the last terminal seen (fast.cpp:66-77)
    const uint32_t mlen = last_d;
    bool done = false;
    // ids 0..2 go to registers, later ones straight to the id scratch
    auto put = [&](uint32_t index, int32_t v) {
      WP_CHECK(index < seg_len);  // a segment never has more ids than bytes
      if (index == 0) t0 = v;
      else if (index == 1) t1 = v;
      else if (index == 2) t2 = v;
      else out[index] = v;
    };
    if (flags & SEG_HAN_FIRST) {
      flags = 0;
      nid = 1;
      if (mlen == 0) {
        t0 = V.unk_id;
        if (V.han_swallow) {
          done = true;  // fast.cpp:85-88: begin += word_len swallows the run
        } else {
          word_first = 1;
          p += first_len;
        }
      } else {
        t0 = last_id;
        p += mlen;
        if (mlen == first_len) {
          word_first = 1;  // fast.cpp:89-91: the next position follows a spacing char => new word
        } else {
          kind = WP_KIND_SUFFIX;
        }
      }
    } else if (mlen == 0) {  // fast.cpp:79-88: whole-word UNK, earlier pieces rolled back
      put(word_first, V.unk_id);
      nid = word_first + 1;
      done = true;
    } else {
      put(nid, last_id);
      nid++;
      p += mlen;
      kind = WP_KIND_SUFFIX;
    }
    if (!done && p < seg_len) {
      raw_cur = mlen ? raw_term : text_at(p);  // (no match: only behind an out-of-vocabulary Han char, fast.cpp:85-88)
      d = 0;
      last_d = 0;
      node = kind;
      ext = true;
      continue;
    }

    // -- the segment is finished.  Result form of the entry (read by K3): up to three ids inline — one 16-byte
    // store and nothing else for most segments — else the count and where the ids sit in the arena
    uint4 res;
    if (nid <= 3) {
      res = make_uint4(nid | SLOW_RESULT_INLINE, static_cast<uint32_t>(t0), static_cast<uint32_t>(t1),
                       static_cast<uint32_t>(t2));
    } else {
      out[0] = t0;
      out[1] = t1;
      out[2] = t2;
      res = make_uint4(nid, area, 0u, 0u);
    }
    *reinterpret_cast<uint4 *>(&P.slow[ent_index]) = res;
    P.seg_result[seg] = SEG_RESULT_SLOW | (min(nid, SEG_SLOW_COUNT_MAX) << SEG_SLOW_INDEX_BITS) | ent_index;
    have = false;
    if (record && seg_len <= WORD_KEY_BYTES && nid <= WORD_MAX_IDS) {
      // record bytes -> ids in the word table so that K1 settles every later occurrence itself
      const uint32_t *tw = P.arena + area + seg_len;
      const uint32_t k0 = tw[0], k1 = seg_len > 4 ? tw[1] : 0u, k2 = seg_len > 8 ? tw[2] : 0u, k3 = seg_len > 12 ? tw[3] : 0u;
      uint32_t idx = word_hash(k0, k1, k2, k3, seg_len, P.word_shift);
      bool placed = false;
      for (uint32_t t = 0; t < WORD_PROBES && !placed; t++) {
        WP_CHECK(idx <= P.word_mask);
        WordSlot *slot = P.words + idx;
        const unsigned int old = atomicCAS(&slot->meta, 0u, WORD_CLAIMED);
        if (old == 0u) {
          // claimed.  The readers that need a complete slot (K1 and K3) run in later kernels; a concurrent K2
          // lane that meets the slot half written can at worst fail to recognise its own word and store a
          // harmless duplicate one slot further.
          *reinterpret_cast<uint4 *>(slot->key) = make_uint4(k0, k1, k2, k3);
          slot->ids[0] = t0;
          slot->ids[1] = t1;
          slot->ids[2] = t2;
          for (uint32_t q = 3; q < nid; q++) slot->ids[q] = __ldcg(out + q);
          __threadfence();
          *reinterpret_cast<volatile unsigned int *>(&slot->meta) = word_meta(seg_len, nid, true);
          placed = true;
        } else if (old == WORD_CLAIMED) {
          placed = true;  // another lane is writing this slot right now (most likely the same word)
        } else if (word_meta_len(old) == seg_len) {
          const uint4 a = __ldcg(reinterpret_cast<const uint4 *>(slot->key));
          if (a.x == k0 && a.y == k1 && a.z == k2 && a.w == k3) placed = true;  // already there
        }
        idx = (idx + 1) & P.word_mask;
      }
      if (!placed) record = false;  // crowded neighbourhood: this lane stops feeding the table
    }
  }
}

// ========================================================= K2L: long segments
//
// A segment that leaves its tile's window (or is longer than LONG_SEGMENT_BYTES) may be arbitrarily long — a
// URL, a base64 blob, a whole text without a space (the reference's own stress shape, tests/tests.cpp:259-272,
// is ONE word of 10 MB) — so it is not walked by one lane.  One CTA per segment:
//   end    : the segment ends at the first spacing char after its start; found by a parallel scan;
//   head   : the first piece (word-initial map; Han-led segments: fast.cpp:85-91) by one thread;
//   rounds of LONG_BLOCK raw bytes:
//     A  every thread takes positions of the block: is it a valid ordinary-char lead, and if so the longest
//        "##" match that starts there (all positions in parallel — only those on the greedy chain are used);
//     B  the chain through the block (position -> first valid lead behind its match) is a linked list; it is
//        ranked by POINTER JUMPING instead of being followed by one thread: jump[k][i] = the piece start 2^k
//        pieces behind i (LONG_LEVELS rounds of doubling), then the start of the chain gets rank 0 and, from
//        the largest stride down, every ranked position ranks the position 2^k behind it — after the last
//        round exactly the positions on the chain carry their piece number.  A chain position without a match
//        turns the whole word into UNK (fast.cpp:79-88);
//     C  the ids of the ranked positions go to the arena at their rank.
constexpr int LONG_THREADS = 256;
constexpr int LONG_BLOCK = 1024;
constexpr int LONG_LEVELS = 10;            // 2^10 = LONG_BLOCK >= the pieces of a chain through one block
constexpr uint32_t LONG_END = 0xFFFFu;     // jump: no successor inside the block; rank: not on the chain
static_assert((1 << LONG_LEVELS) >= LONG_BLOCK, "the strides must reach across a whole block");

struct LongSmem {
  uint16_t jump[LONG_LEVELS][LONG_BLOCK];
  uint16_t rank[LONG_BLOCK];
  uint32_t delta[LONG_BLOCK];  // raw bytes from a piece start to the position behind its longest match (0 = none)
  int32_t id[LONG_BLOCK];
  uint8_t code[LONG_BLOCK];    // 0 = dropped / continuation byte, 1 = lead of an ordinary char
  unsigned long long seg_end;  // raw position of the spacing char that ends the segment (or the text size)
  unsigned long long cur;      // raw position of the next piece
  unsigned long long cur_next;
  uint32_t entry;              // index into the long list
  uint32_t n_round, n_out, word_first, off, finished, failed;
};

__global__ void __launch_bounds__(LONG_THREADS) wp_long_kernel(EncodeParams P) {
  __shared__ LongSmem sm;
  const int tid = threadIdx.x;
  const DeviceVocab &V = P.vocab;
  const TextView tv{P.text, P.n_bytes};
  if (P.call->overflow) return;
  const uint32_t n_long = min(P.counters->n_long, P.long_capacity);
  const uint32_t spill_base = min(P.counters->arena_reserved, P.arena_capacity);
  for (;;) {
    __syncthreads();
    if (tid == 0) sm.entry = atomicAdd(&P.counters->long_ticket, 1u);
    __syncthreads();
    if (sm.entry >= n_long) break;
    const uint32_t si = P.long_list[sm.entry];
    const SlowEntry ent = P.slow[si];
    const size_t start = static_cast<size_t>(ent.pos_lo) | (static_cast<size_t>(ent.meta >> 24) << 32);
    uint32_t len0, cls0;
    gnext(tv, start, &len0, &cls0);  // the start is a valid lead of a non-space class
    if (tid == 0) {
      sm.seg_end = tv.n;
      sm.n_out = 0;
      sm.word_first = 0;
      sm.finished = 0;
      sm.failed = 0;
    }
    __syncthreads();

    // ---- end: the first valid spacing char behind the first char
    for (size_t base = start + len0; base < tv.n; base += 8 * LONG_THREADS) {
      unsigned long long found = ~0ull;
#pragma unroll 1
      for (int j = 0; j < 8; j++) {
        const size_t q = base + static_cast<size_t>(j) * LONG_THREADS + tid;
        if (q >= tv.n) break;
        const uint32_t b0 = tv.t[q];
        if (is_cont_byte(b0) || (b0 < 0x80u && cp_class(b0) == CLS_OTHER)) continue;
        uint32_t cls;
        if (gdecode(tv, q, &cls) && cls != CLS_OTHER) {
          found = q;
          break;
        }
      }
      if (found != ~0ull) atomicMin(&sm.seg_end, found);
      __syncthreads();
      const bool stop = sm.seg_end < base + 8 * LONG_THREADS;
      __syncthreads();
      if (stop) break;
    }
    const size_t seg_end = static_cast<size_t>(sm.seg_end);

    // ---- head (one thread): reserve the id area, match the first piece (and the one behind a lone Han char)
    if (tid == 0) {
      const unsigned long long want = seg_end - start;  // ids <= chars <= bytes
      const unsigned long long off = static_cast<unsigned long long>(spill_base) +
                                     atomicAdd(&P.counters->arena_spill, static_cast<unsigned int>(min(want, 0xFFFFFFFFull)));
      if (off + want > P.arena_capacity) {
        P.call->overflow = 1u;
        sm.finished = 1;
        sm.off = 0;
      } else {
        sm.off = static_cast<uint32_t>(off);
        int32_t *out = reinterpret_cast<int32_t *>(P.arena + off);
        const TextView seg{P.text, seg_end};  // windows never reach past the segment
        int32_t id = 0;
        size_t cur = longest_match_global(V, seg, start, WP_KIND_PREFIX, &id);
        bool need_prefix = false;  // the next piece starts a fresh word (behind a lone Han char)
        if (cls0 == CLS_HAN) {
          if (cur == start) {
            out[0] = V.unk_id;
            if (V.han_swallow) {
              sm.finished = 1;  // fast.cpp:85-88: begin += word_len swallows the run
            } else {
              cur = start + len0;
              need_prefix = true;
            }
          } else {
            out[0] = id;
            need_prefix = cur == start + len0;  // fast.cpp:89-91: the next position follows a spacing char
          }
          sm.n_out = 1;
          if (need_prefix) sm.word_first = 1;
        } else if (cur == start) {  // fast.cpp:79-88
          out[0] = V.unk_id;
          sm.n_out = 1;
          sm.finished = 1;
        } else {
          out[0] = id;
          sm.n_out = 1;
        }
        if (!sm.finished && need_prefix) {
          uint32_t l, c;
          const size_t q = gnext(seg, cur, &l, &c);
          if (q >= seg_end) {
            sm.finished = 1;
          } else {
            cur = longest_match_global(V, seg, q, WP_KIND_PREFIX, &id);
            if (cur == q) {
              out[1] = V.unk_id;
              sm.finished = 1;
            } else {
              out[1] = id;
            }
            sm.n_out = 2;
          }
        }
        sm.cur = cur;
      }
    }
    __syncthreads();

    // ---- rounds
    const TextView seg{P.text, seg_end};
    int32_t *const out = reinterpret_cast<int32_t *>(P.arena + sm.off);
    while (!sm.finished) {
      const size_t b0 = static_cast<size_t>(sm.cur);
      if (b0 >= seg_end) break;
      const uint32_t n = static_cast<uint32_t>(min(seg_end - b0, static_cast<size_t>(LONG_BLOCK)));
      const uint32_t n_out = sm.n_out;
      // A: every position of the block
#pragma unroll 1
      for (uint32_t i = tid; i < n; i += LONG_THREADS) {
        const size_t q = b0 + i;
        uint32_t ch, code = 0, delta = 0;
        int32_t id = 0;
        if (!is_cont_byte(tv.t[q]) && gchar(seg, q, &ch)) {  // a valid lead (no spacing char before seg_end: an ordinary char)
          code = 1;
          delta = static_cast<uint32_t>(longest_match_inside(V, seg, q, WP_KIND_SUFFIX, &id) - q);
        }
        sm.code[i] = static_cast<uint8_t>(code);
        sm.delta[i] = delta;
        sm.id[i] = id;
        sm.rank[i] = static_cast<uint16_t>(LONG_END);
      }
      if (tid == 0) {
        sm.n_round = 0;
        sm.cur_next = b0 + n;  // (a block without a piece start: only dropped bytes)
      }
      __syncthreads();
      // B: successors (the first valid lead at or behind the end of the match), doubled LONG_LEVELS - 1 times
#pragma unroll 1
      for (uint32_t i = tid; i < n; i += LONG_THREADS) {
        uint32_t nx = LONG_END;
        const uint32_t dl = sm.delta[i];
        if (dl != 0 && dl < n - i) {
          uint32_t t = i + dl;
          while (t < n && sm.code[t] == 0) t++;
          if (t < n) nx = t;
        }
        sm.jump[0][i] = static_cast<uint16_t>(nx);
      }
      if (tid == 0) {
        uint32_t t = 0;
        while (t < n && sm.code[t] == 0) t++;
        if (t < n) sm.rank[t] = 0;  // the round's first piece
      }
      __syncthreads();
#pragma unroll 1
      for (int k = 1; k < LONG_LEVELS; k++) {
        for (uint32_t i = tid; i < n; i += LONG_THREADS) {
          const uint32_t j = sm.jump[k - 1][i];
          sm.jump[k][i] = j == LONG_END ? static_cast<uint16_t>(LONG_END) : sm.jump[k - 1][j];
        }
        __syncthreads();
      }
      // (a position ranked during a round may rank its own 2^k-th successor in the same round: the value it
      // writes is right whenever it is written, so rounds need no stricter separation than the barrier)
#pragma unroll 1
      for (int k = LONG_LEVELS - 1; k >= 0; k--) {
        for (uint32_t i = tid; i < n; i += LONG_THREADS) {
          const uint32_t r = sm.rank[i];
          if (r == LONG_END) continue;
          const uint32_t j = sm.jump[k][i];
          WP_CHECK(j == LONG_END || (j < n && j > i && r + (1u << k) < LONG_BLOCK));
          if (j != LONG_END) sm.rank[j] = static_cast<uint16_t>(r + (1u << k));
        }
        __syncthreads();
      }
      // C: ids of the chain; its last piece says where the next round begins
#pragma unroll 1
      for (uint32_t i = tid; i < n; i += LONG_THREADS) {
        const uint32_t r = sm.rank[i];
        if (r == LONG_END) continue;
        const uint32_t dl = sm.delta[i];
        if (dl == 0) {
          sm.failed = 1;  // fast.cpp:79-88 (the chain ends here: a position without a match has no successor)
        } else {
          WP_CHECK(static_cast<unsigned long long>(sm.off) + n_out + r < P.arena_capacity && b0 + i - start >= n_out + r);
          out[n_out + r] = sm.id[i];
          if (sm.jump[0][i] == LONG_END) {
            sm.n_round = r + 1;
            sm.cur_next = b0 + i + dl;
          }
        }
      }
      __syncthreads();
      if (tid == 0) {
        sm.n_out = n_out + sm.n_round;
        sm.cur = sm.cur_next;
        if (sm.failed || sm.cur_next >= seg_end) sm.finished = 1;
      }
      __syncthreads();
    }
    if (tid == 0) {
      uint32_t cnt = sm.n_out;
      if (sm.failed) {  // fast.cpp:79-88: the word's pieces are rolled back, one UNK stands for it
        cnt = sm.word_first + 1;
        P.arena[sm.off + sm.word_first] = static_cast<uint32_t>(V.unk_id);
      }
      if (P.call->overflow) cnt = 0;
      *reinterpret_cast<uint4 *>(&P.slow[si]) = make_uint4(cnt, sm.off, 0u, 0u);  // result form, not inline
      P.seg_result[ent.seg] = SEG_RESULT_SLOW | (min(cnt, SEG_SLOW_COUNT_MAX) << SEG_SLOW_INDEX_BITS) | si;
    }
  }
}

// ============================================================== K3: scatter

struct ScatterSmem {
  int32_t stage[SCATTER_STAGE];
  uint32_t desc_pos[SCATTER_SEGS];     // segments not settled by K1: stage position << 16 | id count
  uint32_t desc_src[SCATTER_SEGS];     // ... and their seg_result word (where the ids are)
  uint32_t n_desc;
  uint32_t n_big;                      // segments with more than SCATTER_BIG ids: copied by the whole block
  uint16_t big[SCATTER_STAGE / (SCATTER_BIG < 6144 ? SCATTER_BIG : 6144) + 2];  // staged path: their indices in desc_pos / desc_src
  uint32_t warp_sums[SCATTER_THREADS / 32];
  uint32_t block_index[2];
  unsigned long long base;
};

// ids of one segment that K1 did not settle with a single id -> dst[0..cnt): inline in the slow entry, from
// the arena, or from the word-table slot
template <class Params>
__device__ __forceinline__ void scatter_fetch(const Params &P, uint32_t res, uint32_t cnt, int32_t *dst) {
  if (res & SEG_RESULT_SLOW) {
    const uint32_t si = res & SEG_SLOW_INDEX_MASK;
    if (si >= P.slow_capacity) return;
    const uint4 e = *reinterpret_cast<const uint4 *>(&P.slow[si]);
    if (e.x & SLOW_RESULT_INLINE) {
      dst[0] = static_cast<int32_t>(e.y);
      if (cnt > 1) dst[1] = static_cast<int32_t>(e.z);
      if (cnt > 2) dst[2] = static_cast<int32_t>(e.w);
    } else if (static_cast<unsigned long long>(e.y) + cnt <= P.arena_capacity) {
      const int32_t *src = reinterpret_cast<const int32_t *>(P.arena + e.y);
      for (uint32_t t = 0; t < cnt; t++) dst[t] = src[t];
    }
  } else {
    const WordSlot *slot = P.words + (res & SEG_WORD_SLOT_MASK);
    const uint4 e = *reinterpret_cast<const uint4 *>(&slot->meta);  // {meta, id0, id1, id2}
    dst[0] = static_cast<int32_t>(e.y);
    if (cnt > 1) dst[1] = static_cast<int32_t>(e.z);
    if (cnt > 2) dst[2] = static_cast<int32_t>(e.w);
    for (uint32_t t = 3; t < cnt; t++) dst[t] = slot->ids[t];
  }
}

// The rare block whose ids do not fit the staging buffer: every thread writes the ids of its own segments
// straight to the output, starting at `out0 + at` (segments with more than SCATTER_BIG ids are only listed).  Rolled (it re-reads its seg_result words instead of indexing registers): it
// must not bloat the kernel's hot loop.
__device__ __forceinline__ void scatter_direct(const EncodeParams &P, unsigned long long first, unsigned long long n_segs,
                                            unsigned long long out0, uint32_t at, uint32_t *big_at, uint32_t *big_si,
                                            uint32_t *n_big) {
  unsigned long long o = out0 + at;
#pragma unroll 1
  for (int j = 0; j < SCATTER_ITEMS; j++) {
    if (first + j >= n_segs) break;
    const uint32_t res = P.seg_result[first + j];
    uint32_t cnt = 1u;
    if (res >= SEG_RESULT_WORD) {
      cnt = (res >> SEG_SLOW_INDEX_BITS) & ((res & SEG_RESULT_SLOW) ? SEG_SLOW_COUNT_MAX : 0xFu);
      if (cnt == SEG_SLOW_COUNT_MAX && (res & SEG_RESULT_SLOW)) {
        const uint32_t si = res & SEG_SLOW_INDEX_MASK;
        cnt = si < P.slow_capacity ? (P.slow[si].off & ~SLOW_RESULT_INLINE) : 0u;
      }
    }
    if (cnt == 0) continue;
    if (res < SEG_RESULT_WORD) {
      if (o < P.capacity) P.ids[o] = static_cast<int32_t>(res) - 1;
    } else if ((res & SEG_RESULT_SLOW) && cnt > SCATTER_BIG && (res & SEG_SLOW_INDEX_MASK) < P.slow_capacity) {
      const uint32_t b = atomicAdd(n_big, 1u);  // left to the whole block (the caller copies the listed segments)
      big_at[b] = static_cast<uint32_t>(o - out0);
      big_si[b] = res & SEG_SLOW_INDEX_MASK;
    } else if (o + cnt <= P.capacity) {
      scatter_fetch(P, res, cnt, P.ids + o);
    } else {
      // the caller's buffer ends inside this segment (the call reports WP_ERR_CAPACITY): id by id
      int32_t tmp[WORD_MAX_IDS];
      if (cnt <= WORD_MAX_IDS) {
        scatter_fetch(P, res, cnt, tmp);
        for (uint32_t t = 0; t < cnt; t++) {
          if (o + t < P.capacity) P.ids[o + t] = tmp[t];
        }
      } else {  // more ids than a word slot holds: a slow entry with its ids in the arena
        const uint32_t si = res & SEG_SLOW_INDEX_MASK;
        if (si < P.slow_capacity) {
          const uint4 e = *reinterpret_cast<const uint4 *>(&P.slow[si]);
          if (static_cast<unsigned long long>(e.y) + cnt <= P.arena_capacity) {
            for (uint32_t t = 0; t < cnt; t++) {
              if (o + t < P.capacity) P.ids[o + t] = static_cast<int32_t>(P.arena[e.y + t]);
            }
          }
        }
      }
    }
    o += cnt;
  }
}

// A block whose ids do not fit the staging buffer because of a few LONG segments (URLs, blobs: hundreds of ids
// each) among ordinary ones — the usual shape of such a block.  The ids of the ordinary segments are staged
// densely (they fit), the long ones are left out of the buffer: staged id i goes to out0 + i + shift, where
// shift = the ids of all long segments before it.  Every long segment k records key_k = the staged ids before
// it and shift_k = the shift that holds behind it; the keys ascend, so a binary search finds the shift of a
// staged id.  Then the staged ids go out in order (coalesced but for the jumps) and every long segment is
// copied from the arena by one warp.  Returns false (uniform, nothing written) when the ordinary ids alone do
// not fit or there are too many long segments: the caller falls back to scatter_direct.  Out of line: rare.
constexpr uint32_t MIXED_MAX_BIG = SCATTER_SEGS / 2;  // keys in desc_pos[0..), shifts in desc_pos[MAX_BIG..), slow indices in desc_src

// what scatter_mixed needs of the kernel's parameters, by value (a reference to the parameter struct would make the
// kernel keep a copy of all of it in local memory)
struct ScatterView {
  const uint32_t *seg_result;
  const SlowEntry *slow;
  const uint32_t *arena;
  const WordSlot *words;
  volatile unsigned long long *block_state;
  CallCounters *call;
  int32_t *ids;
  unsigned long long capacity;
  uint32_t slow_capacity, arena_capacity, range_parity;
};

__device__ __noinline__ bool scatter_mixed(const ScatterView P, ScatterSmem &sm, unsigned long long first,
                                           unsigned long long n_segs, uint32_t b, uint32_t n_blocks,
                                           unsigned long long ids_in, uint32_t total, uint32_t at) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  auto count_of = [&](uint32_t res) -> uint32_t {
    if (res < SEG_RESULT_WORD) return 1u;
    uint32_t c = (res >> SEG_SLOW_INDEX_BITS) & ((res & SEG_RESULT_SLOW) ? SEG_SLOW_COUNT_MAX : 0xFu);
    if (c == SEG_SLOW_COUNT_MAX && (res & SEG_RESULT_SLOW)) {
      const uint32_t si = res & SEG_SLOW_INDEX_MASK;
      c = si < P.slow_capacity ? (P.slow[si].off & ~SLOW_RESULT_INLINE) : 0u;
    }
    return c;
  };
  auto is_big = [&](uint32_t res, uint32_t c) {
    return (res & SEG_RESULT_SLOW) && res >= SEG_RESULT_WORD && c > SCATTER_BIG && (res & SEG_SLOW_INDEX_MASK) < P.slow_capacity;
  };
  // pass 1: my ordinary ids and my long segments
  uint32_t my_small = 0, my_big = 0;
#pragma unroll 1
  for (int j = 0; j < SCATTER_ITEMS; j++) {
    if (first + j >= n_segs) break;
    const uint32_t res = P.seg_result[first + j];
    const uint32_t c = count_of(res);
    if (is_big(res, c)) my_big++;
    else my_small += c;
  }
  uint32_t totals;
  const uint32_t ex = block_exclusive_scan<SCATTER_THREADS / 32>(sm.warp_sums, my_small | (my_big << 16), &totals);
  const uint32_t n_small = totals & 0xFFFFu, n_big = totals >> 16;  // (at most 2048 x 15 ordinary ids: 16 bits hold them)
  if (n_small > SCATTER_STAGE || n_big > MIXED_MAX_BIG || n_big == 0) return false;  // uniform
  if (warp == 0) {
    const unsigned long long base = lookback_walk(P.block_state, b, total, lane);
    if (lane == 0) {
      sm.base = base;
      if (b == n_blocks - 1) P.call->ids_total[P.range_parity ^ 1u] = ids_in + base + total;
    }
  }
  // pass 2: stage the ordinary ids, list the long segments
  uint32_t spos = ex & 0xFFFFu, bk = ex >> 16, pos = at;
#pragma unroll 1
  for (int j = 0; j < SCATTER_ITEMS; j++) {
    if (first + j >= n_segs) break;
    const uint32_t res = P.seg_result[first + j];
    const uint32_t c = count_of(res);
    if (c == 0) continue;
    if (res < SEG_RESULT_WORD) {
      sm.stage[spos++] = static_cast<int32_t>(res) - 1;
    } else if (is_big(res, c)) {
      WP_CHECK(bk < MIXED_MAX_BIG);
      sm.desc_pos[bk] = spos;                          // key: staged ids before this segment
      sm.desc_pos[MIXED_MAX_BIG + bk] = pos + c - spos;  // shift of the staged ids behind it
      sm.desc_src[bk] = res & SEG_SLOW_INDEX_MASK;
      bk++;
    } else {
      WP_CHECK(spos + c <= SCATTER_STAGE);
      scatter_fetch(P, res, c, sm.stage + spos);
      spos += c;
    }
    pos += c;
  }
  __syncthreads();
  const unsigned long long out0 = ids_in + sm.base;
  // the staged ids
  for (uint32_t i = tid; i < n_small; i += SCATTER_THREADS) {
    uint32_t lo = 0, hi = n_big;  // number of keys <= i
    while (lo < hi) {
      const uint32_t mid = (lo + hi) >> 1;
      if (sm.desc_pos[mid] <= i) lo = mid + 1;
      else hi = mid;
    }
    const uint32_t shift = lo ? sm.desc_pos[MIXED_MAX_BIG + lo - 1] : 0u;
    const unsigned long long o = out0 + i + shift;
    WP_CHECK(i + shift < total);
    if (o < P.capacity) P.ids[o] = sm.stage[i];
  }
  // the long segments, one warp each
  for (uint32_t k = warp; k < n_big; k += SCATTER_THREADS / 32) {
    const uint32_t si = sm.desc_src[k];
    const uint4 e = *reinterpret_cast<const uint4 *>(&P.slow[si]);
    const uint32_t cnt = e.x & ~SLOW_RESULT_INLINE;
    if ((e.x & SLOW_RESULT_INLINE) || static_cast<unsigned long long>(e.y) + cnt > P.arena_capacity) continue;
    const unsigned long long o = out0 + (sm.desc_pos[MIXED_MAX_BIG + k] - cnt + sm.desc_pos[k]);
    WP_CHECK(sm.desc_pos[MIXED_MAX_BIG + k] + sm.desc_pos[k] <= total && sm.desc_pos[MIXED_MAX_BIG + k] + sm.desc_pos[k] >= cnt);
    for (uint32_t t = lane; t < cnt; t += 32) {
      if (o + t < P.capacity) P.ids[o + t] = static_cast<int32_t>(P.arena[e.y + t]);
    }
  }
  return true;
}

__global__ void __launch_bounds__(SCATTER_THREADS, WP_K3_BLOCKS) wp_scatter_kernel(EncodeParams P) {
  __shared__ ScatterSmem sm;
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  const unsigned long long n_segs = min(P.counters->n_segs, static_cast<unsigned long long>(P.seg_capacity));
  const uint32_t n_blocks = static_cast<uint32_t>((n_segs + SCATTER_SEGS - 1) / SCATTER_SEGS);
  const unsigned long long ids_in = P.call->ids_total[P.range_parity];
  if (P.call->overflow) return;  // uniform over the grid (K1 and K2 are done): the host retries the call
  if (n_blocks == 0) {
    if (blockIdx.x == 0 && tid == 0) P.call->ids_total[P.range_parity ^ 1u] = ids_in;
    return;
  }
  // The ticket of the NEXT block is taken when only the stores of this one are left, so that its round trip is
  // hidden behind them (two slots, used alternately).  Not earlier: every CTA with a later ticket waits in its
  // look-back for the total of the block whose ticket is being held, and a block that copies the ids of long
  // segments holds it for a long time (on blob-heavy text a quarter of the kernel's instructions were that spin).
  if (tid == 0) sm.block_index[0] = atomicAdd(&P.counters->scatter_ticket, 1u);
  for (uint32_t it = 0;; it++) {
    __syncthreads();
    const uint32_t b = sm.block_index[it & 1u];
    if (b >= n_blocks) break;
    if (tid == 0) {
      sm.n_desc = 0;
      sm.n_big = 0;
    }
    const unsigned long long first = static_cast<unsigned long long>(b) * SCATTER_SEGS + tid * SCATTER_ITEMS;
    {
      // blocks are handed out in order to gridDim.x CTAs: pull the words of the block two rounds ahead into L2
      const unsigned long long pf = (static_cast<unsigned long long>(b) + 2ull * gridDim.x) * SCATTER_SEGS + tid * 32ull;
      if (tid < SCATTER_SEGS / 32 && pf < n_segs) prefetch_l2(P.seg_result + pf);
    }

    // per-segment id counts, straight from the seg_result words (K1: 1; word table and slow: count bits).
    // Items past the last segment get a word that counts zero ids (SEG_RESULT_WORD with count 0).
    uint32_t res[SCATTER_ITEMS], cnt[SCATTER_ITEMS];
    if (first + SCATTER_ITEMS <= n_segs) {
      const uint4 a = *reinterpret_cast<const uint4 *>(P.seg_result + first);
      const uint4 c = *reinterpret_cast<const uint4 *>(P.seg_result + first + 4);
      res[0] = a.x; res[1] = a.y; res[2] = a.z; res[3] = a.w;
      res[4] = c.x; res[5] = c.y; res[6] = c.z; res[7] = c.w;
    } else {
#pragma unroll
      for (int j = 0; j < SCATTER_ITEMS; j++) res[j] = first + j < n_segs ? P.seg_result[first + j] : SEG_RESULT_WORD;
    }
    uint32_t mine = 0, n_other = 0;
#pragma unroll
    for (int j = 0; j < SCATTER_ITEMS; j++) {
      uint32_t c = 1u;
      if (res[j] >= SEG_RESULT_WORD) {
        c = (res[j] >> SEG_SLOW_INDEX_BITS) & ((res[j] & SEG_RESULT_SLOW) ? SEG_SLOW_COUNT_MAX : 0xFu);
        if (c == SEG_SLOW_COUNT_MAX && (res[j] & SEG_RESULT_SLOW)) {  // rare: 31 ids or more
          const uint32_t si = res[j] & SEG_SLOW_INDEX_MASK;
          c = si < P.slow_capacity ? (P.slow[si].off & ~SLOW_RESULT_INLINE) : 0u;  // word 0 of the result form
        }
        n_other += c != 0u;
      }
      cnt[j] = c;
      mine += c;
    }
    uint32_t total;
    uint32_t at = block_exclusive_scan<SCATTER_THREADS / 32>(sm.warp_sums, mine, &total);

    if (tid == 0) lookback_publish(P.block_state, b, total);

    if (total <= SCATTER_STAGE) {
      // stage in shared memory, then write out coalesced.  Ids settled by K1 are placed at once; the other
      // segments are listed (one reservation per warp) and fetched one per thread, all lanes busy (inline
      // they would leave most lanes of a warp idle behind the few that have one).
      uint32_t d = n_other;  // exclusive prefix within the warp, then + the warp's place in the list
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(FULL, d, o);
        if (lane >= o) d += y;
      }
      uint32_t wbase = 0;
      if (lane == 31 && d) wbase = smem_add(&sm.n_desc, d);
      d = d - n_other + __shfl_sync(FULL, wbase, 31);
#pragma unroll
      for (int j = 0; j < SCATTER_ITEMS; j++) {
        WP_CHECK(at + cnt[j] <= total && total <= SCATTER_STAGE);
        if (res[j] < SEG_RESULT_WORD) {
          sm.stage[at] = static_cast<int32_t>(res[j]) - 1;
        } else if (cnt[j] != 0) {
          WP_CHECK(d < SCATTER_SEGS);
          sm.desc_pos[d] = (at << 16) | cnt[j];
          sm.desc_src[d] = res[j];
          d++;
        }
        at += cnt[j];
      }
      __syncthreads();
      const uint32_t n_desc = sm.n_desc;
      for (uint32_t i = tid; i < n_desc; i += SCATTER_THREADS) {
        const uint32_t dp = sm.desc_pos[i], src = sm.desc_src[i];
        if ((src & SEG_RESULT_SLOW) && (dp & 0xFFFFu) > SCATTER_BIG) {
          const uint32_t slot = atomicAdd(&sm.n_big, 1u);  // (ids in the arena; one thread would take ages)
          WP_CHECK(slot < SCATTER_STAGE / SCATTER_BIG + 2);
          sm.big[slot] = static_cast<uint16_t>(i);
        } else {
          scatter_fetch(P, src, dp & 0xFFFFu, sm.stage + (dp >> 16));
        }
      }
      // the ids are staged; only now the block needs its place in the output
      if (warp == 0) {
        const unsigned long long base = lookback_walk(P.block_state, b, total, lane);
        if (lane == 0) {
          sm.base = base;
          if (b == n_blocks - 1) P.call->ids_total[P.range_parity ^ 1u] = ids_in + base + total;
        }
      }
      __syncthreads();
      if (sm.n_big) {  // uniform: the longer segments of this block, one warp each
        for (uint32_t bi = warp; bi < sm.n_big; bi += SCATTER_THREADS / 32) {
          const uint32_t dp = sm.desc_pos[sm.big[bi]], si = sm.desc_src[sm.big[bi]] & SEG_SLOW_INDEX_MASK;
          if (si >= P.slow_capacity) continue;
          const uint4 e = *reinterpret_cast<const uint4 *>(&P.slow[si]);
          const uint32_t cnt = dp & 0xFFFFu;
          if ((e.x & SLOW_RESULT_INLINE) || static_cast<unsigned long long>(e.y) + cnt > P.arena_capacity) continue;
          for (uint32_t t = lane; t < cnt; t += 32) sm.stage[(dp >> 16) + t] = static_cast<int32_t>(P.arena[e.y + t]);
        }
        __syncthreads();
      }
      if (tid == 0) sm.block_index[(it + 1u) & 1u] = atomicAdd(&P.counters->scatter_ticket, 1u);
      const unsigned long long out0 = ids_in + sm.base;
      if (out0 + total <= P.capacity) {
        // 16-byte stores: a scalar head up to the first 16-byte boundary of the output, vectors, a scalar tail
        int32_t *dst = P.ids + out0;
        const uint32_t head = min(total, static_cast<uint32_t>((4u - ((reinterpret_cast<uintptr_t>(dst) >> 2) & 3u)) & 3u));
        const uint32_t n_vec = (total - head) >> 2;
        if (tid < head) dst[tid] = sm.stage[tid];
        for (uint32_t q = tid; q < n_vec; q += SCATTER_THREADS) {
          const uint32_t i = head + 4u * q;
          *reinterpret_cast<int4 *>(dst + i) = make_int4(sm.stage[i], sm.stage[i + 1], sm.stage[i + 2], sm.stage[i + 3]);
        }
        const uint32_t done = head + 4u * n_vec;
        if (tid < total - done) dst[done + tid] = sm.stage[done + tid];
      } else {
        for (uint32_t i = tid; i < total; i += SCATTER_THREADS) {
          if (out0 + i < P.capacity) P.ids[out0 + i] = sm.stage[i];
        }
      }
    } else {
      // a block with unusually many ids (long words cut into many pieces).  Usually a few long segments among
      // ordinary ones: those are kept out of the staging buffer (scatter_mixed)
      const ScatterView view{P.seg_result, P.slow, P.arena, P.words, P.block_state, P.call, P.ids,
                             static_cast<unsigned long long>(P.capacity), P.slow_capacity, P.arena_capacity, P.range_parity};
      if (scatter_mixed(view, sm, first, n_segs, b, n_blocks, ids_in, total, at)) {  // uniform
        if (tid == 0) sm.block_index[(it + 1u) & 1u] = atomicAdd(&P.counters->scatter_ticket, 1u);
        continue;
      }
      // otherwise: write directly
      if (warp == 0) {
        const unsigned long long base = lookback_walk(P.block_state, b, total, lane);
        if (lane == 0) {
          sm.base = base;
          if (b == n_blocks - 1) P.call->ids_total[P.range_parity ^ 1u] = ids_in + base + total;
        }
      }
      __syncthreads();
      const unsigned long long out0 = ids_in + sm.base;
      scatter_direct(P, first, n_segs, out0, at, sm.desc_pos, sm.desc_src, &sm.n_big);
      __syncthreads();
      for (uint32_t bi = warp; bi < sm.n_big; bi += SCATTER_THREADS / 32) {  // its longer segments: (offset in the block's ids, slow index)
        const uint32_t si = sm.desc_src[bi];
        const unsigned long long o = out0 + sm.desc_pos[bi];
        const uint4 e = *reinterpret_cast<const uint4 *>(&P.slow[si]);
        const uint32_t cnt = e.x & ~SLOW_RESULT_INLINE;
        if ((e.x & SLOW_RESULT_INLINE) || static_cast<unsigned long long>(e.y) + cnt > P.arena_capacity) continue;
        for (uint32_t t = lane; t < cnt; t += 32) {
          if (o + t < P.capacity) P.ids[o + t] = static_cast<int32_t>(P.arena[e.y + t]);
        }
      }
      if (tid == 0) sm.block_index[(it + 1u) & 1u] = atomicAdd(&P.counters->scatter_ticket, 1u);
    }
  }
}

// ======================================================= K5: text id offsets
//
// Batch calls (wp_encode_batch, wp_encode_batch_device): where do the ids of every text begin?  K1 has numbered
// the first segment of every text (bound_seg); the ids before segment s are the inclusive prefix K3 left in
// block_state for the block before s's, plus the id counts of the segments of s's block that lie before s.  One
// warp per text.  The texts [i0, i1) that start in the range come from the host (a grid that covers them), or,
// `from_tiles`, from the tile index on the device (a fixed grid that strides over them).
__device__ __forceinline__ uint32_t seg_id_count(const EncodeParams &P, uint32_t res) {
  if (res < SEG_RESULT_WORD) return 1u;
  uint32_t c = (res >> SEG_SLOW_INDEX_BITS) & ((res & SEG_RESULT_SLOW) ? SEG_SLOW_COUNT_MAX : 0xFu);
  if (c == SEG_SLOW_COUNT_MAX && (res & SEG_RESULT_SLOW)) {  // rare: 31 ids or more, the count is in the slow entry
    const uint32_t si = res & SEG_SLOW_INDEX_MASK;
    c = si < P.slow_capacity ? (P.slow[si].off & ~SLOW_RESULT_INLINE) : 0u;
  }
  return c;
}

constexpr int OFFSET_THREADS = 128;

__global__ void __launch_bounds__(OFFSET_THREADS) wp_text_offsets_kernel(EncodeParams P, uint32_t i0, uint32_t i1,
                                                                         uint32_t from_tiles) {
  const int lane = threadIdx.x & 31;
  if (from_tiles) {
    i0 = P.tile_bound[P.first_tile];
    i1 = P.tile_bound[P.first_tile + P.n_tiles];
  }
  if (P.call->overflow) return;
  const unsigned long long n_segs = min(P.counters->n_segs, static_cast<unsigned long long>(P.seg_capacity));
  const uint32_t warps = gridDim.x * (OFFSET_THREADS / 32);
#pragma unroll 1
  for (uint32_t i = i0 + blockIdx.x * (OFFSET_THREADS / 32) + (threadIdx.x >> 5); i < i1; i += warps) {
    const unsigned long long s = min(static_cast<unsigned long long>(P.bound_seg[i]), n_segs);
    const uint32_t blk = static_cast<uint32_t>(s / SCATTER_SEGS);
    const unsigned long long first = static_cast<unsigned long long>(blk) * SCATTER_SEGS;
    unsigned long long sum = 0;
    for (unsigned long long k = first + lane; k < s; k += 32) sum += seg_id_count(P, P.seg_result[k]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(FULL, sum, o);
    if (lane == 0) {
      const unsigned long long before = blk ? (P.block_state[blk - 1] & ((1ull << 62) - 1)) : 0ull;
      P.id_offsets[i] = P.call->ids_total[P.range_parity] + before + sum;  // ([parity] still holds the range's first id)
    }
  }
}

cudaError_t launch_text_offsets(const EncodeParams &P, uint32_t i0, uint32_t i1, cudaStream_t stream, uint64_t *launches) {
  if (i1 <= i0) return cudaSuccess;
  const uint32_t per = OFFSET_THREADS / 32;
  wp_text_offsets_kernel<<<(i1 - i0 + per - 1) / per, OFFSET_THREADS, 0, stream>>>(P, i0, i1, 0u);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

cudaError_t launch_text_offsets_device(const EncodeParams &P, int sm_count, cudaStream_t stream, uint64_t *launches) {
  if (sm_count <= 0) sm_count = 148;
  // (the host does not know how many texts start in the range: 16 x 4 warps per SM stride over them)
  wp_text_offsets_kernel<<<sm_count * 16, OFFSET_THREADS, 0, stream>>>(P, 0u, 0u, 1u);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

// ================================================= device string column -> packed text (wp_encode_batch_device)
//
// A column (Arrow layout: text i = chars[offsets[i] .. offsets[i + 1])) is packed as wp_encode_batch packs host
// texts: text i at start(i) = offsets[i] - offsets[0] + i, followed by one space; the tail up to the packed length
// n_chars + n_texts is spaces.  The source byte of a text byte at packed position p is p + offsets[0] - j, j its
// text: the copy shifts by one at every separator.  Check first, then pack: a column whose offsets do not ascend
// within [0, n_chars] sets *bad, and the packer then lays out n_texts empty texts (all spaces, start(i) = i) and
// reads no char, so the kernels that follow index nothing out of range.

constexpr int COLUMN_THREADS = 256;  // packer: 16 bytes of one tile per thread

__global__ void __launch_bounds__(COLUMN_THREADS) wp_column_check_kernel(ColumnArgs A) {
  const unsigned long long i = static_cast<unsigned long long>(blockIdx.x) * COLUMN_THREADS + threadIdx.x;
  if (i >= A.n_texts) return;
  const unsigned long long a = A.offsets[i], b = A.offsets[i + 1];
  if (a > b || b > A.n_chars) *A.bad = 1u;
}

struct ColumnSmem {
  uint4 src[TILE / 16 + 2];   // the tile's source chars, from the 16-byte unit that holds the first one
  uint32_t sep[TILE / 32];    // bit p: packed position ts + p is a separator
  uint32_t scan[TILE / 32];   // separators in the words before
  uint32_t warp_sum[4];
  uint32_t found[2];          // the first text that starts at or after ts (te)
};

__global__ void __launch_bounds__(COLUMN_THREADS) wp_column_pack_kernel(ColumnArgs A) {
  __shared__ ColumnSmem sm;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t t = blockIdx.x, n = A.n_texts;
  const bool bad = *A.bad != 0u;
  const unsigned long long off0 = bad ? 0ull : A.offsets[0];
  // start(j) for j in [0, n]; start(n) = the end of the last separator
  auto start = [&](uint32_t j) -> unsigned long long {
    WP_CHECK(j <= n);
    return bad ? static_cast<unsigned long long>(j) : A.offsets[j] - off0 + j;
  };
  const unsigned long long ts = static_cast<unsigned long long>(t) * TILE, te = ts + TILE;
  if (tid < TILE / 32) sm.sep[tid] = 0u;
  if (warp < 2) {
    // the first j in [0, n) with start(j) >= x (n if none): a 32-way search, warp 0 for ts, warp 1 for te
    const unsigned long long x = warp ? te : ts;
    uint32_t lo = 0, hi = n;
    while (hi > lo) {
      const uint32_t span = hi - lo;
      const uint32_t p = lo + static_cast<uint32_t>(static_cast<unsigned long long>(span) * lane / 32);
      const uint32_t ge = __ballot_sync(FULL, start(p) >= x);
      const int k = ge ? __ffs(ge) - 1 : 32;  // lanes probe ascending positions: the first lane at or past x
      const uint32_t nhi = k < 32 ? lo + static_cast<uint32_t>(static_cast<unsigned long long>(span) * k / 32) : hi;
      lo = k > 0 ? lo + static_cast<uint32_t>(static_cast<unsigned long long>(span) * (k - 1) / 32) + 1 : lo;
      hi = nhi;
    }
    if (lane == 0) sm.found[warp] = lo;
  }
  __syncthreads();
  const uint32_t a = sm.found[0], b = sm.found[1];
  WP_CHECK(a <= b && b <= n);
  const unsigned long long end = start(n);
  const uint32_t j0 = (a > 0 && start(a) > ts) ? a - 1 : a;  // the text that holds position ts (n: the tail)
  // text starts and the tile index
  for (uint32_t i = a + tid; i < b; i += COLUMN_THREADS) {
    WP_CHECK(i < n);
    A.bounds[i] = start(i);
  }
  if (tid == 0) {
    WP_CHECK(t < A.n_tiles);
    A.tile_bound[t] = a;
    if (t + 1 == A.n_tiles) A.tile_bound[t + 1] = b;  // (= n: every text starts before the packed length)
  }
  // separators in the tile: those of the texts [j0, b)
  const uint32_t j_end = b < n ? b : n;
  for (uint32_t j = j0 + tid; j < j_end; j += COLUMN_THREADS) {
    const unsigned long long s = start(j + 1) - 1;
    if (s >= ts && s < te) atomicOr(&sm.sep[(s - ts) >> 5], 1u << ((s - ts) & 31u));
  }
  __syncthreads();
  if (warp < 4) {  // exclusive scan of the separator counts of the 128 words
    const uint32_t c = __popc(sm.sep[tid]);
    uint32_t inc = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t y = __shfl_up_sync(FULL, inc, o);
      if (lane >= o) inc += y;
    }
    sm.scan[tid] = inc - c;
    if (lane == 31) sm.warp_sum[warp] = inc;
  }
  __syncthreads();
  if (warp < 4) {
    for (int w = 0; w < warp; w++) sm.scan[tid] += sm.warp_sum[w];
  }
  const uint32_t n_sep = sm.warp_sum[0] + sm.warp_sum[1] + sm.warp_sum[2] + sm.warp_sum[3];
  // the source chars of the tile: [src_lo, src_lo + count), count = the positions before the tail that are no
  // separator (every separator of the tile lies before the tail)
  const unsigned long long tail = end > ts ? end - ts : 0ull;  // local position where the tail begins
  const unsigned long long lim = tail < static_cast<unsigned long long>(TILE) ? tail : static_cast<unsigned long long>(TILE);
  unsigned long long src_lo = j0 < n ? ts + off0 - j0 : 0ull;
  unsigned long long src_hi = j0 < n && lim > n_sep ? src_lo + (lim - n_sep) : src_lo;
  if (src_hi > A.n_chars) src_hi = A.n_chars;  // (clamps: only a malformed column, which reads nothing, could exceed)
  if (src_lo > src_hi) src_lo = src_hi;
  const uintptr_t lo_addr = reinterpret_cast<uintptr_t>(A.chars) + src_lo;
  const uintptr_t hi_addr = reinterpret_cast<uintptr_t>(A.chars) + src_hi;
  const uintptr_t base = lo_addr & ~uintptr_t(15);
  const uint32_t lead = static_cast<uint32_t>(lo_addr - base);
  __syncthreads();
  {
    const uint32_t units = static_cast<uint32_t>((hi_addr - base + 15) / 16);
    WP_CHECK(units <= TILE / 16 + 2);
    for (uint32_t u = tid; u < units; u += COLUMN_THREADS) {
      const uintptr_t at = base + 16u * u;
      if (at >= lo_addr && at + 16 <= hi_addr) {
        sm.src[u] = ldg_stream(reinterpret_cast<const uint4 *>(at));
      } else {  // a unit the column only partly covers: its bytes in [src_lo, src_hi) one by one
        uint8_t *d = reinterpret_cast<uint8_t *>(&sm.src[u]);
        for (int k = 0; k < 16; k++)
          if (at + k >= lo_addr && at + k < hi_addr) d[k] = *reinterpret_cast<const uint8_t *>(at + k);
      }
    }
  }
  __syncthreads();
  // 16 packed bytes per thread, one 16-byte store
  const uint32_t lp0 = 16u * tid;
  const uint32_t bits = (sm.sep[tid >> 1] >> (16u * (tid & 1))) & 0xFFFFu;
  uint32_t before = sm.scan[tid >> 1] + ((tid & 1) ? __popc(sm.sep[tid >> 1] & 0xFFFFu) : 0u);
  const uint8_t *src = reinterpret_cast<const uint8_t *>(sm.src);
  uint32_t out[4];
  if (bits == 0 && lp0 + 16u <= lim) {  // text only: 16 consecutive source chars
    const uint32_t q = lp0 - before + lead;
    WP_CHECK(q + 16u <= 16u * (TILE / 16 + 2));
    const uint32_t *w = reinterpret_cast<const uint32_t *>(sm.src) + (q >> 2);
    const uint32_t sh = 8u * (q & 3u);
#pragma unroll
    for (int k = 0; k < 4; k++) out[k] = sh ? __funnelshift_r(w[k], w[k + 1], sh) : w[k];
  } else {
#pragma unroll
    for (int k = 0; k < 4; k++) out[k] = 0u;
#pragma unroll
    for (int k = 0; k < 16; k++) {
      const uint32_t lp = lp0 + k;
      uint32_t c = 0x20u;
      if ((bits >> k) & 1u) {
        before++;
      } else if (lp < lim) {
        const uint32_t q = lp - before + lead;
        WP_CHECK(q < 16u * (TILE / 16 + 2) && base + q < hi_addr);
        c = src[q];
      }
      out[k >> 2] |= c << (8 * (k & 3));
    }
  }
  *reinterpret_cast<uint4 *>(A.text + ts + lp0) = make_uint4(out[0], out[1], out[2], out[3]);
}

cudaError_t launch_column_pack(const ColumnArgs &A, cudaStream_t stream, uint64_t *launches) {
  wp_column_check_kernel<<<static_cast<unsigned>((A.n_texts + COLUMN_THREADS - 1) / COLUMN_THREADS), COLUMN_THREADS, 0,
                           stream>>>(A);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  wp_column_pack_kernel<<<A.n_tiles, COLUMN_THREADS, 0, stream>>>(A);
  if (launches) *launches += 2;
  return cudaGetLastError();
}

// ============================================================== K4: format
//
// ids -> the reference's output wire format, every id in decimal followed by one space (fast.cpp:214-216,
// utils.cpp:30-35: `"id id id "`), for the streaming entry point (encodeExternal).  Two kernels: the total
// length, then the text (per-block scan of the lengths, decoupled look-back, chars staged in shared memory).

constexpr int FORMAT_THREADS = 256;
constexpr int FORMAT_ITEMS = 8;
constexpr int FORMAT_IDS = FORMAT_THREADS * FORMAT_ITEMS;  // 2048 ids per block iteration
constexpr int FORMAT_MAX_CHARS = 12;                       // "-2147483648 "

__device__ __forceinline__ uint32_t decimal_chars(int32_t v) {  // digits + sign + the trailing space
  const uint32_t a = v < 0 ? 0u - static_cast<uint32_t>(v) : static_cast<uint32_t>(v);
  uint32_t n = 2u + (v < 0 ? 1u : 0u);
  n += a >= 10u;
  n += a >= 100u;
  n += a >= 1000u;
  n += a >= 10000u;
  n += a >= 100000u;
  n += a >= 1000000u;
  n += a >= 10000000u;
  n += a >= 100000000u;
  n += a >= 1000000000u;
  return n;
}

__global__ void __launch_bounds__(FORMAT_THREADS) wp_format_total_kernel(const int32_t *__restrict__ ids,
                                                                         unsigned long long n,
                                                                         unsigned long long *total) {
  __shared__ unsigned long long warp_sums[FORMAT_THREADS / 32];
  unsigned long long mine = 0;
  for (unsigned long long i = static_cast<unsigned long long>(blockIdx.x) * FORMAT_THREADS + threadIdx.x; i < n;
       i += static_cast<unsigned long long>(gridDim.x) * FORMAT_THREADS)
    mine += decimal_chars(ids[i]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(FULL, mine, o);
  if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = mine;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long s = 0;
    for (int w = 0; w < FORMAT_THREADS / 32; w++) s += warp_sums[w];
    if (s) atomicAdd(total, s);
  }
}

struct FormatSmem {
  uint8_t stage[FORMAT_IDS * FORMAT_MAX_CHARS];
  uint32_t warp_sums[FORMAT_THREADS / 32];
  uint32_t block_index;
  unsigned long long base;
};

__global__ void __launch_bounds__(FORMAT_THREADS) wp_format_kernel(const int32_t *__restrict__ ids, unsigned long long n,
                                                                   char *__restrict__ out, unsigned long long *block_state,
                                                                   unsigned int *ticket) {
  __shared__ FormatSmem sm;
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const uint32_t n_blocks = static_cast<uint32_t>((n + FORMAT_IDS - 1) / FORMAT_IDS);
  for (;;) {
    __syncthreads();
    if (tid == 0) sm.block_index = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint32_t b = sm.block_index;
    if (b >= n_blocks) break;
    const unsigned long long first = static_cast<unsigned long long>(b) * FORMAT_IDS + tid * FORMAT_ITEMS;
    int32_t v[FORMAT_ITEMS];
    uint32_t len[FORMAT_ITEMS], mine = 0;
#pragma unroll
    for (int j = 0; j < FORMAT_ITEMS; j++) {
      v[j] = first + j < n ? ids[first + j] : 0;
      len[j] = first + j < n ? decimal_chars(v[j]) : 0u;
      mine += len[j];
    }
    uint32_t total;
    uint32_t at = block_exclusive_scan<FORMAT_THREADS / 32>(sm.warp_sums, mine, &total);
    if (tid == 0) lookback_publish(block_state, b, total);
#pragma unroll
    for (int j = 0; j < FORMAT_ITEMS; j++) {
      if (len[j] == 0) continue;
      uint32_t a = v[j] < 0 ? 0u - static_cast<uint32_t>(v[j]) : static_cast<uint32_t>(v[j]);
      uint32_t p = at + len[j] - 1;
      sm.stage[p--] = ' ';
      do {
        sm.stage[p--] = static_cast<uint8_t>('0' + a % 10u);
        a /= 10u;
      } while (a != 0u);
      if (v[j] < 0) sm.stage[p] = '-';
      at += len[j];
    }
    __syncthreads();
    if (tid < 32) {
      const unsigned long long base = lookback_walk(block_state, b, total, lane);
      if (lane == 0) sm.base = base;
    }
    __syncthreads();
    char *dst = out + sm.base;
    for (uint32_t i = tid; i < total; i += FORMAT_THREADS) dst[i] = static_cast<char>(sm.stage[i]);
  }
}

cudaError_t launch_format_total(const int32_t *ids, size_t n, unsigned long long *total, int sm_count,
                                cudaStream_t stream, uint64_t *launches) {
  if (sm_count <= 0) sm_count = 148;
  wp_format_total_kernel<<<sm_count * 8, FORMAT_THREADS, 0, stream>>>(ids, n, total);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

cudaError_t launch_format(const int32_t *ids, size_t n, char *out, unsigned long long *block_state, unsigned int *ticket,
                          int sm_count, cudaStream_t stream, uint64_t *launches) {
  if (sm_count <= 0) sm_count = 148;
  wp_format_kernel<<<sm_count * 4, FORMAT_THREADS, 0, stream>>>(ids, n, out, block_state, ticket);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

uint32_t format_block_ids() { return FORMAT_IDS; }

// ============================================================== decode
//
// ids -> one entry per id of the token text fast::decode gives it (fast.cpp:165-187), empty where the reference
// skips the id.  The shape of K4: a length pass (total bytes, skipped ids, the id == size flag), then blocks by
// ticket that scan their ids' lengths, publish the block total, write their offsets and copy their bytes.  The
// bytes of one block go out through a shared-memory stage in WINDOWS of DECODE_STAGE bytes aligned to 16 bytes of
// the output: for each window every id copies the part of its token that falls inside it, then the window is
// stored with 16-byte stores (byte stores only at the two ends of the block's range, which neighbours share).
// Any block output size takes the same path: a block of 2 048 tokens of 400 bytes is 50 windows.

constexpr int DECODE_THREADS = 256;
constexpr int DECODE_ITEMS = 8;
constexpr int DECODE_IDS = DECODE_THREADS * DECODE_ITEMS;  // 2048 ids per block iteration
constexpr int DECODE_STAGE = 16384;                        // bytes per window (= DECODE_IDS offsets of 8 bytes)
constexpr int DECODE_BLOCKS = 4;                           // CTAs per SM (launch bound and grid)
static_assert(DECODE_STAGE == DECODE_IDS * 8, "the stage holds the block's relative offsets before its bytes");

// bytes of id's entry (0 if skipped); *bad |= id == size
__device__ __forceinline__ uint2 decode_entry(const DecodeArgs &A, int32_t id, bool *bad) {
  if (id < 0 || static_cast<uint32_t>(id) >= A.vocab_size) {
    *bad |= static_cast<uint32_t>(id) == A.vocab_size;
    return make_uint2(0u, 0u);
  }
  WP_CHECK(static_cast<uint32_t>(id) < A.vocab_size);
  const uint2 d = A.desc[id];
  return (d.y & DECODE_SKIP) ? make_uint2(0u, 0u) : d;
}

__global__ void __launch_bounds__(DECODE_THREADS) wp_decode_total_kernel(DecodeArgs A) {
  __shared__ unsigned long long sums[2][DECODE_THREADS / 32];
  unsigned long long bytes = 0, skipped = 0;
  bool bad = false;
  for (unsigned long long i = static_cast<unsigned long long>(blockIdx.x) * DECODE_THREADS + threadIdx.x; i < A.n_ids;
       i += static_cast<unsigned long long>(gridDim.x) * DECODE_THREADS) {
    const uint32_t len = decode_entry(A, A.ids[i], &bad).y;
    bytes += len;
    skipped += len == 0u;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    bytes += __shfl_xor_sync(FULL, bytes, o);
    skipped += __shfl_xor_sync(FULL, skipped, o);
  }
  bad = __syncthreads_or(bad);
  if ((threadIdx.x & 31) == 0) {
    sums[0][threadIdx.x >> 5] = bytes;
    sums[1][threadIdx.x >> 5] = skipped;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long b = 0, s = 0;
    for (int w = 0; w < DECODE_THREADS / 32; w++) {
      b += sums[0][w];
      s += sums[1][w];
    }
    if (b) atomicAdd(&A.work[0], b);
    if (s) atomicAdd(&A.work[1], s);
    if (bad) atomicOr(&A.work[2], 1ull);
  }
}

struct DecodeSmem {
  __align__(16) uint8_t stage[DECODE_STAGE];
  unsigned long long warp_sums[DECODE_THREADS / 32];
  uint32_t block_index;
  unsigned long long base;
};

__global__ void __launch_bounds__(DECODE_THREADS, DECODE_BLOCKS) wp_decode_kernel(DecodeArgs A) {
  __shared__ DecodeSmem sm;
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const unsigned long long n = A.n_ids;
  // (an async call that needs more than capacity, or met an id == size, writes nothing but the void count)
  if (A.work[2] != 0ull || A.work[0] > A.capacity) {
    if (blockIdx.x == 0 && tid == 0) A.offsets[n] = ~0ull;
    return;
  }
  unsigned long long *const block_state = A.work + 4;
  unsigned int *const ticket = reinterpret_cast<unsigned int *>(A.work + 3);
  unsigned long long *const rel = reinterpret_cast<unsigned long long *>(sm.stage);
  const uint32_t n_blocks = static_cast<uint32_t>((n + DECODE_IDS - 1) / DECODE_IDS);
  for (;;) {
    __syncthreads();
    if (tid == 0) sm.block_index = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint32_t b = sm.block_index;
    if (b >= n_blocks) break;
    const unsigned long long block_first = static_cast<unsigned long long>(b) * DECODE_IDS;
    const uint32_t count = static_cast<uint32_t>(n - block_first < DECODE_IDS ? n - block_first : DECODE_IDS);
    const uint32_t first = tid * DECODE_ITEMS;  // within the block
    uint2 e[DECODE_ITEMS];
    unsigned long long mine = 0;
    bool bad = false;
#pragma unroll
    for (int j = 0; j < DECODE_ITEMS; j++) {
      e[j] = first + j < count ? decode_entry(A, A.ids[block_first + first + j], &bad) : make_uint2(0u, 0u);
      mine += e[j].y;
    }
    unsigned long long total;
    unsigned long long at = block_exclusive_scan<DECODE_THREADS / 32>(sm.warp_sums, mine, &total);
    if (tid == 0) lookback_publish(A.work + 4, b, total);
#pragma unroll
    for (int j = 0; j < DECODE_ITEMS; j++) {
      if (first + j < count) {
        WP_CHECK(first + j < DECODE_IDS);
        rel[first + j] = at;
      }
      at += e[j].y;
    }
    __syncthreads();
    if (tid < 32) {
      const unsigned long long base = lookback_walk(block_state, b, total, lane);
      if (lane == 0) sm.base = base;
    }
    __syncthreads();
    const unsigned long long base = sm.base;
    for (uint32_t i = tid; i < count; i += DECODE_THREADS) {
      WP_CHECK(block_first + i < n);
      A.offsets[block_first + i] = base + rel[i];
    }
    if (block_first + count == n && tid == 0) A.offsets[n] = base + total;
    // the block's bytes [base, base + total) of the output, in windows aligned to 16 bytes of the output address
    WP_CHECK(base + total <= A.capacity);
    const uintptr_t lo = reinterpret_cast<uintptr_t>(A.out) + base, hi = lo + total;
    at -= mine;  // back to this thread's first entry
    for (uintptr_t w = lo & ~static_cast<uintptr_t>(15); w < hi; w += DECODE_STAGE) {
      __syncthreads();  // (the stage: the offsets above, or the previous window, have been stored)
      const uintptr_t w_end = w + DECODE_STAGE < hi ? w + DECODE_STAGE : hi;
      unsigned long long s = at;
#pragma unroll
      for (int j = 0; j < DECODE_ITEMS; j++) {
        const uintptr_t t0 = lo + s, t1 = t0 + e[j].y;
        const uintptr_t c0 = t0 > w ? t0 : w, c1 = t1 < w_end ? t1 : w_end;
        const uint8_t *src = A.bytes + e[j].x + (c0 - t0);
#pragma unroll 4
        for (uintptr_t c = c0; c < c1; c++, src++) {
          WP_CHECK(c - w < DECODE_STAGE && src < A.bytes + e[j].x + e[j].y);
          sm.stage[c - w] = *src;
        }
        s += e[j].y;
      }
      __syncthreads();
      for (uintptr_t u = w + 16u * tid; u < w_end; u += 16u * DECODE_THREADS) {
        WP_CHECK(u - w + 16u <= DECODE_STAGE);
        if (u >= lo && u + 16u <= hi) {
          *reinterpret_cast<uint4 *>(u) = *reinterpret_cast<const uint4 *>(sm.stage + (u - w));
        } else {
          for (uintptr_t k = u; k < u + 16u; k++)
            if (k >= lo && k < hi) {
              WP_CHECK(k - reinterpret_cast<uintptr_t>(A.out) < A.capacity);
              *reinterpret_cast<uint8_t *>(k) = sm.stage[k - w];
            }
        }
      }
    }
  }
}

uint32_t decode_block_ids() { return DECODE_IDS; }

cudaError_t launch_decode_total(const DecodeArgs &A, int sm_count, cudaStream_t stream, uint64_t *launches) {
  if (sm_count <= 0) sm_count = 148;
  wp_decode_total_kernel<<<sm_count * 8, DECODE_THREADS, 0, stream>>>(A);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

cudaError_t launch_decode(const DecodeArgs &A, int sm_count, cudaStream_t stream, uint64_t *launches) {
  if (sm_count <= 0) sm_count = 148;
  wp_decode_kernel<<<sm_count * DECODE_BLOCKS, DECODE_THREADS, 0, stream>>>(A);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

// ============================================================== model-input rows
//
// Per-text ids (ids + Arrow id offsets) -> fixed-length rows of max_len ids: [cls]? content [sep]? pad ..., and a
// mask that is 1 on cls, content and sep.  Text t of n_t ids has r_t = 1 row if stride == 0 or n_t <= W, else
// 1 + ceil((n_t - W) / stride); row k holds the text's ids [k stride, min(k stride + W, n_t)).  The shape of the
// decode pair: a scan kernel hands out blocks of 2 048 texts by ticket, counts their rows, scans them (64-bit block
// scan, decoupled look-back) and writes the row offsets; the fill kernel is driven by ROW, so that one text of
// millions of rows spreads over the whole GPU.  Each CTA takes tiles of ROWS_TILE consecutive rows: one 32-way
// search over the row offsets finds the tile's first text, the tile's texts (at most ROWS_TILE, every text has a
// row) are staged in shared memory, and each warp writes whole rows.  A row is a span of the flat output: its
// interior goes out in 16-byte stores, only its ends (< 16 bytes each) in 4-byte (ids) or 1-byte (mask) stores.

constexpr int ROWS_THREADS = 256;
constexpr int ROWS_ITEMS = 8;
constexpr int ROWS_TEXTS = ROWS_THREADS * ROWS_ITEMS;  // 2048 texts per scan block
constexpr int ROWS_SCAN_BLOCKS = 4;                    // scan CTAs per SM (launch bound and grid)
constexpr int ROWS_TILE = 128;                         // rows per fill tile
constexpr int ROWS_FILL_BLOCKS = 6;                    // fill CTAs per SM (launch bound and grid)

// rows of text t; *bad |= its offsets descend or end past n_ids (such a text counts one row: the call is void)
__device__ __forceinline__ unsigned long long rows_of_text(const RowsArgs &A, unsigned long long t, bool *bad) {
  WP_CHECK(t < A.n_texts);
  const unsigned long long a = A.id_offsets[t], b = A.id_offsets[t + 1];
  if (a > b || b > A.n_ids) {
    *bad = true;
    return 1ull;
  }
  const unsigned long long n = b - a;
  return A.stride == 0u || n <= A.width ? 1ull : 1ull + (n - A.width + A.stride - 1u) / A.stride;
}

struct RowsScanSmem {
  unsigned long long rel[ROWS_TEXTS];  // the block's row offsets relative to its first row
  unsigned long long warp_sums[ROWS_THREADS / 32];
  uint32_t block_index;
  unsigned long long base;
};

__global__ void __launch_bounds__(ROWS_THREADS, ROWS_SCAN_BLOCKS) wp_rows_scan_kernel(RowsArgs A) {
  __shared__ RowsScanSmem sm;
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const unsigned long long n = A.n_texts;
  unsigned long long *const block_state = A.work + 3;
  unsigned int *const ticket = reinterpret_cast<unsigned int *>(A.work + 2);
  const uint32_t n_blocks = static_cast<uint32_t>((n + ROWS_TEXTS - 1) / ROWS_TEXTS);
  bool bad = false;
  for (;;) {
    __syncthreads();
    if (tid == 0) sm.block_index = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint32_t b = sm.block_index;
    if (b >= n_blocks) break;
    const unsigned long long block_first = static_cast<unsigned long long>(b) * ROWS_TEXTS;
    const uint32_t count = static_cast<uint32_t>(n - block_first < ROWS_TEXTS ? n - block_first : ROWS_TEXTS);
    const uint32_t first = tid * ROWS_ITEMS;  // within the block
    unsigned long long r[ROWS_ITEMS], mine = 0;
#pragma unroll
    for (int j = 0; j < ROWS_ITEMS; j++) {
      r[j] = first + j < count ? rows_of_text(A, block_first + first + j, &bad) : 0ull;
      mine += r[j];
    }
    unsigned long long total;
    unsigned long long at = block_exclusive_scan<ROWS_THREADS / 32>(sm.warp_sums, mine, &total);
    if (tid == 0) lookback_publish(block_state, b, total);
#pragma unroll
    for (int j = 0; j < ROWS_ITEMS; j++) {
      if (first + j < count) {
        WP_CHECK(first + j < ROWS_TEXTS);
        sm.rel[first + j] = at;
      }
      at += r[j];
    }
    __syncthreads();
    if (tid < 32) {
      const unsigned long long base = lookback_walk(block_state, b, total, lane);
      if (lane == 0) sm.base = base;
    }
    __syncthreads();
    const unsigned long long base = sm.base;
    for (uint32_t i = tid; i < count; i += ROWS_THREADS) {
      WP_CHECK(block_first + i < n);
      A.row_offsets[block_first + i] = base + sm.rel[i];
    }
    if (block_first + count == n && tid == 0) {
      A.row_offsets[n] = base + total;
      A.work[0] = base + total;
    }
  }
  bad = __syncthreads_or(bad);
  if (bad && tid == 0) atomicOr(&A.work[1], 1ull);
}

struct RowsFillSmem {
  unsigned long long row_off[ROWS_TILE + 1];  // row and id offsets of the texts t0 .. t0 + n_local
  unsigned long long id_off[ROWS_TILE + 1];
  unsigned long long t0;                      // the text of the tile's first row
};

// 16 mask bytes starting at column c: byte i is 1 if c + i < valid
__device__ __forceinline__ uint4 mask_unit(uint32_t c, uint32_t valid) {
  const uint32_t ones = valid > c ? (valid - c < 16u ? valid - c : 16u) : 0u;
  uint32_t w[4];
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const uint32_t m = ones > 4u * k ? (ones - 4u * k < 4u ? ones - 4u * k : 4u) : 0u;
    w[k] = m == 4u ? 0x01010101u : 0x01010101u & ((1u << (8u * m)) - 1u);
  }
  return make_uint4(w[0], w[1], w[2], w[3]);
}

__global__ void __launch_bounds__(ROWS_THREADS, ROWS_FILL_BLOCKS) wp_rows_fill_kernel(RowsArgs A) {
  __shared__ RowsFillSmem sm;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned long long total = A.work[0];
  // (an async call whose offsets are malformed, or that needs more rows than capacity, writes only the void count)
  if (A.work[1] != 0ull || total > A.capacity) {
    if (blockIdx.x == 0 && tid == 0) A.row_offsets[A.n_texts] = ~0ull;
    return;
  }
  const uint32_t L = A.max_len;
  const unsigned long long n_tiles = (total + ROWS_TILE - 1) / ROWS_TILE;
  for (unsigned long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const unsigned long long r0 = tile * ROWS_TILE;
    const unsigned long long r1 = total - r0 < ROWS_TILE ? total : r0 + ROWS_TILE;
    __syncthreads();  // (the previous tile's texts are no longer read)
    if (warp == 0) {
      // the first j in [1, n_texts) with row_offsets[j] > r0 (n_texts if none): a 32-way search; the row offsets
      // ascend strictly (every text has a row), so text j - 1 holds row r0
      unsigned long long lo = 1, hi = A.n_texts;
      while (hi > lo) {
        const unsigned long long span = hi - lo;
        const unsigned long long p = lo + span * lane / 32;
        WP_CHECK(p < A.n_texts);
        const uint32_t gt = __ballot_sync(FULL, A.row_offsets[p] > r0);
        const int k = gt ? __ffs(gt) - 1 : 32;  // lanes probe ascending positions: the first lane past r0
        const unsigned long long nhi = k < 32 ? lo + span * k / 32 : hi;
        lo = k > 0 ? lo + span * (k - 1) / 32 + 1 : lo;
        hi = nhi;
      }
      if (lane == 0) sm.t0 = lo - 1;
    }
    __syncthreads();
    const unsigned long long t0 = sm.t0;
    const uint32_t n_local = static_cast<uint32_t>(A.n_texts - t0 < ROWS_TILE ? A.n_texts - t0 : ROWS_TILE);
    for (uint32_t i = tid; i <= n_local; i += ROWS_THREADS) {
      WP_CHECK(t0 + i <= A.n_texts);
      sm.row_off[i] = A.row_offsets[t0 + i];
      sm.id_off[i] = A.id_offsets[t0 + i];
    }
    __syncthreads();
    for (unsigned long long r = r0 + warp; r < r1; r += ROWS_THREADS / 32) {
      // the row's text: the last i with row_off[i] <= r (row_off[0] <= r0 <= r < r1 <= row_off[n_local])
      uint32_t lo = 0, hi = n_local;
      while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (sm.row_off[mid] <= r) lo = mid;
        else hi = mid;
      }
      const unsigned long long k = r - sm.row_off[lo];
      const unsigned long long n_t = sm.id_off[lo + 1] - sm.id_off[lo];
      const unsigned long long from = sm.id_off[lo] + k * A.stride;  // (k = 0 when stride == 0)
      WP_CHECK(k * A.stride <= n_t);
      const uint32_t len = static_cast<uint32_t>(n_t - k * A.stride < A.width ? n_t - k * A.stride : A.width);
      const uint32_t valid = A.cls + len + A.sep;
      auto value = [&](uint32_t c) -> int32_t {
        if (c < A.cls) return A.cls_id;
        const uint32_t j = c - A.cls;
        if (j < len) {
          WP_CHECK(from + j < A.n_ids);
          return __ldg(A.ids + from + j);
        }
        return j == len && A.sep ? A.sep_id : A.pad_id;
      };
      WP_CHECK(r < A.capacity);
      // ids: [0, head) and [body, L) one by one, [head, body) in 16-byte units
      int32_t *const row = A.rows + r * L;
      uint32_t head = ((16u - (reinterpret_cast<uintptr_t>(row) & 15u)) & 15u) >> 2;
      head = head < L ? head : L;
      const uint32_t body = head + ((L - head) & ~3u);
      for (uint32_t e = lane; e < head + (L - body); e += 32) {
        const uint32_t c = e < head ? e : body + (e - head);
        WP_CHECK(c < L);
        row[c] = value(c);
      }
      for (uint32_t c = head + 4u * lane; c < body; c += 128u) {
        WP_CHECK(c + 4u <= L);
        *reinterpret_cast<int4 *>(row + c) = make_int4(value(c), value(c + 1), value(c + 2), value(c + 3));
      }
      if (A.mask != nullptr) {
        uint8_t *const mrow = A.mask + r * L;
        uint32_t mhead = (16u - (reinterpret_cast<uintptr_t>(mrow) & 15u)) & 15u;
        mhead = mhead < L ? mhead : L;
        const uint32_t mbody = mhead + ((L - mhead) & ~15u);
        for (uint32_t e = lane; e < mhead + (L - mbody); e += 32) {
          const uint32_t c = e < mhead ? e : mbody + (e - mhead);
          WP_CHECK(c < L);
          mrow[c] = c < valid ? 1u : 0u;
        }
        for (uint32_t c = mhead + 16u * lane; c < mbody; c += 512u) {
          WP_CHECK(c + 16u <= L);
          *reinterpret_cast<uint4 *>(mrow + c) = mask_unit(c, valid);
        }
      }
    }
  }
}

uint32_t rows_block_texts() { return ROWS_TEXTS; }

cudaError_t launch_rows_scan(const RowsArgs &A, int sm_count, cudaStream_t stream, uint64_t *launches) {
  if (sm_count <= 0) sm_count = 148;
  wp_rows_scan_kernel<<<sm_count * ROWS_SCAN_BLOCKS, ROWS_THREADS, 0, stream>>>(A);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

cudaError_t launch_rows_fill(const RowsArgs &A, int sm_count, cudaStream_t stream, uint64_t *launches) {
  if (sm_count <= 0) sm_count = 148;
  wp_rows_fill_kernel<<<sm_count * ROWS_FILL_BLOCKS, ROWS_THREADS, 0, stream>>>(A);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

// ------------------------------------------------------------ word-table seed
// Every encode call that records words starts from a working table that holds exactly the static words.
__global__ void wp_seed_words_kernel(const WordSlot *__restrict__ image, uint32_t image_slots, WordSlot *work,
                                     uint32_t mask, uint32_t shift) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= image_slots) return;
  const uint4 *src = reinterpret_cast<const uint4 *>(image + i);
  const uint4 key = src[0], lo = src[1];
  if (lo.x == 0) return;
  uint32_t idx = word_hash(key.x, key.y, key.z, key.w, word_meta_len(lo.x), shift);
  while (atomicCAS(&work[idx].meta, 0u, WORD_CLAIMED) != 0u) idx = (idx + 1) & mask;
  uint4 *dst = reinterpret_cast<uint4 *>(work + idx);
  dst[0] = key;
  dst[2] = src[2];
  dst[3] = src[3];
  dst[1] = lo;  // meta last (no reader runs concurrently; the order only keeps CLAIMED until the slot is whole)
}

cudaError_t launch_seed_words(const WordSlot *image, uint32_t image_slots, WordSlot *work, uint32_t work_slots_log2,
                              cudaStream_t stream, uint64_t *launches) {
  cudaError_t e = cudaMemsetAsync(work, 0, (size_t(1) << work_slots_log2) * sizeof(WordSlot), stream);
  if (e != cudaSuccess) return e;
  wp_seed_words_kernel<<<(image_slots + 255) / 256, 256, 0, stream>>>(image, image_slots, work,
                                                                      (1u << work_slots_log2) - 1u, 32 - work_slots_log2);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

// ------------------------------------------------------------ async id count
// The count of an asynchronous call for its caller: UINT64_MAX if a scratch capacity was exceeded (the ids
// are incomplete then and the caller must repeat the call through a synchronous entry, which retries with
// more scratch), else the number of ids.
__global__ void wp_publish_count_kernel(const CallCounters *call, uint32_t parity, unsigned long long *out,
                                        const unsigned int *invalid) {
  *out = (call->overflow || (invalid && *invalid)) ? ~0ull : call->ids_total[parity];
}

cudaError_t launch_publish_count(const CallCounters *call, uint32_t parity, unsigned long long *d_out, cudaStream_t stream,
                                 uint64_t *launches, const unsigned int *invalid) {
  wp_publish_count_kernel<<<1, 1, 0, stream>>>(call, parity, d_out, invalid);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

// -------------------------------------------------------------------- launch

uint32_t encode_tile_bytes() { return TILE; }
uint32_t scatter_block_segments() { return SCATTER_SEGS; }
size_t kernel_geometry(uint32_t *out, size_t cap) {
  const uint32_t g[] = {TILE, LONG_SEGMENT_BYTES, WP_K1_SEG_CAP, SCATTER_SEGS, SCATTER_STAGE, SCATTER_BIG, MIXED_MAX_BIG,
                        LONG_BLOCK, WORD_KEY_BYTES, WORD_MAX_IDS, SEG_SLOW_COUNT_MAX,
                        3u /* ids K2's result form of a slow entry holds inline (wp_match_kernel) */};
  const size_t n = sizeof(g) / sizeof(g[0]);
  for (size_t i = 0; i < n && i < cap; i++) out[i] = g[i];
  return n;
}

cudaError_t launch_encode_range(const EncodeParams &P, int sm_count, cudaStream_t stream, uint64_t *launches,
                                cudaEvent_t *timing) {
  // the opt-in to > 48 KB of dynamic shared memory is per device (K1 stays below it, but keep it explicit)
  static bool configured[64] = {false};
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (dev < 0 || dev >= 64 || !configured[dev]) {
    e = cudaFuncSetAttribute(wp_split_kernel<WP_K1_SEG_CAP>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             static_cast<int>(sizeof(TileSmemT<WP_K1_SEG_CAP>)));
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(wp_split_kernel<TILE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             static_cast<int>(sizeof(TileSmemT<TILE>)));
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < 64) configured[dev] = true;
  }
  if (sm_count <= 0) sm_count = 148;
  // K1 and K3 read the word table at random, K2 the edge table: ask L2 to keep the one a kernel uses resident
  // while text, ids and the intermediates stream through (access policy window, everything else streaming).
  cudaLaunchAttribute attr[1];
  auto window = [&](const void *base, size_t bytes, float ratio) -> unsigned {
    if (bytes == 0) return 0;
    attr[0].id = cudaLaunchAttributeAccessPolicyWindow;
    attr[0].val.accessPolicyWindow.base_ptr = const_cast<void *>(base);
    attr[0].val.accessPolicyWindow.num_bytes = bytes;
    attr[0].val.accessPolicyWindow.hitRatio = ratio;
    attr[0].val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    attr[0].val.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    return 1;
  };
  cudaLaunchConfig_t cfg{};
  cfg.stream = stream;
  cfg.attrs = attr;

  if (timing) cudaEventRecord(timing[0], stream);
  cfg.gridDim = dim3(P.n_tiles);
  cfg.blockDim = dim3(THREADS);
  cfg.numAttrs = window(P.words, P.persist_words_bytes, P.persist_words_ratio);
  if (P.dense_tiles) {
    cfg.dynamicSmemBytes = sizeof(TileSmemT<TILE>);
    e = cudaLaunchKernelEx(&cfg, wp_split_kernel<TILE>, P);
  } else {
    cfg.dynamicSmemBytes = sizeof(TileSmemT<WP_K1_SEG_CAP>);
    e = cudaLaunchKernelEx(&cfg, wp_split_kernel<WP_K1_SEG_CAP>, P);
  }
  if (e != cudaSuccess) return e;
  if (launches) *launches += 1;
  if (timing) cudaEventRecord(timing[1], stream);

  // = resident capacity (see the launch bound): one wave, large shares; a small range (a 4 KiB call is ONE tile)
  // gets a grid to match — a tile has at most MAX_TILE_SLOW unsettled segments, 8 warps x 32 lanes take 256 at a time
  cfg.gridDim = dim3(min(static_cast<unsigned>(sm_count * WP_K2_BLOCKS), P.n_tiles * 4u));
  cfg.blockDim = dim3(MATCH_THREADS);
  cfg.dynamicSmemBytes = 0;
  cfg.numAttrs = window(P.vocab.edges, P.persist_edges_bytes, P.persist_edges_ratio);
  e = cudaLaunchKernelEx(&cfg, wp_match_kernel, P);
  if (e != cudaSuccess) return e;

  cfg.gridDim = dim3(min(static_cast<unsigned>(sm_count * 8), P.n_tiles * 2u + 2u));  // (one CTA per long segment, by ticket)
  cfg.blockDim = dim3(LONG_THREADS);
  e = cudaLaunchKernelEx(&cfg, wp_long_kernel, P);
  if (e != cudaSuccess) return e;
  if (launches) *launches += 2;
  if (timing) cudaEventRecord(timing[2], stream);

  cfg.gridDim = dim3(min(static_cast<unsigned>(sm_count * WP_K3_BLOCKS), P.n_tiles * 2u));  // a tile has at most two blocks of segments
  cfg.blockDim = dim3(SCATTER_THREADS);
  cfg.dynamicSmemBytes = 0;
  cfg.numAttrs = window(P.words, P.persist_words_bytes, P.persist_words_ratio);
  e = cudaLaunchKernelEx(&cfg, wp_scatter_kernel, P);
  if (e != cudaSuccess) return e;
  if (launches) *launches += 1;
  if (timing) cudaEventRecord(timing[3], stream);
  return cudaSuccess;
}

}  // namespace wp
