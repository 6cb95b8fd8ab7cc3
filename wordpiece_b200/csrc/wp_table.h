// Device vocabulary tables, shared by the host builder (wp_vocab.cpp) and the
// kernels (wp_encode.cu).
//
// The reference keeps two unordered_map<VectorSegment,int> (word-initial and
// "##" continuation, fast.cpp:21-35) and finds the longest match by probing the
// window longest -> shortest (fast.cpp:66-77), O(window) probes per piece.  The
// dictionary semantics are exact (utf8.hpp:60-70), so any exact structure that
// returns the same longest match yields the same ids.  Two structures here,
// both over canonical UTF-8 BYTES:
//
//   E  the EDGE TRIE (K2, the walker): every CHAR-prefix of a kept token is a
//      node; an edge (parent node, char) -> child node lives in one open-
//      addressed table of 16-byte slots, hashed on the pair.  The char is its
//      UTF-8 bytes packed into a word, so Cyrillic, kana and Han text walks one
//      edge per char instead of two or three per char (tokens are whole chars,
//      utils.cpp:81-85, so nothing ever ends inside one).  The edge carries the
//      id of the token that ends at the child (term_id), so a longest match is a
//      descent that remembers the last terminal seen: one dependent 16-byte
//      load per char, no key material, no length limit (tokens of any length are
//      just deeper paths).  Node 0 is the root of the word-initial map, node 1
//      the root of the "##" map.
//
//   W  the WORD TABLE (K1): whole segment bytes (<= 16) -> the segment's ids.
//      Its STATIC part is built from the vocabulary: a segment whose bytes are
//      exactly a word-initial token is that token (the longest candidate of
//      fast.cpp:66-72 is the whole window) — ~80 % of English running words,
//      one 32-byte load.  Its DYNAMIC part is filled per encode call by K2 with
//      the words it had to match piece by piece (exact bytes -> exact ids, so a
//      hit is the same ids the matcher would produce): text repeats its words,
//      and every later occurrence is settled by K1's single lookup.
#pragma once
#include <stdint.h>

#include "wp_utf8.h"

namespace wp {

constexpr int32_t WP_NO_ID = -2;             // "no token ends here" (ids are >= 0, UNK may be -1)
constexpr uint32_t WP_KIND_PREFIX = 0;       // word-initial map (prefix_to_id); also the root node of that map
constexpr uint32_t WP_KIND_SUFFIX = 1;       // "##" map (suffix_to_id); also its root node

// ------------------------------------------------------------------ edge trie
struct Edge {
  uint32_t parent;   // node the edge leaves; EDGE_EMPTY = free slot
  uint32_t ch;       // the char: its 1..4 UTF-8 bytes, first byte in the low bits
  uint32_t child;    // node reached (low 24 bits) | EDGE_HAS_CHILDREN: a descent that reaches a leaf stops without another probe
  int32_t term_id;   // token that ends at the child (WP_NO_ID if none); duplicates: last index wins (fast.cpp:34)
};
static_assert(sizeof(Edge) == 16, "an edge is one 16-byte load");
constexpr uint32_t EDGE_EMPTY = 0xFFFFFFFFu;
constexpr uint32_t EDGE_HAS_CHILDREN = 0x80000000u;
constexpr uint32_t EDGE_CHILD_MASK = 0x00FFFFFFu;
constexpr uint32_t EDGE_MAX_NODES = 1u << 24;

// Multiply-add over the pair, one fold, index from the HIGH bits (shift = 32 - log2(slots)).
WP_HD uint32_t edge_hash(uint32_t parent, uint32_t ch, uint32_t shift) {
  uint32_t h = parent * 0x9E3779B1u + ch * 0x85EBCA77u;
  h ^= h >> 15;
  return (h * 0x2C1B3C6Du) >> shift;
}
// The char that starts with byte b0 of the little-endian word `raw` (bytes behind the char are ignored).
WP_HD uint32_t edge_char(uint32_t raw, uint32_t lead_len) {
  return lead_len >= 4u ? raw : (raw & ((1u << (8u * lead_len)) - 1u));
}

// ----------------------------------------------------------------- word table
constexpr uint32_t WORD_KEY_BYTES = 16;
constexpr uint32_t WORD_MAX_IDS = 11;
struct WordSlot {
  uint32_t key[4];   // the segment's bytes, zero padded
  uint32_t meta;     // 0 = empty, WORD_CLAIMED = being written, else WORD_READY | flags | count << 8 | byte length
  int32_t ids[WORD_MAX_IDS];
};
static_assert(sizeof(WordSlot) == 64, "a word slot is two 32-byte sectors; K1 reads only the first");
constexpr uint32_t WORD_CLAIMED = 1u;
constexpr uint32_t WORD_READY = 0x80000000u;
constexpr uint32_t WORD_DYNAMIC = 0x40000000u;   // recorded by K2 during this call (statistics only)
WP_HD uint32_t word_meta_len(uint32_t meta) { return meta & 0x1Fu; }
WP_HD uint32_t word_meta_count(uint32_t meta) { return (meta >> 8) & 0xFu; }
WP_HD uint32_t word_meta(uint32_t len, uint32_t count, bool dynamic) {
  return WORD_READY | (dynamic ? WORD_DYNAMIC : 0u) | (count << 8) | len;
}
// Multiply-add over the four key words and the length (five IMADs), one fold, index from the high bits.
WP_HD uint32_t word_hash(uint32_t k0, uint32_t k1, uint32_t k2, uint32_t k3, uint32_t len, uint32_t shift) {
  uint32_t h = k0 * 0x9E3779B1u + k1 * 0x85EBCA77u + k2 * 0xC2B2AE3Du + k3 * 0x27D4EB2Fu + len * 0x165667B1u;
  h ^= h >> 15;
  return (h * 0x2C1B3C6Du) >> shift;
}
// A K1 lookup looks at this many consecutive slots before it gives up and leaves the segment to K2 (a
// single-char segment, which K2 never sees, follows the probe sequence to its end instead — rare).
constexpr uint32_t WORD_PROBES = 4;

// Everything a kernel needs to know about a vocabulary (device pointers).
struct DeviceVocab {
  const Edge *edges;            // n_edge_slots entries, a power of two
  uint32_t edge_mask;           // n_edge_slots - 1
  uint32_t edge_shift;          // 32 - log2(n_edge_slots)
  int32_t unk_id;               // utils.hpp:30 / utils.cpp:112-114
  uint32_t han_swallow;         // 1 iff max_len >= 2 (SURVEY A.2: an OOV Han char swallows the following run)
};

}  // namespace wp
