"""Parity at the kernels' structural limits.

Random text rarely reaches the places where the kernels switch paths or pack a number into a few bits: K3's
staged / mixed / direct block paths, the id-count fields of ``seg_result`` and of the slow entries, the 16-byte
word key, K2L's 1024-byte rounds, K1's list capacities, the scratch spill and positions past 4 GiB.  Every case
here is built to sit on one side of such a limit, from the values the library reports it was compiled with
(``wp_debug_kernel_geometry``), so the cases follow a variant build (e.g. ``-DWP_SCATTER_BIG=16``).  Each GPU
case compares the whole id array with the oracle, bit-exact.

The CPU tests check the construction itself: that every block the GPU tests build lands on its intended side
of STAGE, BIG and MIXED_MAX_BIG (the planner below restates how K1 numbers segments and K3 cuts them into
blocks, for text of ASCII words separated by single spaces, with the word memo off).
"""
from __future__ import annotations

import random
import re

import numpy as np
import pytest

import cases
from _oracle import Oracle

LETTERS = "abcdefghijklmnopqrstuvwxyz"
# every lowercase letter word-initial and as a continuation: a word of n letters is n ids
LETTER_VOCAB = ["[UNK]"] + list(LETTERS) + ["##" + c for c in LETTERS]
COUNTS = (1, 2, 3, 4, 8, 9, 11, 12, 15, 16, 30, 31, 32, 100)
LONG_HEAD = "P" * 300  # one word-initial token of 300 bytes: a word behind it is LONG and adds no id of its own
BLOCK_VOCAB = LETTER_VOCAB + [LONG_HEAD]

_GEO = None


def geo() -> dict:
    global _GEO
    if _GEO is None:
        from wordpiece_b200._capi import kernel_geometry

        _GEO = kernel_geometry()
    return _GEO


def _first_mismatch(exp, got, tag):
    n = min(len(exp), len(got))
    k = int(np.argmax(exp[:n] != got[:n])) if n and not np.array_equal(exp[:n], got[:n]) else n
    return (f"{tag}: ids differ (oracle {len(exp)} vs gpu {len(got)}), first mismatch at {k}: "
            f"oracle {np.asarray(exp[max(0, k - 3):k + 5]).tolist()} gpu {np.asarray(got[max(0, k - 3):k + 5]).tolist()}")


def _same(exp, got, tag):
    exp, got = np.asarray(exp), np.asarray(got)
    assert len(exp) == len(got) and np.array_equal(exp, got), _first_mismatch(exp, got, tag)


# ---------------------------------------------------------------------------------------------------- planner

class Words:
    """Random letter words by length (a small pool per length, so that the ids vary but the oracle sees few
    distinct words)."""

    def __init__(self, seed):
        self.rng = random.Random(seed)
        self.pool = {}

    def __call__(self, n):
        p = self.pool.setdefault(n, [])
        if len(p) < 24:
            p.append("".join(self.rng.choice(LETTERS) for _ in range(n)))
            return p[-1]
        return self.rng.choice(p)


def fill(n_segs, total, most):
    """n_segs id counts, each in [1, most], adding up to total (as even as possible)."""
    base, rem = divmod(total, n_segs)
    assert base >= 1 and base + (rem > 0) <= most, (n_segs, total, most)
    return [base + 1] * rem + [base] * (n_segs - rem)


def block_shapes(g):
    """[(name, intended path, id count per segment)] of every K3 block the GPU tests build.  The order
    alternates the paths, so that a wrong total in the look-back shifts every later id."""
    S, G, B, M = g["scatter_stage"], g["scatter_segs"], g["scatter_big"], g["mixed_max_big"]
    big = B + 1
    shapes = []
    shapes.append(("staged_stage_minus_1", "staged", fill(G, S - 1, B)))
    one_big = fill(G - 1, S, B)
    shapes.append(("mixed_small_stage_one_big", "mixed", one_big[:G // 3] + [big] + one_big[G // 3:]))
    shapes.append(("direct_stage_plus_1_no_big", "direct", fill(G, S + 1, B)))
    shapes.append(("staged_stage", "staged", fill(G, S, B)))
    edge = fill(G - 4, S - 10, B)
    shapes.append(("mixed_big_first_last_adjacent", "mixed", [big] + edge[:G // 2] + [big, big] + edge[G // 2:] + [big]))
    small_big = fill(G - 1, S + 1, B)
    shapes.append(("direct_small_stage_plus_1", "direct", small_big[:7] + [big] + small_big[7:]))
    n_at, n_over = 100, 100
    thr = [B] * n_at + [big] * n_over
    random.Random(3).shuffle(thr)
    shapes.append(("staged_big_threshold", "staged", thr + [1] * (G - len(thr))))
    shapes.append(("mixed_max_big", "mixed", [x for _ in range(M) for x in (big, 1)] + [1] * (G - 2 * M)))
    over = [big] * (M + 1) + [1] * (G - M - 1)
    random.Random(4).shuffle(over)
    shapes.append(("direct_max_big_plus_1", "direct", over))
    shapes.append(("staged_tail", "staged", fill(G // 3, G, B)))  # a partial last block
    return shapes


def block_path(counts, g):
    """The path K3 takes for a block whose segments have these id counts (memo off: every segment with more
    than one id is a slow segment, and it is copied warp-wise when it has more than BIG ids)."""
    B = g["scatter_big"]
    total = sum(counts)
    n_big = sum(1 for c in counts if c > B)
    n_small = total - sum(c for c in counts if c > B)
    if total <= g["scatter_stage"]:
        return "staged", total, n_small, n_big
    if n_small <= g["scatter_stage"] and 1 <= n_big <= g["mixed_max_big"]:
        return "mixed", total, n_small, n_big
    return "direct", total, n_small, n_big


def long_segments_of(counts, g):
    """Segments of a block that build_blocks_text makes LONG (behind LONG_HEAD, same id count): the middle
    segment of 3 ids, and the first warp-copied one."""
    three = [i for i, c in enumerate(counts) if c == 3]
    bigs = [i for i, c in enumerate(counts) if c > g["scatter_big"]]
    return set(three[len(three) // 2:len(three) // 2 + 1] + bigs[:1])


def build_blocks_text(g, seed=1):
    """The text of block_shapes (vocabulary BLOCK_VOCAB): every block's words, then spaces up to the next multiple
    of RANGE bytes (so that a call cut into ranges of RANGE bytes has exactly one block per range).  Returns
    (text, words, starts, range_bytes, shapes)."""
    shapes = block_shapes(g)
    w = Words(seed)
    tile = g["tile"]
    pieces = []
    for _, _, counts in shapes:
        longs = long_segments_of(counts, g)
        pieces.append(" ".join(LONG_HEAD + w(c - 1) if i in longs else w(c) for i, c in enumerate(counts)))
    rb = (max(len(p) for p in pieces) + 1 + tile - 1) // tile * tile
    text, words, starts = [], [], []
    pos = 0
    for p in pieces:
        for m in re.finditer(r"\S+", p):
            words.append(m.group())
            starts.append(pos + m.start())
        text.append(p + " " * (rb - len(p)))
        pos += rb
    return "".join(text).encode(), words, starts, rb, shapes


def plan(counts, starts, g, range_bytes=None):
    """K3 blocks of a call: [(range, block, path, total, n_small, n_big, first segment)].  K1 numbers the segments
    of a range in text order (segment i = word i here) and K3 cuts them into blocks of SCATTER_SEGS."""
    G = g["scatter_segs"]
    by_range = {}
    for i, s in enumerate(starts):
        by_range.setdefault(s // range_bytes if range_bytes else 0, []).append(i)
    out = []
    for r in sorted(by_range):
        segs = by_range[r]
        for b in range(0, len(segs), G):
            idx = segs[b:b + G]
            out.append((r, b // G, *block_path([counts[i] for i in idx], g), idx[0]))
    return out


def word_counts(words, oracle):
    """The oracle's id count of every word."""
    memo = {}
    for x in set(words):
        memo[x] = len(oracle.encode(x))
    return [memo[x] for x in words]


def test_block_planner_hits_every_side_of_each_limit():
    """The K3 blocks the GPU tests build take the path they are meant to take, and sit exactly on the limit
    they are meant to sit on (STAGE - 1, STAGE, STAGE + 1 ids; BIG and BIG + 1 ids; MIXED_MAX_BIG and one more
    warp-copied segments), computed with the oracle's id counts and the compiled geometry."""
    g = geo()
    S, B, M, G = g["scatter_stage"], g["scatter_big"], g["mixed_max_big"], g["scatter_segs"]
    text, words, starts, rb, shapes = build_blocks_text(g)
    counts = word_counts(words, Oracle(BLOCK_VOCAB))
    assert counts == [c for _, _, cs in shapes for c in cs]
    longs = [i for i, x in enumerate(words) if x.startswith(LONG_HEAD)]
    assert len(longs) == sum(len(long_segments_of(cs, g)) for _, _, cs in shapes) >= len(shapes) and all(len(words[i]) > g["long_segment_bytes"] for i in longs)
    blocks = plan(counts, starts, g)
    assert len(blocks) == len(shapes)
    got = {name: blk for (name, _, _), blk in zip(shapes, blocks)}
    for (name, want, cs), blk in zip(shapes, blocks):
        assert blk[2] == want, (name, blk)
    assert got["staged_stage_minus_1"][3] == S - 1 and got["staged_stage"][3] == S
    assert got["direct_stage_plus_1_no_big"][3:6] == (S + 1, S + 1, 0)
    assert got["mixed_small_stage_one_big"][4:6] == (S, 1)
    assert got["mixed_max_big"][5] == M and got["direct_max_big_plus_1"][5] == M + 1
    assert got["direct_small_stage_plus_1"][4] == S + 1 and got["direct_small_stage_plus_1"][5] >= 1
    cs = dict((n, c) for n, _, c in shapes)
    e = cs["mixed_big_first_last_adjacent"]
    assert e[0] == e[-1] == B + 1 and any(e[i] == e[i + 1] == B + 1 for i in range(1, G - 2))
    assert min(c for c in e if c > B) == B + 1
    thr = cs["staged_big_threshold"]
    assert thr.count(B) == 100 and thr.count(B + 1) == 100 and got["staged_big_threshold"][2] == "staged"
    # one block per range at RANGE bytes: the last block of a range takes each path
    per_range = plan(counts, starts, g, rb)
    assert [b[2] for b in per_range] == [b[2] for b in blocks] and all(b[1] == 0 for b in per_range)
    # the batch cuts of test_k3_block_paths fall inside mixed and direct blocks
    firsts = [b[6] for b in blocks]
    paths = set()
    for c in batch_cuts(blocks, shapes, g):
        i = max(j for j, f in enumerate(firsts) if f <= c)
        assert firsts[i] < c < firsts[i] + len(shapes[i][2]), c
        paths.add(blocks[i][2])
    assert paths == {"mixed", "direct"}


def batch_cuts(blocks, shapes, g):
    """Word indices at which the batch of test_k3_block_paths starts a new text: inside every mixed and direct
    block (mid-block, right before and right behind a warp-copied segment)."""
    B = g["scatter_big"]
    cuts = set()
    for (r, b, path, total, n_small, n_big, first), (_, _, counts) in zip(blocks, shapes):
        if path == "staged":
            continue
        cuts.add(first + len(counts) // 2)
        bigs = [i for i, c in enumerate(counts) if c > B]
        if bigs:
            cuts.add(first + max(bigs[0], 1))
            cuts.add(first + bigs[len(bigs) // 2] + 1)
    return sorted(cuts)


def test_geometry_hook():
    """wp_debug_kernel_geometry reports the compiled limits (a variant build may change SCATTER_BIG and
    WP_K1_SEG_CAP; the rest are fixed by the kernels' data layouts)."""
    g = geo()
    assert g["tile"] == 4096 and g["long_segment_bytes"] == 256 and g["scatter_segs"] == 2048
    assert g["scatter_stage"] == 6144 and g["mixed_max_big"] == g["scatter_segs"] // 2 and g["long_block"] == 1024
    assert g["word_key_bytes"] == 16 and g["word_max_ids"] == 11 and g["seg_slow_count_max"] == 31
    assert g["inline_ids"] == 3 and 1 <= g["scatter_big"] and g["seg_cap"] <= g["tile"]
    import wordpiece_b200

    assert wordpiece_b200.tile_bytes() == g["tile"]


def test_word_key_chars_have_the_intended_class():
    """The chars the word-key cases build their 15..17-byte words from are ordinary chars (not space, punctuation
    or Han) of 1, 2, 3 and 4 bytes, so that each word is one segment."""
    L = Oracle.lib()
    for ch, n in zip(WIDE, (1, 2, 3, 4)):
        b = ch.encode()
        assert len(b) == n
        cp = ord(ch)
        assert not (L.wpo_is_space(cp) or L.wpo_is_punct(cp) or L.wpo_is_han(cp)), ch


# ------------------------------------------------------------------------------------------------- GPU helpers

def _vocab(tokens, dev):
    from wordpiece_b200 import Vocab

    return Vocab(tokens, device=dev)


def _encode_all_ways(v, text, exp, tag):
    """encode (host), encode_into, encode_device: every entry point returns the oracle's ids."""
    import torch

    _same(exp, v.encode(text), tag + " encode")
    out = np.full(len(exp) + 3, -7, np.int32)
    n = v.encode_into(text, out)
    assert n == len(exp) and (out[n:] == -7).all(), tag
    _same(exp, out[:n], tag + " encode_into")
    d_text = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda(v.device)
    d_ids, n = v.encode_device(d_text)
    _same(exp, d_ids[:n].cpu().numpy(), tag + " encode_device")


# ---------------------------------------------------------------------------------------- A. K3 block paths

@pytest.mark.gpu
def test_k3_block_paths(gpu_device, monkeypatch):
    """Staged, mixed and direct blocks at their limits, in one text; then the same text cut into ranges (one
    block per range, so that the last block of a range takes each path; and ranges that cut through blocks),
    and as a batch whose text borders lie inside mixed and direct blocks (K5's offsets)."""
    g = geo()
    monkeypatch.setenv("WORDPIECE_B200_MEMO", "0")
    text, words, starts, rb, shapes = build_blocks_text(g)
    o = Oracle(BLOCK_VOCAB)
    exp = o.encode(text)
    v = _vocab(BLOCK_VOCAB, gpu_device)
    _encode_all_ways(v, text, exp, "blocks")
    for range_bytes in (rb, 2 * g["tile"], 3 * g["tile"]):
        monkeypatch.setenv("WORDPIECE_B200_RANGE_BYTES", str(range_bytes))
        _same(exp, v.encode(text), f"blocks, ranges of {range_bytes} bytes")
    monkeypatch.delenv("WORDPIECE_B200_RANGE_BYTES")
    counts = word_counts(words, o)
    blocks = plan(counts, starts, g)
    cuts = batch_cuts(blocks, shapes, g)
    bounds = [0] + [starts[c] for c in cuts] + [len(text)]
    texts = [text[a:b] for a, b in zip(bounds, bounds[1:])]
    ids, offs = v.encode_batch(texts)
    for i, t in enumerate(texts):
        _same(o.encode(t), ids[int(offs[i]):int(offs[i + 1])], f"batch text {i} of {len(texts)}")
    v.close()


# ------------------------------------------------------------------------------------ B. id-count fields

def count_words(w, counts=COUNTS, long=False):
    """One word per id count: n letters (n ids), or LONG_HEAD + n - 1 letters (n ids, a LONG segment)."""
    return [LONG_HEAD + w(c - 1) if long else w(c) for c in counts]


@pytest.mark.gpu
def test_id_count_fields_in_every_lane(gpu_device, monkeypatch):
    """Segments of 1..100 ids across the 3-id inline form, the 4-bit word count (11 ids in a slot, 12 never
    recorded) and the 5-bit slow count (31 = read the slow entry): through K2 (memo off), through memo hits
    (memo on, several ranges, repeats in later ranges), through K2L (each word behind a 300-byte token), and
    through a batch whose texts start right behind such segments (K5)."""
    g = geo()
    vocab = LETTER_VOCAB + [LONG_HEAD]
    o = Oracle(vocab)
    v = _vocab(vocab, gpu_device)
    w = Words(7)
    assert g["inline_ids"] in COUNTS and g["word_max_ids"] in COUNTS and g["word_max_ids"] + 1 in COUNTS
    assert g["seg_slow_count_max"] in COUNTS and g["seg_slow_count_max"] + 1 in COUNTS
    # K2, memo off
    monkeypatch.setenv("WORDPIECE_B200_MEMO", "0")
    text = " ".join(" ".join(count_words(w)) + " a bc" for _ in range(40)).encode()
    _same(o.encode(text), v.encode(text), "K2 counts")
    # memo hits: the same words again and again over ranges of one tile
    monkeypatch.setenv("WORDPIECE_B200_MEMO", "1")
    monkeypatch.setenv("WORDPIECE_B200_RANGE_BYTES", str(g["tile"]))
    fixed = count_words(Words(8))
    rng = random.Random(9)
    parts = []
    for _ in range(120):
        ws = fixed[:]
        rng.shuffle(ws)
        parts.append(" ".join(ws))
    text = " ".join(parts).encode()
    assert len(text) > 8 * g["tile"]
    _same(o.encode(text), v.encode(text), "memo counts")
    assert v.stats().memo_hits > 0
    monkeypatch.delenv("WORDPIECE_B200_RANGE_BYTES")
    # K2L
    monkeypatch.setenv("WORDPIECE_B200_MEMO", "0")
    text = " ".join(" ".join(count_words(w, long=True)) + " a" for _ in range(6)).encode()
    _same(o.encode(text), v.encode(text), "K2L counts")
    assert v.stats().long_segments >= 6 * len(COUNTS)
    # batch: every text starts right behind a segment of each count (several per K3 block)
    texts = []
    for long in (False, True):
        for c, word in zip(COUNTS, count_words(w, long=long)):
            texts += ["ab " + word, "c " + w(3), word]
    texts += texts[::-1]
    ids, offs = v.encode_batch(texts)
    for i, t in enumerate(texts):
        _same(o.encode(t), ids[int(offs[i]):int(offs[i + 1])], f"batch text {i}")
    v.close()


# ------------------------------------------------------------------------------------------- C. word key

WIDE = ("a", "é", "か", "\U0001D400")  # 1, 2, 3 and 4 bytes; not space, punctuation or Han


def key_words():
    """Words of 15, 16 and 17 bytes from chars of each width (the remainder in 1-byte chars, before or after)."""
    out = []
    for ch in WIDE:
        n = len(ch.encode())
        for L in (15, 16, 17):
            k, r = divmod(L, n)
            out.append(ch * k + "b" * r)
            out.append("c" * r + ch * k)
    mixed = "".join(WIDE)  # 10 bytes
    for L in (15, 16, 17):
        out.append(mixed + "d" * (L - 10))
    return [x.encode() for x in out]


def nul_pair(log2, slot_of, rng, length, text_has_nul):
    """A word W (letters) such that W and W + NUL share a probe sequence of K1's lookup: the token's slot is the
    home slot of the segment.  text_has_nul: the token is W and the text holds W + NUL, else the other way."""
    from _model import word_hash_py

    while True:
        w = "".join(rng.choice(LETTERS) for _ in range(length)).encode()
        tok, seg = (w, w + b"\0") if text_has_nul else (w + b"\0", w)
        if slot_of(tok) == word_hash_py(seg, log2):
            return tok, seg


@pytest.mark.gpu
def test_word_key_edges(gpu_device, monkeypatch):
    """K1's whole-segment lookup at the 16-byte key: words of 15, 16 and 17 bytes in chars of 1..4 bytes, each
    as a vocabulary word (a static hit) and not; a segment ending in NUL next to a token of the same bytes
    without it (both ways round, placed so that both share a probe sequence); a 16-byte word with invalid bytes
    inside it in a dirty tile.  Memo off and on."""
    from _model import word_hash_py
    from wordpiece_b200 import Vocab

    rng = random.Random(11)
    kw = key_words()
    half = kw[::2]
    chars = sorted({c for x in kw for c in x.decode()} - set(LETTERS))
    base = LETTER_VOCAB + chars + ["##" + c for c in chars] + [x.decode() for x in half] + ["\0", "##\0"]
    # NUL pairs (token, segment) whose token's slot is the segment's home slot; the search is repeated with the
    # final vocabulary until every pair holds there (a token may be displaced by the others)
    shapes = [(n, has) for n in (3, 7, 14, 15) for has in (True, False)]
    pairs = [None] * len(shapes)
    for _ in range(50):
        vocab = base + [(p[0] if p else b"%02d" % i).decode() for i, p in enumerate(pairs)]
        host = Vocab(vocab, device=-1)
        slots = host.table_info["word_slots"]
        log2 = slots.bit_length() - 1
        bad = 0
        for i, (n, has) in enumerate(shapes):
            p = pairs[i]
            found = host.debug_word_lookup(p[0]) if p else None
            if p and found and host.debug_word_lookup(p[1]) is None and \
                    (word_hash_py(p[0], log2) + found[1]) % slots == word_hash_py(p[1], log2):
                continue
            pairs[i] = nul_pair(log2, lambda t: word_hash_py(t, log2), rng, n, has)
            bad += 1
        host.close()
        if not bad:
            break
    assert not bad, "no placement of the NUL pairs found"
    v = _vocab(vocab, gpu_device)
    o = Oracle(vocab)
    segs = kw + [s for _, s in pairs] + [t for t, _ in pairs]
    text = b" ".join(segs[i % len(segs)] for i in range(3 * len(segs)))
    dirty = b" ".join([b"abcdefgh\xffijklmnop", b"abcdefghijklmnop", b"abc\xc3defghijklmnop\x80", b"\xe4\xb8xyz"])
    for memo in ("0", "1"):
        monkeypatch.setenv("WORDPIECE_B200_MEMO", memo)
        monkeypatch.setenv("WORDPIECE_B200_RANGE_BYTES", str(geo()["tile"]))
        for t in (text, text * 40, dirty + b" " + text):
            _same(o.encode(t), v.encode(t), f"word key, memo {memo}, {len(t)} bytes")
    # the dirty 16-byte word as a static hit
    v.close()
    vocab2 = vocab + ["abcdefghijklmnop", "##xyz"]
    v = _vocab(vocab2, gpu_device)
    for memo in ("0", "1"):
        monkeypatch.setenv("WORDPIECE_B200_MEMO", memo)
        t = (dirty + b" ") * 300
        _same(Oracle(vocab2).encode(t), v.encode(t), f"dirty key, memo {memo}")
        assert v.stats().dirty_tiles > 0
    v.close()


# ------------------------------------------------------------------------------------------- D. K2L rounds

def _word(rng, n, alphabet=LETTERS):
    return "".join(rng.choice(alphabet) for _ in range(n)).encode()


def k2l_cases(g):
    """(name, text, extra vocab) for the long-segment lane; every text holds at least one LONG segment."""
    rng = random.Random(21)
    LB, tile, ls = g["long_block"], g["tile"], g["long_segment_bytes"]
    out = []
    for L in (1, 2, 3):
        for d in (-1, 0, 1):
            out.append((f"len {L}*{LB}{d:+d}", _word(rng, L * LB + d), []))
    out.append(("token longer than a round", _word(rng, 10) + b"q" * (LB + 500) + _word(rng, 700) + b"q" * 30, ["##" + "q" * (LB + 300)]))
    for at in range(LB - 3, LB + 3):
        w = bytearray(_word(rng, 3 * LB))
        w[at:at + 3] = b"xyz"
        out.append((f"piece across the round border at {at}", bytes(w), ["##xyz"]))
    n = 3 * LB
    for at in (0, n - 1, LB - 1, LB, LB + 1):
        w = bytearray(_word(rng, n))
        w[at] = ord("Z")
        out.append((f"UNK at byte {at}", bytes(w), []))
    for ch in ("é", "か", "\U0001D400"):
        for at in range(LB - 4, LB + 1):
            out.append((f"{ch!r} across the border at {at}", _word(rng, at) + ch.encode() * 3 + _word(rng, LB), ["##" + ch]))
    for junk in (b"\xff", b"\xe4\xb8", b"\xf0\x9f\x98", b"\x80" * 5):
        for at in (LB - 2, LB - 1, LB):
            out.append((f"{junk!r} across the border at {at}", _word(rng, at) + junk * 3 + _word(rng, 2 * LB), []))
    out.append(("a round of dropped bytes only", _word(rng, 1000) + b"\xff" * (2 * LB + 100) + _word(rng, 700), []))
    han = cases.ZH.encode()
    out.append(("Han head, fused window", han + b"ab" + _word(rng, 2 * LB), [cases.ZH, cases.ZH + "ab", cases.ZH + "a"]))
    out.append(("Han head, OOV, swallows", "文".encode() + _word(rng, 2 * LB), ["ab"]))
    out.append(("Han head, matched alone, rest fails", han + _word(rng, LB + 50) + b"Z" + _word(rng, 40), [cases.ZH]))
    out.append(("Han head, matched alone, rest matches", han + _word(rng, LB + 50), [cases.ZH]))
    # starts at TILE - k of a tile, lengths around the LONG limit and the window
    for k in (1, 2, 31, 255, 256, 257):
        for length in (ls - 1, ls, ls + 1, tile + ls - 1, tile + ls + 1):
            pre = b"ab " * ((tile - k) // 3)
            pre += b" " * (tile - k - len(pre))
            out.append((f"start TILE-{k} len {length}", pre + _word(rng, length) + b" a", []))
    # the worst case of K1's long list: words of LONG + 1 bytes, one per LONG + 2 bytes of text
    out.append(("tiles of LONG+1-byte words", b" ".join(_word(rng, ls + 1) for _ in range(80)), []))
    return out


def k2l_han_cases(g):
    """Han-led LONG segments whose vocabulary decides the head (one needs max_len 1)."""
    rng = random.Random(22)
    LB = g["long_block"]
    han = cases.ZH.encode()
    single = ["[UNK]"] + list(LETTERS) + ["##" + c for c in LETTERS]  # max_len 1: an OOV Han char swallows nothing
    return [("Han head, OOV, max_len 1", han + _word(rng, 2 * LB + 3), single),
            ("Han head, OOV, max_len 1, fails later", han + _word(rng, LB) + b"Z" + _word(rng, 9), single)]


@pytest.mark.gpu
def test_k2l_rounds(gpu_device):
    """K2L's 1024-byte rounds: lengths around multiples of a round, a token longer than a round, pieces, UNK,
    multi-byte chars and invalid bytes at the round border, a round of dropped bytes, the four Han-led heads
    (each case's ids against the oracle; the roll-back of a failed word keeps the Han id in front of the UNK),
    segment starts just before a tile border at lengths around LONG and the window, the densest long list."""
    g = geo()
    base = LETTER_VOCAB + ["é", "か", "\U0001D400"]
    for name, text, extra in k2l_cases(g):
        vocab = base + extra
        v = _vocab(vocab, gpu_device)
        t = text + b" ef " + text[::-1] + b" g"
        _same(Oracle(vocab).encode(t), v.encode(t), name)
        if max(len(x) for x in text.split()) >= 2 * g["long_segment_bytes"]:
            assert v.stats().long_segments >= 1, name
        v.close()
    for name, text, vocab in k2l_han_cases(g):
        v = _vocab(vocab, gpu_device)
        assert v.max_len == 1
        t = b"ab " + text + b" c"
        _same(Oracle(vocab).encode(t), v.encode(t), name)
        assert v.stats().long_segments >= 1, name
        v.close()


@pytest.mark.gpu
def test_quirks_as_long_segments(gpu_device):
    """Every behaviour of cases.QUIRKS again, with its last word padded past LONG_SEGMENT_BYTES and past the tile
    window by a continuation piece, so that the same rule is checked in K2L as in K2."""
    g = geo()
    for name, text, vocab in cases.QUIRKS:
        for pad in (g["long_segment_bytes"] + 1, g["tile"] + g["long_segment_bytes"] + 1):
            voc = list(vocab) + ["##x"]
            t = text + b"x" * pad
            v = _vocab(voc, gpu_device)
            _same(Oracle(voc).encode(t), v.encode(t), f"{name} + {pad} x")
            assert v.stats().long_segments >= 1, name
            v.close()


@pytest.mark.gpu
def test_k1_segment_list_capacity(gpu_device):
    """A tile with SEG_CAP - 1, SEG_CAP and SEG_CAP + 1 segments that start in it (one punctuation char each; K1
    counts the segments that START in its tile against its lists): the last one takes the dense-tile retry."""
    g = geo()
    tile, cap = g["tile"], g["seg_cap"]
    vocab = LETTER_VOCAB + [",", ".", "ab"]
    o = Oracle(vocab)
    for n in (cap - 1, cap, cap + 1):
        if n > tile:
            continue
        head = b"ab " * (tile // 3)
        head += b" " * (tile - len(head))
        body = (b",." * tile)[:n] + b" " * (tile - n)
        t = head + body + b"ab cd, ef " * 50
        v = _vocab(vocab, gpu_device)  # a fresh handle each time (the dense retry is sticky per handle)
        _same(o.encode(t), v.encode(t), f"{n} segments in a tile")
        v.close()


# ----------------------------------------------------------------------------------- E. scratch and capacity

@pytest.mark.gpu
def test_arena_spill_overflow_and_retry(gpu_device, monkeypatch):
    """Ranges of one tile and a word far longer than a range: its ids outgrow the spill part of the arena (the
    range plus one tile).  encode / encode_into / encode_device retry with a larger spill and return the oracle's
    ids; encode_device_async publishes UINT64_MAX and writes nothing past its capacity; the next call is exact."""
    import torch

    g = geo()
    monkeypatch.setenv("WORDPIECE_B200_RANGE_BYTES", str(g["tile"]))
    rng = random.Random(31)
    text = b"ab cd " * 2000 + _word(rng, 12 * g["tile"]) + b" ef " + b"gh " * 3000
    o = Oracle(LETTER_VOCAB)
    exp = o.encode(text)
    v = _vocab(LETTER_VOCAB, gpu_device)
    _encode_all_ways(v, text, exp, "spill overflow")
    d_text = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda(gpu_device)
    guard = 64
    d_out = torch.full((len(exp) + guard,), -7, dtype=torch.int32, device=d_text.device)
    d_cnt = torch.zeros(1, dtype=torch.int64, device=d_text.device)
    v.encode_device_async(d_text, d_out[:len(exp)], d_cnt)
    torch.cuda.synchronize()
    assert int(d_cnt.item()) == -1  # UINT64_MAX
    assert (d_out[len(exp):] == -7).all()
    d_ids, n = v.encode_device(d_text)
    _same(exp, d_ids[:n].cpu().numpy(), "after the async overflow")
    v.close()


def _encode_device_raw(v, d_text, d_ids, capacity):
    import ctypes as C

    import torch

    cnt = C.c_size_t()
    st = v._L.wp_encode_device(v._h, d_text.data_ptr(), d_text.numel(), d_ids.data_ptr(), capacity, C.byref(cnt),
                               torch.cuda.current_stream(d_text.device).cuda_stream)
    return st, int(cnt.value)


@pytest.mark.gpu
def test_capacity_cuts_inside_segments(gpu_device, monkeypatch):
    """wp_encode_device with a capacity of n - 1, n, and cuts inside segments of each kind (inline, arena, LONG,
    warp-copied) in staged, mixed and direct blocks, and inside memo hits (word slots): WP_ERR_CAPACITY with the
    exact count, nothing written past the capacity, and the oracle's prefix before it."""
    import torch

    from wordpiece_b200._capi import WP_ERR_CAPACITY, WP_OK

    g = geo()
    B = g["scatter_big"]
    text, words, starts, rb, shapes = build_blocks_text(g)
    vocab = BLOCK_VOCAB
    o = Oracle(vocab)
    counts = word_counts(words, o)
    exp = o.encode(text)
    assert len(exp) == sum(counts)
    blocks = plan(counts, starts, g)
    at = np.concatenate([[0], np.cumsum(counts)])
    cuts = {len(exp) - 1, len(exp), 1}
    for (r, bi, path, total, n_small, n_big, first), (_, _, cs) in zip(blocks, shapes):
        kinds = {"inline": lambda i: 2 <= counts[i] <= g["inline_ids"], "arena": lambda i: g["inline_ids"] < counts[i] <= B,
                 "big": lambda i: counts[i] > B, "LONG": lambda i: words[i].startswith(LONG_HEAD)}
        for kind, pred in kinds.items():
            hit = [first + i for i in range(len(cs)) if pred(first + i)]
            if hit:
                s = hit[len(hit) // 2]
                cuts.update({int(at[s]) + 1, int(at[s + 1]) - 1})
    monkeypatch.setenv("WORDPIECE_B200_MEMO", "0")
    v = _vocab(vocab, gpu_device)
    d_text = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda(gpu_device)
    guard = 256
    d_ids = torch.empty(len(exp) + guard, dtype=torch.int32, device=d_text.device)
    exp_t = torch.from_numpy(exp).to(d_text.device)
    for cap in sorted(cuts):
        d_ids.fill_(-7)
        st, n = _encode_device_raw(v, d_text, d_ids, cap)
        assert n == len(exp), (cap, n)
        assert st == (WP_OK if cap >= len(exp) else WP_ERR_CAPACITY), (cap, st)
        assert (d_ids[cap:] == -7).all(), f"capacity {cap}: written past the capacity"
        assert torch.equal(d_ids[:cap], exp_t[:cap]), _first_mismatch(exp[:cap], d_ids[:cap].cpu().numpy(), f"capacity {cap}")
    v.close()
    # word slots: memo hits of 4..11 ids cut in the middle (several ranges, so the repeats hit)
    monkeypatch.setenv("WORDPIECE_B200_MEMO", "1")
    monkeypatch.setenv("WORDPIECE_B200_RANGE_BYTES", str(g["tile"]))
    ws = count_words(Words(41), counts=(4, 7, 11, 12))
    t = " ".join(" ".join(ws) for _ in range(200)).encode()
    e = o.encode(t)
    v = _vocab(vocab, gpu_device)
    d_t = torch.frombuffer(bytearray(t), dtype=torch.uint8).cuda(gpu_device)
    d_ids = torch.empty(len(e) + guard, dtype=torch.int32, device=d_t.device)
    e_t = torch.from_numpy(e).to(d_t.device)
    per = 4 + 7 + 11 + 12
    for cap in [len(e) - per + x for x in (2, 6, 9, 15, 20, 25)] + [len(e) // 2 + 1]:
        d_ids.fill_(-7)
        st, n = _encode_device_raw(v, d_t, d_ids, cap)
        assert st == WP_ERR_CAPACITY and n == len(e), (cap, st, n)
        assert (d_ids[cap:] == -7).all() and torch.equal(d_ids[:cap], e_t[:cap]), cap
        assert v.stats().memo_hits > 0
    v.close()


@pytest.mark.gpu
def test_slow_slots_reused_after_long_segments(gpu_device):
    """Regression shape of the K2 load-path bug (K2 read its slow entries through the non-coherent cache while
    rewriting the same array): one handle encodes text with many LONG segments, then text whose plain slow entries
    take the same slots, back and forth."""
    rng = random.Random(51)
    vocab = LETTER_VOCAB + [LONG_HEAD]
    o = Oracle(vocab)
    longs = b" ".join((LONG_HEAD + _word(rng, rng.randint(1, 40)).decode()).encode() for _ in range(400))
    plain = b" ".join(_word(rng, rng.randint(2, 40)) for _ in range(30000))
    e_long, e_plain = o.encode(longs), o.encode(plain)
    v = _vocab(vocab, gpu_device)
    for rep in range(3):
        _same(e_long, v.encode(longs), f"long {rep}")
        _same(e_plain, v.encode(plain), f"plain {rep}")
    v.close()


# --------------------------------------------------------------------------------- F. positions past 4 GiB

@pytest.mark.gpu
def test_positions_past_4_gib(gpu_device):
    """A LONG entry keeps its text position in 32 + 8 bits.  A 4.3 GiB device text of 15-byte filler words (one
    K1 static hit each) holds windows with long segments (multi-round chains, invalid bytes, Han heads) that start
    just before 2^32, at 2^32, at 2^32 + 1 and straddle it; the ids are the filler ids plus the oracle's ids of
    each window at offsets known from the construction."""
    import torch

    rng = random.Random(61)
    filler = b"abcdefghijklmno "
    vocab = LETTER_VOCAB + [filler[:-1].decode(), cases.ZH, "##" + "é", "é"]
    o = Oracle(vocab)
    filler_id = len(LETTER_VOCAB)
    G32 = 1 << 32
    n = G32 + (256 << 20)
    # four LONG segments: a multi-round UNK, a multi-round chain with invalid bytes, a Han head, multi-byte chars
    win = (b"Z" + _word(rng, 2000) + b" " + _word(rng, 1500) + b"\xff\xfe" + _word(rng, 900) + b" " +
           cases.ZH.encode() + _word(rng, 1300) + b" " + "é".encode() * 400 + _word(rng, 600) + b"\xe4\xb8" + b" ab")
    dev = torch.device("cuda", gpu_device)
    unit = torch.from_numpy(np.frombuffer(filler, np.uint8).copy()).to(dev)
    torch.cuda.reset_peak_memory_stats(dev)
    d_text = unit.repeat(n // 16)
    d_ids = torch.empty(n // 16 + len(win), dtype=torch.int32, device=dev)
    v = _vocab(vocab, gpu_device)
    # the window starts just before 2^32 (its first segment straddles it), at 2^32, at 2^32 + 1, 700 bytes before
    # it (a later segment straddles it), and near the end of the text; it sits in a region of whole filler words
    for s in (G32 - 5, G32, G32 + 1, G32 - 700, n - len(win) - 100):
        r0 = (s - 1) // 16 * 16
        r1 = (s + len(win) + 1 + 15) // 16 * 16
        region = b" " * (s - r0) + win + b" " * (r1 - s - len(win))
        saved = d_text[r0:r1].clone()
        d_text[r0:r1] = torch.from_numpy(np.frombuffer(region, np.uint8).copy()).to(dev)
        region_ids = torch.from_numpy(o.encode(region)).to(dev)
        before, after = r0 // 16, (n - r1) // 16
        total = before + len(region_ids) + after
        d_ids.fill_(-7)
        _, cnt = v.encode_device(d_text, d_ids)
        assert cnt == total, (s, cnt, total)
        assert v.stats().long_segments == 4, (s, v.stats())
        got = d_ids[before:before + len(region_ids)]
        if not torch.equal(got, region_ids):
            k = int(torch.nonzero(got != region_ids)[0].item())
            raise AssertionError(f"window at {s}: first mismatch at its id {k}: expected {region_ids[k:k + 6].tolist()} "
                                 f"got {got[k:k + 6].tolist()}")
        assert bool((d_ids[:before] == filler_id).all()) and bool((d_ids[before + len(region_ids):total] == filler_id).all()), s
        d_text[r0:r1] = saved
    assert torch.cuda.max_memory_allocated(dev) < 12e9
    v.close()
