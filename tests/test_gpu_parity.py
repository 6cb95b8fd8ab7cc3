"""GPU parity: the CUDA path (through the C ABI) against the oracle, bit-exact.

Every test calls libwordpiece_b200.so -> sm_100a kernels and compares the id
array with oracle/wp_oracle.c on the same bytes.  Nothing here reads
/root/reference; golden vectors are tests/golden/*.json and tests/cases.py.
"""
from __future__ import annotations

import json
import os
import random

import numpy as np
import pytest

import cases
import textgen
from _oracle import EmptyVocabWord, Oracle

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


def _vocab(tokens, dev):
    from wordpiece_b200 import Vocab

    return Vocab(tokens, device=dev)


def _check(text, tokens, dev, tag=""):
    if isinstance(text, str):
        text = text.encode("utf-8")
    exp = Oracle(tokens).encode(text)
    v = _vocab(tokens, dev)
    got = v.encode(text)
    st = v.stats()
    v.close()
    if not np.array_equal(exp, got):
        k = int(np.argmax(exp[: min(len(exp), len(got))] != got[: min(len(exp), len(got))])) if len(exp) and len(got) else 0
        raise AssertionError(
            f"{tag}: ids differ (oracle {len(exp)} vs gpu {len(got)}), first mismatch at {k}: "
            f"oracle {exp[max(0, k - 3):k + 5].tolist()} gpu {got[max(0, k - 3):k + 5].tolist()}; text[:80]={text[:80]!r}"
        )
    return st


def test_reference_golden_vectors(gpu_device):
    """tests/tests.cpp:137-217 — the reference's own 28 known-answer cases."""
    for text, vocab, expected in cases.REFERENCE_GOLDEN:
        v = _vocab(vocab, gpu_device)
        got = v.encode(text).tolist()
        v.close()
        assert got == expected, (text, vocab, expected, got)


def test_reference_differential_cases(gpu_device):
    for text, vocab in cases.REFERENCE_DIFFERENTIAL:
        _check(text, vocab, gpu_device, "differential")


def test_quirks_match_recorded_reference_output(gpu_device):
    """SURVEY A.3 behaviours; expected ids were produced by the compiled reference (tests/golden/quirks.json)."""
    with open(os.path.join(HERE, "golden", "quirks.json")) as f:
        golden = json.load(f)
    names = {name for name, _, _ in cases.QUIRKS}
    assert names == set(golden), "regenerate tests/golden (make_golden.py)"
    for name, text, vocab in cases.QUIRKS:
        v = _vocab(vocab, gpu_device)
        got = v.encode(text).tolist()
        v.close()
        assert got == golden[name]["ids"], (name, golden[name]["ids"], got)


def test_empty_and_degenerate_inputs(gpu_device):
    v = _vocab(["a", "[UNK]"], gpu_device)
    assert v.encode(b"").size == 0                      # fast.cpp:145
    assert v.encode(b"   \n\t ").size == 0
    assert v.encode(b"\xff\xfe\x80").size == 0          # decodes to nothing (reference: SIGFPE; we return {})
    assert v.encode(b"a").tolist() == [0]
    assert v.encode(b" a ").tolist() == [0]
    v.close()
    # no usable token at all (reference divides by zero, fast.cpp:45): every word is UNK
    v = _vocab(["[UNK]", "[CLS]"], gpu_device)
    assert v.encode("ab, 中c".encode()).tolist() == Oracle(["[UNK]", "[CLS]"]).encode("ab, 中c".encode()).tolist()
    v.close()


def test_empty_vocab_word_is_an_error(gpu_device):
    from wordpiece_b200 import WordPieceError

    for vocab in (["a", "##"], ["a", ""], ["\xff".encode("latin1")]):
        with pytest.raises(EmptyVocabWord):
            Oracle(vocab)
        with pytest.raises(WordPieceError) as ei:
            _vocab(vocab, gpu_device)
        assert ei.value.status == 2 and "Vocab word is empty" in str(ei.value)


def test_hostile_fuzz_tiny(gpu_device):
    """SURVEY A.5: tiny vocabularies over a hostile alphabet, invalid bytes included."""
    rng = random.Random(20240517)
    n = 0
    for i in range(2500):
        text, vocab = cases.fuzz_case(rng)
        try:
            Oracle(vocab)
        except EmptyVocabWord:
            continue
        _check(text, vocab, gpu_device, f"fuzz#{i}")
        n += 1
    assert n > 2000


def test_random_split_small(gpu_device):
    """tests.cpp:257-258 — random [a-z] strings cut into vocab pieces, positive and negative."""
    rng = random.Random(17)
    for text_len in range(10, 301, 10):
        for parts in (2, 3, 7, 20, 55, 100):
            if parts > text_len:
                continue
            for positive in (True, False):
                s, vocab = cases.random_split_case(rng, text_len, parts, positive)
                _check(s, vocab, gpu_device, f"split L={text_len} parts={parts} pos={positive}")


@pytest.mark.parametrize("seed,n_bytes", [(11, 5000), (12, 8192), (13, 8193), (14, 8191), (17, 4096), (18, 4097), (19, 4095),
                                          (15, 40000), (16, 300000)])
def test_multilingual_multi_tile(gpu_device, seed, n_bytes):
    import wordpiece_b200

    text, vocab = textgen.case(seed, n_bytes)
    st = _check(text, vocab, gpu_device, f"mixed seed={seed}")
    tile = wordpiece_b200.tile_bytes()
    assert st.n_tiles == (len(text) + tile - 1) // tile


@pytest.mark.parametrize("seed,n_bytes,rate", [(21, 3000, 0.3), (22, 30000, 0.05), (23, 100000, 0.01), (24, 60000, 0.5)])
def test_invalid_utf8_is_dropped(gpu_device, seed, n_bytes, rate):
    """utf8.cpp:130-147: invalid bytes vanish before word splitting, across tile borders too."""
    text, vocab = textgen.case(seed, n_bytes, invalid_rate=rate)
    st = _check(text, vocab, gpu_device, f"dirty seed={seed}")
    assert st.dirty_tiles > 0


def test_invalid_runs_across_tile_borders(gpu_device):
    vocab = ["ab", "##cd", "abcd", "x", "中", "[UNK]"]
    import wordpiece_b200

    tile = wordpiece_b200.tile_bytes()
    for junk in (b"\xff", b"\x80", b"\xe4\xb8", b"\xf0\x9f\x98"):
        for pad in list(range(tile - 12, tile + 8)) + list(range(2 * tile - 12, 2 * tile + 8, 3)):
            text = b"x " * (pad // 2) + b"ab" + junk * 7 + b"cd" + junk * 40 + " 中".encode() + junk + b" x"
            _check(text, vocab, gpu_device, f"junk={junk!r} pad={pad}")
    # a run of invalid bytes longer than a whole tile between the halves of one word
    text = b"ab" + b"\xff" * 20000 + b"cd x"
    _check(text, vocab, gpu_device, "long junk")


def test_multibyte_chars_straddle_tile_borders(gpu_device):
    vocab = ["中", "文", "中文", "при", "##вет", "かな", "##かな", "a", "##a", "[UNK]"]
    unit = "中文 привет かなかな a ".encode()
    for shift in range(0, 12):
        text = b"a" * shift + unit * 700
        _check(text, vocab, gpu_device, f"shift={shift}")


@pytest.mark.parametrize("seed,n_bytes", [(31, 50000), (32, 200000)])
def test_long_segments_leave_the_window(gpu_device, seed, n_bytes):
    """Words longer than a tile's halo are walked from global memory (at most one per tile)."""
    text, vocab = textgen.case(seed, n_bytes, long_run_rate=0.08, long_tokens=40)
    st = _check(text, vocab, gpu_device, f"long seed={seed}")
    assert st.long_segments > 0


def test_giant_single_word(gpu_device):
    """tests.cpp:259-272 shape: one space-free word far longer than a tile, vocab = a random cut of it."""
    rng = random.Random(5)
    for text_len, parts, positive in ((20000, 300, True), (20000, 300, False), (100000, 2000, True)):
        s, vocab = cases.random_split_case(rng, text_len, parts, positive)
        st = _check(s, vocab, gpu_device, f"giant L={text_len}")
        assert st.long_segments >= 1


def test_long_dirty_word(gpu_device):
    """A long word with invalid bytes sprinkled in: the global walker must drop them on the fly."""
    rng = random.Random(8)
    s, vocab = cases.random_split_case(rng, 30000, 500, True)
    b = bytearray(s.encode())
    for _ in range(300):
        b.insert(rng.randint(0, len(b)), 0xFF)
    _check(bytes(b), vocab, gpu_device, "long dirty")


def test_capacity_and_encode_into(gpu_device):
    from wordpiece_b200 import WordPieceError

    text, vocab = textgen.case(41, 50000)
    exp = Oracle(vocab).encode(text)
    v = _vocab(vocab, gpu_device)
    out = np.full(len(exp) + 10, -7, np.int32)
    n = v.encode_into(text, out)
    assert n == len(exp) and np.array_equal(out[:n], exp) and (out[n:] == -7).all()
    small = np.zeros(len(exp) // 2, np.int32)
    with pytest.raises(WordPieceError) as ei:
        v.encode_into(text, small)
    assert ei.value.status == 5
    v.close()


def test_device_resident_entry_point(gpu_device):
    import torch

    text, vocab = textgen.case(42, 120000, invalid_rate=0.01)
    exp = Oracle(vocab).encode(text)
    v = _vocab(vocab, gpu_device)
    d_text = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda(gpu_device)
    d_ids, n = v.encode_device(d_text)
    assert n == len(exp) and np.array_equal(d_ids[:n].cpu().numpy(), exp)
    # misaligned device pointer (a slice): falls back to byte loads, same ids
    for off in (1, 3, 8, 13):
        sub = d_text[off:]
        e2 = Oracle(vocab).encode(text[off:])
        ids2, n2 = v.encode_device(sub)
        assert n2 == len(e2) and np.array_equal(ids2[:n2].cpu().numpy(), e2), off
    # async variant
    d_cnt = torch.zeros(1, dtype=torch.int64, device=d_text.device)
    d_out = torch.empty(len(text), dtype=torch.int32, device=d_text.device)
    v.encode_device_async(d_text, d_out, d_cnt)
    torch.cuda.synchronize()
    assert int(d_cnt.item()) == len(exp) and np.array_equal(d_out[: len(exp)].cpu().numpy(), exp)
    v.close()


def test_handle_reuse_and_order_independence(gpu_device):
    """One handle, many texts of different sizes: scratch is reset between calls."""
    text, vocab = textgen.case(43, 90000)
    o = Oracle(vocab)
    v = _vocab(vocab, gpu_device)
    for cut in (90000, 17, 8192, 50000, 1, 33333, 90000):
        assert np.array_equal(v.encode(text[:cut]), o.encode(text[:cut])), cut
    v.close()


def test_several_ranges_per_call(gpu_device, monkeypatch):
    """Large texts are encoded range by range (bounded scratch); force small ranges to cover the hand-over:
    segments that straddle a range border, the running id offset, slow-list and look-back state resets."""
    import wordpiece_b200

    tile = wordpiece_b200.tile_bytes()
    text, vocab = textgen.case(61, 30 * tile + 123, invalid_rate=0.004, long_run_rate=0.02, long_tokens=10)
    exp = Oracle(vocab).encode(text)
    v = _vocab(vocab, gpu_device)
    for range_bytes in (tile, 3 * tile, 7 * tile + 1):
        monkeypatch.setenv("WORDPIECE_B200_RANGE_BYTES", str(range_bytes))
        got = v.encode(text)
        assert np.array_equal(exp, got), range_bytes
        assert v.stats().kernel_launches >= 3 * (len(text) // (range_bytes + tile))
    monkeypatch.delenv("WORDPIECE_B200_RANGE_BYTES")
    assert np.array_equal(exp, v.encode(text))
    v.close()


def test_host_buffer_pipeline(gpu_device, monkeypatch):
    """wp_encode_into on large texts runs a three-stage pipeline (copy in / encode / copy out) over chunks
    cut after a space; force small chunks so that many of them — and a text with a stretch that has no
    space to cut at, which must fall back to the single-shot path — are covered."""
    text, vocab = textgen.case(71, 400_000, invalid_rate=0.003)
    o = Oracle(vocab)
    exp = o.encode(text)
    v = _vocab(vocab, gpu_device)
    out = np.full(len(exp) + 5, -9, np.int32)
    for chunk in (4096, 30_000, 150_000):
        monkeypatch.setenv("WORDPIECE_B200_PIPE_CHUNK", str(chunk))
        out[:] = -9
        n = v.encode_into(text, out)
        assert n == len(exp) and np.array_equal(out[:n], exp) and (out[n:] == -9).all(), chunk
        assert v.stats().kernel_launches >= 3 * (len(text) // chunk)
    # the chunks of one call share the word memo: the first clears and warms it, later ones only use it
    monkeypatch.setenv("WORDPIECE_B200_MEMO", "1")
    monkeypatch.setenv("WORDPIECE_B200_PIPE_CHUNK", "30000")
    for _ in range(2):
        out[:] = -9
        n = v.encode_into(text, out)
        assert n == len(exp) and np.array_equal(out[:n], exp) and (out[n:] == -9).all()
    monkeypatch.delenv("WORDPIECE_B200_MEMO")
    # too small a buffer: exact count reported
    from wordpiece_b200 import WordPieceError

    with pytest.raises(WordPieceError) as ei:
        v.encode_into(text, np.zeros(len(exp) // 3, np.int32))
    assert ei.value.status == 5
    # pinned id buffer, also not 16-byte aligned
    import torch

    pin = torch.full((len(exp) + 5,), -9, dtype=torch.int32).pin_memory()
    pout = pin.numpy()
    for off in (0, 1, 3):
        pout[:] = -9
        n = v.encode_into(text, pout[off:])
        assert n == len(exp) and np.array_equal(pout[off:off + n], exp) and (pout[:off] == -9).all()
    # no space within a chunk: falls back, same ids
    monkeypatch.setenv("WORDPIECE_B200_PIPE_CHUNK", "4096")
    glued = text[:50_000] + b"x" * 9000 + text[50_000:]
    e2 = o.encode(glued)
    out2 = np.zeros(len(e2) + 8, np.int32)
    n2 = v.encode_into(glued, out2)
    assert n2 == len(e2) and np.array_equal(out2[:n2], e2)
    v.close()


def test_hostile_bytes_at_chunk_borders(gpu_device):
    """K1 classifies 32-byte chunks; a UTF-8 sequence that breaks just before a chunk border leaves stray
    continuation bytes just behind it (E2 's' | 80).  Random hostile byte runs are laid over every 32-byte
    border of a text (and over 4 KiB tile borders), in words that need several pieces, so that a single kept
    stray byte changes the ids."""
    rng = random.Random(77)
    vocab = ["[UNK]"] + [c for c in "abcdefghijklmnopqrstuvwxyz"] + ["##" + c for c in "abcdefghijklmnopqrstuvwxyz"] + \
            ["re", "##tc", "##s", "ab", "##cd", "é", "##é", "中", "文", "か", "##か", ",", "."]
    hostile = [b"\xe2", b"\x80", b"\xbf", b"\xc3", b"\xe4\xb8", b"\xf0\x9f", b"\xf0\x9f\x98", b"\xed\xa0", b"\xc0", b"\xff",
               "é".encode(), "中".encode(), "か".encode(), b"s", b"tc", b" ", b"a", b"", b"", b"\xe2\x96\x81", b"\xe2\x80\x94"]
    for trial in range(4):
        buf = bytearray()
        while len(buf) < 150_000:
            # fill up to a few bytes before the next 32-byte border with letters and spaces, then hostile bytes
            border = (len(buf) // 32 + 1) * 32
            lead_in = border - len(buf) - rng.randint(0, 5)
            while lead_in > 0:
                w = "".join(rng.choice("abcdrestc") for _ in range(rng.randint(1, 7))).encode()[:lead_in]
                buf += w
                lead_in -= len(w)
                if lead_in > 0 and rng.random() < 0.6:
                    buf += b" "
                    lead_in -= 1
            for _ in range(rng.randint(1, 5)):
                buf += rng.choice(hostile)
        text = bytes(buf)
        _check(text, vocab, gpu_device, f"chunk-border fuzz #{trial}")
        _check(b"xy " * trial + text, vocab, gpu_device, f"chunk-border fuzz #{trial} shifted")
    # the case that was found in the dirty-web text: the stray byte is the first byte of a chunk
    for shift in range(0, 40):
        t = b"a" * shift + b" re\xbftc\xe2s\x80 brarbad ci teas"
        _check(t * 300, vocab, gpu_device, f"E2 s | 80 at shift {shift}")


def test_cpp_drop_in_runner(gpu_device, tmp_path):
    """The C++ entry points (include/word_piece.hpp) through the runner CLI with the reference's argv
    contract (tests/runner.cpp:13-65): `fast` prints "Total ids N" and writes "id id id "; `fast-external`
    streams the file in batches cut at a space (fast.cpp:189-220)."""
    import subprocess

    from wordpiece_b200 import synth

    root = os.path.dirname(HERE)
    runner = os.path.join(root, "wordpiece_b200", "lib", "runner")
    g = synth.generator("en")
    text = g.generate(3_000_000, seed=9).tobytes()
    vocab = g.spec.vocab
    tf, vf = tmp_path / "text.txt", tmp_path / "vocab.txt"
    tf.write_bytes(text)
    synth.write_vocab_file(str(vf), vocab)
    exp = Oracle(vocab).encode(text)
    want = "".join(f"{i} " for i in exp.tolist())

    out1 = tmp_path / "ids_fast.txt"
    r = subprocess.run([runner, "fast", str(tf), str(vf), "8", str(out1)], capture_output=True, text=True, check=True)
    assert r.stdout.strip() == f"Total ids {len(exp)}"
    assert out1.read_text() == want
    r = subprocess.run([runner, "fast", str(tf), str(vf), "8"], capture_output=True, text=True, check=True)
    assert r.stdout.strip() == f"Total ids {len(exp)}"

    out2 = tmp_path / "ids_ext.txt"
    # memory_limit_mb >= 50 is enforced by the CLI; the text is 3 MB, so also drive the library entry directly
    subprocess.run([runner, "fast-external", str(tf), str(vf), "8", str(out2), "50"], check=True)
    assert out2.read_text() == want
    import wordpiece_b200

    out3 = tmp_path / "ids_ext_small.txt"
    wordpiece_b200.encode_external(str(tf), str(vf), str(out3), 200_000)  # 100 kB batches
    assert out3.read_text() == want
    # stateless Python mirrors of fast::encode
    assert np.array_equal(wordpiece_b200.encode_files(str(tf), str(vf)), exp)
    assert np.array_equal(wordpiece_b200.encode(text[:100_000], vocab), Oracle(vocab).encode(text[:100_000]))
    # unknown modes are rejected like the reference does for bad argv
    bad = subprocess.run([runner, "linear", str(tf), str(vf)], capture_output=True, text=True)
    assert bad.returncode != 0


def test_displaced_single_char_words(gpu_device, monkeypatch):
    """A single-char segment is always settled by K1 (the slow-list capacities assume >= 2 bytes per entry):
    a word-table hit, "absent => UNK" (the static part is complete), or — when its slot lies further from
    home than K1's lookup looks — the rare probe-sequence walk.  The vocabulary is built so that some
    single chars are displaced by 1..3 slots and one by more than that.
    Worst case text: nothing but such a char (one segment per byte)."""
    import string
    import wordpiece_b200
    from _model import word_hash_py

    rng = random.Random(0)
    words = list(dict.fromkeys("".join(rng.choice(string.ascii_lowercase) for _ in range(rng.randint(2, 6)))
                               for _ in range(3000)))
    singles = list(string.ascii_lowercase) + list(string.punctuation)
    n_short = len(words) + len(singles) + 8
    log2 = 6
    while (1 << log2) < 4 * n_short:
        log2 += 1
    # six words that hash to the home slot of "q" and come BEFORE it in the vocabulary: "q" ends up >= 6 away
    home = word_hash_py(b"q", log2)
    crowd = []
    while len(crowd) < 6:
        w = "".join(rng.choice(string.ascii_lowercase) for _ in range(rng.randint(7, 12)))
        if word_hash_py(w.encode(), log2) == home and w not in words:
            crowd.append(w)
    vocab = ["[UNK]"] + crowd + words + ["##" + w for w in words[:500]] + singles
    v = _vocab(vocab, gpu_device)
    assert v.table_info["word_slots"] == 1 << log2
    near = [chr(c) for c in v.debug_displaced_singles(1) if c < 128]
    far = [chr(c) for c in v.debug_displaced_singles(4) if c < 128]
    assert "q" in far and len(near) >= 2, (near, far)
    ora = Oracle(vocab)
    tile = wordpiece_b200.tile_bytes()
    texts = [("q" * (5 * tile + 17)).encode(), ("".join(near) * (tile // 2)).encode()]
    parts = []
    for _ in range(60000):
        x = rng.random()
        parts.append(rng.choice(near) if x < 0.3 else rng.choice(string.punctuation) if x < 0.4
                     else rng.choice(words + crowd) if x < 0.8 else " ")
    texts.append("".join(parts).encode())
    for memo in ("0", "1"):
        monkeypatch.setenv("WORDPIECE_B200_MEMO", memo)
        monkeypatch.setenv("WORDPIECE_B200_RANGE_BYTES", str(8 * tile))
        for t in texts:
            assert np.array_equal(ora.encode(t), v.encode(t)), (memo, len(t))
    v.close()
    # a crowded working table (no larger than the static image): recorded words and static words share
    # probe sequences, lookups run past WORD_PROBES slots, inserts fail — not one id may change
    monkeypatch.setenv("WORDPIECE_B200_WORD_SLOTS_LOG2", "6")
    monkeypatch.setenv("WORDPIECE_B200_MEMO", "1")
    monkeypatch.setenv("WORDPIECE_B200_RANGE_BYTES", str(2 * tile))
    text, vocab2 = textgen.case(91, 60 * tile)
    v = _vocab(vocab2, gpu_device)
    assert np.array_equal(Oracle(vocab2).encode(text), v.encode(text))
    v.close()
    monkeypatch.delenv("WORDPIECE_B200_WORD_SLOTS_LOG2")
    # multi-byte chars: the displaced single chars of the 120k vocabulary (CJK, their own segments) in running text
    from wordpiece_b200 import synth

    g = synth.generator("zh")
    v = _vocab(g.spec.vocab, gpu_device)
    d = [chr(c) for c in v.debug_displaced_singles(1)]
    assert d
    base = g.generate(1 << 20, seed=5).tobytes().decode("utf-8", "ignore")
    mixed = []
    for i in range(0, len(base), 50):
        mixed.append(base[i:i + 50])
        mixed.append(rng.choice(d) + rng.choice(["", " ", ",", rng.choice(d)]))
    t = "".join(mixed).encode()
    monkeypatch.delenv("WORDPIECE_B200_MEMO")
    assert np.array_equal(Oracle(g.spec.vocab).encode(t), v.encode(t))
    v.close()


def test_word_memo(gpu_device, monkeypatch):
    """The dynamic part of the word table (K2 records bytes -> ids of short unsettled segments, K1 of later
    ranges settles repeats with its one lookup) must not change a single id.  Small ranges maximise the traffic
    through it; dirty tiles, walked segments and Han-led segments ride along."""
    import wordpiece_b200

    tile = wordpiece_b200.tile_bytes()
    monkeypatch.setenv("WORDPIECE_B200_MEMO", "1")
    for seed, n, kw in [(81, 40 * tile, {}), (82, 25 * tile + 77, dict(invalid_rate=0.01)),
                        (83, 30 * tile, dict(long_run_rate=0.03, long_tokens=12))]:
        text, vocab = textgen.case(seed, n, **kw)
        exp = Oracle(vocab).encode(text)
        v = _vocab(vocab, gpu_device)
        hits = []
        for range_bytes in (tile, 4 * tile, 1 << 30):
            monkeypatch.setenv("WORDPIECE_B200_RANGE_BYTES", str(range_bytes))
            got = v.encode(text)
            assert np.array_equal(exp, got), (seed, range_bytes)
            hits.append(v.stats().memo_hits)
        # one range: nothing recorded yet when K1 runs; many ranges: repeats hit (also in tiles with invalid bytes)
        assert hits[2] == 0 and hits[0] > 0, hits
        # the memo is reset per call: same ids and same hit count when the call is repeated
        monkeypatch.setenv("WORDPIECE_B200_RANGE_BYTES", str(tile))
        assert np.array_equal(exp, v.encode(text)) and v.stats().memo_hits == hits[0]
        monkeypatch.setenv("WORDPIECE_B200_MEMO", "0")
        assert np.array_equal(exp, v.encode(text)) and v.stats().memo_hits == 0
        monkeypatch.setenv("WORDPIECE_B200_MEMO", "1")
        v.close()
    # English-like corpus with its Zipf repeats, memo on by size (>= 4 MiB), against the oracle
    monkeypatch.delenv("WORDPIECE_B200_MEMO")
    monkeypatch.setenv("WORDPIECE_B200_RANGE_BYTES", str(1 << 20))
    from wordpiece_b200 import synth

    g = synth.generator("en")
    text = g.generate(6 << 20, seed=12).tobytes()
    v = _vocab(g.spec.vocab, gpu_device)
    assert np.array_equal(Oracle(g.spec.vocab).encode(text), v.encode(text))
    assert v.stats().memo_hits > 10000
    v.close()
    # random strings never repeat: the memo is switched off in the middle of the call (the decision is taken
    # per tile while other tiles move the counters), and not one id may change
    g = synth.generator("adv")
    text = g.generate(8 << 20, seed=13).tobytes()
    monkeypatch.setenv("WORDPIECE_B200_RANGE_BYTES", str(256 << 10))
    v = _vocab(g.spec.vocab, gpu_device)
    exp = Oracle(g.spec.vocab).encode(text)
    for _ in range(3):
        assert np.array_equal(exp, v.encode(text))
    v.close()


def test_full_size_properties(gpu_device):
    """BASELINE configs[1] at full size (1 GiB of English-like text, 29k vocabulary), checked through
    properties that do not need the CPU oracle at that size: the call is deterministic; the text cut after
    a space encodes piecewise to the same ids (the reference's own chunk + concat rule, fast.cpp:113-138);
    the host-buffer pipeline returns the device-resident ids; head and tail agree with the oracle."""
    import torch

    from wordpiece_b200 import synth

    mib = 1 << 20
    n = 1024 * mib
    g = synth.generator("en")
    h_text = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    g.fill(h_text.numpy(), seed=2, first_block=0, n_threads=os.cpu_count() or 8)
    dev = torch.device("cuda", gpu_device)
    d_text = h_text.to(dev)
    v = _vocab(g.spec.vocab, gpu_device)
    cap = n // 2
    ids_a = torch.empty(cap, dtype=torch.int32, device=dev)
    _, n_a = v.encode_device(d_text, ids_a)
    assert 0 < n_a <= cap and v.stats().n_tiles == n // 4096 and v.stats().dirty_tiles == 0
    # deterministic
    ids_b = torch.empty(cap, dtype=torch.int32, device=dev)
    _, n_b = v.encode_device(d_text, ids_b)
    assert n_b == n_a and torch.equal(ids_a[:n_a], ids_b[:n_a])
    # piecewise: the generator's 1 MiB blocks end with a space, so any block boundary is a legal cut
    cuts = [0, 1, 3, 4, 131, 400, 401, 777, 1023, 1024]
    at = 0
    for lo, hi in zip(cuts, cuts[1:]):
        assert h_text[hi * mib - 1].item() in (0x20, 0x0A)
        piece = torch.empty((hi - lo) * mib // 2, dtype=torch.int32, device=dev)
        _, k = v.encode_device(d_text[lo * mib:hi * mib], piece)
        assert torch.equal(piece[:k], ids_a[at:at + k]), (lo, hi)
        at += k
    assert at == n_a
    del ids_b, piece
    # host-buffer entry point (three-stage pipeline over PCIe)
    h_ids = torch.empty(cap, dtype=torch.int32, pin_memory=True)
    k = v.encode_into(h_text.numpy(), h_ids.numpy())
    assert k == n_a and torch.equal(h_ids[:k], ids_a[:k].cpu())
    # head and tail against the oracle
    o = Oracle(g.spec.vocab)
    head = o.encode(h_text[:8 * mib].numpy().tobytes())
    assert np.array_equal(head, ids_a[:len(head)].cpu().numpy())
    tail = o.encode(h_text[-4 * mib:].numpy().tobytes())
    assert np.array_equal(tail, ids_a[n_a - len(tail):n_a].cpu().numpy())
    v.close()


def test_id_text_formatted_on_device(gpu_device):
    """wp_encode_text: the ids as ``"id id id "`` (fast.cpp:214-216 / utils.cpp:30-35), formatted by a kernel.
    Covers -1 (no [UNK] in the vocabulary), ids of every decimal length up to six digits, block borders of
    the formatter, and the empty text."""
    rng = random.Random(3)
    alphabet = "abcdefghijklmnopqrstuvwxyz"
    # 150 000 distinct tokens: ids span 1..6 decimal digits; no [UNK] => unknown words are -1
    vocab, seen = [], set()
    while len(vocab) < 150_000:
        w = "".join(rng.choice(alphabet) for _ in range(rng.randint(1, 5)))
        if w not in seen:
            seen.add(w)
            vocab.append(w)
    words = [rng.choice(vocab) if rng.random() < 0.9 else "".join(rng.choice("XYZ") for _ in range(4))
             for _ in range(120_000)]
    text = " ".join(words).encode()
    o = Oracle(vocab)
    v = _vocab(vocab, gpu_device)
    for cut in (len(text), 2048 * 3, 4096, 7, 1):
        t = text[:cut]
        while t and t[-1:] != b" " and cut != len(text):
            t = t[:-1]
        exp = o.encode(t) if t else np.zeros(0, np.int32)
        want = b"".join(b"%d " % i for i in exp.tolist())
        got = v.encode_text(t)
        assert got == want, (cut, got[:60], want[:60])
    exp = o.encode(text)
    assert (exp == -1).any() and (exp >= 100_000).any() and (exp < 10).any()
    assert v.encode_text(b"") == b""
    v.close()


def test_ticket_mode_is_exact(gpu_device, monkeypatch):
    """K1's fallback order of tiles (an atomic ticket instead of the block index; the host switches to it when a
    look-back walk gives up waiting) gives the same ids: several ranges, dirty tiles, long segments."""
    monkeypatch.setenv("WORDPIECE_B200_TICKET", "1")
    monkeypatch.setenv("WORDPIECE_B200_RANGE_BYTES", str(256 * 1024))
    text, vocab = textgen.case(41, 1_500_000, invalid_rate=0.002, long_run_rate=0.01, long_tokens=4)
    st = _check(text, vocab, gpu_device, "ticket mode")
    assert st.n_tiles > 300


def test_dense_tiles_fall_back_to_full_lists(gpu_device):
    """A tile of punctuation holds one segment per byte — more than the segment lists of the regular K1 (3 072 per
    4 KiB tile, which is what lets eight tiles share an SM).  The call is flagged dense and repeated with the
    full-capacity kernel; ids are the oracle's, also for later calls on the same handle and for a batch."""
    from wordpiece_b200 import Vocab

    vocab = ["[UNK]", ".", ",", "!", "?", "a", "b", "ab", "##b", "(", ")", "中"]
    dense = (b".,!?()" * 3000)[:15000]
    text = b"ab ab " + dense + b" ab a" + "中中中".encode() * 700 + b" b " + dense[:5000]
    o = Oracle(vocab)
    v = Vocab(vocab, device=gpu_device)
    assert np.array_equal(o.encode(text), v.encode(text))
    assert np.array_equal(o.encode(b"ab ab. a"), v.encode(b"ab ab. a"))      # the handle stays usable (and exact)
    ids, offs = v.encode_batch([b"ab", dense, b"", b"a.b"])
    for i, t in enumerate([b"ab", dense, b"", b"a.b"]):
        assert np.array_equal(o.encode(t), ids[int(offs[i]):int(offs[i + 1])]), i
    v.close()
    v2 = Vocab(vocab, device=gpu_device)                                        # a fresh handle, dense batch first
    ids, offs = v2.encode_batch([dense[:9000], b"ab"])
    assert np.array_equal(o.encode(dense[:9000]), ids[int(offs[0]):int(offs[1])])
    assert np.array_equal(o.encode(b"ab"), ids[int(offs[1]):int(offs[2])])
    import torch

    d_text = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda(gpu_device)
    v3 = Vocab(vocab, device=gpu_device)                                        # device-resident entry
    d_ids, n = v3.encode_device(d_text)
    assert np.array_equal(o.encode(text), d_ids[:n].cpu().numpy())
    v2.close()
    v3.close()


def test_repeated_calls_on_one_handle_with_long_runs(gpu_device):
    """Regression (round 2): the last segment of a tile may have no end inside the tile's window; its end entry in
    shared memory was then never written, and when the stale value there happened to be the "undecided single
    char" marker, K1's pass for those overwrote the START of the long segment with a token id — wrong ids that
    depended on the kernels that had run before.  Found by the randomised sweep (seed 1140); this is its small
    form: texts with several long space-free runs, three calls each on ONE handle (the first call was right,
    later ones wrong)."""
    import re

    from wordpiece_b200 import Vocab

    text, vocab = textgen.case(1140, 1_192_536, invalid_rate=0.0, long_run_rate=0.02, long_tokens=5)
    o = Oracle(vocab)
    v = Vocab(vocab, device=gpu_device)
    runs = [(m.start(), m.end()) for m in re.finditer(rb"[^ \n\t\r]{257,}", text)]
    assert len(runs) > 100
    for a, b in runs[:120:4]:
        lo, hi = max(0, a - 3000), min(len(text), b + 3000)
        while lo > 0 and text[lo - 1:lo] not in (b" ", b"\n"):
            lo -= 1
        while hi < len(text) and text[hi:hi + 1] not in (b" ", b"\n"):
            hi += 1
        t = text[lo:hi]
        exp = o.encode(t)
        for rep in range(3):
            got = v.encode(t)
            assert np.array_equal(exp, got), (a, b, rep, len(exp), len(got))
    v.close()


def test_two_handles_in_two_host_threads(gpu_device):
    """Handles are independent: two host threads, each with its own handle (own stream, scratch and word memo) on
    the same device, encoding at the same time (ctypes releases the GIL during the calls) — device-resident
    calls, host-buffer calls large enough for the chunk pipeline (shared copy pool), and batches."""
    import threading

    import torch

    from wordpiece_b200 import Vocab

    os.environ["WORDPIECE_B200_PIPE_CHUNK"] = "150000"
    os.environ["WORDPIECE_B200_BATCH_PART"] = "65536"
    try:
        jobs = []
        for seed in (4101, 4102):
            text, vocab = textgen.case(seed, 900_000, invalid_rate=0.001, long_run_rate=0.01, long_tokens=5)
            o = Oracle(vocab)
            cuts = sorted(random.Random(seed).sample(range(len(text)), 40))
            pieces = [text[a:b] for a, b in zip([0] + cuts, cuts + [len(text)])]
            jobs.append((text, vocab, o.encode(text), pieces, [o.encode(p) for p in pieces]))
        errors = []

        def work(i):
            try:
                text, vocab, exp, pieces, exp_pieces = jobs[i]
                v = Vocab(vocab, device=gpu_device)
                out = np.zeros(exp.size + 1, np.int32)
                pinned = torch.zeros(exp.size + 1, dtype=torch.int32).pin_memory()
                for rep in range(6):
                    assert np.array_equal(v.encode(text), exp), (i, rep, "encode")
                    for tag, buf in (("into", out), ("into pinned", pinned.numpy())):
                        n = v.encode_into(text, buf)
                        assert n == exp.size and np.array_equal(buf[:n], exp), (i, rep, tag)
                    ids, offs = v.encode_batch(pieces)
                    for k, e in enumerate(exp_pieces):
                        assert np.array_equal(ids[int(offs[k]):int(offs[k + 1])], e), (i, rep, "batch", k)
                v.close()
            except BaseException as e:  # noqa: BLE001
                errors.append(e)

        threads = [threading.Thread(target=work, args=(i,)) for i in range(2)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        assert not errors, errors[0]
    finally:
        os.environ.pop("WORDPIECE_B200_PIPE_CHUNK", None)
        os.environ.pop("WORDPIECE_B200_BATCH_PART", None)
