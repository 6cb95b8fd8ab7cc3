"""CPU tests of the product's host side: the C ABI surface, the vocabulary builder and its
table image (through the host mirror of the device probe), decode, the synthetic corpora
and the sharding plan.  No encode call is made here — that needs a GPU (tests -m gpu)."""
from __future__ import annotations

import ctypes
import os
import random
import re

import numpy as np
import pytest

import cases
import textgen
from _model import model_encode
from _oracle import EmptyVocabWord, Oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    import wordpiece_b200
    from wordpiece_b200._capi import EXPORTED_SYMBOLS

    header = open(os.path.join(ROOT, "include", "wordpiece_b200.h")).read()
    declared = set(re.findall(r"\b(wp_[a-z0-9_]+)\s*\(", header))
    assert declared == set(EXPORTED_SYMBOLS), declared ^ set(EXPORTED_SYMBOLS)
    lib = wordpiece_b200.load_library()
    for name in declared:
        assert hasattr(lib, name), name


def test_cpp_entry_points_are_exported():
    """The reference's C++ signatures (src/word_piece.hpp:25-34) exist in the shared library."""
    import subprocess

    out = subprocess.check_output(["nm", "-DC", "--defined-only", os.path.join(ROOT, "wordpiece_b200", "lib",
                                                                              "libwordpiece_b200.so")], text=True)
    for sig in ("word_piece::fast::encode(std::__cxx11::basic_string", "word_piece::fast::decode(",
                "word_piece::fast::encodeExternal(", "utils::writeToFile(", "utils::globalThreadPool("):
        assert sig in out, sig


def test_runner_argv_contract_without_a_device(tmp_path):
    """tests/runner.cpp:13-65 — everything the CLI decides before it encodes: argument count, the 50 MB floor of
    memory_limit_mb, external mode without a limit, unknown and out-of-scope modes; errors are uncaught
    std::runtime_error like the reference's (non-zero exit, message on stderr).  And with valid arguments but no
    CUDA device (this container) `fast` must fail loudly — there is no CPU path behind the CLI either."""
    import subprocess

    import torch

    runner = os.path.join(ROOT, "wordpiece_b200", "lib", "runner")
    if not os.path.exists(runner):
        pytest.skip("runner not built")
    tf, vf = tmp_path / "t.txt", tmp_path / "v.txt"
    tf.write_bytes(b"hello world")
    vf.write_bytes(b"[UNK]\nhello\nworld\n")

    def run(*argv):
        r = subprocess.run([runner, *map(str, argv)], capture_output=True, text=True)
        return r.returncode, r.stdout, r.stderr

    for argv, message in [
        (("fast", tf), "Usage: ./runner <mode> <text_file> <vocab_file>"),
        (("fast", tf, vf, 8, "o", 50, "extra"), "Usage: ./runner"),
        (("fast-external", tf, vf, 8, tmp_path / "o.txt", 49), "memory_limit cannot be less than 50Mb"),
        (("fast-external", tf, vf, 8, tmp_path / "o.txt"), "For external mode provide out_file and memory_limit"),
        (("fast-external", tf, vf), "For external mode provide out_file and memory_limit"),
        (("linear", tf, vf), "not part of wordpiece_b200"),
        (("linear-external", tf, vf, 8, tmp_path / "o.txt", 50), "not part of wordpiece_b200"),
        (("slow", tf, vf), "Unknown mode"),
    ]:
        rc, out, err = run(*argv)
        assert rc != 0 and message in err and out == "", (argv, rc, out, err)
    assert not (tmp_path / "o.txt").exists()
    if not torch.cuda.is_available():
        rc, out, err = run("fast", tf, vf, 8)
        assert rc != 0 and "Total ids" not in out and err.strip(), (rc, out, err)


def test_no_device_fails_loudly():
    """Without a CUDA device (this container) creation on device 0 must fail — never fall back to a CPU path."""
    import torch

    import wordpiece_b200

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(wordpiece_b200.WordPieceError) as ei:
        wordpiece_b200.Vocab(["a", "[UNK]"], device=0)
    assert ei.value.status == 4
    v = wordpiece_b200.Vocab(["a", "[UNK]"], device=-1)
    with pytest.raises(wordpiece_b200.WordPieceError) as ei:
        v.encode(b"a")
    assert ei.value.status == 4 and "no CPU path" in str(ei.value)


def test_vocab_builder_matches_oracle_classification():
    from wordpiece_b200 import Vocab, WordPieceError

    rng = random.Random(7)
    for _ in range(400):
        _, vocab = cases.fuzz_case(rng)
        try:
            o = Oracle(vocab)
        except EmptyVocabWord:
            with pytest.raises(WordPieceError) as ei:
                Vocab(vocab, device=-1)
            assert ei.value.status == 2 and str(ei.value) == "Vocab word is empty"
            continue
        v = Vocab(vocab, device=-1)
        assert (v.unk_id, v.max_len, len(v)) == (o.unk_id, o.max_len, len(vocab))
        for i in range(len(vocab)):
            assert (v.token_flags(i) & 7) == o.token_flags(i)


def test_table_image_against_oracle_through_the_model():
    """The byte-domain plan of the kernel (tests/_model.py) over the table image == oracle."""
    from wordpiece_b200 import Vocab

    for text, vocab, expected in cases.REFERENCE_GOLDEN:
        assert model_encode(Vocab(vocab, device=-1), text.encode()) == expected
    for name, text, vocab in cases.QUIRKS:
        assert model_encode(Vocab(vocab, device=-1), text) == Oracle(vocab).encode(text).tolist(), name
    rng = random.Random(31)
    for _ in range(3000):
        text, vocab = cases.fuzz_case(rng)
        try:
            o = Oracle(vocab)
        except EmptyVocabWord:
            continue
        assert model_encode(Vocab(vocab, device=-1), text) == o.encode(text).tolist(), (text, vocab)
    for i in range(60):  # long tokens (> 22 bytes) hang off depth-22 nodes
        s, vocab = cases.random_split_case(rng, rng.randint(40, 600), rng.randint(2, 14), i % 3 != 0)
        v = Vocab(vocab, device=-1)
        assert model_encode(v, s.encode()) == Oracle(vocab).encode(s).tolist()
    text, vocab = textgen.case(3, 20000, long_run_rate=0.05, long_tokens=20)
    v = Vocab(vocab, device=-1)
    assert v.table_info["long_tokens"] >= 20
    assert model_encode(v, text) == Oracle(vocab).encode(text).tolist()


def test_table_image_shape():
    from wordpiece_b200 import Vocab

    v = Vocab(["ab", "abc", "##abc", "b", "[UNK]", "x" * 30, "x" * 40, "x" * 30], device=-1)
    info = v.table_info
    assert info["slots"] >= 2 * info["nodes"] and info["slots"] & (info["slots"] - 1) == 0
    assert info["long_tokens"] == 2  # the duplicate long token is stored once
    assert v.debug_longest_match(b"abcd", 0) == (3, 1)
    assert v.debug_longest_match(b"abcd", 1) == (3, 2)
    assert v.debug_longest_match(b"ab", 0) == (2, 0)
    assert v.debug_longest_match(b"a", 0) == (0, -2)
    assert v.debug_longest_match(b"x" * 50, 0) == (40, 6)
    assert v.debug_longest_match(b"x" * 39, 0) == (30, 7)  # last duplicate wins
    assert v.debug_longest_match(b"x" * 29, 0) == (0, -2)


def test_decode_matches_reference_rules(tmp_path):
    """fast.cpp:165-187."""
    import wordpiece_b200

    vocab = ["[PAD]", "a", "##b", "--", "[UNK]", "中", "##かな"]
    v = wordpiece_b200.Vocab(vocab, device=-1)
    assert v.decode([1, 2, 5, 6, 0, 4]) == [b"a", b"##b", "中".encode(), "##かな".encode(), b"[PAD]", b"[UNK]"]
    assert v.decode([-1, 1, 3, 8, 2]) == [b"a", b"##b"]  # negative, malformed and > size are skipped
    with pytest.raises(wordpiece_b200.WordPieceError) as ei:
        v.decode([7])  # id == size: the reference's .at() throws
    assert ei.value.status == 8
    p = tmp_path / "vocab.txt"
    p.write_bytes(b"\n".join(t.encode() for t in vocab) + b"\n")
    assert wordpiece_b200.decode(str(p), [1, 2]) == [b"a", b"##b"]


def test_vocab_file_reader_semantics(tmp_path):
    """utils.cpp:123-137: getline — '\\r' stays, blank line throws, last line need not end in '\\n'."""
    import wordpiece_b200

    p = tmp_path / "v.txt"
    p.write_bytes(b"a\r\n[UNK]\nb")
    v = wordpiece_b200.Vocab.from_file(str(p), device=-1)
    assert len(v) == 3 and v.unk_id == 1
    assert v.decode([0, 2]) == [b"a\r", b"b"]
    p.write_bytes(b"a\n\nb\n")
    with pytest.raises(wordpiece_b200.WordPieceError) as ei:
        wordpiece_b200.Vocab.from_file(str(p), device=-1)
    assert ei.value.status == 2
    with pytest.raises(wordpiece_b200.WordPieceError) as ei:
        wordpiece_b200.Vocab.from_file(str(tmp_path / "missing.txt"), device=-1)
    assert ei.value.status == 6


def test_synthetic_corpus_is_deterministic_and_shardable():
    from wordpiece_b200 import synth

    g = synth.generator("en")
    whole = g.generate(3 * synth.BLOCK + 12345, seed=4, n_threads=3)
    again = g.generate(3 * synth.BLOCK + 12345, seed=4, n_threads=1)
    assert np.array_equal(whole, again)
    part = g.generate(synth.BLOCK + 12345, seed=4, first_block=2)
    assert np.array_equal(whole[2 * synth.BLOCK:], part)
    assert not np.array_equal(whole[:1000], g.generate(1000, seed=5))
    vocab = g.spec.vocab
    assert len(vocab) == 28996 and len(set(vocab)) == 28996 and vocab[100] == b"[UNK]"
    o = Oracle(vocab)
    ids = o.encode(whole[: 1 << 20])
    ratio = ids.size / (1 << 20)
    assert 0.2 < ratio < 0.35, ratio
    assert 0.002 < float((ids == o.unk_id).mean()) < 0.05


def test_shard_plan_preserves_ids():
    """wp_plan_shards: cuts at safe starts leave the concatenated ids unchanged (fast.cpp:113-115, SURVEY
    8(e)) — on mixed text, on text with invalid bytes, and on space-free CJK text, where the cuts fall at
    punctuation and Han chars."""
    from wordpiece_b200 import global_offsets, plan_shards, shard_ranges

    texts = [textgen.case(seed, 70000, **kw) for seed, kw in
             ((51, {}), (52, dict(invalid_rate=0.02)), (53, dict(long_run_rate=0.05, long_tokens=10)))]
    rng = __import__("random").Random(54)
    _, vocab = texts[0]
    cjk = "".join(rng.choice("中文字漢語日本人大小山川田かなあいうえお。、abc-") for _ in range(40000)).encode()
    texts.append((cjk, vocab))
    texts.append((cjk[:30000] + b"\xe4\xb8" + cjk[30000:33000] + b"\xff\xe5" + cjk[33000:], vocab))
    for ti, (text, vocab) in enumerate(texts):
        o = Oracle(vocab)
        whole = o.encode(text)
        for n_shards in (2, 3, 8, 64):
            cuts = plan_shards(text, n_shards)
            assert cuts[0] == 0 and cuts[-1] == len(text) and cuts == sorted(cuts) and len(cuts) == n_shards + 1
            sizes = [b - a for a, b in shard_ranges(text, n_shards)]
            assert max(sizes) - min(sizes) < 2000, (ti, n_shards, sizes)
            parts = [o.encode(text[a:b]) for a, b in shard_ranges(text, n_shards)]
            offs = global_offsets([p.size for p in parts])
            out = np.empty(sum(p.size for p in parts), np.int32)
            for off, p in zip(offs, parts):
                out[off:off + p.size] = p
            assert np.array_equal(out, whole), (ti, n_shards)
    # a text without any safe cut is one shard plus empty ones; tiny texts give empty shards
    assert plan_shards(b"x" * 1000, 4) == [0, 1000, 1000, 1000, 1000]
    assert plan_shards(b"", 3) == [0, 0, 0, 0]
    assert plan_shards(b"a b", 8)[-1] == 3


def test_pipeline_chunk_plan():
    """Host-buffer pipeline (wp_encode_into on large texts): chunks end right after an ASCII space — the
    reference's serial state is reset there (fast.cpp:89-91,113-115) — cover the text exactly, ramp up from
    chunk/8 at the start and down again at the end, and a stretch without a space makes the plan fail (the
    caller then encodes in one shot)."""
    import random

    from wordpiece_b200._capi import debug_plan_chunks

    rng = random.Random(4)
    words = ["".join(rng.choice("abcdefgh") for _ in range(rng.randint(1, 12))) for _ in range(400)]
    text = " ".join(rng.choice(words) for _ in range(200_000)).encode()
    for chunk in (4096, 30_000, 150_000):
        cuts = debug_plan_chunks(text, chunk)
        assert cuts[0] == 0 and cuts[-1] == len(text) and cuts == sorted(set(cuts))
        sizes = [b - a for a, b in zip(cuts, cuts[1:])]
        assert max(sizes) <= chunk
        for c in cuts[1:-1]:
            assert text[c - 1:c] == b" "
        small = chunk // 8
        # ramp up: about chunk/8, /4, /2, then full chunks; and the mirror image at the end
        assert sizes[0] <= small < sizes[1] <= 2 * small < sizes[2] <= 4 * small < sizes[3]
        assert sizes[-1] <= small + 1 and sizes[-2] <= 2 * small + 16
        assert sum(1 for s in sizes if s > chunk // 2) >= len(sizes) - 10
    # a text shorter than the smallest chunk is one piece
    assert debug_plan_chunks(text[:300], 4096) == [0, 300]
    # no space to cut at within half a chunk: no plan
    glued = text[:50_000] + b"x" * 9000 + text[50_000:]
    assert debug_plan_chunks(glued, 4096) == []


def test_batch_packing_rule_is_exact():
    """wp_encode_batch packs its texts into one buffer, each followed by one space, and encodes the buffer once.
    The rule it rests on, checked here with the oracle alone (no device): the ids of the packed buffer are the
    ids of the texts one after the other — also when a text ends inside a UTF-8 sequence, in an open word or in
    a Han char (fast.cpp:89-91: a space resets the matcher; utf8.cpp:130-147: a cut sequence stays invalid)."""
    import random

    import textgen

    hand = [b"ab", b"", b"a", b"b c", b"\xe4\xb8", b"\xad abc", b"ab\xc3", b"\xa9", b"\xe4\xb8\xad", b"a",
            b"\xe6\x96\x87", b"", b"abc.", b".", b"   ", b"\xff", b"abc\xe2\x96", b"\x81x", "中a".encode(), b"xyz"]
    hand_vocab = ["[UNK]", "a", "b", "ab", "##b", "##c", "abc", "中", "中a", "##a", "é", "##é", ".", "文"]
    jobs = [(hand_vocab, hand)]
    for seed in (1, 2, 3):
        rng = random.Random(seed)
        vocab = textgen.mixed_vocab(rng, 300, long_tokens=3)
        texts = []
        for _ in range(300):
            n = rng.randint(0, 300)
            t = textgen.mixed_text(rng, n, vocab, invalid_rate=0.02, long_run_rate=0.01) if n else b""
            if t and rng.random() < 0.3:
                t = t[: rng.randint(0, len(t))]
            texts.append(t)
        jobs.append((vocab, texts))
    for vocab, texts in jobs:
        o = Oracle(vocab)
        whole = o.encode(b"".join(t + b" " for t in texts))
        parts = np.concatenate([o.encode(t) for t in texts])
        assert np.array_equal(whole, parts)


def test_staging_copies_are_exact():
    """The copies that stage caller memory into pinned buffers (batch packer, pooled copy) with ordinary and with
    streaming stores: byte-exact for every alignment and size, including texts that share a cache line, empty
    texts, pieces longer than the writer's gather buffer, and shares cut across the pool's threads."""
    import random

    from wordpiece_b200._capi import debug_stage

    rng = random.Random(5)
    blob = bytes(rng.randrange(256) for _ in range(70000))

    def piece(n):
        a = rng.randrange(0, len(blob) - n + 1) if n <= len(blob) else 0
        return (blob * (n // len(blob) + 2))[a:a + n]

    shapes = [
        [],
        [b""],
        [b"", b"", b""],
        [b"a"],
        [piece(n) for n in (1, 2, 62, 63, 64, 65, 127, 128, 129, 0, 255, 256, 257)],
        [piece(rng.randrange(0, 40)) for _ in range(3000)],               # many texts per cache line
        [piece(rng.randrange(0, 9000)) for _ in range(300)],              # around the gather buffer's size
        [piece(8192), piece(8191), piece(8193), piece(16384), piece(100000), b"x", piece(70001)],
        [piece(rng.randrange(3000, 5000)) for _ in range(700)],           # > 1 MiB: packed by the whole pool
        [piece(1), piece(3 << 20), piece(5)],                             # one long text across the shares
    ]
    for texts in shapes:
        want = b"".join(t + b" " for t in texts)
        for mode in (0, 1):
            assert debug_stage(texts, mode) == want, (mode, len(texts))
    for n in (0, 1, 63, 64, 255, 256, 257, 4096, 1 << 20, (1 << 20) + 1, (3 << 20) + 77):
        src = piece(n)
        for mode in (2, 3):
            assert debug_stage([src], mode) == src, (mode, n)
