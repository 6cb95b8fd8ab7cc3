"""GPU parity of the batch entry point (wp_encode_batch): every text of a batch must get exactly the ids the
oracle gives that text ALONE — one packed copy and one pass of the kernels must not leak anything across a text
border (an unfinished UTF-8 sequence, an open word, a Han char waiting for its run)."""
from __future__ import annotations

import random

import numpy as np
import pytest

import cases
import textgen
from _oracle import Oracle

pytestmark = pytest.mark.gpu


def _check_batch(v, oracle, texts, tag):
    ids, offs = v.encode_batch(texts)
    assert offs.size == len(texts) + 1 and int(offs[0]) == 0 and int(offs[-1]) == ids.size, tag
    for i, t in enumerate(texts):
        exp = oracle.encode(t if isinstance(t, bytes) else t.encode("utf-8"))
        got = ids[int(offs[i]):int(offs[i + 1])]
        assert np.array_equal(exp, got), (tag, i, t[:60], exp[:12].tolist(), got[:12].tolist())


def test_batch_hand_made_borders(gpu_device):
    """Text ends that try to reach into the next text: truncated sequences, open words, lone Han chars."""
    from wordpiece_b200 import Vocab

    vocab = ["[UNK]", "a", "b", "ab", "##b", "##c", "abc", "中", "中a", "##a", "é", "##é", ".", "文"]
    texts = [b"ab", b"", b"a", b"b c", b"\xe4\xb8", b"\xad abc", b"ab\xc3", b"\xa9", b"\xe4\xb8\xad", b"a", b"\xe4\xb8\xad",
             b"\xe6\x96\x87", b"", b"", b"abc.", b".", b" ", b"   ", b"ab ab ab", b"\xff", b"abc\xe2\x96", b"\x81x",
             "中a".encode(), "中".encode(), b"a", b"xyz", b"b"]
    v = Vocab(vocab, device=gpu_device)
    o = Oracle(vocab)
    _check_batch(v, o, texts, "hand-made")
    _check_batch(v, o, [b""], "one empty text")
    _check_batch(v, o, [b"", b"", b""], "only empty texts")
    _check_batch(v, o, [b"ab"], "one text")
    ids, offs = v.encode_batch([])
    assert ids.size == 0 and offs.tolist() == [0]
    v.close()


def test_batch_reference_golden_vectors(gpu_device):
    """The reference's own known-answer texts (tests/tests.cpp:137-217), grouped by vocabulary, as batches."""
    from wordpiece_b200 import Vocab

    by_vocab = {}
    for text, vocab, expected in cases.REFERENCE_GOLDEN:
        by_vocab.setdefault(tuple(vocab), []).append((text, expected))
    for vocab, items in by_vocab.items():
        v = Vocab(list(vocab), device=gpu_device)
        ids, offs = v.encode_batch([t for t, _ in items])
        for i, (t, expected) in enumerate(items):
            assert ids[int(offs[i]):int(offs[i + 1])].tolist() == expected, (t, expected)
        v.close()


@pytest.mark.parametrize("seed,n_texts,max_len,invalid", [(1, 300, 200, 0.0), (2, 2000, 64, 0.01), (3, 64, 20000, 0.003),
                                                          (4, 5000, 9, 0.02), (5, 40, 70000, 0.0)])
def test_batch_random_texts(gpu_device, seed, n_texts, max_len, invalid):
    """Hostile random texts of very different lengths (many per tile; several tiles per text; dirty tiles)."""
    from wordpiece_b200 import Vocab

    rng = random.Random(seed)
    vocab = textgen.mixed_vocab(rng, 300, long_tokens=3)
    texts = []
    for _ in range(n_texts):
        n = rng.randint(0, max_len)
        t = textgen.mixed_text(rng, n, vocab, invalid_rate=invalid, long_run_rate=0.01) if n else b""
        if t and rng.random() < 0.3:
            t = t[: rng.randint(0, len(t))]  # cut anywhere, also inside a multi-byte sequence
        texts.append(t)
    v = Vocab(vocab, device=gpu_device)
    _check_batch(v, Oracle(vocab), texts, f"random seed {seed}")
    st = v.stats()
    assert st.n_ids > 0
    v.close()


def test_batch_large_goes_through_several_ranges(gpu_device, monkeypatch):
    """A batch that spans several kernel ranges (range size forced down) and uses the word memo."""
    from wordpiece_b200 import Vocab

    monkeypatch.setenv("WORDPIECE_B200_RANGE_BYTES", str(64 * 1024))
    monkeypatch.setenv("WORDPIECE_B200_MEMO", "1")
    rng = random.Random(11)
    vocab = textgen.mixed_vocab(rng, 400)
    texts = [textgen.mixed_text(rng, rng.randint(1, 3000), vocab, invalid_rate=0.002) for _ in range(600)]
    v = Vocab(vocab, device=gpu_device)
    _check_batch(v, Oracle(vocab), texts, "several ranges")
    v.close()


def test_batch_capacity_error_reports_the_count(gpu_device):
    from wordpiece_b200 import Vocab, WordPieceError

    v = Vocab(["a", "[UNK]"], device=gpu_device)
    out = np.zeros(2, np.int32)
    with pytest.raises(WordPieceError):
        v.encode_batch([b"a a a", b"a a"], out=out)
    ids, offs = v.encode_batch([b"a a a", b"a a"])
    assert ids.tolist() == [0] * 5 and offs.tolist() == [0, 3, 5]
    v.close()


@pytest.mark.parametrize("part", [4096, 50_000])
def test_batch_pipeline_of_parts(gpu_device, monkeypatch, part):
    """A batch cut into many parts (part size forced down): packed, copied and encoded in a pipeline over three
    buffer sets; offsets of later parts are rebased on the ids of the earlier ones."""
    from wordpiece_b200 import Vocab

    monkeypatch.setenv("WORDPIECE_B200_BATCH_PART", str(part))
    rng = random.Random(part)
    vocab = textgen.mixed_vocab(rng, 300, long_tokens=2)
    texts = []
    for _ in range(700):
        n = rng.choice([0, 1, 5, 40, 300, 2000, 9000])
        texts.append(textgen.mixed_text(rng, rng.randint(0, n), vocab, invalid_rate=0.005, long_run_rate=0.01) if n else b"")
    v = Vocab(vocab, device=gpu_device)
    o = Oracle(vocab)
    _check_batch(v, o, texts, f"parts of {part}")
    _check_batch(v, o, texts[:5], "then a small batch on the same handle")
    v.close()


def test_batch_repeat_after_void_part_switches_k1_mode(gpu_device, monkeypatch):
    """A pipelined batch whose part 0 overflows the default id spill of its first range (a space-free word of
    40 000 ids) while part 1, never finished before the whole batch is repeated as one part, holds a tile of
    4 096 segments: the repeat trips the dense-tile flag of the regular K1 and must itself be repeated with the
    full-capacity K1, as a single call would be."""
    from wordpiece_b200 import Vocab

    monkeypatch.setenv("WORDPIECE_B200_RANGE_BYTES", "4096")
    monkeypatch.setenv("WORDPIECE_B200_MEMO", "0")
    monkeypatch.setenv("WORDPIECE_B200_BATCH_PART", "4096")
    vocab = ["[UNK]", "a", "##a", "!"]
    v = Vocab(vocab, device=gpu_device)
    _check_batch(v, Oracle(vocab), [b"a" * 40000, b"!" * 8192], "void part, then a dense tile")
    v.close()
