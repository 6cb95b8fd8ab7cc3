"""The device batch entry point (wp_encode_batch_device[_async]): a string column in GPU memory (chars + Arrow
offsets) in, per-text ids and id offsets in GPU memory out.  Every text must get exactly the ids the oracle gives
that text alone, and the same ids and offsets as wp_encode_batch gives the same texts from host memory.  The column
is packed on the device, so its layout (where the texts lie in the buffer, its alignment) must not matter, and a
malformed column must fail cleanly instead of reading out of range."""
from __future__ import annotations

import ctypes as C
import random

import numpy as np
import pytest

import cases
import textgen
from _oracle import Oracle

HAND_MADE_VOCAB = ["[UNK]", "a", "b", "ab", "##b", "##c", "abc", "中", "中a", "##a", "é", "##é", ".", "文"]
HAND_MADE_TEXTS = [b"ab", b"", b"a", b"b c", b"\xe4\xb8", b"\xad abc", b"ab\xc3", b"\xa9", b"\xe4\xb8\xad", b"a",
                   b"\xe4\xb8\xad", b"\xe6\x96\x87", b"", b"", b"abc.", b".", b" ", b"   ", b"ab ab ab", b"\xff",
                   b"abc\xe2\x96", b"\x81x", "中a".encode(), "中".encode(), b"a", b"xyz", b"b"]
UINT64_MAX_AS_INT64 = -1


def _column(texts, device, lead=0, trail=0, odd=False):
    """(d_chars, d_offsets) of `texts`, with `lead` unused bytes before the first text and `trail` after the last;
    `odd`: d_chars starts at an odd address (a slice of a larger tensor)."""
    import torch

    blob = b"\x00" * (1 if odd else 0) + b"x" * lead + b"".join(texts) + b"y" * trail
    base = torch.frombuffer(bytearray(blob), dtype=torch.uint8).cuda(device) if blob else \
        torch.empty(0, dtype=torch.uint8, device=f"cuda:{device}")
    d_chars = base[1:] if odd else base
    offs = np.zeros(len(texts) + 1, np.int64)
    offs[0] = lead
    offs[1:] = lead + np.cumsum([len(t) for t in texts], dtype=np.int64)
    return d_chars, torch.from_numpy(offs).cuda(device)


def _check(v, oracle, texts, tag, **layout):
    import torch

    d_chars, d_offsets = _column(texts, v.device, **layout)
    d_ids, d_id_offsets, n = v.encode_batch_device(d_chars, d_offsets)
    ids = d_ids[:n].cpu().numpy()
    offs = d_id_offsets.cpu().numpy()
    assert offs.size == len(texts) + 1 and offs[0] == 0 and offs[-1] == n, tag
    for i, t in enumerate(texts):
        exp = oracle.encode(t)
        got = ids[offs[i]:offs[i + 1]]
        assert np.array_equal(exp, got), (tag, i, t[:60], exp[:12].tolist(), got[:12].tolist())
    st = v.stats()  # (the packed column: n_chars + one separator per text)
    assert st.n_ids == n and st.n_bytes == d_chars.numel() + len(texts), (tag, st)
    if texts:
        h_ids, h_offs = v.encode_batch(texts)
        assert np.array_equal(h_ids, ids) and np.array_equal(h_offs.astype(np.int64), offs), (tag, "differs from encode_batch")
    torch.cuda.synchronize()
    return ids, offs


def _random_texts(seed, n_texts, max_len, invalid):
    rng = random.Random(seed)
    vocab = textgen.mixed_vocab(rng, 300, long_tokens=3)
    texts = []
    for _ in range(n_texts):
        n = rng.randint(0, max_len)
        t = textgen.mixed_text(rng, n, vocab, invalid_rate=invalid, long_run_rate=0.01) if n else b""
        if t and rng.random() < 0.3:
            t = t[: rng.randint(0, len(t))]
        texts.append(t)
    return vocab, texts


# ---- parity ---------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_batch_device_hand_made_borders(gpu_device):
    from wordpiece_b200 import Vocab

    v = Vocab(HAND_MADE_VOCAB, device=gpu_device)
    o = Oracle(HAND_MADE_VOCAB)
    _check(v, o, HAND_MADE_TEXTS, "hand-made")
    _check(v, o, HAND_MADE_TEXTS, "hand-made, odd address, unused bytes around", lead=7, trail=5, odd=True)
    v.close()


@pytest.mark.gpu
def test_batch_device_reference_golden_vectors(gpu_device):
    from wordpiece_b200 import Vocab

    by_vocab = {}
    for text, vocab, expected in cases.REFERENCE_GOLDEN:
        by_vocab.setdefault(tuple(vocab), []).append((text, expected))
    for vocab, items in by_vocab.items():
        v = Vocab(list(vocab), device=gpu_device)
        texts = [t if isinstance(t, bytes) else t.encode("utf-8") for t, _ in items]
        d_chars, d_offsets = _column(texts, gpu_device, lead=3)
        d_ids, d_id_offsets, n = v.encode_batch_device(d_chars, d_offsets)
        ids, offs = d_ids[:n].cpu().tolist(), d_id_offsets.cpu().tolist()
        for i, (t, expected) in enumerate(items):
            assert ids[offs[i]:offs[i + 1]] == expected, (t, expected)
        v.close()


@pytest.mark.gpu
@pytest.mark.parametrize("seed,n_texts,max_len,invalid", [(1, 300, 200, 0.0), (2, 2000, 64, 0.01), (3, 64, 20000, 0.003),
                                                          (4, 5000, 9, 0.02), (5, 40, 70000, 0.0)])
def test_batch_device_random_texts(gpu_device, seed, n_texts, max_len, invalid):
    from wordpiece_b200 import Vocab

    vocab, texts = _random_texts(seed, n_texts, max_len, invalid)
    v = Vocab(vocab, device=gpu_device)
    _check(v, Oracle(vocab), texts, f"random seed {seed}", lead=seed * 3, trail=seed, odd=seed % 2 == 1)
    v.close()


# ---- layout ---------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_batch_device_layouts(gpu_device):
    """Offsets that do not start at 0, unused bytes on both sides, an odd address; all texts empty; one text."""
    from wordpiece_b200 import Vocab

    rng = random.Random(21)
    vocab = textgen.mixed_vocab(rng, 300, long_tokens=2)
    texts = [textgen.mixed_text(rng, rng.randint(0, 900), vocab, invalid_rate=0.005) for _ in range(200)]
    v = Vocab(vocab, device=gpu_device)
    o = Oracle(vocab)
    ids0, offs0 = _check(v, o, texts, "plain")
    for lead, trail, odd in [(1, 0, False), (4097, 13, False), (0, 0, True), (5, 4099, True), (15, 1, True)]:
        ids, offs = _check(v, o, texts, f"lead {lead} trail {trail} odd {odd}", lead=lead, trail=trail, odd=odd)
        assert np.array_equal(ids, ids0) and np.array_equal(offs, offs0)
    _check(v, o, [b""] * 5000, "all empty")
    _check(v, o, [b""], "one empty text", lead=3, trail=2)
    _check(v, o, [texts[3]], "one text", lead=2, odd=True)
    v.close()


@pytest.mark.gpu
def test_batch_device_no_texts(gpu_device):
    import torch
    from wordpiece_b200 import Vocab

    v = Vocab(HAND_MADE_VOCAB, device=gpu_device)
    d_chars = torch.zeros(10, dtype=torch.uint8, device=f"cuda:{gpu_device}")
    d_offsets = torch.tensor([4], dtype=torch.int64, device=f"cuda:{gpu_device}")
    d_id_offsets = torch.full((1,), 77, dtype=torch.int64, device=f"cuda:{gpu_device}")
    _, offs, n = v.encode_batch_device(d_chars, d_offsets, d_id_offsets=d_id_offsets)
    assert n == 0 and offs.tolist() == [0] and v.stats().kernel_launches == 0
    d_id_offsets.fill_(77)
    v.encode_batch_device_async(d_chars, d_offsets, torch.empty(1, dtype=torch.int32, device=d_chars.device), d_id_offsets)
    torch.cuda.synchronize()
    assert d_id_offsets.tolist() == [0]
    v.close()


@pytest.mark.gpu
def test_batch_device_large_text_among_tiny_ones(gpu_device):
    """A text of several tiles next to thousands of 1-9 byte texts (dozens of texts per tile of the packed column)."""
    from wordpiece_b200 import Vocab

    rng = random.Random(8)
    vocab = textgen.mixed_vocab(rng, 300, long_tokens=2)
    tiny = [textgen.mixed_text(rng, rng.randint(1, 9), vocab, invalid_rate=0.01)[:9] for _ in range(6000)]
    big = textgen.mixed_text(rng, 5 * 4096 + 77, vocab, invalid_rate=0.002, long_run_rate=0.01)
    texts = tiny[:3000] + [big] + tiny[3000:]
    v = Vocab(vocab, device=gpu_device)
    _check(v, Oracle(vocab), texts, "big among tiny", lead=9, trail=33, odd=True)
    v.close()


# ---- ranges, void calls, capacity ----------------------------------------------------------------------------

@pytest.mark.gpu
def test_batch_device_several_ranges(gpu_device, monkeypatch):
    """Small ranges: texts start in every range and one text spans several, so K5 takes each range's texts from
    the tile index on the device."""
    from wordpiece_b200 import Vocab

    monkeypatch.setenv("WORDPIECE_B200_RANGE_BYTES", str(64 * 1024))
    monkeypatch.setenv("WORDPIECE_B200_MEMO", "1")
    rng = random.Random(12)
    vocab = textgen.mixed_vocab(rng, 400)
    texts = [textgen.mixed_text(rng, rng.randint(1, 3000), vocab, invalid_rate=0.002) for _ in range(300)]
    texts.insert(150, textgen.mixed_text(rng, 200_000, vocab, invalid_rate=0.001))
    v = Vocab(vocab, device=gpu_device)
    _check(v, Oracle(vocab), texts, "several ranges", lead=100, trail=3, odd=True)
    assert v.stats().n_tiles > 3 * 16
    v.close()


@pytest.mark.gpu
def test_batch_device_repeat_after_void_call(gpu_device, monkeypatch):
    """A 40 000-id word overflows the first id spill and a tile of 4 096 segments trips the dense-tile flag: the sync
    call repeats until its ids are exact; the async call on a fresh handle reports the void call in its last offset."""
    import torch
    from wordpiece_b200 import Vocab

    monkeypatch.setenv("WORDPIECE_B200_RANGE_BYTES", "4096")
    monkeypatch.setenv("WORDPIECE_B200_MEMO", "0")
    vocab = ["[UNK]", "a", "##a", "!"]
    texts = [b"a" * 40000, b"!" * 8192]
    v = Vocab(vocab, device=gpu_device)
    _check(v, Oracle(vocab), texts, "void call, then a dense tile")
    v.close()
    v = Vocab(vocab, device=gpu_device)
    d_chars, d_offsets = _column(texts, gpu_device)
    d_ids = torch.empty(d_chars.numel(), dtype=torch.int32, device=d_chars.device)
    d_id_offsets = torch.zeros(3, dtype=torch.int64, device=d_chars.device)
    v.encode_batch_device_async(d_chars, d_offsets, d_ids, d_id_offsets)
    torch.cuda.synchronize()
    assert int(d_id_offsets[-1]) == UINT64_MAX_AS_INT64
    v.close()


@pytest.mark.gpu
def test_batch_device_capacity_error_reports_the_count(gpu_device):
    import torch
    from wordpiece_b200 import Vocab, WordPieceError
    from wordpiece_b200._capi import WP_ERR_CAPACITY

    v = Vocab(["a", "[UNK]"], device=gpu_device)
    d_chars, d_offsets = _column([b"a a a", b"a a", b"", b"aa"], gpu_device, lead=2)
    d_ids = torch.empty(2, dtype=torch.int32, device=d_chars.device)
    d_id_offsets = torch.zeros(5, dtype=torch.int64, device=d_chars.device)
    cnt = C.c_size_t()
    st = v._L.wp_encode_batch_device(v._h, d_chars.data_ptr(), d_chars.numel(), d_offsets.data_ptr(), 4, d_ids.data_ptr(),
                                     2, d_id_offsets.data_ptr(), C.byref(cnt), None)
    assert st == WP_ERR_CAPACITY and cnt.value == 6
    assert d_id_offsets.tolist() == [0, 3, 5, 5, 6]
    with pytest.raises(WordPieceError):
        v.encode_batch_device(d_chars, d_offsets, d_ids=d_ids)
    d_ids, offs, n = v.encode_batch_device(d_chars, d_offsets)
    assert n == 6 and d_ids[:n].tolist() == [0, 0, 0, 0, 0, 1] and offs.tolist() == [0, 3, 5, 5, 6]
    v.close()


# ---- malformed columns --------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("offsets", [[0, 5, 3, 8], [0, 3, 11], [9, 2], [0, 4, 4, 1 << 40]])
def test_batch_device_malformed_column(gpu_device, offsets):
    """Offsets that decrease or pass n_chars: the sync call fails with WP_ERR_INVALID_ARG, the async call leaves
    UINT64_MAX in the last offset, and neither reads out of range; the next valid call is exact."""
    import torch
    from wordpiece_b200 import Vocab, WordPieceError
    from wordpiece_b200._capi import WP_ERR_INVALID_ARG

    v = Vocab(HAND_MADE_VOCAB, device=gpu_device)
    o = Oracle(HAND_MADE_VOCAB)
    dev = f"cuda:{gpu_device}"
    d_chars = torch.frombuffer(bytearray(b"ab abc ab a"[:10]), dtype=torch.uint8).to(dev)
    d_offsets = torch.tensor(offsets, dtype=torch.int64, device=dev)
    with pytest.raises(WordPieceError) as e:
        v.encode_batch_device(d_chars, d_offsets)
    assert e.value.status == WP_ERR_INVALID_ARG
    _check(v, o, HAND_MADE_TEXTS, "valid call after a malformed one (sync)")
    d_ids = torch.empty(16, dtype=torch.int32, device=dev)
    d_id_offsets = torch.zeros(len(offsets), dtype=torch.int64, device=dev)
    v.encode_batch_device_async(d_chars, d_offsets, d_ids, d_id_offsets)
    torch.cuda.synchronize()
    assert int(d_id_offsets[-1]) == UINT64_MAX_AS_INT64
    _check(v, o, HAND_MADE_TEXTS, "valid call after a malformed one (async)", lead=1)
    v.close()


# ---- streams --------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_batch_device_async_on_the_producing_stream(gpu_device):
    """The column is produced by torch ops on a side stream and the async call is enqueued on that stream."""
    import torch
    from wordpiece_b200 import Vocab

    vocab, texts = _random_texts(31, 400, 600, 0.005)
    v = Vocab(vocab, device=gpu_device)
    o = Oracle(vocab)
    dev = torch.device(f"cuda:{gpu_device}")
    blob = b"".join(texts)
    h_chars = torch.frombuffer(bytearray(blob), dtype=torch.uint8).pin_memory()
    lens = torch.tensor([len(t) for t in texts], dtype=torch.int64)
    s = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(s):
        d_chars = h_chars.to(dev, non_blocking=True).clone()
        d_offsets = torch.zeros(len(texts) + 1, dtype=torch.int64, device=dev)
        d_offsets[1:] = torch.cumsum(lens.to(dev, non_blocking=True), 0)
        d_ids = torch.empty(len(blob), dtype=torch.int32, device=dev)
        d_id_offsets = torch.empty(len(texts) + 1, dtype=torch.int64, device=dev)
        v.encode_batch_device_async(d_chars, d_offsets, d_ids, d_id_offsets, stream=s.cuda_stream)
    s.synchronize()
    offs = d_id_offsets.cpu().numpy()
    ids = d_ids[: int(offs[-1])].cpu().numpy()
    for i, t in enumerate(texts):
        assert np.array_equal(o.encode(t), ids[offs[i]:offs[i + 1]]), i
    v.close()


@pytest.mark.gpu
def test_batch_device_two_async_calls_on_two_streams(gpu_device):
    """Two async calls on one handle, on different streams, with different columns: the library orders them, and
    each gives exact results."""
    import torch
    from wordpiece_b200 import Vocab

    vocab, texts_a = _random_texts(41, 3000, 300, 0.005)
    _, texts_b = _random_texts(42, 50, 30000, 0.002)
    v = Vocab(vocab, device=gpu_device)
    o = Oracle(vocab)
    dev = torch.device(f"cuda:{gpu_device}")
    out = []
    streams = [torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)]
    for texts, s, lead in [(texts_a, streams[0], 5), (texts_b, streams[1], 0)]:
        d_chars, d_offsets = _column(texts, gpu_device, lead=lead, odd=lead > 0)
        torch.cuda.synchronize()
        d_ids = torch.empty(max(d_chars.numel(), 1), dtype=torch.int32, device=dev)
        d_id_offsets = torch.empty(len(texts) + 1, dtype=torch.int64, device=dev)
        v.encode_batch_device_async(d_chars, d_offsets, d_ids, d_id_offsets, stream=s.cuda_stream)
        out.append((texts, d_chars, d_ids, d_id_offsets))
    torch.cuda.synchronize()
    for texts, _, d_ids, d_id_offsets in out:
        offs = d_id_offsets.cpu().numpy()
        ids = d_ids[: int(offs[-1])].cpu().numpy()
        for i, t in enumerate(texts):
            assert np.array_equal(o.encode(t), ids[offs[i]:offs[i + 1]]), i
    v.close()


# ---- host only (no GPU) ---------------------------------------------------------------------------------------

def test_batch_device_host_only_handle_and_null_arguments():
    from wordpiece_b200 import Vocab
    from wordpiece_b200._capi import WP_ERR_INVALID_ARG, WP_ERR_NO_DEVICE

    v = Vocab(HAND_MADE_VOCAB, device=-1)
    L, h = v._L, v._h
    fake = 0x1000  # never dereferenced: the handle fails before any device work
    cnt = C.c_size_t(5)
    assert L.wp_encode_batch_device(h, fake, 8, fake, 2, fake, 8, fake, C.byref(cnt), None) == WP_ERR_NO_DEVICE
    assert cnt.value == 0
    assert L.wp_encode_batch_device_async(h, fake, 8, fake, 2, fake, 8, fake, None) == WP_ERR_NO_DEVICE
    assert b"host-only" in L.wp_last_error()
    for args in [(None, fake, 8, fake, 2, fake, 8, fake), (h, None, 8, fake, 2, fake, 8, fake),
                 (h, fake, 8, None, 2, fake, 8, fake), (h, fake, 8, fake, 2, None, 8, fake),
                 (h, fake, 8, fake, 2, fake, 8, None)]:
        assert L.wp_encode_batch_device(*args, C.byref(cnt), None) == WP_ERR_INVALID_ARG, args
        assert L.wp_encode_batch_device_async(*args, None) == WP_ERR_INVALID_ARG, args
    assert L.wp_encode_batch_device(h, fake, 8, fake, 2, fake, 8, fake, None, None) == WP_ERR_INVALID_ARG
    v.close()


def test_batch_device_symbols_are_exported():
    from wordpiece_b200._capi import EXPORTED_SYMBOLS, load_library

    L = load_library()
    for name in ("wp_encode_batch_device", "wp_encode_batch_device_async"):
        assert name in EXPORTED_SYMBOLS and hasattr(L, name)
