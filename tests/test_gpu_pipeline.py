"""GPU parity of the host pipeline (wp_encode_into on large texts, wp_encode_batch on large batches): the rare
paths of the slots — a void part that makes the whole call run again, ids that outgrow the pinned id staging,
slots whose buffers grow while the pipeline runs — must return exactly the oracle's ids."""
from __future__ import annotations

import random

import numpy as np
import pytest

import textgen
from _oracle import Oracle

pytestmark = pytest.mark.gpu

_WORDS = [b"the", b"cat", b"sat", b"on", b"a", b"mat", b"cats", b"mats"]
_VOCAB = ["[UNK]", "the", "cat", "sat", "on", "a", "##a", "mat", "##s", ".", ",", "!", "?", "(", ")"]


def _filler(rng, n):
    out = bytearray()
    while len(out) < n:
        out += rng.choice(_WORDS) + rng.choice([b" ", b" ", b" ", b". "])
    return bytes(out[:n]) + b" "


def _check_into(v, text, exp, out, tag, repeated=False):
    out[:] = -9
    n = v.encode_into(text, out)
    assert n == exp.size and np.array_equal(out[:n], exp) and (out[n:] == -9).all(), tag
    assert v.stats().n_ids == exp.size and v.stats().n_bytes == len(text), tag
    if repeated:  # the ids came from one call over the whole text, not from chunks (each rounds up to whole tiles)
        import wordpiece_b200

        tile = wordpiece_b200.tile_bytes()
        assert v.stats().n_tiles == (len(text) + tile - 1) // tile, tag


def _void_chunk_text(seed, tile, dense):
    """~620 KB of text with a space-free word of 12 tiles in the middle: its ids outgrow the default id spill of a
    one-tile range (range + tile = 2 tiles of ids), so the chunk that holds it is void.  `dense`: a later chunk
    also holds a tile of punctuation, more segments than the regular K1's lists hold."""
    rng = random.Random(seed)
    text = _filler(rng, 300_000) + b"a" * (12 * tile) + b" " + _filler(rng, 150_000)
    if dense:
        text += b".,!?()" * (tile // 3) + b" "
    return text + _filler(rng, 120_000)


def test_into_void_chunk_repeats_whole_call(gpu_device, monkeypatch):
    """A middle chunk of a pipelined encode_into overflows the id spill: the call is repeated in one piece and its
    ids and statistics are exact; a second call on the same handle as well."""
    import wordpiece_b200
    from wordpiece_b200 import Vocab
    from wordpiece_b200._capi import debug_plan_chunks

    tile = wordpiece_b200.tile_bytes()
    monkeypatch.setenv("WORDPIECE_B200_RANGE_BYTES", str(tile))
    monkeypatch.setenv("WORDPIECE_B200_PIPE_CHUNK", "150000")
    text = _void_chunk_text(11, tile, dense=False)
    cuts = debug_plan_chunks(text, 150_000)
    assert len(cuts) > 3, "the text must be pipelined"
    exp = Oracle(_VOCAB).encode(text)
    v = Vocab(_VOCAB, device=gpu_device)
    out = np.full(exp.size + 7, -9, np.int32)
    _check_into(v, text, exp, out, "first call", repeated=True)
    _check_into(v, text, exp, out, "second call", repeated=True)
    v.close()


@pytest.mark.parametrize("pinned_out", [False, True])
def test_into_void_chunk_then_dense_tile(gpu_device, monkeypatch, pinned_out):
    """The same with a later chunk holding a dense tile, on a fresh handle: the repeat of the whole call trips the
    dense-tile flag and is repeated once more with the full-capacity K1."""
    import wordpiece_b200
    from wordpiece_b200 import Vocab

    tile = wordpiece_b200.tile_bytes()
    monkeypatch.setenv("WORDPIECE_B200_RANGE_BYTES", str(tile))
    monkeypatch.setenv("WORDPIECE_B200_PIPE_CHUNK", "150000")
    text = _void_chunk_text(12, tile, dense=True)
    exp = Oracle(_VOCAB).encode(text)
    v = Vocab(_VOCAB, device=gpu_device)
    if pinned_out:
        import torch

        pin = torch.full((exp.size + 7,), -9, dtype=torch.int32).pin_memory()
        out = pin.numpy()
    else:
        out = np.full(exp.size + 7, -9, np.int32)
    _check_into(v, text, exp, out, f"pinned output {pinned_out}", repeated=True)
    _check_into(v, text, exp, out, f"pinned output {pinned_out}, again", repeated=True)
    v.close()


def test_into_more_ids_than_staging_slot(gpu_device, monkeypatch):
    """Pageable output and chunks with more ids than a pinned staging slot holds (half an id per chunk byte): one
    id per byte, copied out piece by piece."""
    import wordpiece_b200
    from wordpiece_b200 import Vocab

    vocab = ["[UNK]", "a", "##b", "."]
    monkeypatch.setenv("WORDPIECE_B200_PIPE_CHUNK", "30000")
    text = b"ab." * 100_000  # three ids and two segments per three bytes, a safe cut at every "."
    exp = Oracle(vocab).encode(text)
    assert exp.size == len(text)
    v = Vocab(vocab, device=gpu_device)
    out = np.full(exp.size + 7, -9, np.int32)
    _check_into(v, text, exp, out, "first call")
    _check_into(v, text, exp, out, "second call")
    tile = wordpiece_b200.tile_bytes()
    assert v.stats().n_tiles > (len(text) + tile - 1) // tile, "pipelined in chunks, not repeated"
    v.close()


def test_batch_parts_grow_while_pipelined(gpu_device, monkeypatch):
    """A pipelined batch whose parts grow from a few bytes to tens of KiB: every slot grows while the slots
    before and after it are in flight."""
    from wordpiece_b200 import Vocab

    monkeypatch.setenv("WORDPIECE_B200_BATCH_PART", "4096")
    rng = random.Random(21)
    vocab = textgen.mixed_vocab(rng, 300, long_tokens=2)
    texts = [textgen.mixed_text(rng, int(6 * 1.4 ** i), vocab, invalid_rate=0.003, long_run_rate=0.01) for i in range(30)]
    assert sum(len(t) for t in texts) > 100_000
    o = Oracle(vocab)
    exp = [o.encode(t) for t in texts]
    v = Vocab(vocab, device=gpu_device)
    for rep in range(2):
        ids, offs = v.encode_batch(texts)
        assert offs.size == len(texts) + 1 and int(offs[-1]) == ids.size, rep
        for i, e in enumerate(exp):
            assert np.array_equal(ids[int(offs[i]):int(offs[i + 1])], e), (rep, i)
        assert v.stats().n_ids == ids.size, rep
    v.close()
