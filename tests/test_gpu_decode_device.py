"""Device decode (wp_decode_device[_async]): token ids in GPU memory to one token string per id in GPU memory (chars +
n + 1 Arrow offsets).  Every non-empty entry must be what the host wp_decode gives that id, the empty entries exactly
the ids it skips, and the offsets exact at every block border, across many stage windows and past 4 GiB."""
from __future__ import annotations

import ctypes as C
import random

import numpy as np
import pytest

import textgen

# test_host.py's hand-made vocabulary (test_decode_matches_reference_rules), plus a token that ends in "\r", a
# duplicate, a token whose invalid UTF-8 bytes the decoded word drops, and a continuation token of one char
RULES_VOCAB = [b"[PAD]", b"a", b"##b", b"--", b"[UNK]", "中".encode(), "##かな".encode(), b"a\r", b"a", b"x\xffy\xc3",
               b"##\xe4\xb8z", b"##q"]
UINT64_MAX_AS_INT64 = -1


def _dev(gpu_device):
    import torch

    return torch.device(f"cuda:{gpu_device}")


def _ids(ids, gpu_device):
    import torch

    return torch.tensor(np.asarray(ids, dtype=np.int32), dtype=torch.int32, device=_dev(gpu_device))


def _entries(d_chars, d_char_offsets, n_ids):
    chars = d_chars.cpu().numpy().tobytes()
    offs = d_char_offsets[: n_ids + 1].cpu().numpy()
    return [chars[int(offs[i]):int(offs[i + 1])] for i in range(n_ids)], offs


def _check(v, ids, gpu_device, tag):
    """decode_device of `ids` (a host list/array) against the host decode of the same ids, id by id."""
    import torch

    ids = np.asarray(ids, dtype=np.int32)
    d_chars, d_offs, n_chars, n_skipped = v.decode_device(_ids(ids, gpu_device))
    got, offs = _entries(d_chars, d_offs, ids.size)
    assert offs[0] == 0 and offs[-1] == n_chars == d_chars.numel(), tag
    skipped = 0
    cache = {}
    for i, x in enumerate(ids.tolist()):
        if x not in cache:
            cache[x] = v.decode([x])
        exp = cache[x]
        if exp == []:
            skipped += 1
            assert got[i] == b"", (tag, i, x, got[i])
        else:
            assert [got[i]] == exp, (tag, i, x, got[i], exp)
    assert n_skipped == skipped, (tag, n_skipped, skipped)
    assert [e for e in got if e] == v.decode(ids), tag
    # the async form gives the same column
    d_chars2 = torch.full((n_chars + 7,), 0xEE, dtype=torch.uint8, device=d_chars.device)
    d_offs2 = torch.empty(ids.size + 1, dtype=torch.int64, device=d_chars.device)
    v.decode_device_async(_ids(ids, gpu_device), d_chars2, d_offs2)
    torch.cuda.synchronize()
    assert torch.equal(d_offs2, d_offs[: ids.size + 1]), tag
    assert torch.equal(d_chars2[:n_chars], d_chars) and bool((d_chars2[n_chars:] == 0xEE).all()), tag
    return got, offs


# ---- rules ------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_decode_device_reference_rules(gpu_device):
    from wordpiece_b200 import Vocab

    v = Vocab(RULES_VOCAB, device=gpu_device)
    size = len(v)
    ids = [i for i in range(-3, size + 3) if i != size]
    got, _ = _check(v, ids, gpu_device, "every id")
    by_id = dict(zip(ids, got))
    assert by_id[1] == b"a" and by_id[2] == b"##b" and by_id[3] == b"" and by_id[0] == b"[PAD]"
    assert by_id[7] == b"a\r" and by_id[8] == b"a" and by_id[9] == b"xy" and by_id[10] == b"##z" and by_id[11] == b"##q"
    assert by_id[-1] == b"" and by_id[size + 1] == b""
    rng = random.Random(3)
    _check(v, [rng.choice(ids) for _ in range(5000)], gpu_device, "random")
    v.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["en", "ja", "adv"])
def test_decode_device_bench_vocabularies(gpu_device, name):
    """The 29k, the 120k and the long-m100 vocabulary, random ids (out-of-range ones included)."""
    from wordpiece_b200 import Vocab, synth

    vocab = synth.generator(name).spec.vocab
    v = Vocab(vocab, device=gpu_device)
    size = len(v)
    rng = np.random.default_rng(11)
    ids = rng.integers(-3, size + 3, 30000).astype(np.int32)
    ids[ids == size] = size + 1
    _check(v, ids, gpu_device, name)
    v.close()


# ---- round trip of a column ------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_decode_device_round_trip_of_a_column(gpu_device):
    import torch
    from wordpiece_b200 import Vocab

    rng = random.Random(5)
    vocab = textgen.mixed_vocab(rng, 400, long_tokens=3)
    texts = []
    for k in range(600):
        n = rng.choice([0, 0, 1, 5, 40, 300, 3000])
        texts.append(textgen.mixed_text(rng, n, vocab, invalid_rate=0.01, long_run_rate=0.01)[:n] if n else b"")
    v = Vocab(vocab, device=gpu_device)
    dev = _dev(gpu_device)
    blob = b"".join(texts)
    d_chars = torch.frombuffer(bytearray(blob), dtype=torch.uint8).to(dev)
    d_offsets = torch.from_numpy(np.concatenate([[0], np.cumsum([len(t) for t in texts])]).astype(np.int64)).to(dev)
    d_ids, d_id_offsets, n_ids = v.encode_batch_device(d_chars, d_offsets)
    tok_chars, tok_offs, _, _ = v.decode_device(d_ids[:n_ids])
    entries, _ = _entries(tok_chars, tok_offs, n_ids)
    id_offs = d_id_offsets.cpu().numpy()
    for t, text in enumerate(texts):
        mine = [e for e in entries[int(id_offs[t]):int(id_offs[t + 1])] if e]
        assert mine == v.decode(v.encode(text)), (t, text[:40])
    v.close()


# ---- block borders, stage windows ------------------------------------------------------------------------------

def _longest_adv_token(v, vocab):
    lens = [len(b"".join(v.decode([i]))) for i in range(len(vocab))]
    return int(np.argmax(lens)), max(lens)


@pytest.mark.gpu
def test_decode_device_block_borders(gpu_device):
    from wordpiece_b200 import Vocab, synth

    block = 2048  # ids per block of the scatter kernel
    vocab = synth.generator("adv").spec.vocab
    v = Vocab(vocab, device=gpu_device)
    size = len(v)
    long_id, long_len = _longest_adv_token(v, vocab)
    assert long_len >= 100
    rng = np.random.default_rng(2)
    for n in [0, 1, block - 1, block, block + 1, 3 * block - 1, 37 * block + 5]:
        ids = rng.integers(-2, size + 2, n).astype(np.int32)
        ids[ids == size] = -1
        if n == 0:
            d_chars, d_offs, n_chars, n_skipped = v.decode_device(_ids(ids, gpu_device))
            assert d_offs.tolist() == [0] and n_chars == 0 and n_skipped == 0
            continue
        _check(v, ids, gpu_device, f"n = {n}")
    # every id the longest token: each block writes 2048 x ~100 bytes through a 16 KiB stage, about 13 windows
    _check(v, np.full(3 * block + 17, long_id, np.int32), gpu_device, "all long")
    # long and short tokens mixed: long tokens cross window borders at many phases
    short = [i for i in range(1000, 1400) if v.decode([i])]
    ids = np.array([long_id if rng.random() < 0.4 else rng.choice(short) for _ in range(5 * block + 3)], np.int32)
    _check(v, ids, gpu_device, "mixed long and short")
    v.close()


# ---- errors -----------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("where", [0, 5000, -1])
def test_decode_device_id_equal_to_size(gpu_device, where):
    """An id == size in the first, a middle or the last block: WP_ERR_ID_RANGE (sync), UINT64_MAX (async)."""
    import torch
    from wordpiece_b200 import Vocab, WordPieceError
    from wordpiece_b200._capi import WP_ERR_ID_RANGE

    v = Vocab(RULES_VOCAB, device=gpu_device)
    size = len(v)
    ids = np.random.default_rng(4).integers(0, size, 3 * 2048 + 100).astype(np.int32)
    ids[where] = size
    d_ids = _ids(ids, gpu_device)
    with pytest.raises(WordPieceError) as e:
        v.decode_device(d_ids)
    assert e.value.status == WP_ERR_ID_RANGE
    d_chars = torch.full((ids.size * 10,), 0xEE, dtype=torch.uint8, device=d_ids.device)
    d_offs = torch.zeros(ids.size + 1, dtype=torch.int64, device=d_ids.device)
    v.decode_device_async(d_ids, d_chars, d_offs)
    torch.cuda.synchronize()
    assert int(d_offs[-1]) == UINT64_MAX_AS_INT64 and bool((d_chars == 0xEE).all())
    ids[where] = 1
    _check(v, ids, gpu_device, "valid after an id == size")
    v.close()


@pytest.mark.gpu
def test_decode_device_capacity(gpu_device):
    """capacity = needed - 1: WP_ERR_CAPACITY with the exact count (sync), UINT64_MAX (async); a canary after the
    capacity stays untouched in both.  A size query with d_chars = NULL."""
    import torch
    from wordpiece_b200 import Vocab, synth
    from wordpiece_b200._capi import WP_ERR_CAPACITY, WP_OK

    v = Vocab(synth.generator("en").spec.vocab, device=gpu_device)
    ids = np.random.default_rng(6).integers(-1, len(v), 9000).astype(np.int32)
    d_ids = _ids(ids, gpu_device)
    _, _, need, skipped = v.decode_device(d_ids)
    L, h = v._L, v._h
    d_offs = torch.zeros(ids.size + 1, dtype=torch.int64, device=d_ids.device)
    cnt, sk = C.c_size_t(), C.c_size_t()
    assert L.wp_decode_device(h, d_ids.data_ptr(), ids.size, None, 0, d_offs.data_ptr(), C.byref(cnt), C.byref(sk),
                              None) == WP_ERR_CAPACITY
    assert cnt.value == need and sk.value == skipped
    big = torch.full((need + 64,), 0xEE, dtype=torch.uint8, device=d_ids.device)
    assert L.wp_decode_device(h, d_ids.data_ptr(), ids.size, big.data_ptr(), need - 1, d_offs.data_ptr(), C.byref(cnt),
                              None, None) == WP_ERR_CAPACITY
    torch.cuda.synchronize()
    assert cnt.value == need and bool((big == 0xEE).all()) and bool((d_offs == 0).all())
    v.decode_device_async(d_ids, big[: need - 1], d_offs)
    torch.cuda.synchronize()
    assert int(d_offs[-1]) == UINT64_MAX_AS_INT64 and bool((big == 0xEE).all())
    assert L.wp_decode_device(h, d_ids.data_ptr(), ids.size, big.data_ptr(), need, d_offs.data_ptr(), C.byref(cnt),
                              None, None) == WP_OK
    torch.cuda.synchronize()
    assert int(d_offs[-1]) == need and bool((big[need:] == 0xEE).all())
    v.close()


# ---- ordering on one handle -------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_decode_device_between_async_encodes_on_two_streams(gpu_device):
    """encode_device_async on stream A, decode_device_async of its ids on stream B, another encode on A: the handle
    orders them (they share its scratch) and all three results are right."""
    import torch
    from wordpiece_b200 import Vocab
    from _oracle import Oracle

    rng = random.Random(9)
    vocab = textgen.mixed_vocab(rng, 500, long_tokens=3)
    text1 = textgen.mixed_text(rng, 3_000_000, vocab, invalid_rate=0.001, long_run_rate=0.01)
    text2 = textgen.mixed_text(rng, 2_000_000, vocab, invalid_rate=0.001)
    o = Oracle(vocab)
    exp1, exp2 = o.encode(text1), o.encode(text2)
    v = Vocab(vocab, device=gpu_device)
    dev = _dev(gpu_device)
    sa, sb = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    d_t1 = torch.frombuffer(bytearray(text1), dtype=torch.uint8).to(dev)
    d_t2 = torch.frombuffer(bytearray(text2), dtype=torch.uint8).to(dev)
    d_ids1 = torch.zeros(len(text1), dtype=torch.int32, device=dev)
    d_ids2 = torch.zeros(len(text2), dtype=torch.int32, device=dev)
    c1, c2 = torch.zeros(1, dtype=torch.int64, device=dev), torch.zeros(1, dtype=torch.int64, device=dev)
    n = exp1.size
    exp_tokens = v.decode(exp1)
    d_chars = torch.empty(sum(len(t) for t in exp_tokens), dtype=torch.uint8, device=dev)
    d_offs = torch.empty(n + 1, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    v.encode_device_async(d_t1, d_ids1, c1, stream=sa.cuda_stream)
    sb.wait_stream(sa)  # (the ids are the caller's to order; the scratch is the library's)
    v.decode_device_async(d_ids1[:n], d_chars, d_offs, stream=sb.cuda_stream)
    v.encode_device_async(d_t2, d_ids2, c2, stream=sa.cuda_stream)
    torch.cuda.synchronize()
    assert int(c1) == exp1.size and np.array_equal(d_ids1[: exp1.size].cpu().numpy(), exp1)
    assert int(c2) == exp2.size and np.array_equal(d_ids2[: exp2.size].cpu().numpy(), exp2)
    offs = d_offs.cpu().numpy()
    assert offs[-1] == d_chars.numel()
    chars = d_chars.cpu().numpy().tobytes()
    got = [chars[int(offs[i]):int(offs[i + 1])] for i in range(n)]
    assert [e for e in got if e] == exp_tokens
    v.close()


# ---- offsets past 4 GiB -----------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_decode_device_offsets_past_4gib(gpu_device):
    """About 45 M ids of a 100-byte token (with shorter and skipped ids among them): more than 2^32 output bytes."""
    import torch
    from wordpiece_b200 import Vocab

    vocab = [b"[UNK]", b"x" * 99 + b"y", b"##z", b"--"]
    v = Vocab(vocab, device=gpu_device)
    dev = _dev(gpu_device)
    n = 45_000_000
    rng = np.random.default_rng(8)
    ids = np.ones(n, np.int32)
    pick = rng.integers(0, n, 200_000)
    ids[pick] = rng.choice(np.array([0, 2, 3, -1, 7], np.int32), pick.size)
    lens = np.array([5, 100, 3, 0], np.int64)
    entry = np.where((ids >= 0) & (ids < 4), lens[np.clip(ids, 0, 3)], 0)
    exp_offs = np.concatenate([[0], np.cumsum(entry)])
    assert exp_offs[-1] > (1 << 32)
    d_ids = torch.from_numpy(ids).to(dev)
    d_chars, d_offs, n_chars, n_skipped = v.decode_device(d_ids)
    assert n_chars == exp_offs[-1] and n_skipped == int((entry == 0).sum())
    assert np.array_equal(d_offs.cpu().numpy(), exp_offs)
    table = {0: b"[UNK]", 1: b"x" * 99 + b"y", 2: b"##z"}
    for i in list(range(5)) + rng.integers(0, n, 3000).tolist() + list(range(n - 5, n)):
        a, b = int(exp_offs[i]), int(exp_offs[i + 1])
        got = d_chars[a:b].cpu().numpy().tobytes()
        assert got == table.get(int(ids[i]), b""), (i, int(ids[i]), got[:20])
    del d_chars, d_offs
    v.close()
    torch.cuda.empty_cache()


# ---- host only (no GPU) -----------------------------------------------------------------------------------------

def test_decode_device_host_only_handle_and_null_arguments():
    """No device: WP_ERR_NO_DEVICE; null or inconsistent arguments: WP_ERR_INVALID_ARG; neither launches a kernel."""
    from wordpiece_b200 import Vocab, kernel_launch_count
    from wordpiece_b200._capi import WP_ERR_INVALID_ARG, WP_ERR_NO_DEVICE

    v = Vocab(RULES_VOCAB, device=-1)
    L, h = v._L, v._h
    launches = kernel_launch_count()
    fake = 0x1000  # never dereferenced: the call fails before any device work
    cnt, sk = C.c_size_t(5), C.c_size_t(5)
    assert L.wp_decode_device(h, fake, 8, fake, 8, fake, C.byref(cnt), C.byref(sk), None) == WP_ERR_NO_DEVICE
    assert cnt.value == 0 and sk.value == 0 and b"host-only" in L.wp_last_error()
    assert L.wp_decode_device_async(h, fake, 8, fake, 8, fake, None) == WP_ERR_NO_DEVICE
    assert L.wp_decode_device(h, fake, 0, None, 0, fake, C.byref(cnt), None, None) == WP_ERR_NO_DEVICE
    for args in [(None, fake, 8, fake, 8, fake),   # no handle
                 (h, None, 8, fake, 8, fake),      # ids missing
                 (h, fake, 8, None, 8, fake),      # capacity without chars
                 (h, fake, 8, fake, 8, None)]:     # offsets missing
        assert L.wp_decode_device(*args, C.byref(cnt), None, None) == WP_ERR_INVALID_ARG, args
        assert L.wp_decode_device_async(*args, None) == WP_ERR_INVALID_ARG, args
    assert L.wp_decode_device(h, fake, 8, fake, 8, fake, None, None, None) == WP_ERR_INVALID_ARG  # no n_chars
    assert kernel_launch_count() == launches
    v.close()


def test_decode_device_python_host_only_handle():
    """Vocab.decode_device on a host-only handle raises with WP_ERR_NO_DEVICE (the library's status)."""
    import torch
    from wordpiece_b200 import Vocab, WordPieceError
    from wordpiece_b200._capi import WP_ERR_NO_DEVICE

    v = Vocab(RULES_VOCAB, device=-1)

    class FakeCuda:  # a stand-in for a CUDA tensor on a machine without one: only its metadata is read
        is_cuda = True

        def __init__(self, dtype, n):
            self.dtype, self._n = dtype, n
            self.device = "cuda:0"

        def dim(self):
            return 1

        def is_contiguous(self):
            return True

        def numel(self):
            return self._n

        def data_ptr(self):
            return 0x1000

    with pytest.raises(WordPieceError) as e:
        v.decode_device(FakeCuda(torch.int32, 4), FakeCuda(torch.uint8, 16), FakeCuda(torch.int64, 5), stream=0)
    assert e.value.status == WP_ERR_NO_DEVICE
    v.close()


def test_decode_device_symbols_are_exported():
    from wordpiece_b200._capi import EXPORTED_SYMBOLS, load_library

    L = load_library()
    for name in ("wp_decode_device", "wp_decode_device_async"):
        assert name in EXPORTED_SYMBOLS and hasattr(L, name)
