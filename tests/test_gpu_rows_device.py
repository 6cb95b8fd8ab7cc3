"""Model-input rows (wp_rows_device[_async], Vocab.rows_device, Vocab.encode_rows_device): per-text ids in GPU memory
(ids + Arrow id offsets) to fixed-length rows of max_len ids, [CLS]? content [SEP]? pad ..., with an attention mask,
truncated or cut into overlapping windows.  Every row, mask and row offset must equal the numpy model below bit for
bit: at every combination of special tokens and strides, at unaligned row starts, scan block borders, a text of a
million windows, output past 4 GiB, and on the ids the encoder gives real text."""
from __future__ import annotations

import ctypes as C

import numpy as np
import pytest

from _oracle import Oracle

UINT64_MAX_AS_INT64 = -1
BLOCK = 2048  # texts per block of the scan kernel


# ---- the reference model --------------------------------------------------------------------------------------

def row_count(n_t: int, width: int, stride: int) -> int:
    """Rows of a text of n_t ids: 1 when truncating or when it fits, else 1 + ceil((n_t - W) / stride)."""
    if stride == 0 or n_t <= width:
        return 1
    return 1 + (n_t - width + stride - 1) // stride


def model(ids, id_offsets, max_len, stride=0, pad_id=0, cls_id=None, sep_id=None, rows=None):
    """(rows [k, L] int32, mask [k, L] uint8, row_offsets [n_texts + 1] int64) of the semantics in
    include/wordpiece_b200.h, for the row numbers `rows` (default: all of them)."""
    ids = np.asarray(ids, np.int32)
    offs = np.asarray(id_offsets, np.int64)
    c, s = int(cls_id is not None), int(sep_id is not None)
    width = max_len - c - s
    assert width >= 1 and 0 <= stride <= width
    n_t = np.diff(offs)
    if stride == 0:
        counts = np.ones(n_t.size, np.int64)
    else:
        counts = np.where(n_t <= width, 1, 1 + (n_t - width + stride - 1) // stride)
    row_offs = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    if rows is None:
        rows = np.arange(row_offs[-1], dtype=np.int64)
    rows = np.asarray(rows, np.int64)
    t = np.searchsorted(row_offs, rows, side="right") - 1
    k = rows - row_offs[t]
    start = k * stride
    length = np.minimum(n_t[t] - start, width)
    col = np.arange(max_len, dtype=np.int64)[None, :]
    j = col - c
    content = (j >= 0) & (j < length[:, None])
    src = np.clip(offs[t][:, None] + start[:, None] + j, 0, max(ids.size - 1, 0))
    out = np.full((rows.size, max_len), pad_id, np.int32)
    if ids.size:
        out[content] = ids[src[content]]
    if c:
        out[:, 0] = cls_id
    if s:
        out[np.arange(rows.size), c + length] = sep_id
    mask = (col < (c + length + s)[:, None]).astype(np.uint8)
    return out, mask, row_offs


def texts_to_column(texts):
    ids = np.concatenate([np.asarray(x, np.int32) for x in texts]) if texts else np.zeros(0, np.int32)
    offs = np.concatenate([[0], np.cumsum([len(x) for x in texts])]).astype(np.int64)
    return ids, offs


# ---- the model on hand-written cases (no GPU) ------------------------------------------------------------------

@pytest.mark.parametrize("width,stride", [(5, 0), (5, 1), (5, 2), (5, 5), (1, 1), (126, 64)])
def test_rows_model_row_counts(width, stride):
    for n_t, exp in [(0, 1), (width, 1), (width + 1, 1 if stride == 0 else 2),
                     (width + max(stride, 1), 1 if stride == 0 else 2),
                     (width + max(stride, 1) + 1, 1 if stride == 0 else 3)]:
        assert row_count(n_t, width, stride) == exp, (n_t, width, stride)
        ids = np.arange(100, 100 + n_t, dtype=np.int32)
        rows, _, row_offs = model(ids, [0, n_t], width + 2, stride, pad_id=0, cls_id=1, sep_id=2)
        assert row_offs.tolist() == [0, exp] and rows.shape == (exp, width + 2)
        if n_t:  # windows start `stride` ids apart and the last one ends at n_t (truncation: at W)
            assert rows[-1][rows[-1] >= 100][-1] == 100 + (n_t if stride else min(n_t, width)) - 1
            for r in range(exp):
                assert rows[r, 1] == 100 + r * stride


def test_rows_model_hand_written_rows():
    # L = 6, CLS 101, SEP 102, pad 0: W = 4; SEP right after the content, not at the end of the row
    ids, offs = texts_to_column([[7, 8], [], [1, 2, 3, 4, 5, 6], [-1, 9]])
    rows, mask, row_offs = model(ids, offs, 6, stride=2, pad_id=0, cls_id=101, sep_id=102)
    assert row_offs.tolist() == [0, 1, 2, 4, 5]
    assert rows.tolist() == [[101, 7, 8, 102, 0, 0],
                             [101, 102, 0, 0, 0, 0],
                             [101, 1, 2, 3, 4, 102],
                             [101, 3, 4, 5, 6, 102],
                             [101, -1, 9, 102, 0, 0]]
    assert mask.tolist() == [[1, 1, 1, 1, 0, 0], [1, 1, 0, 0, 0, 0], [1] * 6, [1] * 6, [1, 1, 1, 1, 0, 0]]
    # truncation, no specials, pad -5
    rows, mask, row_offs = model(ids, offs, 3, stride=0, pad_id=-5)
    assert row_offs.tolist() == [0, 1, 2, 3, 4]
    assert rows.tolist() == [[7, 8, -5], [-5, -5, -5], [1, 2, 3], [-1, 9, -5]]
    assert mask.tolist() == [[1, 1, 0], [0, 0, 0], [1, 1, 1], [1, 1, 0]]
    # SEP only, windows of W = 2 with stride 1
    rows, _, row_offs = model([1, 2, 3, 4], [0, 4], 3, stride=1, sep_id=9)
    assert row_offs.tolist() == [0, 3] and rows.tolist() == [[1, 2, 9], [2, 3, 9], [3, 4, 9]]


# ---- the C ABI without a GPU -----------------------------------------------------------------------------------

def _spec(max_len, stride=0, pad_id=0, cls_id=None, sep_id=None):
    from wordpiece_b200._capi import RowsSpec

    return RowsSpec.make(max_len, stride, pad_id, cls_id, sep_id)


def test_rows_device_host_only_handle_and_argument_errors():
    """Null arguments and bad specs: WP_ERR_INVALID_ARG, found before the device check; a host-only handle with good
    arguments: WP_ERR_NO_DEVICE.  No kernel is launched."""
    from wordpiece_b200 import Vocab, kernel_launch_count
    from wordpiece_b200._capi import WP_ERR_INVALID_ARG, WP_ERR_NO_DEVICE, RowsSpec

    v = Vocab(["[UNK]", "a"], device=-1)
    L, h = v._L, v._h
    launches = kernel_launch_count()
    fake = 0x1000  # never dereferenced: every call fails before any device work
    n = C.c_size_t(7)
    good = _spec(8, 2, 0, 101, 102)

    def sync(*a, spec=good, rows=fake, mask=fake, cap=4, row_offs=fake, n_rows=C.byref(n)):
        return L.wp_rows_device(h, *a, C.byref(spec) if spec is not None else None, rows, mask, cap, row_offs, n_rows, None)

    def asyn(*a, spec=good, rows=fake, mask=fake, cap=4, row_offs=fake):
        return L.wp_rows_device_async(h, *a, C.byref(spec) if spec is not None else None, rows, mask, cap, row_offs, None)

    base = (fake, 16, fake, 3)
    assert sync(*base) == WP_ERR_NO_DEVICE and n.value == 0 and b"host-only" in L.wp_last_error()
    assert asyn(*base) == WP_ERR_NO_DEVICE
    assert sync(*base, mask=None) == WP_ERR_NO_DEVICE  # (the mask is optional)
    assert sync(fake, 0, fake, 0, rows=None, cap=0) == WP_ERR_NO_DEVICE
    bad_args = [dict(a=(None, 16, fake, 3)),          # ids missing
                dict(a=(fake, 16, None, 3)),          # id offsets missing
                dict(a=base, spec=None),              # spec missing
                dict(a=base, rows=None),              # capacity without rows
                dict(a=base, row_offs=None),          # row offsets missing
                dict(a=base, rows=fake + 2),          # rows not 4-byte aligned
                dict(a=base, spec=_spec(2, 0, 0, 101, 102)),         # W = 0
                dict(a=base, spec=_spec(1, 0, 0, 101)),              # W = 0
                dict(a=base, spec=_spec(0)),                         # W = 0
                dict(a=base, spec=_spec(8, 7, 0, 101, 102)),         # stride = W + 1
                dict(a=base, spec=_spec(1, 2)),                      # stride = W + 1
                dict(a=base, spec=RowsSpec(8, 0, 0, 0, 0, 4)),       # unknown flag
                dict(a=base, cap=(1 << 62) // 8)]                    # capacity * L * 4 overflows
    for kw in bad_args:
        a = kw.pop("a")
        assert sync(*a, **kw) == WP_ERR_INVALID_ARG, kw
        assert asyn(*a, **kw) == WP_ERR_INVALID_ARG, kw
    assert sync(*base, n_rows=None) == WP_ERR_INVALID_ARG  # no n_rows
    assert L.wp_rows_device(None, *base, C.byref(good), fake, fake, 4, fake, C.byref(n), None) == WP_ERR_INVALID_ARG
    # W = 1 and stride = W are allowed
    assert sync(*base, spec=_spec(3, 1, 0, 101, 102)) == WP_ERR_NO_DEVICE
    assert sync(*base, spec=_spec(1, 1)) == WP_ERR_NO_DEVICE
    assert kernel_launch_count() == launches
    v.close()


def test_rows_device_symbols_are_exported():
    from wordpiece_b200._capi import EXPORTED_SYMBOLS, load_library

    L = load_library()
    for name in ("wp_rows_device", "wp_rows_device_async"):
        assert name in EXPORTED_SYMBOLS and hasattr(L, name)


# ---- on the GPU ------------------------------------------------------------------------------------------------

def _dev(gpu_device):
    import torch

    return torch.device(f"cuda:{gpu_device}")


def _to(x, dtype, gpu_device):
    import torch

    return torch.from_numpy(np.ascontiguousarray(x)).to(dtype=dtype, device=_dev(gpu_device))


def _check(v, ids, offs, gpu_device, tag, max_len, stride=0, pad_id=0, cls_id=None, sep_id=None, d_ids=None, d_offs=None):
    """rows_device (sync, with and without mask) and rows_device_async against the model, bit for bit."""
    import torch

    kw = dict(stride=stride, pad_id=pad_id, cls_id=cls_id, sep_id=sep_id)
    exp_rows, exp_mask, exp_offs = model(ids, offs, max_len, **kw)
    if d_ids is None:
        d_ids, d_offs = _to(ids, torch.int32, gpu_device), _to(offs, torch.int64, gpu_device)
    d_rows, d_mask, d_row_offs, n_rows = v.rows_device(d_ids, d_offs, max_len, **kw)
    assert n_rows == exp_rows.shape[0], tag
    assert np.array_equal(d_row_offs.cpu().numpy(), exp_offs), tag
    assert np.array_equal(d_rows.cpu().numpy(), exp_rows), tag
    assert np.array_equal(d_mask.cpu().numpy(), exp_mask), tag
    # async into preallocated buffers with one spare row (left untouched)
    rows2 = torch.full(((n_rows + 1) * max_len,), 0x7EEEEEEE, dtype=torch.int32, device=d_ids.device)
    mask2 = torch.full(((n_rows + 1) * max_len,), 0xEE, dtype=torch.uint8, device=d_ids.device)
    offs2 = torch.zeros(offs.size, dtype=torch.int64, device=d_ids.device)
    v.rows_device_async(d_ids, d_offs, rows2, offs2, max_len, d_mask=mask2, **kw)
    torch.cuda.synchronize()
    assert np.array_equal(offs2.cpu().numpy(), exp_offs), tag
    assert np.array_equal(rows2[: n_rows * max_len].view(n_rows, max_len).cpu().numpy(), exp_rows), tag
    assert np.array_equal(mask2[: n_rows * max_len].view(n_rows, max_len).cpu().numpy(), exp_mask), tag
    assert bool((rows2[n_rows * max_len:] == 0x7EEEEEEE).all()) and bool((mask2[n_rows * max_len:] == 0xEE).all()), tag
    return d_rows, d_mask, d_row_offs, n_rows


def _random_texts(rng, width, n_texts, vocab_size=30000):
    lens = [0, 1, max(width - 1, 0), width, width + 1, 2 * width + 3, 3 * width + 7]
    texts = []
    for _ in range(n_texts):
        n = int(rng.choice(lens)) if rng.random() < 0.6 else int(rng.integers(0, 3 * width + 10))
        texts.append(rng.integers(-2, vocab_size + 5, n).astype(np.int32))
    return texts


@pytest.mark.gpu
@pytest.mark.parametrize("specials", ["none", "cls", "sep", "both"])
@pytest.mark.parametrize("max_len", ["w1", 3, 128, 509, 512])
def test_rows_device_specials_strides_lengths(gpu_device, specials, max_len):
    """Every combination of CLS / SEP present, stride in {0, 1, W - 1, W}, L in {specials + 1 (W = 1), 3, 128, 509,
    512}; odd L puts row starts at every 16-byte phase."""
    from wordpiece_b200 import Vocab

    cls_id = 101 if specials in ("cls", "both") else None
    sep_id = 102 if specials in ("sep", "both") else None
    n_spec = (cls_id is not None) + (sep_id is not None)
    L = n_spec + 1 if max_len == "w1" else max_len
    width = L - n_spec
    if width < 1:
        pytest.skip("W < 1")
    v = Vocab(["[UNK]", "a"], device=gpu_device)
    rng = np.random.default_rng(L * 7 + n_spec)
    ids, offs = texts_to_column(_random_texts(rng, width, 300))
    for stride in sorted({0, 1, width - 1, width}):
        _check(v, ids, offs, gpu_device, f"L={L} {specials} stride={stride}", L, stride=stride, pad_id=-9,
               cls_id=cls_id, sep_id=sep_id)
    v.close()


@pytest.mark.gpu
def test_rows_device_misaligned_outputs_with_canaries(gpu_device):
    """d_rows and d_mask as views at every offset into larger buffers; the canaries before and after stay."""
    import torch
    from wordpiece_b200 import Vocab

    v = Vocab(["[UNK]", "a"], device=gpu_device)
    rng = np.random.default_rng(3)
    for L, stride in [(509, 200), (13, 5), (3, 1), (128, 0)]:
        ids, offs = texts_to_column(_random_texts(rng, L - 2, 150))
        exp_rows, exp_mask, exp_offs = model(ids, offs, L, stride, 0, 101, 102)
        n = exp_rows.shape[0]
        d_ids, d_offs = _to(ids, torch.int32, gpu_device), _to(offs, torch.int64, gpu_device)
        for lead_ids, lead_mask in [(1, 1), (2, 7), (3, 15), (0, 3), (1, 0)]:
            big_rows = torch.full((n * L + 8,), 0x7EEEEEEE, dtype=torch.int32, device=d_ids.device)
            big_mask = torch.full((n * L + 32,), 0xEE, dtype=torch.uint8, device=d_ids.device)
            rows = big_rows[lead_ids: lead_ids + n * L]
            mask = big_mask[lead_mask: lead_mask + n * L]
            r, m, ro, k = v.rows_device(d_ids, d_offs, L, stride, 0, 101, 102, d_rows=rows, d_mask=mask)
            tag = (L, stride, lead_ids, lead_mask)
            assert k == n and np.array_equal(ro.cpu().numpy(), exp_offs), tag
            assert np.array_equal(r.cpu().numpy(), exp_rows) and np.array_equal(m.cpu().numpy(), exp_mask), tag
            assert bool((big_rows[:lead_ids] == 0x7EEEEEEE).all()) and bool((big_rows[lead_ids + n * L:] == 0x7EEEEEEE).all()), tag
            assert bool((big_mask[:lead_mask] == 0xEE).all()) and bool((big_mask[lead_mask + n * L:] == 0xEE).all()), tag
    v.close()


@pytest.mark.gpu
def test_rows_device_offset_base_and_ids_copied_verbatim(gpu_device):
    """d_id_offsets that start past 0 (ids before and after the column unused), and ids that are negative or past
    the vocabulary: copied as they are."""
    import torch
    from wordpiece_b200 import Vocab

    v = Vocab(["[UNK]", "a"], device=gpu_device)
    rng = np.random.default_rng(4)
    texts = _random_texts(rng, 30, 500)
    for x in texts[::7]:
        if x.size:
            x[0] = -1
            x[-1] = 2**31 - 1
    ids, offs = texts_to_column(texts)
    lead, trail = 37, 11
    all_ids = np.concatenate([np.full(lead, 5, np.int32), ids, np.full(trail, 6, np.int32)])
    base_offs = offs + lead
    for stride in (0, 7, 30):
        _check(v, all_ids, base_offs, gpu_device, f"base stride={stride}", 32, stride=stride, cls_id=-3, sep_id=2**31 - 1,
               pad_id=-2**31)
    v.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["en", "ja"])
def test_encode_rows_device_end_to_end(gpu_device, name):
    """A string column of bench text through encode_rows_device, against the oracle's per-text ids through the
    model."""
    import torch
    from wordpiece_b200 import Vocab, synth

    g = synth.generator(name)
    text = g.generate(2 << 20, seed=5).tobytes()
    rng = np.random.default_rng(6)
    cuts = np.sort(rng.integers(0, len(text), 700))
    bounds = np.concatenate([[0], cuts, [len(text)]]).astype(np.int64)
    texts = [text[bounds[i]:bounds[i + 1]] for i in range(bounds.size - 1)]
    o = Oracle(g.spec.vocab)
    ids, offs = texts_to_column([o.encode(t) for t in texts])
    v = Vocab(g.spec.vocab, device=gpu_device)
    d_chars, d_offsets = _to(np.frombuffer(bytearray(text), np.uint8), torch.uint8, gpu_device), _to(bounds, torch.int64, gpu_device)
    for L, stride in [(512, 384), (128, 0), (64, 1)]:
        exp_rows, exp_mask, exp_offs = model(ids, offs, L, stride, 0, 2, 3)
        d_rows, d_mask, d_row_offs, n = v.encode_rows_device(d_chars, d_offsets, L, stride=stride, pad_id=0, cls_id=2,
                                                             sep_id=3)
        assert n == exp_rows.shape[0] and np.array_equal(d_row_offs.cpu().numpy(), exp_offs), (name, L, stride)
        assert np.array_equal(d_rows.cpu().numpy(), exp_rows), (name, L, stride)
        assert np.array_equal(d_mask.cpu().numpy(), exp_mask), (name, L, stride)
    v.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n_texts", [BLOCK - 1, BLOCK, BLOCK + 1, 3 * BLOCK + 1])
def test_rows_device_scan_block_borders(gpu_device, n_texts):
    from wordpiece_b200 import Vocab

    v = Vocab(["[UNK]", "a"], device=gpu_device)
    rng = np.random.default_rng(n_texts)
    ids, offs = texts_to_column(_random_texts(rng, 14, n_texts))
    for stride in (0, 3):
        _check(v, ids, offs, gpu_device, f"n_texts={n_texts} stride={stride}", 16, stride=stride, cls_id=1, sep_id=2)
    v.close()


@pytest.mark.gpu
def test_rows_device_one_text_of_a_million_windows(gpu_device):
    """One text of 1.2 M ids with stride 1 (about as many rows), between two short texts: checked row by row in
    chunks."""
    import torch
    from wordpiece_b200 import Vocab

    v = Vocab(["[UNK]", "a"], device=gpu_device)
    rng = np.random.default_rng(8)
    ids, offs = texts_to_column([rng.integers(0, 30000, 5), rng.integers(-1, 30000, 1_200_000), rng.integers(0, 9, 3)])
    L = 128
    d_rows, d_mask, d_row_offs, n = v.rows_device(_to(ids, torch.int32, gpu_device), _to(offs, torch.int64, gpu_device), L,
                                                  stride=1, cls_id=101, sep_id=102)
    _, _, exp_offs = model(ids, offs, L, 1, 0, 101, 102, rows=[])
    assert n == exp_offs[-1] == 1 + (1_200_000 - 126 + 1) + 1 and np.array_equal(d_row_offs.cpu().numpy(), exp_offs)
    for a in range(0, n, 1 << 16):
        rows = np.arange(a, min(n, a + (1 << 16)))
        exp_rows, exp_mask, _ = model(ids, offs, L, 1, 0, 101, 102, rows=rows)
        assert np.array_equal(d_rows[a:a + rows.size].cpu().numpy(), exp_rows), a
        assert np.array_equal(d_mask[a:a + rows.size].cpu().numpy(), exp_mask), a
    v.close()


@pytest.mark.gpu
def test_rows_device_capacity(gpu_device):
    """Exact capacity works; one row short gives WP_ERR_CAPACITY with the exact count and offsets and writes no
    row or mask byte (sync), UINT64_MAX and nothing written (async); d_rows NULL with capacity 0 is a size query."""
    import torch
    from wordpiece_b200 import Vocab
    from wordpiece_b200._capi import WP_ERR_CAPACITY, WP_OK

    v = Vocab(["[UNK]", "a"], device=gpu_device)
    L, h = v._L, v._h
    rng = np.random.default_rng(9)
    ids, offs = texts_to_column(_random_texts(rng, 30, 3000))
    ML = 33
    exp_rows, exp_mask, exp_offs = model(ids, offs, ML, 8, 0, 1, 2)
    need = exp_rows.shape[0]
    d_ids, d_offs = _to(ids, torch.int32, gpu_device), _to(offs, torch.int64, gpu_device)
    spec = _spec(ML, 8, 0, 1, 2)
    row_offs = torch.zeros(offs.size, dtype=torch.int64, device=d_ids.device)
    n = C.c_size_t()

    def sync(rows, mask, cap):
        return L.wp_rows_device(h, d_ids.data_ptr(), ids.size, d_offs.data_ptr(), offs.size - 1, C.byref(spec),
                                rows, mask, cap, row_offs.data_ptr(), C.byref(n), None)

    assert sync(None, None, 0) == WP_ERR_CAPACITY and n.value == need
    assert np.array_equal(row_offs.cpu().numpy(), exp_offs)
    rows = torch.full((need * ML,), 0x7EEEEEEE, dtype=torch.int32, device=d_ids.device)
    mask = torch.full((need * ML,), 0xEE, dtype=torch.uint8, device=d_ids.device)
    row_offs.zero_()
    assert sync(rows.data_ptr(), mask.data_ptr(), need - 1) == WP_ERR_CAPACITY and n.value == need
    torch.cuda.synchronize()
    assert np.array_equal(row_offs.cpu().numpy(), exp_offs)
    assert bool((rows == 0x7EEEEEEE).all()) and bool((mask == 0xEE).all())
    v.rows_device_async(d_ids, d_offs, rows[: (need - 1) * ML], row_offs, ML, 8, 0, 1, 2, d_mask=mask)
    torch.cuda.synchronize()
    assert int(row_offs[-1]) == UINT64_MAX_AS_INT64
    assert bool((rows == 0x7EEEEEEE).all()) and bool((mask == 0xEE).all())
    assert sync(rows.data_ptr(), mask.data_ptr(), need) == WP_OK and n.value == need
    torch.cuda.synchronize()
    assert np.array_equal(row_offs.cpu().numpy(), exp_offs)
    assert np.array_equal(rows.view(need, ML).cpu().numpy(), exp_rows)
    assert np.array_equal(mask.view(need, ML).cpu().numpy(), exp_mask)
    v.close()


@pytest.mark.gpu
@pytest.mark.parametrize("how", ["descending", "past_n_ids", "first_past_n_ids"])
def test_rows_device_malformed_offsets(gpu_device, how):
    """Offsets that descend or end past n_ids, in a middle block: WP_ERR_INVALID_ARG (sync); UINT64_MAX and no row
    or mask byte written (async).  A good call on the same handle afterwards is right."""
    import torch
    from wordpiece_b200 import Vocab, WordPieceError
    from wordpiece_b200._capi import WP_ERR_INVALID_ARG

    v = Vocab(["[UNK]", "a"], device=gpu_device)
    rng = np.random.default_rng(10)
    ids, offs = texts_to_column(_random_texts(rng, 20, 3 * BLOCK))
    bad = offs.copy()
    if how == "descending":
        bad[BLOCK + 5] = bad[BLOCK + 4] - 1
    elif how == "past_n_ids":
        bad[-1] = ids.size + 1
    else:
        bad[0] = ids.size + 1
    d_ids, d_bad = _to(ids, torch.int32, gpu_device), _to(bad, torch.int64, gpu_device)
    with pytest.raises(WordPieceError) as e:
        v.rows_device(d_ids, d_bad, 24, 4, cls_id=1, sep_id=2)
    assert e.value.status == WP_ERR_INVALID_ARG
    rows = torch.full((ids.size * 24,), 0x7EEEEEEE, dtype=torch.int32, device=d_ids.device)
    mask = torch.full((ids.size * 24,), 0xEE, dtype=torch.uint8, device=d_ids.device)
    row_offs = torch.zeros(offs.size, dtype=torch.int64, device=d_ids.device)
    v.rows_device_async(d_ids, d_bad, rows, row_offs, 24, 4, 0, 1, 2, d_mask=mask)
    torch.cuda.synchronize()
    assert int(row_offs[-1]) == UINT64_MAX_AS_INT64
    assert bool((rows == 0x7EEEEEEE).all()) and bool((mask == 0xEE).all())
    _check(v, ids, offs, gpu_device, "after malformed", 24, 4, cls_id=1, sep_id=2)
    v.close()


@pytest.mark.gpu
def test_rows_device_without_mask_and_without_texts(gpu_device):
    import torch
    from wordpiece_b200 import Vocab, kernel_launch_count

    v = Vocab(["[UNK]", "a"], device=gpu_device)
    rng = np.random.default_rng(11)
    ids, offs = texts_to_column(_random_texts(rng, 10, 500))
    exp_rows, _, exp_offs = model(ids, offs, 12, 5, 0, 1, 2)
    d_ids, d_offs = _to(ids, torch.int32, gpu_device), _to(offs, torch.int64, gpu_device)
    d_rows, d_mask, d_row_offs, n = v.rows_device(d_ids, d_offs, 12, 5, cls_id=1, sep_id=2, mask=False)
    assert d_mask is None and n == exp_rows.shape[0]
    assert np.array_equal(d_rows.cpu().numpy(), exp_rows) and np.array_equal(d_row_offs.cpu().numpy(), exp_offs)
    # n_texts == 0: one offset, 0, and no kernel
    launches = kernel_launch_count()
    d_rows, d_mask, d_row_offs, n = v.rows_device(d_ids, _to(np.array([3], np.int64), torch.int64, gpu_device), 12)
    assert n == 0 and d_row_offs.tolist() == [0] and tuple(d_rows.shape) == (0, 12) and tuple(d_mask.shape) == (0, 12)
    ro = torch.full((1,), 77, dtype=torch.int64, device=d_ids.device)
    v.rows_device_async(d_ids, _to(np.array([0], np.int64), torch.int64, gpu_device), d_rows, ro, 12)
    torch.cuda.synchronize()
    assert ro.tolist() == [0] and kernel_launch_count() == launches
    v.close()


@pytest.mark.gpu
def test_rows_device_after_async_encode_on_another_stream(gpu_device):
    """encode_batch_device_async on stream A, then rows_device_async of its ids on stream B with no synchronisation
    by the caller: the handle orders the two (the rows call waits for the encode), and the rows are right."""
    import torch
    from wordpiece_b200 import Vocab, synth

    g = synth.generator("en")
    text = g.generate(1 << 20, seed=12).tobytes()
    rng = np.random.default_rng(12)
    bounds = np.concatenate([[0], np.sort(rng.integers(0, len(text), 300)), [len(text)]]).astype(np.int64)
    o = Oracle(g.spec.vocab)
    ids, offs = texts_to_column([o.encode(text[bounds[i]:bounds[i + 1]]) for i in range(bounds.size - 1)])
    exp_rows, exp_mask, exp_offs = model(ids, offs, 256, 128, 0, 2, 3)
    v = Vocab(g.spec.vocab, device=gpu_device)
    dev = _dev(gpu_device)
    sa, sb = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    d_chars, d_offsets = _to(np.frombuffer(bytearray(text), np.uint8), torch.uint8, gpu_device), _to(bounds, torch.int64, gpu_device)
    d_ids = torch.empty(len(text), dtype=torch.int32, device=dev)
    d_id_offs = torch.empty(bounds.size, dtype=torch.int64, device=dev)
    cap = exp_rows.shape[0] + 10
    rows = torch.empty(cap * 256, dtype=torch.int32, device=dev)
    mask = torch.empty(cap * 256, dtype=torch.uint8, device=dev)
    row_offs = torch.empty(bounds.size, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    v.encode_batch_device_async(d_chars, d_offsets, d_ids, d_id_offs, stream=sa.cuda_stream)
    # (the ids tensor is the full-capacity buffer: the rows call reads only what the offsets name)
    v.rows_device_async(d_ids, d_id_offs, rows, row_offs, 256, 128, 0, 2, 3, d_mask=mask, stream=sb.cuda_stream)
    torch.cuda.synchronize()
    n = exp_rows.shape[0]
    assert np.array_equal(row_offs.cpu().numpy(), exp_offs)
    assert np.array_equal(rows[: n * 256].view(n, 256).cpu().numpy(), exp_rows)
    assert np.array_equal(mask[: n * 256].view(n, 256).cpu().numpy(), exp_mask)
    v.close()


@pytest.mark.gpu
def test_rows_device_output_past_4gib(gpu_device):
    """2.2 M rows of L = 512 (4.5 GB of ids) from windows over a few long texts: the row offsets exactly, the rows
    around the 4 GiB byte boundary of d_rows, the last rows and sampled rows against the model."""
    import torch
    from wordpiece_b200 import Vocab

    v = Vocab(["[UNK]", "a"], device=gpu_device)
    rng = np.random.default_rng(13)
    L, stride = 512, 2
    ids, offs = texts_to_column([rng.integers(-1, 30000, n).astype(np.int32) for n in (1_000_000, 7, 1_500_000, 3333, 2_000_000)])
    d_ids, d_offs = _to(ids, torch.int32, gpu_device), _to(offs, torch.int64, gpu_device)
    d_rows, d_mask, d_row_offs, n = v.rows_device(d_ids, d_offs, L, stride=stride, pad_id=0, cls_id=101, sep_id=102)
    _, _, exp_offs = model(ids, offs, L, stride, 0, 101, 102, rows=[])
    assert n == exp_offs[-1] and n * L * 4 > (1 << 32) and np.array_equal(d_row_offs.cpu().numpy(), exp_offs)
    r4g = (1 << 32) // (L * 4)
    sample = np.unique(np.concatenate([np.arange(0, 50), np.arange(r4g - 100, r4g + 100), np.arange(n - 50, n),
                                       rng.integers(0, n, 5000)]))
    exp_rows, exp_mask, _ = model(ids, offs, L, stride, 0, 101, 102, rows=sample)
    idx = torch.from_numpy(sample).to(d_rows.device)
    assert np.array_equal(d_rows[idx].cpu().numpy(), exp_rows)
    assert np.array_equal(d_mask[idx].cpu().numpy(), exp_mask)
    del d_rows, d_mask
    v.close()
    torch.cuda.empty_cache()
