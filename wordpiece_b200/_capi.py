"""ctypes binding of include/wordpiece_b200.h.  No tokenisation logic lives here."""
from __future__ import annotations

import ctypes as C
import hashlib
import mmap
import os
import threading
from dataclasses import dataclass
from typing import Iterable, List, Optional, Sequence, Union

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# (WORDPIECE_B200_LIB: another build of the same library, e.g. a tuning variant from `make variant`)
LIB_PATH = os.environ.get("WORDPIECE_B200_LIB") or os.path.join(_HERE, "lib", "libwordpiece_b200.so")

WP_OK = 0
WP_ERR_INVALID_ARG = 1
WP_ERR_EMPTY_VOCAB_WORD = 2
WP_ERR_CUDA = 3
WP_ERR_NO_DEVICE = 4
WP_ERR_CAPACITY = 5
WP_ERR_IO = 6
WP_ERR_NOMEM = 7
WP_ERR_ID_RANGE = 8

KIND_PREFIX = 0
KIND_SUFFIX = 1


class WordPieceError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(message)
        self.status = status


class _StatsStruct(C.Structure):
    _fields_ = [
        ("n_bytes", C.c_uint64),
        ("n_ids", C.c_uint64),
        ("n_tiles", C.c_uint64),
        ("dirty_tiles", C.c_uint64),
        ("long_segments", C.c_uint64),
        ("kernel_launches", C.c_uint64),
        ("memo_hits", C.c_uint64),
    ]


WP_ROWS_CLS = 1
WP_ROWS_SEP = 2


class RowsSpec(C.Structure):
    """``wp_rows_spec``: row length, window stride (0 = truncate), pad / cls / sep ids, WP_ROWS_* flags."""

    _fields_ = [
        ("max_len", C.c_uint32),
        ("stride", C.c_uint32),
        ("pad_id", C.c_int32),
        ("cls_id", C.c_int32),
        ("sep_id", C.c_int32),
        ("flags", C.c_uint32),
    ]

    @classmethod
    def make(cls, max_len, stride=0, pad_id=0, cls_id=None, sep_id=None) -> "RowsSpec":
        flags = (WP_ROWS_CLS if cls_id is not None else 0) | (WP_ROWS_SEP if sep_id is not None else 0)
        return cls(max_len, stride, pad_id, 0 if cls_id is None else cls_id, 0 if sep_id is None else sep_id, flags)


@dataclass
class Stats:
    n_bytes: int
    n_ids: int
    n_tiles: int
    dirty_tiles: int
    long_segments: int
    kernel_launches: int
    memo_hits: int = 0


# every symbol include/wordpiece_b200.h declares (tests check that all are exported)
EXPORTED_SYMBOLS = [
    "wp_last_error",
    "wp_kernel_launch_count",
    "wp_tile_bytes",
    "wp_vocab_create",
    "wp_vocab_create_from_file",
    "wp_vocab_destroy",
    "wp_vocab_size",
    "wp_vocab_unk_id",
    "wp_vocab_max_len",
    "wp_vocab_device",
    "wp_vocab_token_flags",
    "wp_vocab_device_bytes",
    "wp_encode",
    "wp_encode_text",
    "wp_encode_into",
    "wp_encode_device",
    "wp_encode_device_async",
    "wp_plan_shards",
    "wp_next_safe_cut",
    "wp_encode_sharded",
    "wp_encode_sharded_gather",
    "wp_encode_batch",
    "wp_encode_batch_device",
    "wp_encode_batch_device_async",
    "wp_last_stats",
    "wp_set_kernel_timing",
    "wp_last_kernel_ms",
    "wp_decode",
    "wp_decode_device",
    "wp_decode_device_async",
    "wp_rows_device",
    "wp_rows_device_async",
    "wp_free",
    "wp_debug_longest_match",
    "wp_debug_table_slots",
    "wp_debug_table_nodes",
    "wp_debug_long_tokens",
    "wp_debug_displaced_singles",
    "wp_debug_word_slots",
    "wp_debug_static_words",
    "wp_debug_word_lookup",
    "wp_debug_kernel_geometry",
    "wp_debug_plan_chunks",
    "wp_debug_stage",
]

_lib = None


def load_library() -> C.CDLL:
    """Load libwordpiece_b200.so; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise WordPieceError(
            WP_ERR_NO_DEVICE,
            f"{LIB_PATH} is missing: build it with `make -C wordpiece_b200/csrc` "
            "(or `python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback.",
        )
    L = C.CDLL(LIB_PATH)
    vp, sz, i32p = C.c_void_p, C.c_size_t, C.POINTER(C.c_int32)
    L.wp_last_error.restype = C.c_char_p
    L.wp_kernel_launch_count.restype = C.c_uint64
    L.wp_tile_bytes.restype = C.c_uint32
    L.wp_vocab_create.argtypes = [C.POINTER(C.c_char_p), C.POINTER(sz), sz, C.c_int, C.POINTER(vp)]
    L.wp_vocab_create.restype = C.c_int
    L.wp_vocab_create_from_file.argtypes = [C.c_char_p, C.c_int, C.POINTER(vp)]
    L.wp_vocab_create_from_file.restype = C.c_int
    L.wp_vocab_destroy.argtypes = [vp]
    L.wp_vocab_destroy.restype = None
    L.wp_vocab_size.argtypes = [vp]
    L.wp_vocab_size.restype = sz
    L.wp_vocab_unk_id.argtypes = [vp]
    L.wp_vocab_unk_id.restype = C.c_int32
    L.wp_vocab_max_len.argtypes = [vp]
    L.wp_vocab_max_len.restype = sz
    L.wp_vocab_device.argtypes = [vp]
    L.wp_vocab_device.restype = C.c_int
    L.wp_vocab_token_flags.argtypes = [vp, sz]
    L.wp_vocab_token_flags.restype = C.c_int
    L.wp_vocab_device_bytes.argtypes = [vp]
    L.wp_vocab_device_bytes.restype = sz
    L.wp_encode.argtypes = [vp, vp, sz, C.POINTER(i32p), C.POINTER(sz)]
    L.wp_encode.restype = C.c_int
    L.wp_encode_into.argtypes = [vp, vp, sz, vp, sz, C.POINTER(sz)]
    L.wp_encode_into.restype = C.c_int
    L.wp_encode_device.argtypes = [vp, vp, sz, vp, sz, C.POINTER(sz), vp]
    L.wp_encode_device.restype = C.c_int
    if hasattr(L, "wp_encode_batch"):  # (an older build loaded through WORDPIECE_B200_LIB for a bisect may lack it)
        L.wp_encode_batch.argtypes = [vp, vp, vp, sz, vp, sz, vp, C.POINTER(sz)]
        L.wp_encode_batch.restype = C.c_int
    L.wp_encode_device_async.argtypes = [vp, vp, sz, vp, sz, vp, vp]
    L.wp_encode_device_async.restype = C.c_int
    if hasattr(L, "wp_encode_batch_device"):  # (as wp_encode_batch: an older build may lack it)
        L.wp_encode_batch_device.argtypes = [vp, vp, sz, vp, sz, vp, sz, vp, C.POINTER(sz), vp]
        L.wp_encode_batch_device.restype = C.c_int
        L.wp_encode_batch_device_async.argtypes = [vp, vp, sz, vp, sz, vp, sz, vp, vp]
        L.wp_encode_batch_device_async.restype = C.c_int
    L.wp_plan_shards.argtypes = [vp, sz, sz, C.POINTER(sz)]
    L.wp_plan_shards.restype = sz
    L.wp_next_safe_cut.argtypes = [vp, sz, sz]
    L.wp_next_safe_cut.restype = sz
    L.wp_encode_sharded.argtypes = [vp, sz, vp, sz, vp, sz, C.POINTER(sz), vp]
    L.wp_encode_sharded.restype = C.c_int
    L.wp_encode_sharded_gather.argtypes = [vp, sz, vp, sz, sz, vp, sz, C.POINTER(sz), vp, C.POINTER(C.c_float)]
    L.wp_encode_sharded_gather.restype = C.c_int
    L.wp_last_stats.argtypes = [vp, C.POINTER(_StatsStruct)]
    L.wp_last_stats.restype = C.c_int
    L.wp_set_kernel_timing.argtypes = [vp, C.c_int]
    L.wp_encode_text.argtypes = [vp, vp, sz, C.POINTER(vp), C.POINTER(sz), C.POINTER(sz)]
    L.wp_encode_text.restype = C.c_int
    L.wp_set_kernel_timing.restype = C.c_int
    L.wp_last_kernel_ms.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_uint32)]
    L.wp_last_kernel_ms.restype = C.c_int
    L.wp_decode.argtypes = [vp, vp, sz, C.POINTER(vp), C.POINTER(vp), C.POINTER(sz), C.POINTER(sz)]
    L.wp_decode.restype = C.c_int
    if hasattr(L, "wp_decode_device"):  # (as wp_encode_batch: an older build may lack it)
        L.wp_decode_device.argtypes = [vp, vp, sz, vp, sz, vp, C.POINTER(sz), C.POINTER(sz), vp]
        L.wp_decode_device.restype = C.c_int
        L.wp_decode_device_async.argtypes = [vp, vp, sz, vp, sz, vp, vp]
        L.wp_decode_device_async.restype = C.c_int
    if hasattr(L, "wp_rows_device"):
        L.wp_rows_device.argtypes = [vp, vp, sz, vp, sz, C.POINTER(RowsSpec), vp, vp, sz, vp, C.POINTER(sz), vp]
        L.wp_rows_device.restype = C.c_int
        L.wp_rows_device_async.argtypes = [vp, vp, sz, vp, sz, C.POINTER(RowsSpec), vp, vp, sz, vp, vp]
        L.wp_rows_device_async.restype = C.c_int
    L.wp_free.argtypes = [vp]
    L.wp_free.restype = None
    L.wp_debug_longest_match.argtypes = [vp, C.c_char_p, sz, C.c_int, C.POINTER(C.c_uint32), C.POINTER(C.c_int32)]
    L.wp_debug_longest_match.restype = C.c_int
    for f in ("wp_debug_table_slots", "wp_debug_table_nodes", "wp_debug_long_tokens", "wp_debug_word_slots",
              "wp_debug_static_words"):
        getattr(L, f).argtypes = [vp]
        getattr(L, f).restype = sz
    L.wp_debug_plan_chunks.argtypes = [vp, sz, sz, C.POINTER(sz), sz]
    L.wp_debug_plan_chunks.restype = sz
    L.wp_debug_stage.argtypes = [C.POINTER(C.c_char_p), C.POINTER(sz), sz, vp, sz, C.c_int]
    L.wp_debug_stage.restype = sz
    L.wp_debug_displaced_singles.argtypes = [vp, C.c_uint32, C.POINTER(C.c_uint32), sz]
    L.wp_debug_displaced_singles.restype = sz
    L.wp_debug_word_lookup.argtypes = [vp, C.c_char_p, sz, C.POINTER(C.c_int32), C.POINTER(C.c_uint32)]
    L.wp_debug_word_lookup.restype = C.c_uint32
    L.wp_debug_kernel_geometry.argtypes = [C.POINTER(C.c_uint32), sz]
    L.wp_debug_kernel_geometry.restype = sz
    _lib = L
    return L


def _check(status: int) -> None:
    if status != WP_OK:
        msg = load_library().wp_last_error()
        raise WordPieceError(status, (msg or b"").decode("utf-8", "replace") or f"wp_status {status}")


def kernel_launch_count() -> int:
    return int(load_library().wp_kernel_launch_count())


def tile_bytes() -> int:
    return int(load_library().wp_tile_bytes())


KERNEL_GEOMETRY_FIELDS = ("tile", "long_segment_bytes", "seg_cap", "scatter_segs", "scatter_stage", "scatter_big",
                          "mixed_max_big", "long_block", "word_key_bytes", "word_max_ids", "seg_slow_count_max",
                          "inline_ids")


def kernel_geometry() -> dict:
    """The limits the kernels were compiled with (``wp_debug_kernel_geometry``, test hook, no device):
    ``KERNEL_GEOMETRY_FIELDS`` -> value."""
    L = load_library()
    n = int(L.wp_debug_kernel_geometry(None, 0))
    buf = (C.c_uint32 * n)()
    L.wp_debug_kernel_geometry(buf, n)
    assert n == len(KERNEL_GEOMETRY_FIELDS), n
    return {k: int(buf[i]) for i, k in enumerate(KERNEL_GEOMETRY_FIELDS)}


def _as_bytes(x) -> bytes:
    if isinstance(x, str):
        return x.encode("utf-8")
    if isinstance(x, np.ndarray):
        return x.tobytes()
    return bytes(x)


def _buffer_address(buf) -> tuple:
    """(address, nbytes, keepalive) of a bytes-like / numpy uint8 / mmap object, without copying."""
    if isinstance(buf, np.ndarray):
        a = np.ascontiguousarray(buf).view(np.uint8)
        return a.ctypes.data, a.size, a
    if isinstance(buf, bytes):
        return C.cast(C.c_char_p(buf), C.c_void_p).value or 0, len(buf), buf
    a = np.frombuffer(buf, dtype=np.uint8)
    return a.ctypes.data, a.size, a


class Vocab:
    """A vocabulary resident on one GPU (``wp_vocab`` handle).

    ``tokens[i]`` is the token with id ``i`` (str or bytes), as in
    ``utils::parseVocab`` (utils.cpp:108-121).  ``device=-1`` builds a host-only
    handle (queries and decode only).
    """

    def __init__(self, tokens: Sequence[Union[str, bytes]], device: int = 0):
        L = load_library()
        toks = [_as_bytes(t) for t in tokens]
        n = len(toks)
        arr = (C.c_char_p * max(n, 1))(*toks)
        lens = (C.c_size_t * max(n, 1))(*[len(t) for t in toks])
        h = C.c_void_p()
        self._h = None
        _check(L.wp_vocab_create(arr, lens, n, device, C.byref(h)))
        self._h = h
        self._L = L

    @classmethod
    def from_file(cls, vocab_file: str, device: int = 0) -> "Vocab":
        L = load_library()
        h = C.c_void_p()
        _check(L.wp_vocab_create_from_file(os.fsencode(vocab_file), device, C.byref(h)))
        self = cls.__new__(cls)
        self._h = h
        self._L = L
        return self

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._L.wp_vocab_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self) -> int:
        return int(self._L.wp_vocab_size(self._h))

    @property
    def unk_id(self) -> int:
        return int(self._L.wp_vocab_unk_id(self._h))

    @property
    def max_len(self) -> int:
        return int(self._L.wp_vocab_max_len(self._h))

    @property
    def device(self) -> int:
        return int(self._L.wp_vocab_device(self._h))

    @property
    def device_bytes(self) -> int:
        return int(self._L.wp_vocab_device_bytes(self._h))

    def token_flags(self, index: int) -> int:
        return int(self._L.wp_vocab_token_flags(self._h, index))

    @property
    def table_info(self) -> dict:
        return {
            "slots": int(self._L.wp_debug_table_slots(self._h)),
            "nodes": int(self._L.wp_debug_table_nodes(self._h)),
            "long_tokens": int(self._L.wp_debug_long_tokens(self._h)),
            "word_slots": int(self._L.wp_debug_word_slots(self._h)),
            "static_words": int(self._L.wp_debug_static_words(self._h)),
        }

    def debug_displaced_singles(self, min_displacement: int = 1) -> list:
        """Code points of single-char word-initial tokens whose word-table slot lies at least
        ``min_displacement`` slots from its home slot (test hook)."""
        n = int(self._L.wp_debug_displaced_singles(self._h, min_displacement, None, 0))
        buf = (C.c_uint32 * max(n, 1))()
        self._L.wp_debug_displaced_singles(self._h, min_displacement, buf, n)
        return [int(buf[i]) for i in range(n)]

    def debug_word_lookup(self, word: bytes):
        """Host mirror of K1's whole-segment lookup in the static word table: (ids, displacement) or None."""
        ids = (C.c_int32 * 11)()
        disp = C.c_uint32()
        n = int(self._L.wp_debug_word_lookup(self._h, word, len(word), ids, C.byref(disp)))
        return ([int(ids[i]) for i in range(n)], int(disp.value)) if n else None

    def debug_longest_match(self, text: bytes, kind: int):
        ln, tid = C.c_uint32(), C.c_int32()
        _check(self._L.wp_debug_longest_match(self._h, text, len(text), kind, C.byref(ln), C.byref(tid)))
        return int(ln.value), int(tid.value)

    # ---- encode ---------------------------------------------------------
    def encode(self, text) -> np.ndarray:
        """Host text (str / bytes / uint8 array / mmap) -> int32 ids (numpy).  ``wp_encode``."""
        if isinstance(text, str):
            text = text.encode("utf-8")
        addr, n, keep = _buffer_address(text)
        ids = C.POINTER(C.c_int32)()
        cnt = C.c_size_t()
        _check(self._L.wp_encode(self._h, addr, n, C.byref(ids), C.byref(cnt)))
        del keep
        if cnt.value == 0:
            if ids:
                self._L.wp_free(ids)
            return np.zeros(0, np.int32)
        out = np.ctypeslib.as_array(ids, shape=(cnt.value,)).copy()
        self._L.wp_free(ids)
        return out

    def encode_text(self, text) -> bytes:
        """Host text -> the ids as decimal text ``b"id id id "`` (formatted on the device).  ``wp_encode_text``."""
        addr, n, keep = _buffer_address(text)
        out, out_len, cnt = C.c_void_p(), C.c_size_t(), C.c_size_t()
        _check(self._L.wp_encode_text(self._h, addr, n, C.byref(out), C.byref(out_len), C.byref(cnt)))
        del keep
        try:
            return C.string_at(out.value, out_len.value)
        finally:
            self._L.wp_free(out)

    def encode_into(self, text, out: np.ndarray) -> int:
        """Host text -> caller's int32 numpy buffer; returns the id count.  ``wp_encode_into``."""
        assert out.dtype == np.int32 and out.flags.c_contiguous
        addr, n, keep = _buffer_address(text)
        cnt = C.c_size_t()
        _check(self._L.wp_encode_into(self._h, addr, n, out.ctypes.data, out.size, C.byref(cnt)))
        del keep
        return int(cnt.value)

    @staticmethod
    def batch_pointers(texts):
        """The C arguments of a batch (pointer and length arrays), built once for repeated calls on the same
        texts: (ptrs, lens, n, total_bytes, keepalive)."""
        bufs = [t.encode("utf-8") if isinstance(t, str) else t for t in texts]
        n = len(bufs)
        keep = []
        ptrs = (C.c_void_p * max(n, 1))()
        lens = (C.c_size_t * max(n, 1))()
        total = 0
        for i, b in enumerate(bufs):
            addr, ln, k = _buffer_address(b)
            keep.append(k)
            ptrs[i] = addr
            lens[i] = ln
            total += ln
        return ptrs, lens, n, total, keep

    def encode_batch(self, texts, out: Optional[np.ndarray] = None, offsets: Optional[np.ndarray] = None, prepared=None):
        """Many host texts in one call -> (ids, offsets): ids of text i are ``ids[offsets[i]:offsets[i + 1]]``,
        each text encoded exactly as ``encode`` would encode it alone.  ``wp_encode_batch``.  ``out`` may be a
        preallocated int32 buffer (pinned memory is fastest); otherwise one id per byte is allocated.
        ``prepared`` = the result of ``batch_pointers(texts)`` (skips the per-text Python work)."""
        ptrs, lens, n, total, keep = prepared if prepared is not None else self.batch_pointers(texts)
        if out is None:
            out = np.empty(max(total, 1), np.int32)
        if offsets is None:
            offsets = np.zeros(n + 1, np.uint64)
        assert out.dtype == np.int32 and out.flags.c_contiguous
        assert offsets.dtype == np.uint64 and offsets.size >= n + 1 and offsets.flags.c_contiguous
        cnt = C.c_size_t()
        _check(self._L.wp_encode_batch(self._h, ptrs, lens, n, out.ctypes.data, out.size, offsets.ctypes.data,
                                       C.byref(cnt)))
        del keep
        return out[: int(cnt.value)], offsets[: n + 1]

    def encode_device(self, d_text, d_ids=None, stream=None):
        """Device text (torch uint8 CUDA tensor) -> (torch int32 CUDA tensor of ids, count).

        ``wp_encode_device``.  ``d_ids`` may be a preallocated int32 tensor (capacity = numel);
        otherwise one id per byte is allocated (always enough).  Synchronises the stream.
        """
        import torch

        assert d_text.is_cuda and d_text.dtype == torch.uint8 and d_text.is_contiguous()
        n = d_text.numel()
        if d_ids is None:
            d_ids = torch.empty(max(n, 1), dtype=torch.int32, device=d_text.device)
        assert d_ids.is_cuda and d_ids.dtype == torch.int32 and d_ids.is_contiguous()
        if stream is None:
            stream = torch.cuda.current_stream(d_text.device).cuda_stream
        cnt = C.c_size_t()
        st = self._L.wp_encode_device(self._h, d_text.data_ptr(), n, d_ids.data_ptr(), d_ids.numel(), C.byref(cnt),
                                      stream)
        _check(st)
        return d_ids, int(cnt.value)

    def encode_device_async(self, d_text, d_ids, d_count, stream=None) -> None:
        """Fully asynchronous variant: count lands in the int64 CUDA tensor ``d_count`` (1 element)."""
        import torch

        assert d_text.is_cuda and d_text.dtype == torch.uint8 and d_text.is_contiguous()
        assert d_ids.is_cuda and d_ids.dtype == torch.int32 and d_ids.is_contiguous()
        assert d_count.is_cuda and d_count.dtype == torch.int64 and d_count.numel() >= 1
        if stream is None:
            stream = torch.cuda.current_stream(d_text.device).cuda_stream
        _check(self._L.wp_encode_device_async(self._h, d_text.data_ptr(), d_text.numel(), d_ids.data_ptr(),
                                              d_ids.numel(), d_count.data_ptr(), stream))

    @staticmethod
    def _column(d_chars, d_offsets, d_ids, d_id_offsets):
        import torch

        assert d_chars.is_cuda and d_chars.dtype == torch.uint8 and d_chars.dim() == 1 and d_chars.is_contiguous()
        assert d_offsets.is_cuda and d_offsets.dtype == torch.int64 and d_offsets.dim() == 1 and d_offsets.is_contiguous()
        assert d_offsets.numel() >= 1, "a column of n texts has n + 1 offsets"
        n_texts = d_offsets.numel() - 1
        if d_ids is None:
            d_ids = torch.empty(max(d_chars.numel(), 1), dtype=torch.int32, device=d_chars.device)
        if d_id_offsets is None:
            d_id_offsets = torch.empty(n_texts + 1, dtype=torch.int64, device=d_chars.device)
        assert d_ids.is_cuda and d_ids.dtype == torch.int32 and d_ids.is_contiguous()
        assert d_id_offsets.is_cuda and d_id_offsets.dtype == torch.int64 and d_id_offsets.is_contiguous()
        assert d_id_offsets.numel() >= n_texts + 1
        return n_texts, d_ids, d_id_offsets

    def encode_batch_device(self, d_chars, d_offsets, d_ids=None, d_id_offsets=None, stream=None):
        """Device string column -> (d_ids, d_id_offsets, n_ids).  ``wp_encode_batch_device``.

        ``d_chars`` is a torch uint8 CUDA tensor, ``d_offsets`` an int64 CUDA tensor of n + 1 entries (Arrow
        layout: text i is ``d_chars[d_offsets[i]:d_offsets[i + 1]]``, ``d_offsets[0]`` need not be 0).  The ids of
        text i are ``d_ids[d_id_offsets[i]:d_id_offsets[i + 1]]`` (int64 CUDA tensor of n + 1 entries), each text
        encoded exactly as ``encode`` would encode it alone.  ``d_ids`` may be a preallocated int32 tensor; otherwise
        one id per char is allocated (always enough).  Synchronises the stream.
        """
        import torch

        n_texts, d_ids, d_id_offsets = self._column(d_chars, d_offsets, d_ids, d_id_offsets)
        if stream is None:
            stream = torch.cuda.current_stream(d_chars.device).cuda_stream
        cnt = C.c_size_t()
        _check(self._L.wp_encode_batch_device(self._h, d_chars.data_ptr(), d_chars.numel(), d_offsets.data_ptr(), n_texts,
                                              d_ids.data_ptr(), d_ids.numel(), d_id_offsets.data_ptr(), C.byref(cnt),
                                              stream))
        return d_ids, d_id_offsets, int(cnt.value)

    def encode_batch_device_async(self, d_chars, d_offsets, d_ids, d_id_offsets, stream=None) -> None:
        """Fully asynchronous variant of ``encode_batch_device``: the total lands in ``d_id_offsets[n]``, which
        reads -1 (UINT64_MAX) if the ids are void or the column is malformed; then repeat the call through
        ``encode_batch_device``.  ``wp_encode_batch_device_async``."""
        import torch

        n_texts, d_ids, d_id_offsets = self._column(d_chars, d_offsets, d_ids, d_id_offsets)
        if stream is None:
            stream = torch.cuda.current_stream(d_chars.device).cuda_stream
        _check(self._L.wp_encode_batch_device_async(self._h, d_chars.data_ptr(), d_chars.numel(), d_offsets.data_ptr(),
                                                    n_texts, d_ids.data_ptr(), d_ids.numel(), d_id_offsets.data_ptr(),
                                                    stream))

    def set_kernel_timing(self, enabled: bool) -> None:
        _check(self._L.wp_set_kernel_timing(self._h, 1 if enabled else 0))

    def last_kernel_ms(self):
        """(ms of K1 split, K2 match, K3 scatter summed over the last call's ranges, number of ranges)."""
        ms = (C.c_float * 3)()
        n = C.c_uint32()
        _check(self._L.wp_last_kernel_ms(self._h, ms, C.byref(n)))
        return [float(ms[0]), float(ms[1]), float(ms[2])], int(n.value)

    def stats(self) -> Stats:
        s = _StatsStruct()
        _check(self._L.wp_last_stats(self._h, C.byref(s)))
        return Stats(s.n_bytes, s.n_ids, s.n_tiles, s.dirty_tiles, s.long_segments, s.kernel_launches, s.memo_hits)

    # ---- decode ---------------------------------------------------------
    def decode(self, ids: Iterable[int]) -> List[bytes]:
        """``word_piece::fast::decode`` (fast.cpp:165-187) -> list of token byte strings."""
        a = np.ascontiguousarray(np.asarray(list(ids) if not isinstance(ids, np.ndarray) else ids, dtype=np.int32))
        buf, offs = C.c_void_p(), C.c_void_p()
        n, skipped = C.c_size_t(), C.c_size_t()
        _check(self._L.wp_decode(self._h, a.ctypes.data, a.size, C.byref(buf), C.byref(offs), C.byref(n),
                                 C.byref(skipped)))
        o = np.ctypeslib.as_array(C.cast(offs, C.POINTER(C.c_size_t)), shape=(n.value + 1,)).copy()
        raw = C.string_at(buf, int(o[-1]))
        self._L.wp_free(buf)
        self._L.wp_free(offs)
        return [raw[int(o[i]):int(o[i + 1])] for i in range(n.value)]

    @staticmethod
    def _decode_column(d_ids, d_chars, d_char_offsets):
        import torch

        assert d_ids.is_cuda and d_ids.dtype == torch.int32 and d_ids.dim() == 1 and d_ids.is_contiguous()
        n_ids = d_ids.numel()
        if d_char_offsets is None:
            d_char_offsets = torch.empty(n_ids + 1, dtype=torch.int64, device=d_ids.device)
        assert d_char_offsets.is_cuda and d_char_offsets.dtype == torch.int64 and d_char_offsets.is_contiguous()
        assert d_char_offsets.numel() >= n_ids + 1, "n ids have n + 1 char offsets"
        if d_chars is not None:
            assert d_chars.is_cuda and d_chars.dtype == torch.uint8 and d_chars.dim() == 1 and d_chars.is_contiguous()
        return n_ids, d_char_offsets

    def decode_device(self, d_ids, d_chars=None, d_char_offsets=None, stream=None):
        """Device ids (torch int32 CUDA tensor) -> (d_chars, d_char_offsets, n_chars, n_skipped).  ``wp_decode_device``.

        Entry i, ``d_chars[d_char_offsets[i]:d_char_offsets[i + 1]]``, is what ``decode`` gives id i, or empty where
        ``decode`` skips the id: one entry per id, so a batch's id offsets index the entries directly.  Dropping the
        empty entries gives ``decode(ids)``.  ``d_chars`` may be a preallocated uint8 tensor (capacity = numel);
        otherwise the call asks for the size first and allocates exactly ``n_chars``.  Synchronises the stream."""
        import torch

        n_ids, d_char_offsets = self._decode_column(d_ids, d_chars, d_char_offsets)
        if stream is None:
            stream = torch.cuda.current_stream(d_ids.device).cuda_stream
        cnt, skipped = C.c_size_t(), C.c_size_t()

        def call(chars):
            return self._L.wp_decode_device(self._h, d_ids.data_ptr(), n_ids, chars.data_ptr() if chars is not None else None,
                                            chars.numel() if chars is not None else 0, d_char_offsets.data_ptr(),
                                            C.byref(cnt), C.byref(skipped), stream)

        st = call(d_chars)
        if d_chars is None:
            if st == WP_ERR_CAPACITY or st == WP_OK:  # (the size query; with 0 bytes needed it was the whole call)
                d_chars = torch.empty(cnt.value, dtype=torch.uint8, device=d_ids.device)
                if st == WP_ERR_CAPACITY:
                    st = call(d_chars)
        _check(st)
        return d_chars, d_char_offsets, int(cnt.value), int(skipped.value)

    def decode_device_async(self, d_ids, d_chars, d_char_offsets, stream=None) -> None:
        """Fully asynchronous variant of ``decode_device``: the total lands in ``d_char_offsets[n]``, which reads -1
        (UINT64_MAX) if an id equals the vocabulary size or ``d_chars`` is too small; then repeat the call through
        ``decode_device`` for the status.  ``wp_decode_device_async``."""
        import torch

        n_ids, d_char_offsets = self._decode_column(d_ids, d_chars, d_char_offsets)
        if stream is None:
            stream = torch.cuda.current_stream(d_ids.device).cuda_stream
        _check(self._L.wp_decode_device_async(self._h, d_ids.data_ptr(), n_ids, d_chars.data_ptr(), d_chars.numel(),
                                              d_char_offsets.data_ptr(), stream))

    # ---- model-input rows ---------------------------------------------
    @staticmethod
    def _rows_args(d_ids, d_id_offsets, d_rows, d_mask, d_row_offsets, max_len):
        """(n_texts, row capacity, d_row_offsets) after checking the tensors; d_row_offsets allocated if None."""
        import torch

        assert d_ids.is_cuda and d_ids.dtype == torch.int32 and d_ids.dim() == 1 and d_ids.is_contiguous()
        assert d_id_offsets.is_cuda and d_id_offsets.dtype == torch.int64 and d_id_offsets.dim() == 1
        assert d_id_offsets.is_contiguous() and d_id_offsets.numel() >= 1, "n texts have n + 1 id offsets"
        n_texts = d_id_offsets.numel() - 1
        if d_row_offsets is None:
            d_row_offsets = torch.empty(n_texts + 1, dtype=torch.int64, device=d_ids.device)
        assert d_row_offsets.is_cuda and d_row_offsets.dtype == torch.int64 and d_row_offsets.is_contiguous()
        assert d_row_offsets.numel() >= n_texts + 1, "n texts have n + 1 row offsets"
        capacity = 0
        if d_rows is not None:
            assert d_rows.is_cuda and d_rows.dtype == torch.int32 and d_rows.is_contiguous()
            capacity = d_rows.numel() // max(max_len, 1)
        if d_mask is not None:
            assert d_mask.is_cuda and d_mask.dtype == torch.uint8 and d_mask.is_contiguous()
            assert d_mask.numel() >= capacity * max_len, "the mask holds as many rows as d_rows"
        return n_texts, capacity, d_row_offsets

    def rows_device(self, d_ids, d_id_offsets, max_len, stride=0, pad_id=0, cls_id=None, sep_id=None, mask=True,
                    d_rows=None, d_mask=None, stream=None):
        """Per-text ids in GPU memory -> fixed-length model-input rows.  ``wp_rows_device``.

        Text t's ids are ``d_ids[d_id_offsets[t]:d_id_offsets[t + 1]]`` (int32 and int64 CUDA tensors, e.g. what
        ``encode_batch_device`` returns).  Every row is ``max_len`` ids: ``[cls_id]? content [sep_id]? pad_id ...``
        (cls / sep present when given), content width W = max_len minus the specials.  ``stride`` 0 truncates each
        text to one row; 1 <= stride <= W cuts it into windows whose starts are ``stride`` ids apart (cuDF's meaning;
        HuggingFace's overlap is W - stride).  Returns ``(d_rows [n_rows, max_len] int32, d_mask [n_rows, max_len]
        uint8 or None, d_row_offsets int64 [n_texts + 1], n_rows)``; text t's rows are
        ``d_row_offsets[t]:d_row_offsets[t + 1]``.  ``d_rows`` / ``d_mask`` may be preallocated contiguous tensors
        (capacity = d_rows.numel() // max_len rows); otherwise the call asks for the row count first and allocates
        exactly.  ``mask=False`` writes no mask.  Synchronises the stream."""
        import torch

        if not mask:
            d_mask = None
        elif d_mask is None and d_rows is not None:
            d_mask = torch.empty(d_rows.numel() // max(max_len, 1) * max_len, dtype=torch.uint8, device=d_rows.device)
        n_texts, capacity, d_row_offsets = self._rows_args(d_ids, d_id_offsets, d_rows, d_mask, None, max_len)
        if stream is None:
            stream = torch.cuda.current_stream(d_ids.device).cuda_stream
        spec = RowsSpec.make(max_len, stride, pad_id, cls_id, sep_id)
        cnt = C.c_size_t()

        def call(rows, msk, cap):
            return self._L.wp_rows_device(self._h, d_ids.data_ptr(), d_ids.numel(), d_id_offsets.data_ptr(), n_texts,
                                          C.byref(spec), rows.data_ptr() if rows is not None else None,
                                          msk.data_ptr() if msk is not None else None, cap, d_row_offsets.data_ptr(),
                                          C.byref(cnt), stream)

        st = call(d_rows, d_mask, capacity)
        if d_rows is None and st in (WP_OK, WP_ERR_CAPACITY):  # the size query (with 0 rows it was the whole call)
            d_rows = torch.empty((cnt.value, max_len), dtype=torch.int32, device=d_ids.device)
            if mask and d_mask is None:
                d_mask = torch.empty((cnt.value, max_len), dtype=torch.uint8, device=d_ids.device)
            if st == WP_ERR_CAPACITY:
                st = call(d_rows, d_mask, cnt.value)
        _check(st)
        n_rows = int(cnt.value)
        d_rows = d_rows.view(-1)[: n_rows * max_len].view(n_rows, max_len)
        if d_mask is not None:
            d_mask = d_mask.view(-1)[: n_rows * max_len].view(n_rows, max_len)
        return d_rows, d_mask, d_row_offsets, n_rows

    def rows_device_async(self, d_ids, d_id_offsets, d_rows, d_row_offsets, max_len, stride=0, pad_id=0, cls_id=None,
                          sep_id=None, d_mask=None, stream=None) -> None:
        """Fully asynchronous variant of ``rows_device`` into preallocated tensors: the row total lands in
        ``d_row_offsets[n_texts]``, which reads -1 (UINT64_MAX) if the id offsets are malformed or ``d_rows`` is too
        small (then nothing is written to ``d_rows`` / ``d_mask``); repeat the call through ``rows_device`` for the
        status.  ``wp_rows_device_async``."""
        import torch

        n_texts, capacity, d_row_offsets = self._rows_args(d_ids, d_id_offsets, d_rows, d_mask, d_row_offsets, max_len)
        if stream is None:
            stream = torch.cuda.current_stream(d_ids.device).cuda_stream
        spec = RowsSpec.make(max_len, stride, pad_id, cls_id, sep_id)
        _check(self._L.wp_rows_device_async(self._h, d_ids.data_ptr(), d_ids.numel(), d_id_offsets.data_ptr(), n_texts,
                                            C.byref(spec), d_rows.data_ptr(), d_mask.data_ptr() if d_mask is not None else None,
                                            capacity, d_row_offsets.data_ptr(), stream))

    def encode_rows_device(self, d_chars, d_offsets, max_len, stride=0, pad_id=0, cls_id=None, sep_id=None, mask=True,
                           stream=None):
        """A string column in GPU memory -> model-input rows: ``encode_batch_device`` then ``rows_device`` (see
        both).  Returns ``(d_rows, d_mask, d_row_offsets, n_rows)``."""
        d_ids, d_id_offsets, n_ids = self.encode_batch_device(d_chars, d_offsets, stream=stream)
        return self.rows_device(d_ids[:n_ids], d_id_offsets, max_len, stride=stride, pad_id=pad_id, cls_id=cls_id,
                                sep_id=sep_id, mask=mask, stream=stream)


# ---- the reference's stateless entry points ---------------------------------

_cache: dict = {}
_cache_lock = threading.Lock()


def _default_device() -> int:
    return int(os.environ.get("WORDPIECE_B200_DEVICE", "0"))


def debug_plan_chunks(text: bytes, chunk: int) -> list:
    """Cut offsets of the host-buffer pipeline for `text` with `chunk`-byte chunks (test hook, no device)."""
    L = load_library()
    cap = len(text) // max(chunk // 16, 1) + 64
    buf = (C.c_size_t * cap)()
    n = int(L.wp_debug_plan_chunks(text, len(text), chunk, buf, cap))
    return [int(buf[i]) for i in range(min(n, cap))]


def debug_stage(texts: Sequence[bytes], mode: int) -> bytes:
    """The library's staging copies run on the host (test hook, no device): mode 0/1 = batch packer with ordinary /
    streaming stores, 2/3 = pooled copy of texts[0] ordinary / streamed."""
    L = load_library()
    n = len(texts)
    ptrs = (C.c_char_p * max(n, 1))(*texts)
    lens = (C.c_size_t * max(n, 1))(*[len(t) for t in texts])
    cap = sum(len(t) for t in texts) + n + 64
    out = C.create_string_buffer(cap)
    k = int(L.wp_debug_stage(ptrs, lens, n, out, cap, mode))
    return out.raw[:k]


def _cached_vocab(tokens: Sequence[Union[str, bytes]], device: Optional[int]) -> Vocab:
    dev = _default_device() if device is None else device
    # content key in one pass over the joined bytes (a per-token Python loop costs ~4 ms for a 29k vocabulary,
    # most of a 4 KiB call); the token count and the byte count keep differently split lists apart
    try:
        blob = b"\n".join(tokens)  # all bytes
    except TypeError:
        try:
            blob = "\n".join(tokens).encode("utf-8")  # all str
        except TypeError:
            blob = b"\n".join(_as_bytes(t) for t in tokens)
    if blob.count(b"\n") == len(tokens) - 1 or not tokens:
        # no token holds the separator, so the joined bytes determine the list; 128-bit digest of the content
        key = (dev, hashlib.blake2b(blob, digest_size=16).digest(), len(blob), len(tokens))
    else:
        key = (dev, tuple(_as_bytes(t) for t in tokens))  # a token with a newline inside: the exact list is the key
    with _cache_lock:
        v = _cache.get(key)
        if v is None:
            if len(_cache) >= 4:
                # (the evicted handle is closed when its last user drops it, not here: another thread may hold it)
                _cache.pop(next(iter(_cache)))
            v = Vocab(tokens, device=dev)
            _cache[key] = v
    return v


def _read_vocab_lines(vocab_file: str) -> List[bytes]:
    # std::getline semantics (utils.cpp:123-137): split at '\n'; no trailing empty token; '\r' stays
    with open(vocab_file, "rb") as f:
        data = f.read()
    lines = data.split(b"\n")
    if lines and lines[-1] == b"":
        lines.pop()
    return lines


def encode(text, vocab: Sequence[Union[str, bytes]], device: Optional[int] = None) -> np.ndarray:
    """``word_piece::fast::encode(text, vocab)`` (fast.cpp:154-157)."""
    return _cached_vocab(vocab, device).encode(text)


def encode_files(text_file: str, vocab_file: str, device: Optional[int] = None) -> np.ndarray:
    """``word_piece::fast::encode(text_file, vocab_file)`` (fast.cpp:159-163)."""
    v = _cached_vocab(_read_vocab_lines(vocab_file), device)
    if os.path.getsize(text_file) == 0:
        return np.zeros(0, np.int32)
    with open(text_file, "rb") as f, mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ) as m:
        a = np.frombuffer(m, dtype=np.uint8)
        try:
            return v.encode(a)
        finally:
            del a


def decode(vocab_file: str, ids: Iterable[int], device: Optional[int] = -1) -> List[bytes]:
    """``word_piece::fast::decode(vocab_file, ids)`` (fast.cpp:165-187)."""
    return _cached_vocab(_read_vocab_lines(vocab_file), device).decode(ids)


def _starts_with_space(b: bytes, pos: int, size_arg: int) -> bool:
    # utf8.cpp:92-96 via :54-90, with the reference's (pointer, remaining) arguments
    c = b[pos]
    if c < 0x80:
        return 0x09 <= c <= 0x0D or c == 0x20
    return size_arg >= 3 and b[pos:pos + 3] == b"\xe2\x96\x81"


def encode_external(text_file: str, vocab_file: str, out_file: str, memory_limit: int,
                    device: Optional[int] = None) -> None:
    """``word_piece::fast::encodeExternal`` (fast.cpp:189-220): batches of at most
    ``memory_limit // 2`` bytes, each extended until its last byte starts a space,
    ids appended to ``out_file`` as ``"id id id "``."""
    v = _cached_vocab(_read_vocab_lines(vocab_file), device)
    max_batch = memory_limit // 2
    size = os.path.getsize(text_file)
    with open(out_file, "wb") as fout:
        if size == 0:
            return
        with open(text_file, "rb") as f, mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ) as m:
            begin = 0
            while size > 0:
                if size > max_batch:
                    batch = max(max_batch, 1)
                    while batch < size and not _starts_with_space(m, begin + batch - 1, size - batch):
                        batch += 1
                else:
                    batch = size
                a = np.frombuffer(m, dtype=np.uint8, count=batch, offset=begin)
                fout.write(v.encode_text(a))
                del a
                begin += batch
                size -= batch
