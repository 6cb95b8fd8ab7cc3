"""wordpiece_b200 — B200-native fast WordPiece encoder (host-side Python mirror).

The product is ``wordpiece_b200/lib/libwordpiece_b200.so`` (hand-written sm_100a
CUDA behind a C ABI, ``include/wordpiece_b200.h``).  This package is the thin
ctypes layer tests and ``bench.py`` use; it mirrors the reference's entry points
(gleb-kov/wordpiece ``src/word_piece.hpp:25-34``):

===========================================  =====================================
reference (C++)                              here
===========================================  =====================================
``word_piece::fast::encode(text, vocab)``    :func:`encode`
``word_piece::fast::encode(tfile, vfile)``   :func:`encode_files`
``word_piece::fast::decode(vfile, ids)``     :func:`decode`
``word_piece::fast::encodeExternal(...)``    :func:`encode_external`
===========================================  =====================================

plus the persistent handle :class:`Vocab` (the reference rebuilds its hash maps
on every call, fast.cpp:21-35; a handle builds the device table once), whose
batch calls the reference lacks: ``Vocab.encode_batch`` (host texts) and
``Vocab.encode_batch_device[_async]`` (a string column in GPU memory: uint8
chars + int64 Arrow offsets in, ids + per-text id offsets in GPU memory out),
``Vocab.decode_device[_async]`` (ids in GPU memory to one token string per
id in the same column layout), and ``Vocab.rows_device[_async]`` /
``Vocab.encode_rows_device`` (per-text ids, or a string column, to the
fixed-length rows, special tokens, padding, overflow windows and attention
mask a BERT-family model takes, in GPU memory).

There is no CPU fallback: if the shared library is missing or no CUDA device is
usable, calls raise.
"""
from __future__ import annotations

from ._capi import (  # noqa: F401
    LIB_PATH,
    Stats,
    Vocab,
    WordPieceError,
    decode,
    encode,
    encode_external,
    encode_files,
    kernel_launch_count,
    load_library,
    tile_bytes,
)
from .sharding import (  # noqa: F401
    Shard,
    encode_sharded,
    encode_sharded_gather,
    global_offsets,
    next_safe_cut,
    plan_shards,
    shard_ranges,
)

__all__ = [
    "LIB_PATH",
    "Stats",
    "Vocab",
    "WordPieceError",
    "decode",
    "encode",
    "encode_external",
    "encode_files",
    "kernel_launch_count",
    "load_library",
    "tile_bytes",
    "Shard",
    "encode_sharded",
    "encode_sharded_gather",
    "global_offsets",
    "next_safe_cut",
    "plan_shards",
    "shard_ranges",
]
