#!/usr/bin/env python3
"""Model-input rows (wp_rows_device) on one GPU, against the torch composition a user would write otherwise:
    python tools/rows_device.py [--out DIR] [--repeats 7] [--short-texts 1048576] [--long-texts 10000]
Workloads, per-text ids already in device memory (encode_batch_device of a string column of bench.py's English
corpus, seed 2, 29k vocabulary):
  - short: the corpus cut into `short-texts` texts of 128 bytes, L = 128, truncation, CLS + SEP
  - long:  the corpus cut into `long-texts` texts of 4 KiB, L = 512, stride 384 (overflow windows), CLS + SEP
Timed with CUDA events around warm calls, interleaved, `repeats` rounds:
  - rows:  Vocab.rows_device_async (scan + fill) into preallocated tensors
  - torch: the same rows, mask and row offsets from torch ops (row counts, cumsum, repeat_interleave, an
           [n_rows, L] int64 index matrix, gather + where, scatter of SEP); its output is compared with the call's
  - encode_rows: Vocab.encode_rows_device end to end (string column -> rows; sync, allocates), next to
           encode_batch: Vocab.encode_batch_device alone (sync, preallocated)
A separate torch.profiler run of the rows call gives each kernel's time.  The fill's write bandwidth is the bytes it
writes (n_rows * L * 4 ids + n_rows * L mask) over its kernel time, as a share of the data sheet's 7.7 TB/s of
HBM3e.  Writes DIR/rows_device.json and DIR/rows_device.txt (with the card and its power limit, read in the same
run)."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import wordpiece_b200  # noqa: E402
from wordpiece_b200 import synth  # noqa: E402

HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU
CLS, SEP, PAD = 2, 3, 0


def card() -> str:
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                       text=True).strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e!r})"


def torch_rows(d_ids, d_id_offsets, L, stride, pad_id, cls_id, sep_id):
    """The rows, mask and row offsets from torch ops: what a caller without wp_rows_device writes."""
    import torch

    c, s = int(cls_id is not None), int(sep_id is not None)
    width = L - c - s
    n_t = d_id_offsets[1:] - d_id_offsets[:-1]
    if stride == 0:
        counts = torch.ones_like(n_t)
    else:
        counts = torch.where(n_t <= width, 1, 1 + torch.div(n_t - width + stride - 1, stride, rounding_mode="floor"))
    row_offs = torch.zeros(n_t.numel() + 1, dtype=torch.int64, device=d_ids.device)
    torch.cumsum(counts, 0, out=row_offs[1:])
    text = torch.repeat_interleave(torch.arange(n_t.numel(), device=d_ids.device), counts)
    k = torch.arange(text.numel(), device=d_ids.device) - row_offs[text]
    start = d_id_offsets[text] + k * stride
    length = torch.minimum(n_t[text] - k * stride, torch.tensor(width, device=d_ids.device))
    j = torch.arange(L, device=d_ids.device) - c
    idx = (start[:, None] + j[None, :]).clamp_(0, max(d_ids.numel() - 1, 0))
    content = (j[None, :] >= 0) & (j[None, :] < length[:, None])
    rows = torch.where(content, d_ids[idx], torch.tensor(pad_id, dtype=torch.int32, device=d_ids.device))
    if c:
        rows[:, 0] = cls_id
    if s:
        rows.scatter_(1, (c + length)[:, None], sep_id)
    mask = (torch.arange(L, device=d_ids.device)[None, :] < (c + length + s)[:, None]).to(torch.uint8)
    return rows, mask, row_offs


def run(args):
    import torch
    from torch.profiler import ProfilerActivity, profile

    dev = torch.device("cuda:0")
    g = synth.generator("en")
    v = wordpiece_b200.Vocab(g.spec.vocab, device=0)
    out = {"card": card(), "repeats": args.repeats, "hbm_bytes_per_s": HBM_BYTES_PER_S, "workloads": []}
    lines = [f"card (name, power limit, max SM clock): {out['card']}", ""]
    stream = torch.cuda.current_stream(dev)

    def timed(fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fn()
        b.record(stream)
        b.synchronize()
        return a.elapsed_time(b)

    for name, n_texts, text_bytes, L, stride in (("short", args.short_texts, 128, 128, 0),
                                                 ("long", args.long_texts, 4096, 512, 384)):
        text = g.generate(n_texts * text_bytes, seed=2)
        d_chars = torch.from_numpy(text).to(dev)
        d_offsets = torch.arange(0, n_texts * text_bytes + 1, text_bytes, dtype=torch.int64, device=dev)
        del text
        d_ids_full = torch.empty(d_chars.numel(), dtype=torch.int32, device=dev)
        d_id_offs = torch.empty(n_texts + 1, dtype=torch.int64, device=dev)
        _, _, n_ids = v.encode_batch_device(d_chars, d_offsets, d_ids_full, d_id_offs)
        d_ids = d_ids_full[:n_ids]
        kw = dict(stride=stride, pad_id=PAD, cls_id=CLS, sep_id=SEP)
        rows, mask, row_offs, n_rows = v.rows_device(d_ids, d_id_offs, L, **kw)
        t_rows, t_mask, t_offs = torch_rows(d_ids, d_id_offs, L, stride, PAD, CLS, SEP)
        same = (torch.equal(rows, t_rows) and torch.equal(mask, t_mask) and torch.equal(row_offs, t_offs))
        del t_rows, t_mask, t_offs
        calls = {
            "rows": lambda: timed(lambda: v.rows_device_async(d_ids, d_id_offs, rows, row_offs, L, d_mask=mask, **kw)),
            "torch": lambda: timed(lambda: torch_rows(d_ids, d_id_offs, L, stride, PAD, CLS, SEP)),
            "encode_rows": lambda: timed(lambda: v.encode_rows_device(d_chars, d_offsets, L, **kw)),
            "encode_batch": lambda: timed(lambda: v.encode_batch_device(d_chars, d_offsets, d_ids_full, d_id_offs)),
        }
        for fn in calls.values():
            fn()
        times = {m: [] for m in calls}
        for _ in range(args.repeats):
            for m, fn in calls.items():
                times[m].append(fn())
        assert int(row_offs[-1]) == n_rows, "async call was void"

        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.profile_calls):
                v.rows_device_async(d_ids, d_id_offs, rows, row_offs, L, d_mask=mask, **kw)
            torch.cuda.synchronize()
        kern = {}
        for e in prof.key_averages():
            t_us = getattr(e, "device_time_total", None)
            if t_us is None:
                t_us = e.cuda_time_total
            if t_us > 0:
                kern[e.key] = kern.get(e.key, 0.0) + t_us / args.profile_calls / 1e3
        fill_ms = sum(t for k, t in kern.items() if "rows_fill" in k)
        written = n_rows * L * 5
        med = {m: float(np.median(t)) for m, t in times.items()}
        res = {"workload": name, "n_texts": n_texts, "text_bytes": text_bytes, "n_ids": n_ids, "max_len": L,
               "stride": stride, "n_rows": n_rows, "fill_bytes_written": written, "rows_equal_torch": bool(same),
               "ms": {m: {"median": med[m], "min": float(np.min(t)), "all": t} for m, t in times.items()},
               "profile_ms_per_call": kern}
        out["workloads"].append(res)
        lines.append(f"{name}: {n_texts} texts x {text_bytes} B -> {n_ids} ids -> {n_rows} rows of L = {L}, stride {stride}, "
                     f"CLS + SEP; rows == torch composition: {same}")
        lines.append(f"  rows call (scan + fill, async)  median {med['rows']:8.3f} ms  min {res['ms']['rows']['min']:8.3f} ms")
        if fill_ms > 0:
            lines.append(f"  fill kernel {fill_ms:8.3f} ms: {written / 1e6:.1f} MB written, {written / (fill_ms * 1e-3) / 1e9:7.1f} GB/s = "
                         f"{written / (fill_ms * 1e-3) / HBM_BYTES_PER_S * 100:5.1f} % of 7.7 TB/s")
        lines.append(f"  torch composition               median {med['torch']:8.3f} ms  (x{med['torch'] / med['rows']:.1f} the rows call)")
        lines.append(f"  encode_rows_device (end to end) median {med['encode_rows']:8.3f} ms;  encode_batch_device alone "
                     f"{med['encode_batch']:8.3f} ms")
        lines.append("  profiler (rows call): " + ", ".join(f"{k} {t:.3f} ms" for k, t in sorted(kern.items())))
        lines.append("")
        print("\n".join(lines[-7:]), flush=True)
        del rows, mask, row_offs, d_ids, d_ids_full, d_id_offs, d_chars, d_offsets
        torch.cuda.empty_cache()
    v.close()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "rows_device.json"), "w") as f:
        json.dump(out, f, indent=1)
    with open(os.path.join(args.out, "rows_device.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "rows_device"))
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--profile-calls", type=int, default=5)
    ap.add_argument("--short-texts", type=int, default=1 << 20)
    ap.add_argument("--long-texts", type=int, default=10000)
    args = ap.parse_args()
    import torch

    assert torch.cuda.is_available(), "tools/rows_device.py measures on a CUDA device; there is no CPU mode"
    run(args)


if __name__ == "__main__":
    main()
