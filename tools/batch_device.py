#!/usr/bin/env python3
"""Device batch (wp_encode_batch_device) against its neighbours, on one GPU:
    python tools/batch_device.py [--out DIR] [--repeats 7] [--workloads 10000x4096,100000x256,...]
A column of English text (wordpiece_b200.synth, 29k vocabulary) cut into n texts of `size` bytes is encoded by
  - batch_device:       wp_encode_batch_device (sync), column and ids in device memory
  - batch_device_async: wp_encode_batch_device_async, same buffers
  - device_packed:      wp_encode_device over the same texts packed as the batch packs them (the ceiling: no packer)
  - host_batch:         wp_encode_batch from host pointers into a pinned id buffer
Every call is warm; the four are interleaved, `repeats` rounds.  Device calls are timed with CUDA events on the
stream they run on, the host-pointer call (which ends in a stream synchronisation) with the host clock.  Then a
separate torch.profiler run of the async call gives each kernel's share of the call.  Writes
DIR/batch_device.json and DIR/batch_device.txt (a table with the card and its power limit)."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import tempfile
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

import wordpiece_b200  # noqa: E402
from wordpiece_b200 import synth  # noqa: E402

METHODS = ("batch_device", "batch_device_async", "device_packed", "host_batch")


def card() -> str:
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                       text=True).strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e!r})"


def workload(n_texts: int, size: int, dev):
    import torch

    g = synth.generator("en")
    text = g.generate(n_texts * size, seed=5)
    offs = np.arange(n_texts + 1, dtype=np.int64) * size
    packed = np.full(n_texts * (size + 1), 0x20, np.uint8)  # the batch packing rule: every text, then one space
    packed.reshape(n_texts, size + 1)[:, :size] = text.reshape(n_texts, size)
    return {
        "text": text,
        "d_chars": torch.from_numpy(text).to(dev),
        "d_offsets": torch.from_numpy(offs).to(dev),
        "d_packed": torch.from_numpy(packed).to(dev),
        "slices": [text[i * size:(i + 1) * size] for i in range(n_texts)],
    }, g.spec.vocab


def run(args):
    import torch

    dev = torch.device("cuda:0")
    out = {"card": card(), "repeats": args.repeats, "workloads": []}
    lines = [f"card (name, power limit, max SM clock): {out['card']}", ""]
    for spec in args.workloads.split(","):
        n_texts, size = (int(x) for x in spec.split("x"))
        w, vocab_tokens = workload(n_texts, size, dev)
        v = wordpiece_b200.Vocab(vocab_tokens, device=0)
        n_chars = n_texts * size
        cap = n_chars // 2 + 4096
        d_ids = torch.empty(cap, dtype=torch.int32, device=dev)
        d_id_offsets = torch.empty(n_texts + 1, dtype=torch.int64, device=dev)
        d_cnt = torch.zeros(1, dtype=torch.int64, device=dev)
        prepared = v.batch_pointers(w["slices"])
        h_out = torch.empty(cap, dtype=torch.int32, pin_memory=True).numpy()
        h_offs = np.zeros(n_texts + 1, np.uint64)
        stream = torch.cuda.current_stream(dev)

        # correctness: the device batch equals the host batch, and the packed ceiling gives the same ids
        _, _, n_ids = v.encode_batch_device(w["d_chars"], w["d_offsets"], d_ids, d_id_offsets)
        ref_ids, ref_offs = v.encode_batch(None, out=h_out, offsets=h_offs, prepared=prepared)
        same = bool(np.array_equal(d_ids[:n_ids].cpu().numpy(), ref_ids)) and bool(
            np.array_equal(d_id_offsets.cpu().numpy(), ref_offs.astype(np.int64)))
        _, n_packed = v.encode_device(w["d_packed"], d_ids)
        same = same and n_packed == n_ids

        def dev_timed(fn):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            fn()
            b.record(stream)
            b.synchronize()
            return a.elapsed_time(b)

        calls = {
            "batch_device": lambda: dev_timed(lambda: v.encode_batch_device(w["d_chars"], w["d_offsets"], d_ids, d_id_offsets)),
            "batch_device_async": lambda: dev_timed(
                lambda: v.encode_batch_device_async(w["d_chars"], w["d_offsets"], d_ids, d_id_offsets)),
            "device_packed": lambda: dev_timed(lambda: v.encode_device(w["d_packed"], d_ids)),
        }

        def host_batch():
            t0 = time.perf_counter()
            v.encode_batch(None, out=h_out, offsets=h_offs, prepared=prepared)
            return (time.perf_counter() - t0) * 1e3

        calls["host_batch"] = host_batch
        for fn in calls.values():  # warm-up of every shape
            fn()
        torch.cuda.synchronize()
        assert int(d_id_offsets[-1]) == n_ids, "async call was void"
        times = {m: [] for m in METHODS}
        for _ in range(args.repeats):
            for m in METHODS:
                times[m].append(calls[m]())
        res = {"n_texts": n_texts, "size": size, "text_bytes": n_chars, "ids": n_ids, "device_equals_host_batch": same,
               "ms": {m: {"median": float(np.median(t)), "min": float(np.min(t)), "all": t} for m, t in times.items()}}

        # kernel shares of the async call, from a separate profiler run
        from torch.profiler import ProfilerActivity, profile

        reps = 5
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                v.encode_batch_device_async(w["d_chars"], w["d_offsets"], d_ids, d_id_offsets)
            torch.cuda.synchronize()
        kern = {}
        for e in prof.key_averages():
            if e.device_type.name == "CUDA" or getattr(e, "device_time_total", 0) > 0:
                name = e.key
                t_us = getattr(e, "device_time_total", None)
                if t_us is None:
                    t_us = e.cuda_time_total
                kern[name] = kern.get(name, 0.0) + t_us / reps / 1e3
        total_k = sum(kern.values())
        pack = sum(t for k, t in kern.items() if "wp_column_" in k)
        k1 = sum(t for k, t in kern.items() if "wp_split_kernel" in k)
        res["profile_ms_per_call"] = kern
        res["profile_summary"] = {"all_kernels_ms": total_k, "check_and_pack_ms": pack, "k1_ms": k1,
                                  "check_and_pack_share": pack / total_k if total_k else None}
        out["workloads"].append(res)
        gbs = {m: n_chars / (res["ms"][m]["median"] * 1e-3) / 1e9 for m in METHODS}
        lines.append(f"{n_texts} x {size} B ({n_chars / 2**20:.1f} MiB, {n_ids} ids, device == host batch: {same})")
        for m in METHODS:
            lines.append(f"  {m:20s} median {res['ms'][m]['median']:9.3f} ms  min {res['ms'][m]['min']:9.3f} ms  "
                         f"{gbs[m]:7.1f} GB/s  {n_texts / (res['ms'][m]['median'] * 1e-3) / 1e6:8.2f} M texts/s")
        ps = res["profile_summary"]
        lines.append(f"  profiler (async call, kernels only): all kernels {ps['all_kernels_ms']:.3f} ms, check + pack "
                     f"{ps['check_and_pack_ms']:.3f} ms ({100 * (ps['check_and_pack_share'] or 0):.1f} %), K1 {ps['k1_ms']:.3f} ms")
        lines.append("")
        print("\n".join(lines[-7:]), flush=True)
        v.close()
        del w, d_ids, d_id_offsets, d_cnt, h_out, prepared
        torch.cuda.empty_cache()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "batch_device.json"), "w") as f:
        json.dump(out, f, indent=1)
    with open(os.path.join(args.out, "batch_device.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "batch_device"))
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--workloads", default="10000x4096,100000x256,1000000x64,16x67108864")
    args = ap.parse_args()
    import torch

    assert torch.cuda.is_available(), "tools/batch_device.py measures on a CUDA device; there is no CPU mode"
    run(args)


if __name__ == "__main__":
    main()
