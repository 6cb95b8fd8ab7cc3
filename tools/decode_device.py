#!/usr/bin/env python3
"""Device decode (wp_decode_device) on one GPU, against the host wp_decode of the same ids:
    python tools/decode_device.py [--out DIR] [--repeats 7] [--en-mib 1024] [--ja-mib 256] [--long-ids 10000000]
Workloads, the ids already in device memory:
  - en:   the ids of bench.py's English corpus (1 GiB, seed 2, 29k vocabulary)
  - ja:   the ids of a Japanese corpus (120k vocabulary)
  - long: every id the longest token of the long-m100 vocabulary (each block's output spans many stage windows)
Only the decode call is timed: CUDA events around warm calls, sync and async interleaved, `repeats` rounds.  The
host wp_decode of the same ids is timed with the host clock.  A separate torch.profiler run gives each kernel's time.
Rates: output GB/s (chars written), ids/s, and the algorithmic bytes 4 n_ids + n_chars + 8 (n_ids + 1) (ids read once,
chars and offsets written once) over the call time as a share of the data sheet's 7.7 TB/s of HBM3e.  Writes
DIR/decode_device.json and DIR/decode_device.txt (a table with the card and its power limit, read in the same run)."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import wordpiece_b200  # noqa: E402
from wordpiece_b200 import synth  # noqa: E402

HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU
MIB = 1 << 20


def card() -> str:
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                       text=True).strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e!r})"


def workloads(args, dev):
    """(name, vocab tokens, device ids) one at a time, so that only one corpus is in memory."""
    import torch

    for name, mib, seed in (("en", args.en_mib, 2), ("ja", args.ja_mib, 21)):
        g = synth.generator(name)
        text = g.generate(mib * MIB, seed=seed)
        v = wordpiece_b200.Vocab(g.spec.vocab, device=0)
        d_ids, n = v.encode_device(torch.from_numpy(text).to(dev))
        v.close()
        del text
        yield f"{name} ({mib} MiB corpus)", g.spec.vocab, d_ids[:n].clone()
        del d_ids
    vocab = synth.generator("adv").spec.vocab
    v = wordpiece_b200.Vocab(vocab, device=-1)
    lens = [len(b"".join(v.decode([i]))) for i in range(len(vocab))]
    v.close()
    long_id = int(np.argmax(lens))
    yield f"long (token {long_id}, {lens[long_id]} bytes)", vocab, torch.full((args.long_ids,), long_id, dtype=torch.int32,
                                                                               device=dev)


def host_decode(L, h, ids: np.ndarray):
    """wp_decode of `ids` on the host: (ms, joined bytes, token count)."""
    buf, offs, n, skipped = C.c_void_p(), C.c_void_p(), C.c_size_t(), C.c_size_t()
    t0 = time.perf_counter()
    st = L.wp_decode(h, ids.ctypes.data, ids.size, C.byref(buf), C.byref(offs), C.byref(n), C.byref(skipped))
    ms = (time.perf_counter() - t0) * 1e3
    assert st == 0, st
    total = np.ctypeslib.as_array(C.cast(offs, C.POINTER(C.c_size_t)), shape=(n.value + 1,))[-1]
    joined = C.string_at(buf, int(total))
    L.wp_free(buf)
    L.wp_free(offs)
    return ms, joined, int(n.value)


def run(args):
    import torch
    from torch.profiler import ProfilerActivity, profile

    dev = torch.device("cuda:0")
    out = {"card": card(), "repeats": args.repeats, "hbm_bytes_per_s": HBM_BYTES_PER_S, "workloads": []}
    lines = [f"card (name, power limit, max SM clock): {out['card']}", ""]
    for name, vocab, d_ids in workloads(args, dev):
        v = wordpiece_b200.Vocab(vocab, device=0)
        n_ids = d_ids.numel()
        d_chars, d_offs, n_chars, n_skipped = v.decode_device(d_ids)  # (builds the decode table)
        stream = torch.cuda.current_stream(dev)

        def timed(fn):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            fn()
            b.record(stream)
            b.synchronize()
            return a.elapsed_time(b)

        calls = {"sync": lambda: timed(lambda: v.decode_device(d_ids, d_chars, d_offs)),
                 "async": lambda: timed(lambda: v.decode_device_async(d_ids, d_chars, d_offs))}
        for fn in calls.values():
            fn()
        assert int(d_offs[-1]) == n_chars, "async call was void"
        times = {m: [] for m in calls}
        for _ in range(args.repeats):
            for m, fn in calls.items():
                times[m].append(fn())

        # the host wp_decode of the same ids, and the same bytes
        h_ids = d_ids.cpu().numpy()
        host_ms, joined, n_tokens = [], None, 0
        for _ in range(args.host_repeats):
            ms, joined, n_tokens = host_decode(v._L, v._h, h_ids)
            host_ms.append(ms)
        same = n_tokens == n_ids - n_skipped and joined == d_chars.cpu().numpy().tobytes()
        del joined, h_ids

        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.profile_calls):
                v.decode_device_async(d_ids, d_chars, d_offs)
            torch.cuda.synchronize()
        kern = {}
        for e in prof.key_averages():
            t_us = getattr(e, "device_time_total", None)
            if t_us is None:
                t_us = e.cuda_time_total
            if t_us > 0:
                kern[e.key] = kern.get(e.key, 0.0) + t_us / args.profile_calls / 1e3

        alg_bytes = 4 * n_ids + n_chars + 8 * (n_ids + 1)
        res = {"workload": name, "n_ids": n_ids, "n_chars": n_chars, "n_skipped": n_skipped, "algorithmic_bytes": alg_bytes,
               "device_equals_host_wp_decode": same,
               "ms": {m: {"median": float(np.median(t)), "min": float(np.min(t)), "all": t} for m, t in times.items()},
               "host_wp_decode_ms": {"median": float(np.median(host_ms)), "all": host_ms},
               "profile_ms_per_call": kern}
        out["workloads"].append(res)
        lines.append(f"{name}: {n_ids} ids -> {n_chars} chars ({n_skipped} skipped), device == host wp_decode: {same}")
        for m in calls:
            t = res["ms"][m]["median"] * 1e-3
            lines.append(f"  {m:6s} median {t * 1e3:9.3f} ms  min {res['ms'][m]['min']:9.3f} ms  {n_chars / t / 1e9:7.1f} GB/s out  "
                         f"{n_ids / t / 1e9:6.2f} G ids/s  HBM share {alg_bytes / t / HBM_BYTES_PER_S * 100:5.1f} %")
        h = res["host_wp_decode_ms"]["median"]
        lines.append(f"  host wp_decode {h:9.1f} ms  (x{h / res['ms']['sync']['median']:.0f} the sync device call)")
        lines.append("  profiler (async call): " + ", ".join(f"{k} {t:.3f} ms" for k, t in sorted(kern.items())))
        lines.append("")
        print("\n".join(lines[-6:]), flush=True)
        v.close()
        del d_ids, d_chars, d_offs
        torch.cuda.empty_cache()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "decode_device.json"), "w") as f:
        json.dump(out, f, indent=1)
    with open(os.path.join(args.out, "decode_device.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "decode_device"))
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--host-repeats", type=int, default=1)
    ap.add_argument("--profile-calls", type=int, default=5)
    ap.add_argument("--en-mib", type=int, default=1024)
    ap.add_argument("--ja-mib", type=int, default=256)
    ap.add_argument("--long-ids", type=int, default=10_000_000)
    args = ap.parse_args()
    import torch

    assert torch.cuda.is_available(), "tools/decode_device.py measures on a CUDA device; there is no CPU mode"
    run(args)


if __name__ == "__main__":
    main()
