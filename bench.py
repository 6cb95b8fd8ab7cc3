#!/usr/bin/env python
"""Benchmark of the fast WordPiece encode path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload en|ru|ja|zh|adv]
                    [--dump-outputs DIR]

One step = one pass of the encode path over one batch of synthetic text.  The text and the vocabulary come
from fixed seeds, so the same arguments give the same inputs in every run; --dump-outputs DIR writes what the
last timed step returned (see dump_outputs) so that two builds can be compared output for output.

* N = 1: the batch is BASELINE.json configs[1] — 1 GiB of English-like text, the 29k-entry bert-shaped
  vocabulary, resident in HBM before the timed region.  The line also carries a compact `configs` object
  (ru / ja / zh / adversarial at 256 MiB, the open-vocabulary and dirty-web shapes, the 4 KiB latency), the
  end-to-end figure through the reference's own C++ signature (`e2e_dropin`) and the whole-process
  `runner fast` time of configs[0].
* N > 1 (launched by torchrun, one rank per GPU): configs[3] — ONE 10 GiB corpus cut into N contiguous byte
  ranges at safe starts (wp_next_safe_cut), replicated vocabulary, no data-path collective => STRONG scaling.
  Every step ends with the per-shard id counts gathered and scanned into global offsets (the only exchange
  the path has); the optional gather of all ids on rank 0 over NCCL/NVLink is timed separately (`gather`).

Prints ONE JSON line (rank 0).  `value` is whole-job GB/s of text with device-resident input; `e2e` is the
same metric through the host-buffer C-ABI call (wp_encode_into: pinned host text -> H2D -> kernels -> D2H
ids), next to the measured PCIe ceiling of the same copies; `roofline` is (text bytes + 4 x ids) / kernel
time against the measured HBM copy peak; `cpu_baseline` is the reference's own CPU fast path on the box's
host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

GIB = 1 << 30
MIB = 1 << 20
METRIC = "GB/s text tokenized"
UNIT = "GB/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="en", choices=["en", "ru", "ja", "zh", "adv"])
    ap.add_argument("--mib", type=int, default=1024, help="text MiB at N = 1 (default 1024 = BASELINE configs[1])")
    ap.add_argument("--corpus-gib", type=int, default=10, help="size of the one corpus sharded over N > 1 GPUs (configs[3])")
    ap.add_argument("--cpu-sample-mib", type=int, default=1024, help="text MiB per step of the CPU reference timing")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the other configurations / latency / drop-in legs")
    ap.add_argument("--no-gather", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the ids of the last timed step as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the GPU path; it is not available with --impl reference")
    return args


def workload_name(args, world: int = 1) -> str:
    vocab = {"en": "bert-cased-29k", "adv": "long-m100"}.get(args.workload, "mbert-120k")
    if world > 1:
        return f"{args.workload}-{args.corpus_gib}GiB-corpus-over-{world}-gpus/{vocab}"
    size = f"{args.mib // 1024}GiB" if args.mib % 1024 == 0 else f"{args.mib}MiB"
    return f"{args.workload}-{size}/{vocab}"


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def traffic_from_profile():
    """dram bytes per launch of the dominant kernel from the committed ncu capture, if any."""
    path = os.path.join(ROOT, "profiles", "dram_traffic.json")
    try:
        with open(path) as f:
            return json.load(f)
    except Exception:
        return None


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU during the timed region (NVML)."""

    def __init__(self, index: int, period: float = 0.01):
        super().__init__(daemon=True)
        self.index = index
        self.period = period
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._halt.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._halt.wait(self.period)

    def stop(self):
        self._halt.set()
        if self.ok:
            self.join(timeout=2)

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def physical_gpu_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


def cpu_reference_timing(text: np.ndarray, vocab, sample_mib: int, threads: int = 0):
    """Time the reference's own CPU fast path (oracle/_ref, else the C port) on the first `sample_mib` MiB."""
    from _oracle import Oracle, Ref

    n = min(text.size, sample_mib * MIB)
    sample = text[:n]
    if n < text.size:  # cut at the last whitespace so the sample is a valid shard
        tail = sample[-4096:].tobytes()
        cut = max(tail.rfind(b" "), tail.rfind(b"\n"))
        if cut >= 0:
            sample = sample[: n - len(tail) + cut + 1]
    b = sample.tobytes()
    whole = "the whole workload" if len(b) == text.size else f"the first {len(b) / MIB:.0f} MiB of the workload"
    if Ref.available():
        Ref.lib(threads or (os.cpu_count() or 1))  # the pool size is frozen by the first call (utils.cpp:25-28)
        ids, sec = Ref.encode(b, vocab, "fast", return_seconds=True)
        return {"kind": "reference", "cores": int(Ref.pool_threads), "seconds": sec, "bytes": len(b), "ids": int(ids.size),
                "sample": f"{whole}, reference fast::encode(text, vocab) in-process (oracle/_ref, -O3 -flto "
                          f"-march=x86-64-v3), {Ref.pool_threads} pool threads, includes its per-call vocab parse + "
                          f"hash-map build"}
    o = Oracle(vocab)
    t0 = time.perf_counter()
    ids = o.encode(b)
    sec = time.perf_counter() - t0
    return {"kind": "port", "cores": 1, "seconds": sec, "bytes": len(b), "ids": int(ids.size),
            "sample": f"{whole}, oracle/wp_oracle.c (scalar port, 1 thread)"}


def cpu_reference_subprocess(workload: str, mib: int, threads: int):
    """The same timing in a fresh process with a pool of `threads` threads (the reference freezes its pool size
    at the first call, so a second thread count needs a second process).  BASELINE.md section 3: n_threads = 8."""
    import subprocess

    code = ("import sys, json; sys.path[:0] = [%r, %r]\n"
            "import bench\nfrom wordpiece_b200 import synth\n"
            "g = synth.generator(%r); t = g.generate(%d * bench.MIB, seed=2)\n"
            "i = bench.cpu_reference_timing(t, g.spec.vocab, %d, threads=%d)\n"
            "print(json.dumps(i))\n") % (ROOT, os.path.join(ROOT, "tests"), workload, mib, mib, threads)
    try:
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
        info = json.loads(r.stdout.strip().splitlines()[-1])
        return {"value": info["bytes"] / info["seconds"] / 1e9, "unit": UNIT, "cores": info["cores"], "kind": info["kind"],
                "sample": info["sample"], "tokens_per_s": info["ids"] / info["seconds"]}
    except Exception as e:  # a reported baseline, never a reason to lose the line
        return {"error": f"{type(e).__name__}: {e}"}


def run_reference(args, rank: int, world: int):
    """--impl reference: the reference's CPU fast path on this box's host cores (rank 0 only), every step the
    whole configs[1] text (1 GiB), all host threads; the n_threads = 8 figure of BASELINE.md rides along."""
    if rank != 0:
        return
    from wordpiece_b200 import synth

    g = synth.generator(args.workload)
    sample_mib = min(args.cpu_sample_mib, args.mib)
    # N = 1: the whole configs[1] text (same generator seed as the GPU arm).  N > 1: the GPU arm shards ONE 10 GiB
    # corpus (seed 4); a CPU step over all of it would take a minute, so every step here is a bounded sample of
    # that corpus — its first args.mib MiB (throughput of this path does not depend on the size at this scale)
    text = g.generate(args.mib * MIB, seed=2 if world == 1 else 4)
    vocab = g.spec.vocab
    times, info = [], None
    for i in range(args.warmup + args.steps):
        info = cpu_reference_timing(text, vocab, sample_mib)
        if i >= args.warmup:
            times.append(info["seconds"])
    total = sum(times)
    gbs = info["bytes"] * len(times) / total / 1e9
    line = {
        "impl": "reference",
        "metric": METRIC, "value": gbs, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": workload_name(args, world), "text_bytes": int(info["bytes"]),
                   "step": f"one reference fast::encode(text, vocab) call over {info['bytes']} bytes"
                           + ("" if world == 1 else f" (bounded sample: the first {args.mib} MiB of the corpus)"),
                   "timing": "steady_clock inside the reference process (host only; no GPU involved)"},
        "tokens_per_s": info["ids"] * len(times) / total,
        "cpu_baseline": {"value": gbs, "unit": UNIT, "cores": info["cores"], "kind": info["kind"],
                         "sample": info["sample"]},
        "cpu_baseline_8_threads": cpu_reference_subprocess(args.workload, sample_mib, 8),
        "e2e": {"value": gbs, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


_REAL_STDOUT = None


def claim_stdout():
    """Keep stdout for the ONE JSON line: everything else that writes to fd 1 from here on (NCCL prints its
    version banner there from C code, libraries may log) goes to stderr; emit() writes to the saved fd."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


DUMP_SAMPLE = 1 << 21  # ids kept by --dump-outputs over all ranks: 2 x 16 MiB of float64 (ids and positions)


def dump_outputs(out_dir: str, d_ids, n_ids: int, vocab_size: int, sample: int = DUMP_SAMPLE, first_id: int = 0):
    """--dump-outputs: what a caller of the timed path receives, the id count and the id array (float64, which
    holds every id and position exactly).  A 1 GiB step yields ~300 M ids, so the array is written as a fixed
    seeded sample of at most `sample` positions (all of them for smaller outputs), next to the histogram of
    ALL ids, which a single changed id anywhere alters:
        n_ids.npy                 [n_ids]
        ids_sample.npy            ids at the positions below
        ids_sample_positions.npy  sorted positions, first_id + index into this call's id array
        id_histogram.npy          occurrences of id -1 (no [UNK] in the vocabulary), 0, 1, ..., vocab_size - 1
    N > 1: every rank writes its shard's files; first_id is the shard's offset in the whole corpus's ids, so
    the positions of all ranks index one array, and `sample` is DUMP_SAMPLE / N to keep the total bounded."""
    import torch

    os.makedirs(out_dir, exist_ok=True)
    ids = d_ids[:n_ids]
    if n_ids <= sample:
        pos = np.arange(n_ids, dtype=np.int64)
    else:
        pos = np.unique(np.random.default_rng(0).integers(0, n_ids, sample))
    values = ids[torch.from_numpy(pos).to(ids.device)].cpu().numpy()
    hist = torch.bincount(ids.long() + 1, minlength=vocab_size + 1).cpu().numpy()
    for name, a in (("n_ids", np.array([n_ids])), ("ids_sample", values), ("ids_sample_positions", first_id + pos),
                    ("id_histogram", hist)):
        np.save(os.path.join(out_dir, f"{name}.npy"), a.astype(np.float64))


# ------------------------------------------------------------------ helper legs (N = 1)

def other_configs(dev_index: int, peak: float):
    """ru / ja / zh / adversarial at 256 MiB plus the open-vocabulary and dirty-web shapes of the English
    workload at 128 MiB: device-resident GB/s, roofline fraction of the whole path, and a parity flag (first
    4 MiB against the CPU checker, bit-exact)."""
    import torch
    import wordpiece_b200
    from _oracle import Oracle
    from wordpiece_b200 import synth

    out = {}
    seeds = {"ru": 31, "ja": 32, "zh": 33, "adv": 5}
    jobs = [(name, name, 256) for name in ("ru", "ja", "zh", "adv")] + [("en-open-vocabulary", "en", 128),
                                                                          ("en-dirty-web", "en", 128)]
    for tag, name, mib in jobs:
        g = synth.generator(name)
        text = g.generate(mib * MIB, seed=seeds.get(name, 21))
        if tag == "en-open-vocabulary":
            text = synth.open_vocabulary(text, seed=23)
        elif tag == "en-dirty-web":
            text = synth.dirty_web(text, seed=22)
        vocab_tokens = g.spec.vocab
        v = wordpiece_b200.Vocab(vocab_tokens, device=dev_index)
        d_text = torch.from_numpy(text).cuda(dev_index)
        # one id per byte is the worst case (ids <= chars <= bytes); the high-UNK and random-alphanumeric shapes
        # pass 0.5 ids per byte
        d_ids = torch.empty(text.size, dtype=torch.int32, device=d_text.device)
        d_cnt = torch.zeros(1, dtype=torch.int64, device=d_text.device)
        _, n_ids = v.encode_device(d_text, d_ids)
        st = v.stats()
        cut = 4 * MIB
        while text[cut - 1] not in (0x20, 0x0A):
            cut -= 1
        parity = bool(np.array_equal(Oracle(vocab_tokens).encode(text[:cut]), v.encode(text[:cut])))
        times = []
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            v.encode_device_async(d_text, d_ids, d_cnt)
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
        v.set_kernel_timing(True)
        v.encode_device_async(d_text, d_ids, d_cnt)
        k_ms, _ = v.last_kernel_ms()
        v.set_kernel_timing(False)
        med = float(np.median(times))
        out[tag] = {"text_mib": mib, "gb_per_s": text.size / (med * 1e-3) / 1e9, "tokens_per_s": n_ids / (med * 1e-3),
                    "roofline_frac": (text.size + 4 * n_ids) / (med * 1e-3) / 1e9 / peak, "parity": parity,
                    "kernel_ms": dict(zip(["split", "match", "scatter"], [round(x, 4) for x in k_ms])),
                    "dirty_tiles": st.dirty_tiles, "long_segments": st.long_segments, "memo_hits": st.memo_hits}
        v.close()
        del d_text, d_ids
    return out


def latency_4k(text: np.ndarray, vocab, n_slices: int = 2000):
    """configs[4]: 4 096-byte slices cut at a space, one call each through the handle (p50 / p99 in microseconds)."""
    import torch

    rng = np.random.default_rng(0)
    slices = []
    for start in rng.integers(0, text.size - 8192, size=n_slices):
        s = int(start)
        while text[s - 1] != 0x20:
            s += 1
        e = s + 4096
        while text[e - 1] != 0x20:
            e -= 1
        slices.append(np.ascontiguousarray(text[s:e]))
    out = np.zeros(4096, np.int32)
    for sl in slices[:50]:
        vocab.encode_into(sl, out)
    t_host = []
    for sl in slices:
        t0 = time.perf_counter()
        vocab.encode_into(sl, out)
        t_host.append((time.perf_counter() - t0) * 1e6)
    d_slices = [torch.from_numpy(sl).cuda() for sl in slices[:1000]]
    d_ids = torch.empty(4096, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    t_dev = []
    for ds in d_slices:
        t0 = time.perf_counter()
        vocab.encode_device(ds, d_ids)
        t_dev.append((time.perf_counter() - t0) * 1e6)
    pct = lambda a, q: float(np.percentile(a, q))  # noqa: E731
    return {"slices": n_slices, "host_buffers_us": {"p50": pct(t_host, 50), "p99": pct(t_host, 99)},
            "device_resident_us": {"p50": pct(t_dev, 50), "p99": pct(t_dev, 99)},
            "call": "wp_encode_into / wp_encode_device, one 4 KiB text per call, handle reused"}


def batch_throughput(text: np.ndarray, vocab, n_texts: int = 10000, size: int = 4096):
    """SURVEY 8(f): many short texts in ONE call (wp_encode_batch): `n_texts` slices of about `size` bytes, host
    pointers in, pinned id buffer out; every copy (packing, H2D, D2H) inside the timed call.  Checked against
    one-call-per-text on a sample."""
    import torch

    rng = np.random.default_rng(1)
    slices = []
    for start in rng.integers(0, text.size - 2 * size, size=n_texts):
        s = int(start)
        while text[s - 1] != 0x20:
            s += 1
        e = s + size
        while text[e - 1] != 0x20:
            e -= 1
        slices.append(text[s:e].tobytes())
    total = sum(len(b) for b in slices)
    prepared = vocab.batch_pointers(slices)
    out = torch.empty(total, dtype=torch.int32, pin_memory=True).numpy()
    offs = np.zeros(n_texts + 1, np.uint64)
    ids, offsets = vocab.encode_batch(slices, out=out, offsets=offs, prepared=prepared)
    ok = True
    for i in range(0, n_texts, max(1, n_texts // 50)):
        one = vocab.encode(slices[i])
        ok = ok and bool(np.array_equal(one, ids[int(offsets[i]):int(offsets[i + 1])]))
    times = []
    for _ in range(5):
        t0 = time.perf_counter()
        vocab.encode_batch(slices, out=out, offsets=offs, prepared=prepared)
        times.append(time.perf_counter() - t0)
    best = min(times)
    return {"texts": n_texts, "text_bytes": total, "ids": int(ids.size), "seconds_best_of_5": best,
            "gb_per_s": total / best / 1e9, "texts_per_s": n_texts / best, "matches_single_calls": ok,
            "call": "wp_encode_batch: host text pointers in (packed by the library into pinned memory), one H2D, "
                    "one pass of the kernels, ids + per-text offsets back into a pinned buffer"}


def dropin_and_process(text: np.ndarray, vocab_tokens, n_ids: int):
    """(1) e2e through the reference's own C++ signature: a small C++ helper (csrc/dropin_bench.cpp) reads the
    text and the vocabulary from files and times word_piece::fast::encode(std::string, std::vector<std::string>)
    — pageable std::string in, std::vector<int> out.  (2) BASELINE configs[0] the way speed_test.py times it:
    wall clock of a whole `runner fast <10 MB text> <vocab> 8` process, this build and the reference."""
    import subprocess
    import tempfile

    res = {}
    shm = "/dev/shm" if os.path.isdir("/dev/shm") else None
    with tempfile.TemporaryDirectory(dir=shm) as d:
        tf, vf = os.path.join(d, "text.txt"), os.path.join(d, "vocab.txt")
        with open(vf, "wb") as f:
            f.write(b"\n".join(t if isinstance(t, bytes) else t.encode() for t in vocab_tokens) + b"\n")
        exe = os.path.join(ROOT, "wordpiece_b200", "lib", "dropin_bench")
        if os.path.exists(exe):
            text.tofile(tf)
            try:
                r = subprocess.run([exe, tf, vf, "3", "10000", "4096"], capture_output=True, text=True, timeout=600)
                info = json.loads(r.stdout.strip().splitlines()[-1])
                ok = info.get("n_ids") == n_ids
                b = info.get("batch")
                if b:
                    res["batch_cpp_10000x4KiB"] = {
                        "texts": b["texts"], "text_bytes": b["bytes"], "ids": b["n_ids"],
                        "gb_per_s_fresh_vector": b["bytes"] / b["fresh_vector_best_seconds"] / 1e9,
                        "gb_per_s_reused_vector": b["bytes"] / b["reused_vector_best_seconds"] / 1e9,
                        "seconds_best_of_5": [b["fresh_vector_best_seconds"], b["reused_vector_best_seconds"]],
                        "call": "word_piece::fast::Encoder::encodeBatch(const std::vector<std::string>&, std::vector<int>&, "
                                "std::vector<size_t>&) (include/word_piece.hpp): pageable strings in, a std::vector<int> "
                                "out (a fresh one / one that keeps its storage between calls)"}
                res["e2e_dropin"] = {"value": text.size / info["best_seconds"] / 1e9, "unit": UNIT,
                                     "call": "word_piece::fast::encode(const std::string&, const std::vector<std::string>&) "
                                             "-> std::vector<int> (include/word_piece.hpp), pageable memory both ways",
                                     "best_of": info["reps"], "seconds": info["seconds"], "ids_match": ok,
                                     "result_vector_fill_seconds": info.get("vector_seconds")}
            except Exception as e:
                res["e2e_dropin"] = {"error": f"{type(e).__name__}: {e}"}
        cut = 10_000_000
        while text[cut - 1] != 0x20:
            cut -= 1
        text[:cut].tofile(tf)
        proc = {"text_bytes": int(cut), "argv": "runner fast <text> <vocab> 8"}
        for tag, exe in (("ours", os.path.join(ROOT, "wordpiece_b200", "lib", "runner")),
                         ("reference", os.path.join(ROOT, "oracle", "_ref", "runner"))):
            if not os.path.exists(exe):
                continue
            best, total = None, None
            for _ in range(3):
                t0 = time.perf_counter()
                r = subprocess.run([exe, "fast", tf, vf, "8"], capture_output=True, text=True)
                dt = time.perf_counter() - t0
                if r.returncode != 0:
                    break
                best = dt if best is None else min(best, dt)
                total = r.stdout.strip()
            proc[tag] = {"wall_s_best_of_3": best, "stdout": total}
        res["process_10MB"] = proc
    return res


def pcie_ceiling(h_in, h_out_bytes: int, dev, barrier, max_over_ranks):
    """The two copies of an e2e step alone, concurrently on two streams, pinned memory: the ceiling of any
    host-buffer entry point on this box (all ranks copy at the same time, as in the e2e loop)."""
    import torch

    h_out = torch.empty(h_out_bytes, dtype=torch.uint8, pin_memory=True)
    d_in = torch.empty(h_in.numel(), dtype=torch.uint8, device=dev)
    d_out = torch.empty(h_out_bytes, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    best = None
    for _ in range(3):
        barrier()
        t0 = time.perf_counter()
        with torch.cuda.stream(s1):
            d_in.copy_(h_in, non_blocking=True)
        with torch.cuda.stream(s2):
            h_out.copy_(d_out, non_blocking=True)
        torch.cuda.synchronize(dev)
        sec = max_over_ranks(time.perf_counter() - t0)
        best = sec if best is None else min(best, sec)
    return best


# ------------------------------------------------------------------------------ main

def main():
    args = parse_args()
    claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    import wordpiece_b200
    from wordpiece_b200 import synth

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU path to measure)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if "WP_NCCL_DEBUG" in os.environ:
            os.environ["NCCL_DEBUG"] = os.environ["WP_NCCL_DEBUG"]
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize(dev)

    def reduce_ranks(x: float, op) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=op)
        return float(t.item())

    def max_over_ranks(x: float) -> float:
        return reduce_ranks(x, dist.ReduceOp.MAX) if world > 1 else x

    def sum_over_ranks(x: float) -> float:
        return reduce_ranks(x, dist.ReduceOp.SUM) if world > 1 else x

    # ---- workload
    g = synth.generator(args.workload)
    vocab_tokens = g.spec.vocab
    threads = max(1, (os.cpu_count() or 8) // max(1, min(world, 8)))
    shard_info = None
    if world == 1:
        n_bytes = args.mib * MIB
        h_text = torch.empty(n_bytes, dtype=torch.uint8, pin_memory=True)
        g.fill(h_text.numpy(), seed=2, n_threads=threads)
    else:
        # configs[3]: this rank's byte range of ONE corpus.  Only the blocks around the range are generated
        # (the generator is block-wise reproducible); both neighbours of a border compute the same safe cut
        # from the same bytes (wp_next_safe_cut looks at a few bytes around a position).
        total = args.corpus_gib * GIB
        total_blocks = total // synth.BLOCK
        lo, hi = total * rank // world, total * (rank + 1) // world
        b_lo = max(0, lo // synth.BLOCK - 1)
        b_hi = min(total_blocks, hi // synth.BLOCK + 2)
        gen = np.empty((b_hi - b_lo) * synth.BLOCK, np.uint8)
        g.fill(gen, seed=4, first_block=b_lo, n_threads=threads)
        base = b_lo * synth.BLOCK
        c_lo = 0 if rank == 0 else wordpiece_b200.next_safe_cut(gen, lo - base)
        c_hi = gen.size if rank == world - 1 else wordpiece_b200.next_safe_cut(gen, hi - base)
        n_bytes = c_hi - c_lo
        h_text = torch.empty(n_bytes, dtype=torch.uint8, pin_memory=True)
        h_text.numpy()[:] = gen[c_lo:c_hi]
        shard_info = {"rank": rank, "begin": int(base + c_lo), "end": int(base + c_hi)}
        del gen
    d_text = h_text.to(dev, non_blocking=False)

    vocab = wordpiece_b200.Vocab(vocab_tokens, device=local_rank)
    cap = n_bytes // 2 + 4096
    d_ids = torch.empty(cap, dtype=torch.int32, device=dev)
    d_cnt = torch.zeros(1, dtype=torch.int64, device=dev)

    # one checked pass (count; also the first warm-up)
    _, n_ids = vocab.encode_device(d_text, d_ids)
    stats = vocab.stats()
    assert n_ids <= cap, "id buffer too small for this workload"

    counts_t = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(world)]
    mine_t = torch.zeros(1, dtype=torch.int64, device=dev)
    offsets = [0]

    def step():
        """One pass.  N > 1: followed by the path's only exchange — the id counts of all shards, scanned into
        global offsets on the host (fast.cpp:125-137 does the same over its threads' vectors)."""
        if world == 1:
            vocab.encode_device_async(d_text, d_ids, d_cnt)
            return
        _, n = vocab.encode_device(d_text, d_ids)
        mine_t.fill_(n)
        dist.all_gather(counts_t, mine_t)
        offsets[:] = wordpiece_b200.global_offsets([int(c.item()) for c in counts_t])

    for _ in range(max(args.warmup, 3) - 1):
        step()
    barrier()

    sampler = ClockSampler(physical_gpu_index(local_rank))
    sampler.start()
    launches0 = wordpiece_b200.kernel_launch_count()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    sampler.stop()
    launches = int(sum_over_ranks(float(wordpiece_b200.kernel_launch_count() - launches0)))
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    ms_step = ms_total / args.steps
    assert int(d_cnt.item()) == n_ids or world > 1
    if args.dump_outputs:
        # the last timed step's own count (d_cnt, or this rank's gathered count) and ids
        n_last = int(d_cnt.item()) if world == 1 else int(counts_t[rank].item())
        dump_outputs(args.dump_outputs if world == 1 else os.path.join(args.dump_outputs, f"rank{rank}"),
                     d_ids, n_last, len(vocab_tokens), sample=DUMP_SAMPLE // world, first_id=offsets[rank])

    total_bytes = sum_over_ranks(float(n_bytes))
    total_ids = sum_over_ranks(float(n_ids))
    value = total_bytes / (ms_step * 1e-3) / 1e9
    tokens_per_s = total_ids / (ms_step * 1e-3)

    # ---- roofline.  Algorithmic bytes = text + 4 x ids (SURVEY 8(d)), this rank.  The path is K1 / K2 (+K2L) / K3
    # per range of at most 64 MiB; their device times come from CUDA events the library records on the launching
    # stream around each launch (wp_set_kernel_timing), in a separate short pass so that the timed loop
    # above carries no extra events.  The roofline object is for the DOMINANT kernel, as the contract asks;
    # `whole_path_frac` is the same bytes over the whole step.
    peak, peak_src = measured_peak()
    algo_bytes = float(n_bytes) + 4.0 * float(n_ids)
    my_ms = e0.elapsed_time(e1) / args.steps
    names = ["wp_split_kernel", "wp_match_kernel", "wp_scatter_kernel"]
    vocab.set_kernel_timing(True)
    k_ms = [0.0, 0.0, 0.0]
    prof_steps = 3
    n_ranges = 1
    for _ in range(prof_steps):
        vocab.encode_device_async(d_text, d_ids, d_cnt)
        ms, n_ranges = vocab.last_kernel_ms()
        k_ms = [a + b for a, b in zip(k_ms, ms)]
    vocab.set_kernel_timing(False)
    k_ms = [x / prof_steps for x in k_ms]
    dom = int(np.argmax(k_ms))
    achieved = algo_bytes / (k_ms[dom] * 1e-3) / 1e9
    prof = traffic_from_profile()
    traffic = None
    if prof and names[dom] in prof.get("per_kernel", {}):
        traffic = prof["per_kernel"][names[dom]].get("dram_bytes")
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "kernel": names[dom],
                "algo_bytes_per_launch": algo_bytes / max(n_ranges, 1), "launches_per_step": n_ranges,
                "kernel_ms_per_launch": k_ms[dom] / max(n_ranges, 1),
                "kernel_ms_per_step": dict(zip(names, k_ms)), "step_ms": my_ms,
                "whole_path_achieved": algo_bytes / (my_ms * 1e-3) / 1e9,
                "whole_path_frac": algo_bytes / (my_ms * 1e-3) / 1e9 / peak,
                "peak_source": peak_src,
                "note": "achieved = (text bytes + 4 x ids) of one range / device time of the dominant kernel for that "
                        "range (CUDA events on the launching stream; wp_match_kernel includes the long-segment "
                        "kernel); a step = launches_per_step x (scratch memset + K1 + K2 + K2L + K3)"}
    if prof:
        # the capture is one launch over a FULL 64 MiB range (a step also has a 2 MiB, an 8 MiB and a tail range)
        roofline["traffic_launch_algo_bytes"] = algo_bytes * min(1.0, 64.0 * MIB / n_bytes)
        roofline["traffic_source"] = prof.get("source")

    # ---- e2e: the host-buffer C-ABI call (pinned host text in, host ids out), copies inside the timed region
    e2e = None
    if not args.no_e2e:
        h_ids = torch.empty(cap, dtype=torch.int32, pin_memory=True)
        h_ids_np = h_ids.numpy()
        h_text_np = h_text.numpy()
        e2e_steps = max(2, min(args.steps, 5))
        vocab.encode_into(h_text_np, h_ids_np)  # warm-up: sizes the library's device staging buffers
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            got = vocab.encode_into(h_text_np, h_ids_np)
        torch.cuda.synchronize(dev)
        sec = time.perf_counter() - t0
        barrier()
        assert got == n_ids
        sec = max_over_ranks(sec)
        e2e = {"value": total_bytes * e2e_steps / sec / 1e9, "unit": UNIT, "h2d_bytes_per_step": int(total_bytes),
               "d2h_bytes_per_step": int(4 * total_ids), "steps": e2e_steps,
               "call": "wp_encode_into (C ABI, include/wordpiece_b200.h) with pinned host text and id buffers",
               "timing": "host wall clock around synchronous calls, max over ranks"}
        # the ids that came back are the ones the device-resident path produced
        assert np.array_equal(h_ids_np[:n_ids], d_ids[:n_ids].cpu().numpy())
        ceil_sec = pcie_ceiling(h_text, 4 * n_ids, dev, barrier, max_over_ranks)
        e2e["pcie_ceiling"] = {"value": total_bytes / ceil_sec / 1e9, "unit": UNIT, "ms": ceil_sec * 1e3,
                               "what": "the step's H2D and D2H bytes as two monolithic concurrent pinned copies per "
                                       "rank, all ranks at once, no kernel: the bound of any host-buffer entry on this box"}
        e2e["frac_of_pcie_ceiling"] = e2e["value"] / e2e["pcie_ceiling"]["value"]
        del h_ids

    # ---- N > 1: the optional gather of every shard's ids on rank 0 (NCCL send/recv over NVLink), timed separately
    gather = None
    shards = None
    if world > 1:
        infos = [None] * world
        dist.all_gather_object(infos, dict(shard_info, n_ids=int(n_ids)))
        offs = wordpiece_b200.global_offsets([i["n_ids"] for i in infos])
        shards = [dict(i, id_offset=int(o)) for i, o in zip(infos, offs)]
        if not args.no_gather:
            tot = int(total_ids)
            d_all = torch.empty(tot if rank == 0 else 1, dtype=torch.int32, device=dev)
            best = None
            for _ in range(3):
                barrier()
                g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                g0.record()
                if rank == 0:
                    d_all[:n_ids].copy_(d_ids[:n_ids])
                    ops = [dist.P2POp(dist.irecv, d_all[offs[r]:offs[r] + infos[r]["n_ids"]], r) for r in range(1, world)]
                else:
                    ops = [dist.P2POp(dist.isend, d_ids[:n_ids], 0)]
                for req in dist.batch_isend_irecv(ops):
                    req.wait()
                g1.record()
                barrier()
                ms = max_over_ranks(g0.elapsed_time(g1))
                best = ms if best is None else min(best, ms)
            ok = None
            if rank == 0:
                ok = bool(torch.equal(d_all[:n_ids], d_ids[:n_ids]))
            gather = {"ms": best, "bytes": 4 * tot, "gb_per_s": 4 * tot / (best * 1e-3) / 1e9, "rank0_part_intact": ok,
                      "how": "grouped ncclSend/ncclRecv (torch batch_isend_irecv), every shard's ids to rank 0's "
                             "device at its scanned offset; not part of `value`"}
            del d_all

    # ---- CPU baseline and the other legs (rank 0, N = 1 only)
    cpu = None
    extra = {}
    if rank == 0 and world == 1:
        if not args.no_cpu_baseline:
            info = cpu_reference_timing(h_text.numpy(), vocab_tokens, min(args.cpu_sample_mib, args.mib))
            cpu = {"value": info["bytes"] / info["seconds"] / 1e9, "unit": UNIT, "cores": info["cores"],
                   "kind": info["kind"], "sample": info["sample"], "tokens_per_s": info["ids"] / info["seconds"]}
        if not args.no_configs:
            try:
                extra["configs"] = other_configs(local_rank, peak)
                extra["configs"]["latency_4KiB"] = latency_4k(h_text.numpy(), vocab)
                extra["configs"]["batch_10000x4KiB"] = batch_throughput(h_text.numpy(), vocab, 10000, 4096)
                extra["configs"]["batch_100000x256B"] = batch_throughput(h_text.numpy(), vocab, 100000, 256)
                extra.update(dropin_and_process(h_text.numpy(), vocab_tokens, n_ids))
            except Exception as e:  # the headline must survive a failing side leg
                extra["configs_error"] = f"{type(e).__name__}: {e}"

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {
                "workload": workload_name(args, world),
                "text_bytes_total": int(total_bytes), "ids_total": int(total_ids), "text_bytes_rank0": n_bytes,
                "vocab_entries": len(vocab_tokens),
                "sharding": "none (1 GPU, BASELINE configs[1])" if world == 1 else
                            f"configs[3]: one {args.corpus_gib} GiB corpus, {world} contiguous byte ranges cut at safe "
                            f"starts (wp_next_safe_cut), replicated vocab, per step: encode + all_gather of the id "
                            f"counts + host exclusive scan; no collective on the data path",
                "shards": shards,
                "l2": "input and output per GPU are far larger than the 126 MB L2; no flush needed",
                "tiles_rank0": stats.n_tiles, "dirty_tiles": stats.dirty_tiles, "long_segments": stats.long_segments,
            },
            "tokens_per_s": tokens_per_s,
            "roofline": roofline,
            "cpu_baseline": cpu,
            "e2e": e2e,
            "gather": gather,
            "gpu_launches": int(launches),
            "clocks": sampler.summary(),
        }
        line.update(extra)
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
