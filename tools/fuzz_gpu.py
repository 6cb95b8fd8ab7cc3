#!/usr/bin/env python3
"""Randomised parity sweep on a B200: hostile texts and vocabularies (tests/textgen.py) through randomly
chosen entry points, range sizes and memo settings, every result compared with the CPU oracle.
    python tools/fuzz_gpu.py [--seconds 120] [--seed0 1000]
Prints one line per failure (with the seed to reproduce) and a summary; exit code 1 if anything differed."""
from __future__ import annotations

import argparse
import os
import random
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import textgen  # noqa: E402
import wordpiece_b200  # noqa: E402
from _oracle import Oracle  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=120.0)
    ap.add_argument("--seed0", type=int, default=1000)
    ap.add_argument("--seeds", type=str, default="", help="comma-separated seeds to run (each --repeat times) instead of a sweep")
    ap.add_argument("--repeat", type=int, default=1)
    args = ap.parse_args()
    tile = wordpiece_b200.tile_bytes()
    t_end = time.time() + args.seconds
    seed, fails, cases, total_bytes = args.seed0, 0, 0, 0
    by_entry = {}
    todo = [int(x) for x in args.seeds.split(",") if x] * args.repeat
    while (todo or not args.seeds) and (args.seeds or time.time() < t_end):
        if args.seeds:
            seed = todo.pop(0)
        rng = random.Random(seed)
        n = int(10 ** rng.uniform(1.0, 6.4))
        kw = dict(invalid_rate=rng.choice([0.0, 0.0, 0.0005, 0.01, 0.2]),
                  long_run_rate=rng.choice([0.0, 0.0, 0.02, 0.1]),
                  long_tokens=rng.choice([0, 0, 5, 40]))
        text, vocab = textgen.case(seed, n, **kw)
        if rng.random() < 0.15:  # no [UNK] => -1
            vocab = [t for t in vocab if t != b"[UNK]"]
        try:
            exp = Oracle(vocab).encode(text)
        except Exception as e:  # outside the reference's domain (e.g. empty vocab word): skip
            seed += 1
            continue
        os.environ["WORDPIECE_B200_MEMO"] = rng.choice(["0", "1", "1"])
        os.environ["WORDPIECE_B200_RANGE_BYTES"] = str(tile * rng.choice([1, 2, 3, 7, 16, 64, 1 << 14]))
        if rng.random() < 0.5:
            os.environ["WORDPIECE_B200_PIPE_CHUNK"] = str(rng.choice([4096, 20000, 150000]))
        else:
            os.environ.pop("WORDPIECE_B200_PIPE_CHUNK", None)
        os.environ["WORDPIECE_B200_TICKET"] = "1" if rng.random() < 0.1 else "0"
        entry = rng.choice(["encode", "encode_into", "encode_into_pinned", "encode_device", "encode_text", "encode_batch",
                            "encode_batch_device"])
        v = wordpiece_b200.Vocab(vocab, device=0)
        if rng.random() < 0.3:  # a handle that has already encoded something else (scratch, memo and shared memory in use)
            other, _ = textgen.case(seed + 77777, min(n, 200000), **kw)
            v.encode(other)
        try:
            if entry in ("encode_batch", "encode_batch_device"):
                # the text cut at arbitrary BYTE positions (also inside a UTF-8 sequence, inside a word): every piece
                # must get the ids the oracle gives that piece alone
                k_cuts = rng.choice([0, 1, 3, 17, 200, 3000])
                cuts = sorted(rng.randrange(0, len(text) + 1) for _ in range(k_cuts)) if text else []
                pieces = [text[a:b] for a, b in zip([0] + cuts, cuts + [len(text)])]
                if rng.random() < 0.5:
                    os.environ["WORDPIECE_B200_BATCH_PART"] = str(rng.choice([256, 5000, 70000]))
                else:
                    os.environ.pop("WORDPIECE_B200_BATCH_PART", None)
                o = Oracle(vocab)
                exp_parts = [o.encode(p) for p in pieces]
                exp = np.concatenate(exp_parts) if exp_parts else np.zeros(0, np.int32)
                if entry == "encode_batch":
                    got, offs = v.encode_batch(pieces)
                else:
                    # the pieces as a slice of a larger column: unused bytes before and after, d_offsets[0] > 0, and
                    # d_chars at any alignment
                    lead, trail, shift = rng.randrange(1, 5000), rng.randrange(0, 5000), rng.randrange(0, 16)
                    blob = bytes(rng.randrange(256) for _ in range(shift + lead)) + text + b"\xff" * trail
                    base = torch.frombuffer(bytearray(blob), dtype=torch.uint8).cuda()
                    d_chars = base[shift:]
                    d_offsets = torch.tensor([lead] + [lead + c for c in cuts] + [lead + len(text)], dtype=torch.int64,
                                             device="cuda")
                    d_ids, d_offs, k = v.encode_batch_device(d_chars, d_offsets)
                    got, offs = d_ids[:k].cpu().numpy(), d_offs.cpu().numpy()
                exp_offs = np.concatenate([[0], np.cumsum([len(e) for e in exp_parts])])
                assert np.array_equal(np.asarray(offs, dtype=np.int64), exp_offs.astype(np.int64)), "text offsets differ"
            elif entry == "encode":
                got = v.encode(text)
            elif entry == "encode_into":
                out = np.full(len(exp) + 3, -7, np.int32)
                k = v.encode_into(text, out)
                got = out[:k]
                assert (out[k:] == -7).all()
            elif entry == "encode_into_pinned":
                pin = torch.full((len(exp) + 3,), -7, dtype=torch.int32).pin_memory()
                k = v.encode_into(text, pin.numpy())
                got = pin.numpy()[:k].copy()
            elif entry == "encode_device":
                d = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda() if text else torch.empty(0, dtype=torch.uint8, device="cuda")
                ids, k = v.encode_device(d)
                got = ids[:k].cpu().numpy()
            else:
                s = v.encode_text(text)
                got = np.array([int(x) for x in s.split()], dtype=np.int32) if s else np.zeros(0, np.int32)
                assert s == b"".join(b"%d " % i for i in got.tolist())
            ok = np.array_equal(exp, got)
        except Exception as e:  # noqa: BLE001
            ok = False
            print(f"EXC seed={seed} entry={entry} n={n} kw={kw}: {e!r}", flush=True)
        if not ok:
            fails += 1
            try:
                m = min(len(exp), len(got))
                diff = np.nonzero(exp[:m] != got[:m])[0]
                k = int(diff[0]) if diff.size else m
                print(f"  sizes oracle {len(exp)} gpu {len(got)}, first mismatch at {k}, mismatches {int(diff.size)}: oracle "
                      f"{exp[max(0, k - 2):k + 6].tolist()} gpu {got[max(0, k - 2):k + 6].tolist()}", flush=True)
            except Exception:  # noqa: BLE001
                pass
            print(f"FAIL seed={seed} entry={entry} n={n} kw={kw} memo={os.environ['WORDPIECE_B200_MEMO']} "
                  f"range={os.environ['WORDPIECE_B200_RANGE_BYTES']} pipe={os.environ.get('WORDPIECE_B200_PIPE_CHUNK')}",
                  flush=True)
        v.close()
        cases += 1
        total_bytes += len(text)
        by_entry[entry] = by_entry.get(entry, 0) + 1
        seed += 1
    print(f"fuzz: {cases} cases, {total_bytes / 1e6:.1f} MB, {fails} failures, seeds {args.seed0}..{seed - 1}, {by_entry}")
    sys.exit(1 if fails else 0)


if __name__ == "__main__":
    main()
