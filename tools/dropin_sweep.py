#!/usr/bin/env python3
"""word_piece::fast::encode(std::string, vector<string>) on 1 GiB through the C++ helper (lib/dropin_bench) under
combinations of the host-copy switches: WORDPIECE_B200_COPY_THREADS, WORDPIECE_B200_STREAM_STORES (staging
copies in); `--set hugepages`: the transparent-huge-page advice on the result vector on / off
(WORDPIECE_B200_HUGEPAGES).   python tools/dropin_sweep.py [--mib 1024] [--set ...]"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from wordpiece_b200 import synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--mib", type=int, default=1024)
ap.add_argument("--set", default="copies", choices=["copies", "hugepages"])
a = ap.parse_args()
g = synth.generator("en")
text = g.generate(a.mib << 20, seed=2)
exe = os.path.join(ROOT, "wordpiece_b200", "lib", "dropin_bench")
shm = "/dev/shm" if os.path.isdir("/dev/shm") else None
with tempfile.TemporaryDirectory(dir=shm) as d:
    tf, vf = os.path.join(d, "text.txt"), os.path.join(d, "vocab.txt")
    text.tofile(tf)
    with open(vf, "wb") as f:
        f.write(b"\n".join(t if isinstance(t, bytes) else t.encode() for t in g.spec.vocab) + b"\n")
    base = [dict(), dict(WORDPIECE_B200_STREAM_STORES="0"), dict(WORDPIECE_B200_COPY_THREADS="16"),
            dict(WORDPIECE_B200_COPY_THREADS="16", WORDPIECE_B200_STREAM_STORES="0"),
            dict(WORDPIECE_B200_COPY_THREADS="8"), dict(WORDPIECE_B200_COPY_THREADS="8", WORDPIECE_B200_STREAM_STORES="0")]
    combos = base * 3  # interleaved and repeated: the box's state drifts between runs
    if a.set == "hugepages":
        for knob in ("enabled", "defrag"):
            try:
                print(json.dumps({"transparent_hugepage/" + knob: open("/sys/kernel/mm/transparent_hugepage/" + knob).read().strip()}))
            except OSError as ex:
                print(json.dumps({"transparent_hugepage/" + knob: repr(ex)}))
        combos = [dict(WORDPIECE_B200_HUGEPAGES="1"), dict()] * 3
    for env in combos:
        e = dict(os.environ)
        e.update(env)
        r = subprocess.run([exe, tf, vf, "4"], capture_output=True, text=True, env=e, timeout=600)
        try:
            info = json.loads(r.stdout.strip().splitlines()[-1])
            print(json.dumps({"env": env, "gb_per_s": round(text.size / info["best_seconds"] / 1e9, 2), "seconds": info["seconds"]}), flush=True)
        except Exception as ex:  # noqa: BLE001
            print(json.dumps({"env": env, "error": repr(ex), "stderr": r.stderr[-300:]}), flush=True)
