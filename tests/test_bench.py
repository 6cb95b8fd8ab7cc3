"""bench.py's own logic: its argument checks and the files --dump-outputs writes (CPU), and that those files hold
what the timed path computed (GPU)."""
from __future__ import annotations

import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

DUMP_FILES = ["id_histogram.npy", "ids_sample.npy", "ids_sample_positions.npy", "n_ids.npy"]


def _load(d, name):
    return np.load(os.path.join(d, f"{name}.npy"))


def test_argument_checks():
    for argv, message in ((["--steps", "0"], "--steps must be at least 1"),
                          (["--impl", "reference", "--dump-outputs", "x"], "not available with --impl reference")):
        r = subprocess.run([sys.executable, os.path.join(bench.ROOT, "bench.py"), *argv], capture_output=True, text=True)
        assert r.returncode != 0 and message in r.stderr, (argv, r.stderr)


def test_dump_outputs(tmp_path, monkeypatch):
    ids = torch.randint(-1, 500, (30_000,), dtype=torch.int32)
    bench.dump_outputs(str(tmp_path / "all"), ids, 20_000, 500)
    assert sorted(os.listdir(tmp_path / "all")) == DUMP_FILES
    assert all(_load(tmp_path / "all", n[:-4]).dtype == np.float64 for n in DUMP_FILES)
    assert _load(tmp_path / "all", "n_ids").tolist() == [20_000]
    assert np.array_equal(_load(tmp_path / "all", "ids_sample"), ids[:20_000].numpy())
    assert np.array_equal(_load(tmp_path / "all", "ids_sample_positions"), np.arange(20_000))
    assert np.array_equal(_load(tmp_path / "all", "id_histogram"), np.bincount(ids[:20_000].numpy() + 1, minlength=501))

    # more ids than the sample holds: a seeded sample, the same in every run
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 1000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), ids, 20_000, 500, sample=bench.DUMP_SAMPLE)
    pos = _load(tmp_path / "a", "ids_sample_positions").astype(np.int64)
    assert 900 < pos.size <= 1000 and np.all(np.diff(pos) > 0) and pos[-1] < 20_000
    assert np.array_equal(_load(tmp_path / "a", "ids_sample"), ids.numpy()[pos])
    assert np.array_equal(_load(tmp_path / "a", "id_histogram"), _load(tmp_path / "all", "id_histogram"))
    for n in ("ids_sample", "ids_sample_positions"):
        assert np.array_equal(_load(tmp_path / "a", n), _load(tmp_path / "b", n))

    # one shard of N: a smaller sample, positions into the whole corpus's ids
    bench.dump_outputs(str(tmp_path / "shard"), ids, 20_000, 500, sample=250, first_id=70_000)
    pos = _load(tmp_path / "shard", "ids_sample_positions").astype(np.int64)
    assert 200 < pos.size <= 250 and pos[0] >= 70_000 and pos[-1] < 90_000
    assert np.array_equal(_load(tmp_path / "shard", "ids_sample"), ids.numpy()[pos - 70_000])


@pytest.mark.gpu
def test_dump_holds_the_timed_steps_ids(gpu_device, tmp_path):
    """bench.py end to end on a small text: the dumped count, sample and histogram are those of the CPU oracle on
    the same seeded text (12 MiB gives more ids than DUMP_SAMPLE, so the sampled form is the one checked)."""
    from _oracle import Oracle
    from wordpiece_b200 import synth

    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(bench.ROOT, "bench.py"), "--gpus", "1", "--steps", "2",
                        "--warmup", "1", "--mib", "12", "--no-cpu-baseline", "--no-e2e", "--no-configs",
                        "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    assert sorted(os.listdir(out)) == DUMP_FILES
    g = synth.generator("en")
    exp = Oracle(g.spec.vocab).encode(g.generate(12 << 20, seed=2))
    assert exp.size > bench.DUMP_SAMPLE
    assert _load(out, "n_ids").tolist() == [exp.size]
    pos = _load(out, "ids_sample_positions").astype(np.int64)
    assert pos.size > 0.6 * bench.DUMP_SAMPLE
    assert np.array_equal(_load(out, "ids_sample"), exp[pos])
    assert np.array_equal(_load(out, "id_histogram"), np.bincount(exp + 1, minlength=len(g.spec.vocab) + 1))
