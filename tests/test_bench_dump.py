"""bench.py --dump-outputs: what the last timed step returned, as float32 / float64 .npy files of at most 64 MB, the same for
the same flags; --steps sets the number of timed batch calls."""
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import helpers as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
bench = importlib.import_module("bench")


class _HostBatch:
    """The fields of swcompression_b200.batch.Batch that dump_outputs reads, on the host: unit i decodes to
    `ln[i]` bytes of value i % 251 followed by stale bytes (0xEE)."""

    def __init__(self, n):
        self.n = n
        self.h_out_off = np.arange(n, dtype=np.uint64) * np.uint64(bench.UNIT)
        self.ln = np.full(n, bench.UNIT, dtype=np.int64)
        self.ln[::7] = 100
        self.d_out = torch.full((n * bench.UNIT,), 0xEE, dtype=torch.uint8)
        for i in range(n):
            self.d_out[i * bench.UNIT: i * bench.UNIT + int(self.ln[i])] = i % 251

    def results(self):
        return np.zeros(self.n, dtype=np.int32), self.ln, self.ln * 3


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_is_float_bounded_seeded_and_zero_past_the_decoded_length(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_TABLE_UNITS", 1000)         # a batch larger than the table sample, at a host-sized n
    b = _HostBatch(1500)
    bench.dump_outputs(b, str(tmp_path / "a"))
    bench.dump_outputs(b, str(tmp_path / "b"))
    a, a2 = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert a.keys() == a2.keys() == {"units", "status", "out_len", "consumed_bits", "output_units", "output"}
    assert all(np.array_equal(a[k], a2[k]) for k in a)
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    rows = a["units"].astype(np.int64)
    assert len(rows) == 1000 and len(set(rows)) == 1000 and rows.max() < b.n
    assert np.array_equal(a["out_len"], b.ln[rows]) and np.array_equal(a["consumed_bits"], 3 * b.ln[rows])
    assert a["output"].shape == (bench.DUMP_OUTPUT_UNITS, bench.UNIT)
    for r, i in enumerate(a["output_units"].astype(np.int64)):
        m = int(b.ln[i])
        assert (a["output"][r, :m] == i % 251).all() and (a["output"][r, m:] == 0).all()


def test_dump_budget_at_the_benched_batch_size_is_at_most_64_MB():
    tables = 5 * 8 * min(bench.N_UNITS, bench.DUMP_TABLE_UNITS)          # 4 columns + the sampled output indices
    assert tables + 4 * bench.UNIT * bench.DUMP_OUTPUT_UNITS <= 64e6


@pytest.mark.gpu
def test_dump_outputs_of_the_product_arm_and_timed_step_count(tmp_path):
    units, distinct = 20480, 64            # >= 20 000 units: the batch takes the benched table-lookup decoder

    def run(steps, d):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
                            "--units", str(units), "--distinct", str(distinct), "--no-e2e", "--no-cpu", "--dump-outputs", str(d)],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, cwd=ROOT, timeout=600)
        assert p.returncode == 0, p.stderr.decode()[-2000:]
        return json.loads(p.stdout.decode())

    one, three = run(1, tmp_path / "one"), run(3, tmp_path / "three")
    assert one["steps"] == 1 and three["steps"] == 3
    assert three["gpu_launches"] == 3 * one["gpu_launches"] > 0
    a, b = _load(tmp_path / "one"), _load(tmp_path / "three")
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)
    assert sum(os.path.getsize(tmp_path / "one" / f) for f in os.listdir(tmp_path / "one")) <= 64e6
    assert np.array_equal(a["units"], np.arange(units))
    assert (a["status"] == 0).all() and (a["out_len"] == bench.UNIT).all() and (a["consumed_bits"] > 0).all()
    for r, i in enumerate(a["output_units"].astype(np.int64)):
        raw = H.textlike(bench.UNIT, 2 + i % distinct)                  # bench.make_corpus: unit i is seed 2 + i % distinct
        assert a["output"][r].astype(np.uint8).tobytes() == raw, i
