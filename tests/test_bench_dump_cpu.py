"""bench.py --dump-outputs: what it writes must fit its byte budget, keep small arrays whole, and sample large ones at the same
positions on every run, so that two builds run with the same arguments can be compared array for array."""
import importlib.util
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_dump_outputs_budget_dtypes_and_fixed_sample(tmp_path):
    bench = _bench()
    bench.DUMP_BYTES = 1 << 20
    g = torch.Generator().manual_seed(0)
    arrays = dict(big=torch.randn(300_000, generator=g), big_bf16=torch.randn(600, 500, generator=g).bfloat16(),
                  small=torch.randn(4, 8, generator=g, dtype=torch.float64), count=torch.tensor(7))
    bench.dump_outputs(str(tmp_path / "a"), arrays)
    bench.dump_outputs(str(tmp_path / "b"), arrays)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["big.npy", "big_bf16.npy", "count.npy", "small.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in names) <= bench.DUMP_BYTES
    a = {n[:-4]: np.load(tmp_path / "a" / n) for n in names}
    for n in names:
        assert np.array_equal(a[n[:-4]], np.load(tmp_path / "b" / n))
    assert a["big"].dtype == a["big_bf16"].dtype == np.float32
    assert a["small"].dtype == a["count"].dtype == np.float64
    assert np.array_equal(a["small"], arrays["small"].numpy()) and a["count"] == 7
    assert 0 < a["big"].size < 300_000 and np.isin(a["big"], arrays["big"].numpy()).all()


def test_steps_must_be_positive(monkeypatch):
    bench = _bench()
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "0"])
    with pytest.raises(SystemExit):
        bench.parse()
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "7", "--dump-outputs", "out"])
    a = bench.parse()
    assert a.steps == 7 and a.dump_outputs == "out"
