"""bench.py's command line and --dump-outputs writer (no GPU: the timed path itself is exercised by bench.py on the device)."""
import os
import sys

import numpy as np
import pytest

import bench


def parse(monkeypatch, *argv):
    monkeypatch.setattr(sys, "argv", ["bench.py"] + list(argv))
    return bench.parse()


def test_steps_and_dump_arguments(monkeypatch):
    a = parse(monkeypatch, "--gpus", "1", "--steps", "7", "--warmup", "2", "--dump-outputs", "out")
    assert a.steps == 7 and a.warmup == 2 and a.dump_outputs == "out"
    with pytest.raises(SystemExit):
        parse(monkeypatch, "--steps", "0")
    with pytest.raises(SystemExit):
        parse(monkeypatch, "--impl", "reference", "--dump-outputs", "out")


def test_dump_outputs_whole_and_sampled(tmp_path):
    small = np.arange(1000, dtype=np.float32)
    bench.dump_outputs(str(tmp_path / "a"), {"hpsi": small})
    got = np.load(tmp_path / "a" / "hpsi.npy")
    assert got.dtype == np.float64 and np.array_equal(got, small)
    big = np.random.default_rng(3).standard_normal(bench.DUMP_BYTES // 8 + 12345)
    for d in ("b", "c"):
        bench.dump_outputs(str(tmp_path / d), {"hpsi": big})
    b, c = np.load(tmp_path / "b" / "hpsi.npy"), np.load(tmp_path / "c" / "hpsi.npy")
    assert np.array_equal(b, c) and b.size < big.size                    # the same fixed sample every time
    assert os.path.getsize(tmp_path / "b" / "hpsi.npy") <= bench.DUMP_BYTES
    assert np.isin(b, big).all()
