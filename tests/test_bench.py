"""CPU checks of bench.py's command line and of the waveform it writes with --dump-outputs."""
import sys

import numpy as np
import pytest
import torch

import bench


def test_dump_waveform_whole_and_seeded_sample(tmp_path, monkeypatch):
    w = torch.arange(5 * 12, dtype=torch.float32).reshape(5, 1, 12)
    bench.dump_waveform(str(tmp_path / "all"), w)
    assert np.array_equal(np.load(tmp_path / "all" / "waveform.npy"), w.numpy())
    monkeypatch.setattr(bench, "DUMP_BYTES", 2 * 12 * 4)
    bench.dump_waveform(str(tmp_path / "a"), w)
    bench.dump_waveform(str(tmp_path / "b"), w)
    a, b = np.load(tmp_path / "a" / "waveform.npy"), np.load(tmp_path / "b" / "waveform.npy")
    assert a.dtype == np.float32 and a.shape == (2, 1, 12) and np.array_equal(a, b)
    assert all(any(np.array_equal(r, x) for x in w.numpy()) for r in a)      # whole utterances of the batch
    monkeypatch.setattr(bench, "DUMP_BYTES", 5 * 4)                           # one utterance is larger than the limit
    bench.dump_waveform(str(tmp_path / "c"), w)
    assert np.load(tmp_path / "c" / "waveform.npy").shape == (1, 1, 5)


def test_steps_and_dump_arguments(monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "7", "--dump-outputs", "out"])
    a = bench.parse()
    assert a.steps == 7 and a.dump_outputs == "out"
    for bad in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        monkeypatch.setattr(sys, "argv", ["bench.py"] + bad)
        with pytest.raises(SystemExit):
            bench.parse()
