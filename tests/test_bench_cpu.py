"""CPU-only: bench.py's argument checks and the writer behind --dump-outputs (no GPU, no compute calls)."""
import os
import sys
import types

import numpy as np
import pytest
import torch

import bench


def _parse(monkeypatch, *argv):
    monkeypatch.setattr(sys, "argv", ["bench.py", *argv])
    return bench.parse()


def test_steps_and_dump_arguments(monkeypatch):
    a = _parse(monkeypatch, "--steps", "4", "--warmup", "0", "--dump-outputs", "d")
    assert (a.steps, a.warmup, a.dump_outputs) == (4, 0, "d")
    for bad in (["--steps", "0"], ["--warmup", "-1"], ["--dump-outputs", "d", "--impl", "reference"],
                ["--dump-outputs", "d", "--workload", "hrnn_convnet"]):
        with pytest.raises(SystemExit):
            _parse(monkeypatch, *bad)


def test_last_step_outputs_are_flat_float_arrays():
    prog = types.SimpleNamespace(last_fx=torch.arange(6, dtype=torch.float64), X=torch.randn(2, 5),
                                 nets={"cw": types.SimpleNamespace(theta=torch.randn(7))})
    out = bench.last_step_outputs(prog)
    assert sorted(out) == ["fx", "theta_cw", "x"]
    assert out["fx"].dtype == np.float64 and out["x"].dtype == np.float32 and out["theta_cw"].dtype == np.float32
    assert out["x"].shape == (10,) and np.array_equal(out["x"], prog.X.numpy().reshape(-1))


def test_dump_keeps_small_arrays_whole_and_samples_large_ones_the_same_way(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 4096)
    rng = np.random.default_rng(1)
    arrays = {"fx": rng.random(11), "x": rng.random(5000).astype(np.float32), "big": rng.random(3000)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    a = {f[:-4]: np.load(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")}
    assert sorted(a) == ["big", "fx", "x"]
    assert np.array_equal(a["fx"], arrays["fx"])                       # fits: written whole
    assert sum(v.nbytes for v in a.values()) <= 4096
    for k in ("x", "big"):
        assert a[k].dtype == arrays[k].dtype and 0 < a[k].size < arrays[k].size
        assert np.isin(a[k], arrays[k]).all()                          # a sample of the array's own elements
        assert np.array_equal(a[k], np.load(tmp_path / "b" / (k + ".npy")))   # the same sample in every run
