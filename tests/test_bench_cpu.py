"""CPU: bench.py's argument checks and `dump_outputs`, the float64 .npy files two builds are compared by."""
import os
import sys

import numpy as np
import pytest

import bench


def test_dump_outputs_layout(tmp_path):
    finals = np.arange(24).reshape(4, 3, 2) * (1 + 2j)
    bench.dump_outputs(str(tmp_path), {"cost": 0.25, "grads": np.ones((5, 2), dtype=np.float32), "final_states": finals})
    assert sorted(os.listdir(tmp_path)) == ["cost.npy", "final_states.npy", "grads.npy"]
    assert np.load(tmp_path / "cost.npy").tolist() == [0.25]
    g = np.load(tmp_path / "grads.npy")
    assert g.dtype == np.float64 and g.shape == (5, 2)
    f = np.load(tmp_path / "final_states.npy")
    assert f.dtype == np.float64 and f.shape == (4, 3, 2, 2)
    np.testing.assert_array_equal(f[..., 0] + 1j * f[..., 1], finals)


def test_dump_outputs_samples_above_the_limit(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 40000)
    a = np.random.default_rng(3).standard_normal((100, 8, 8)) * 1j           # 102400 bytes as float64 pairs
    for d in ("one", "two"):
        bench.dump_outputs(str(tmp_path / d), {"expm": a})
    total = sum(os.path.getsize(tmp_path / "one" / f) for f in os.listdir(tmp_path / "one"))
    assert total < 40000 + 2 * 128                                   # + the two .npy headers
    x, idx = np.load(tmp_path / "one" / "expm.npy"), np.load(tmp_path / "one" / "expm_index.npy")
    assert 0 < len(idx) < 100 and np.all(np.diff(idx) > 0)
    np.testing.assert_array_equal(x[..., 0] + 1j * x[..., 1], a[idx.astype(int)])
    np.testing.assert_array_equal(np.load(tmp_path / "two" / "expm_index.npy"), idx)     # seeded: same sample every run


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]])
def test_bench_rejects_bad_arguments(argv, monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    with pytest.raises(SystemExit) as e:
        bench.main()
    assert e.value.code == 2
