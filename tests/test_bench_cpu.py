"""``bench.py`` without a device: argument checks and the ``--dump-outputs`` writer on host tensors."""

import os
import subprocess
import sys
import types

import numpy as np
import pytest

torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_rejected_arguments(argv):
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True)
    assert proc.returncode == 2 and "error" in proc.stderr


def basis(n, seed):
    gen = torch.Generator().manual_seed(seed)
    return types.SimpleNamespace(h=torch.randn(n, n, dtype=torch.float64, generator=gen),
                                 s=torch.eye(n, dtype=torch.float64),
                                 u=torch.randn((n,) * 4, dtype=torch.float64, generator=gen))


def load(directory):
    return {name[:-4]: np.load(os.path.join(directory, name)) for name in sorted(os.listdir(directory))}


@pytest.mark.parametrize("cap", [100, 10**6])
def test_dump_outputs(tmp_path, monkeypatch, cap):
    """h and s whole; u at a fixed set of flat indices (independent of the data) when it has more than
    ``DUMP_U_SAMPLE`` elements, whole otherwise; everything float64, and the same files for the same input."""
    monkeypatch.setattr(bench, "DUMP_U_SAMPLE", cap)
    b = basis(9, 1)
    for name, which in (("a", b), ("b", b), ("c", basis(9, 2))):
        bench.dump_outputs(str(tmp_path / name), which)
    got, again, other = load(tmp_path / "a"), load(tmp_path / "b"), load(tmp_path / "c")
    assert sorted(got) == ["h", "s", "u_sample", "u_sample_index"]
    assert all(a.dtype == np.float64 for a in got.values())
    assert all(np.array_equal(got[k], again[k]) for k in got)
    np.testing.assert_array_equal(got["u_sample_index"], other["u_sample_index"])
    np.testing.assert_array_equal(got["h"], b.h.numpy())
    np.testing.assert_array_equal(got["s"], b.s.numpy())
    index = got["u_sample_index"].astype(np.int64)
    np.testing.assert_array_equal(got["u_sample"], b.u.numpy().reshape(-1)[index])
    if cap < 9**4:
        assert 0 < len(index) <= cap and np.array_equal(index, np.unique(index))
    else:
        np.testing.assert_array_equal(index, np.arange(9**4))


def test_dump_outputs_stay_under_64_mb():
    n = 128  # the one-GPU workload
    assert (2 * bench.DUMP_U_SAMPLE + 2 * n * n) * 8 <= 64 * 2**20
