"""CPU: bench.py --dump-outputs.  The same arguments must give the same arrays, every array is float32 or float64,
and the dump stays within its byte budget (larger arrays become a fixed, seeded sample).  Runs the CPU reference arm
end to end at a toy size, and dump_outputs itself with a small budget."""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def _run(out):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                        "--warmup", "1", "--size", "64", "--batch", "2", "--dump-outputs", out],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    return {f[:-4]: np.load(os.path.join(out, f)) for f in sorted(os.listdir(out))}


def test_reference_arm_dump_is_reproducible(tmp_path):
    a, b = _run(str(tmp_path / "a")), _run(str(tmp_path / "b"))
    assert sorted(a) == ["buffers", "grads", "loss", "params"]
    assert sum(x.nbytes for x in a.values()) <= bench.DUMP_BYTES
    for k in a:
        assert a[k].dtype in (np.float32, np.float64) and np.isfinite(a[k]).all(), k
        assert np.array_equal(a[k], b[k]), k
    assert a["loss"].shape == (1,) and a["params"].size == bench.DUMP_BYTES // 4 // 4     # sampled to its share


def test_dump_outputs_budget_and_sampling(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 4096)
    big = torch.arange(10000, dtype=torch.int64)
    arrays = {"small": torch.tensor([1.5, 2.5], dtype=torch.float64), "big": big}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    s, g = (np.load(str(tmp_path / "a" / f"{n}.npy")) for n in ("small", "big"))
    assert s.dtype == np.float64 and s.tolist() == [1.5, 2.5]
    assert g.dtype == np.float32 and g.size == 2048 // 4                   # an even share of the budget
    assert np.all(np.diff(g) > 0) and set(g.tolist()) <= set(range(10000))   # distinct elements, in index order
    assert np.array_equal(g, np.load(str(tmp_path / "b" / "big.npy")))
