"""CPU checks of bench.py's --dump-outputs writer and argument checks (the timed path itself needs the GPU)."""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _results(seed):
    g = torch.Generator().manual_seed(seed)
    big = torch.randn(2, 1024, 600, generator=g).bfloat16()               # 1.2 M elements: sampled
    x = torch.randn(2, 1024, 3, 2, generator=g)
    grads = (big.clone(), big.clone(), torch.randn(1024, 1, generator=g), torch.randn(2, 4, 1, 600, generator=g).bfloat16(),
             torch.randn(2, 4, 1, 600, generator=g).bfloat16(), torch.randn(1024, generator=g), None, None)
    return [(big, x, grads)]


def test_dump_writes_float32_samples_at_fixed_places(tmp_path):
    import bench
    res = _results(0)
    bench.dump_outputs(str(tmp_path / "a"), ["w"], res)
    bench.dump_outputs(str(tmp_path / "b"), ["w"], _results(0))
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(f"w.{n}.npy" for n in ("out", "last_state", "du", "ddelta", "dA", "dB", "dC", "dD"))
    total = 0
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float32 and np.array_equal(a, b), f
        total += a.nbytes
    assert total <= bench.DUMP_MAX_BYTES
    out = np.load(tmp_path / "a" / "w.out.npy")
    assert out.shape == (bench.DUMP_MAX_ELEMS,)
    assert np.isin(out, res[0][0].float().numpy()).all()                  # a sample of the array, not something else
    assert np.array_equal(np.load(tmp_path / "a" / "w.last_state.npy"), res[0][1][:, :, -1, 1::2].numpy())
    assert np.array_equal(np.load(tmp_path / "a" / "w.dB.npy"), res[0][2][3].float().numpy())   # small arrays whole


def test_bench_rejects_zero_steps():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True)
    assert r.returncode == 2 and "--steps" in r.stderr
