"""`bench.py --dump-outputs`: the last timed step's outputs as float32 .npy files, from inputs that depend only on the
arguments, so that two builds can be compared output for output."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from _golden import rel_err

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_outputs_cap_and_fixed_sample(tmp_path):
    from bench import DUMP_BYTES, dump_outputs

    big = torch.arange(3 << 19, dtype=torch.float32)[:, None] + torch.arange(16) / 32  # 96 MB, row i holds i + j/32
    small = {"grad": torch.arange(4096.0).reshape(-1, 16), "loss": torch.tensor(1.5, dtype=torch.float64)}
    dump_outputs(str(tmp_path / "a"), {"features": big, **small})
    dump_outputs(str(tmp_path / "b"), {"features": 2 * big, **small})
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert sorted(a) == ["features", "grad", "loss"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= DUMP_BYTES
    assert all(v.dtype == np.float32 for v in a.values())
    assert np.array_equal(a["grad"], small["grad"].numpy()) and a["loss"].shape == () and a["loss"] == 1.5
    f = a["features"]
    assert f.shape[1] == 16 and 0 < f.shape[0] < big.shape[0]
    rows = f[:, 0].astype(np.int64)  # whole rows, in order, no repeats
    assert np.array_equal(f, big.numpy()[rows]) and (np.diff(rows) > 0).all()
    assert np.array_equal(b["features"], 2 * f)  # the same rows for the same shape


@pytest.mark.gpu
def test_bench_dump_outputs_repeat(tmp_path):
    """Two runs with different step counts dump the same outputs of the same inputs (up to the order of the
    gradient atomics), and the loss is the MSE of the dumped features to the bench's seeded target."""
    runs = []
    for steps in (1, 2):
        out = tmp_path / f"steps{steps}"
        subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup",
                        "1", "--width", "64", "--height", "32", "--skip-cpu-baseline", "--skip-in-volume",
                        "--dump-outputs", str(out)], check=True, cwd=str(tmp_path))
        runs.append(_load(out))
    a, b = runs
    assert sorted(a) == ["features", "grad_grid", "grad_harmonic_ray_embedding_linear_bias",
                         "grad_harmonic_ray_embedding_linear_weight", "grad_mlp_params", "loss"]
    assert a["features"].shape == (64 * 32, 3) and a["grad_grid"].shape == (3 * 64 * 64, 16)
    for k in a:
        assert a[k].dtype == np.float32 and np.isfinite(a[k]).all(), k
        assert rel_err(a[k], b[k]) < 1e-5, (k, rel_err(a[k], b[k]))
    target = torch.rand(64 * 32, 3, generator=torch.Generator().manual_seed(0)).numpy()
    assert abs(float(((a["features"] - target) ** 2).mean()) - float(a["loss"])) < 1e-5 * float(a["loss"])
