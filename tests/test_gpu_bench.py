"""bench.py --dump-outputs on the default workload (batch cut to 512 samples, so the dump still has to sample rows): the
files hold the last timed step's outputs in float64 within 64 MB, and two runs with the same arguments dump the same
rows of the same results."""
import json
import pathlib
import subprocess
import sys

import numpy as np
import pytest
import torch

from difffe_physics_lab_b200 import _native

pytestmark = pytest.mark.gpu
ROOT = pathlib.Path(__file__).resolve().parent.parent


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    _native.build()


def run_bench(out_dir):
    cmd = [sys.executable, str(ROOT / "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1", "--batch", "512",
           "--no-e2e", "--no-cpu", "--no-sweep", "--no-parity", "--dump-outputs", str(out_dir)]
    res = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-3000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    return line, {p.stem: np.load(p) for p in sorted(out_dir.glob("*.npy"))}


def test_dump_outputs_repeatable(tmp_path):
    line, a = run_bench(tmp_path / "a")
    assert line["steps"] == 2 and line["config"]["batch_per_gpu"] == 512
    assert set(a) == {"u", "grad_f", "grad_kappa"}
    assert all(v.dtype == np.float64 and np.isfinite(v).all() for v in a.values())
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= 64 * 10 ** 6
    nn = 100001
    assert a["grad_kappa"].shape == (512, 1)
    assert 0 < a["u"].shape[0] < 512 and a["u"].shape == a["grad_f"].shape and a["u"].shape[1] == nn
    assert np.all(a["u"][:, 0] == 0.0) and np.all(a["u"][:, -1] == 0.0)          # the line mesh's Dirichlet ends
    _, b = run_bench(tmp_path / "b")
    for k in a:
        assert a[k].shape == b[k].shape
        np.testing.assert_allclose(b[k], a[k], rtol=1e-12, atol=1e-12 * np.abs(a[k]).max())
