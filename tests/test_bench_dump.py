"""bench.py --dump-outputs: the loss and gradients of the last timed step, written as .npy so that two builds can be compared
output for output on the same seeded inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
from oracle import tc_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load(d):
    return {f[:-len(".npy")]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_dump_writes_the_arrays_and_samples_rows_over_the_budget(tmp_path, monkeypatch):
    g = torch.Generator().manual_seed(3)
    loss, dmu, dlv = torch.tensor(2.5), torch.randn(64, 8, generator=g), torch.randn(64, 8, generator=g)
    bench.dump_outputs(str(tmp_path / "full"), loss, dmu, dlv, 1, 0)
    got = _load(tmp_path / "full")
    assert sorted(got) == ["grad_logvar", "grad_mu", "loss"]
    assert all(a.dtype == np.float32 for a in got.values())
    assert got["loss"].tolist() == [2.5]
    assert np.array_equal(got["grad_mu"], dmu.numpy()) and np.array_equal(got["grad_logvar"], dlv.numpy())

    # room for 20 of the 64 rows: the same seeded sample on every call, its indices in rows.npy, within the budget
    monkeypatch.setattr(bench, "DUMP_BYTES", 4096 + 4 + 20 * (8 * 8 + 8))
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), loss, dmu, dlv, 1, 0)
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert a["rows"].dtype == np.float64 and a["rows"].shape == (20,) and np.array_equal(a["rows"], b["rows"])
    rows = a["rows"].astype(np.int64)
    assert np.array_equal(a["grad_mu"], dmu.numpy()[rows]) and np.array_equal(a["grad_logvar"], dlv.numpy()[rows])
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= bench.DUMP_BYTES


@pytest.mark.gpu
def test_bench_dumps_the_timed_step_on_its_seeded_inputs(tmp_path):
    """bench.py end to end at a small shape: the dumped loss and gradients are the step's on synthetic_latents(B, D),
    against the fp64 CPU oracle at the north-star tolerances."""
    B, D = 256, 32
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0", "--batch", str(B), "--zdim", str(D),
           "--no-cpu-baseline", "--no-train", "--dump-outputs", str(tmp_path)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-3000:]
    assert json.loads(res.stdout.strip().splitlines()[-1])["steps"] == 2
    got = _load(tmp_path)

    mu_c, lv_c, eps_c = (t.double() for t in bench.synthetic_latents(B, D))
    mu, lv = mu_c.requires_grad_(True), lv_c.requires_grad_(True)
    loss = O.kl_loss_simple(O.reparameterize(mu, lv, eps_c), mu, lv, bench.DATASET_SIZE, bench.BETA)
    loss.backward()
    rel = lambda a, b: float(np.abs(a.astype(np.float64) - b.numpy()).max() / b.abs().max().item())     # noqa: E731
    assert got["loss"].shape == (1,) and abs(float(got["loss"][0]) - loss.item()) <= 1e-5 * abs(loss.item())
    assert got["grad_mu"].shape == (B, D) and rel(got["grad_mu"], mu.grad) < 1e-4
    assert got["grad_logvar"].shape == (B, D) and rel(got["grad_logvar"], lv.grad) < 1e-4
