"""bench.py --dump-outputs: what the timed step computed, written so that two builds can be compared row for row."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_sample_is_fixed_paired_and_bounded(tmp_path):
    import torch

    n = bench.DUMP_ROWS + 1000
    nlml = torch.arange(n, dtype=torch.float64)
    grad = nlml[:, None] * torch.ones(2 * bench.DIM + 4, dtype=torch.float64)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), nlml, grad)
    v, g = np.load(tmp_path / "a" / "nlml.npy"), np.load(tmp_path / "a" / "grad.npy")
    assert v.dtype == g.dtype == np.float64 and v.shape == (bench.DUMP_ROWS,) and g.shape == (bench.DUMP_ROWS, 14)
    assert np.all(np.diff(v) > 0) and np.all(g == v[:, None])  # increasing problem order, rows of both files paired
    assert np.array_equal(v, np.load(tmp_path / "b" / "nlml.npy"))
    assert v.nbytes + g.nbytes <= 64 << 20
    bench.dump_outputs(str(tmp_path / "small"), nlml[:10], grad[:10])  # a step that fits is written whole
    assert np.array_equal(np.load(tmp_path / "small" / "nlml.npy"), np.arange(10.0))


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(tmp_path):
    from oracle import mfgp_oracle_torch as otc

    R = 4
    out = tmp_path / "dump"
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--restarts", str(R), "--steps", "3", "--warmup", "1",
                          "--no-cpu-baseline", "--no-extra", "--dump-outputs", str(out)],
                         capture_output=True, text=True, timeout=600, cwd=tmp_path)
    assert res.returncode == 0, res.stderr[-2000:]
    line = json.loads([ln for ln in res.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["steps"] == 3 and line["gpu_launches"] == 3
    nlml, grad = np.load(out / "nlml.npy"), np.load(out / "grad.npy")
    assert nlml.shape == (R * bench.NBINS,) and grad.shape == (R * bench.NBINS, 2 * bench.DIM + 4)
    X, Y = bench.load_hbs()
    th, nz = bench.make_thetas(R, 1000)  # rank 0's hyper-parameter sets
    for b in (0, 77, R * bench.NBINS - 1):
        v, g, gn = otc.gpr_lml_value_and_grad(X, Y[:, b % bench.NBINS:b % bench.NBINS + 1], th[b], nz[b])
        assert abs(nlml[b] + v) < 1e-9 * abs(v), (b, nlml[b], -v)
        want = -np.concatenate([g, [gn]])
        np.testing.assert_allclose(grad[b], want, rtol=1e-7, atol=1e-7 * np.abs(want).max())
