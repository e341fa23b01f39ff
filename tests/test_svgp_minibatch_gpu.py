"""GPU tests: minibatch training in the device-resident SVGP loops.  mfgp_minibatch_gather draws the rows of the NumPy twin
(tests/_minibatch_twin.py) bit for bit; optimize_on_device(minibatch_size=B) follows a host loop that feeds the twin's rows
to value_and_grad and Adam; the data-parallel loop follows the single-GPU minibatch trajectory."""
import copy
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import mfgp_oracle as onp
from tests import _minibatch_twin as twin

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def h():
    from multi_fidelity_gpflow_b200 import _lib

    hh = _lib.Handle(0)
    yield hh
    hh.close()


def _same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


def test_gather_draws_the_twins_rows(h):
    import torch

    ds = onp.load_dataset("hbs")
    N = 53
    rng = np.random.default_rng(3)
    X = np.hstack([np.arange(N, dtype=float)[:, None], ds["X"]])  # column 0 reads the index stream back
    Y = np.hstack([ds["Y"], 0.05 + rng.random(ds["Y"].shape)])   # heteroscedastic layout: 2P columns
    Y[rng.random(Y.shape) < 0.25] = np.nan                        # masked entries travel as they are
    cases = [  # (pos0, step, B, lo, count)
        (40, 0, 16, 0, 16),   # crosses the epoch boundary at 53
        (0, 5, 16, 3, 10),    # B does not divide N; a shard of the batch
        (2 * N - 1, 1, 53, 0, 53),
        (7, 2, 1, 0, 1),
    ]
    for pos0, step, B, lo, count in cases:
        Xb, Yb = h.minibatch_gather(X, Y, 17, pos0, B, lo=lo, count=count, step=step)
        r = twin.batch_rows(N, 17, pos0, step, B, lo, count)
        assert _same_bits(Xb, X[r]) and _same_bits(Yb, Y[r]), (pos0, step, B, lo, count)
    # N = 1, and the step counter on the device
    one = np.array([[4.25, 1.0]])
    Xb, _ = h.minibatch_gather(one, None, 5, 3, 1, step=torch.tensor([9], dtype=torch.int32, device="cuda"))
    assert _same_bits(Xb, one)
    dstep = torch.tensor([6], dtype=torch.int32, device="cuda")
    Xd, Yd = torch.from_numpy(X).cuda(), torch.from_numpy(Y).cuda()
    f64 = dict(dtype=torch.float64, device="cuda")
    Xb_d, Yb_d = torch.empty((9, X.shape[1]), **f64), torch.empty((9, Y.shape[1]), **f64)
    h.minibatch_gather(Xd, Yd, 2**64 - 1, 11, 12, lo=2, count=9, step=dstep, Xb=Xb_d, Yb=Yb_d)
    r = twin.batch_rows(N, 2**64 - 1, 11, 6, 12, 2, 9)
    assert _same_bits(Xb_d.cpu().numpy(), X[r]) and _same_bits(Yb_d.cpu().numpy(), Y[r])
    # a large data set several epochs in (64-bit positions, two-level Feistel domain 2^22)
    Nbig = 2**20 + 3
    Xbig = np.arange(Nbig, dtype=float)[:, None]
    pos0 = 3 * Nbig - 100
    Xb, _ = h.minibatch_gather(Xbig, None, 99, pos0, 1024, step=2)
    np.testing.assert_array_equal(Xb[:, 0].astype(np.int64), twin.batch_rows(Nbig, 99, pos0, 2, 1024))
    for bad in (dict(batch_size=54), dict(batch_size=0), dict(batch_size=16, lo=10, count=7), dict(batch_size=16, pos0=-1)):
        kw = dict(pos0=0)
        kw.update(bad)
        with pytest.raises(ValueError):
            h.minibatch_gather(X, Y, 1, kw.pop("pos0"), kw.pop("batch_size"), **kw)


def _kernels(d=5):
    from multi_fidelity_gpflow_b200.kernels import SquaredExponential

    return SquaredExponential(lengthscales=np.ones(d)), SquaredExponential(lengthscales=np.ones(d))


def _params(model):
    out = [model.q_mu.numpy(), np.tril(model.q_sqrt.numpy()), model.Z.numpy(), np.ravel(model.likelihood.variance.numpy())]
    W = getattr(model.kernel, "W", None)
    if W is not None:
        out.append(W.numpy())
    out.append(np.stack([k.theta(5) for k in model.kernel.kernels]))
    return out


def _model(kind):
    from multi_fidelity_gpflow_b200.linear_svgp import LatentMFCoregionalizationSVGP
    from multi_fidelity_gpflow_b200.singlebin_svgp import SingleBinSVGP

    ds = onp.load_dataset("hbs")
    rng = np.random.default_rng(5)
    X, Y = ds["X"], ds["Y"].copy()
    if kind == "singlebin":
        Y = np.ascontiguousarray(Y[:, :6])
        m = SingleBinSVGP(X, Y, *_kernels(), 6, ds["Z_kmeans50"])
        m.num_data = X.shape[0]
    elif kind == "hetero":
        Y = np.hstack([Y, 0.05 + 0.1 * rng.random(Y.shape)])
        m = LatentMFCoregionalizationSVGP(X, Y, *_kernels(), num_latents=4, num_inducing=20, heterosed=True)
    elif kind == "masked":
        Y[rng.random(Y.shape) < 0.25] = np.nan
        m = LatentMFCoregionalizationSVGP(X, Y, *_kernels(), num_latents=4, num_inducing=20, num_outputs=49, masked=True)
    else:
        m = LatentMFCoregionalizationSVGP(X, Y, *_kernels(), num_latents=4, num_inducing=20, num_outputs=49)
    return X, Y, m


def _host_minibatch_loop(model, X, Y, max_iters, lr, B, seed, klm=1.0):
    """GPflow's minibatch loop: the twin's rows of each step through value_and_grad (scale num_data / B), then Adam."""
    from multi_fidelity_gpflow_b200.optimizers import Adam, CosineDecay

    opt = Adam(CosineDecay(lr, max_iters))
    traced = model.trainable_variables
    losses, kls = [], []
    for t in range(max_iters):
        r = twin.batch_rows(X.shape[0], seed, 0, t, B)
        loss, kl, grads = model.value_and_grad((X[r], Y[r]), traced, klm)
        opt.apply_gradients(zip(grads, traced))
        losses.append(loss)
        kls.append(kl)
    return losses, kls


@pytest.mark.parametrize("kind,klm", [("latent", 1.0), ("latent", 2.5), ("singlebin", 1.0), ("hetero", 1.0), ("masked", 1.0)])
def test_minibatch_device_loop_equals_host_loop(kind, klm):
    X, Y, a = _model(kind)
    b = copy.deepcopy(a)
    losses, kls = _host_minibatch_loop(a, X, Y, 12, 0.01, 16, seed=4, klm=klm)  # 192 rows: more than three epochs of 53
    b.optimize_on_device((X, Y), max_iters=12, initial_lr=0.01, kl_multiplier=klm, minibatch_size=16, seed=4)
    np.testing.assert_allclose(b.loss_history, losses, rtol=1e-10)
    if kind != "singlebin":
        np.testing.assert_allclose(b.kl_history, kls, rtol=1e-10, atol=1e-12)
        assert b.minibatch_position == 12 * 16
    for pa, pb in zip(_params(a), _params(b)):
        np.testing.assert_allclose(pb, pa, rtol=1e-8, atol=1e-10)


def test_resumed_minibatch_calls_continue_the_stream():
    """Two calls with different batch sizes equal one host loop over the concatenated positions (optimizer restarted)."""
    from multi_fidelity_gpflow_b200.optimizers import Adam, CosineDecay

    X, Y, a = _model("latent")
    b = copy.deepcopy(a)
    b.optimize_on_device((X, Y), max_iters=4, initial_lr=0.01, minibatch_size=16, seed=2)
    b.optimize_on_device((X, Y), max_iters=9, initial_lr=0.01, minibatch_size=10, seed=2)
    assert b.minibatch_position == 4 * 16 + 5 * 10
    traced, pos, losses = a.trainable_variables, 0, []
    for steps, B, max_iters in ((range(4), 16, 4), (range(4, 9), 10, 9)):
        opt = Adam(CosineDecay(0.01, max_iters))
        for _ in steps:
            r = twin.rows(pos + np.arange(B), 53, 2)
            pos += B
            loss, _, grads = a.value_and_grad((X[r], Y[r]), traced)
            opt.apply_gradients(zip(grads, traced))
            losses.append(loss)
    np.testing.assert_allclose(b.loss_history, losses, rtol=1e-10)
    for pa, pb in zip(_params(a), _params(b)):
        np.testing.assert_allclose(pb, pa, rtol=1e-8, atol=1e-10)


@pytest.mark.parametrize("B", [16, 12])
def test_minibatch_scaled_expectation_is_unbiased_over_an_epoch(h, B):
    """At fixed parameters the mean over one epoch's N / B batches of scale * VE is the full-data VE (B divides N)."""
    from multi_fidelity_gpflow_b200.linear_svgp import LatentMFCoregionalizationSVGP

    ds = onp.load_dataset("hbs")
    X, Y = np.ascontiguousarray(ds["X"][:48]), np.ascontiguousarray(ds["Y"][:48])
    m = LatentMFCoregionalizationSVGP(X, Y, *_kernels(), num_latents=4, num_inducing=20, num_outputs=49)
    rng = np.random.default_rng(0)
    m.q_mu.assign(0.1 * rng.standard_normal(m.q_mu.shape))
    kl = m.prior_kl()
    full = m.elbo((X, Y)) + kl
    ves = []
    for t in range(48 // B):
        Xb, Yb = h.minibatch_gather(X, Y, 9, 48, B, step=t)  # epoch 1 of the stream
        ves.append(m.elbo((Xb, Yb)) + kl)                  # scale num_data / B = 48 / B
    assert abs(np.mean(ves) - full) < 1e-12 * abs(full)
    assert len(set(ves)) == len(ves)  # the batches really differ


def test_minibatch_of_all_rows_starts_where_the_full_batch_loop_does():
    X, Y, a = _model("latent")
    b = copy.deepcopy(a)
    a.optimize_on_device((X, Y), max_iters=5, initial_lr=0.01)
    b.optimize_on_device((X, Y), max_iters=5, initial_lr=0.01, minibatch_size=53)
    assert abs(b.loss_history[0] - a.loss_history[0]) < 1e-12 * abs(a.loss_history[0])  # the same rows, summed in another order
    np.testing.assert_allclose(b.loss_history, a.loss_history, rtol=1e-9)


def test_minibatch_loop_graph_owns_no_memory(h):
    from multi_fidelity_gpflow_b200 import _lib  # noqa: F401  (loads the runtime libmfgp links)

    rt = ctypes.CDLL("libcudart.so.12")
    val = ctypes.c_uint64(0)

    def reserved():
        assert rt.cudaDeviceGetGraphMemAttribute(0, 2, ctypes.byref(val)) == 0  # cudaGraphMemAttrReservedMemCurrent
        return val.value

    X, Y, m = _model("latent")
    m._handle = h
    m.optimize_on_device((X, Y), max_iters=3, initial_lr=0.01, minibatch_size=16)  # warm the pool
    before = reserved()
    m.optimize_on_device((X, Y), max_iters=20, initial_lr=0.01, minibatch_size=16)  # 20 steps: a captured graph
    assert reserved() == before
    assert len(m.loss_history) == 20 and np.all(np.isfinite(m.loss_history))


def test_data_parallel_minibatch_on_one_rank_equals_device_loop():
    import torch
    import torch.distributed as dist

    created = False
    if not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", str(29500 + os.getpid() % 200))
        torch.cuda.set_device(0)
        dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
        created = True
    try:
        X, Y, a = _model("latent")
        b = copy.deepcopy(a)
        for max_iters, B in ((7, 16), (12, 10)):  # the second call resumes the stream with another batch size
            a.optimize_on_device((X, Y), max_iters=max_iters, initial_lr=0.01, kl_multiplier=1.5, minibatch_size=B, seed=6)
            b.optimize_data_parallel((X, Y), max_iters=max_iters, initial_lr=0.01, kl_multiplier=1.5, minibatch_size=B, seed=6)
        assert a.minibatch_position == b.minibatch_position == 7 * 16 + 5 * 10
        np.testing.assert_allclose(b.loss_history, a.loss_history, rtol=1e-12)
        np.testing.assert_allclose(b.kl_history, a.kl_history, rtol=1e-12, atol=1e-14)
        for pa, pb in zip(_params(a), _params(b)):
            np.testing.assert_allclose(pb, pa, rtol=1e-12, atol=1e-14)
    finally:
        if created:
            dist.destroy_process_group()


WORKER = r'''
import copy, json, os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, %r)
from multi_fidelity_gpflow_b200 import _lib
from multi_fidelity_gpflow_b200.kernels import SquaredExponential
from multi_fidelity_gpflow_b200.linear_svgp import LatentMFCoregionalizationSVGP
from oracle import mfgp_oracle as onp
rank = int(os.environ["RANK"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
h = _lib.Handle(rank)
ds = onp.load_dataset("hbs")
X, Y = ds["X"], ds["Y"]
mk = lambda: LatentMFCoregionalizationSVGP(X, Y, SquaredExponential(lengthscales=np.ones(5)), SquaredExponential(lengthscales=np.ones(5)),
                                           num_latents=4, num_inducing=20, num_outputs=49, handle=h)
m2 = mk()
m2.optimize_data_parallel((X, Y), max_iters=8, initial_lr=0.01, kl_multiplier=1.3, minibatch_size=17, seed=3)
if rank == 0:
    m0 = mk()
    m0.optimize_on_device((X, Y), max_iters=8, initial_lr=0.01, kl_multiplier=1.3, minibatch_size=17, seed=3)
    rel = lambda a, b: float(np.max(np.abs(np.asarray(a) - np.asarray(b))) / np.max(np.abs(np.asarray(b))))
    print("RESULT " + json.dumps({"loss": float(np.max(np.abs(np.array(m2.loss_history) / np.array(m0.loss_history) - 1))),
                                  "q_mu": rel(m2.q_mu.numpy(), m0.q_mu.numpy()), "W": rel(m2.kernel.W.numpy(), m0.kernel.W.numpy())}))
dist.destroy_process_group()
''' % ROOT


def test_two_gpu_minibatch_equals_single_gpu(tmp_path):
    import json

    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "mb_worker.py"
    script.write_text(WORKER)
    res = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                          "127.0.0.1", "--master-port", "29633", str(script)], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    r = json.loads([l for l in res.stdout.splitlines() if l.startswith("RESULT ")][0][7:])
    assert r["loss"] < 1e-12 and r["q_mu"] < 1e-10 and r["W"] < 1e-10, r
