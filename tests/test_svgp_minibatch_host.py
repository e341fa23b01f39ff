"""CPU tests of minibatch training for the device-resident SVGP loops: the shuffled-epoch stream's NumPy twin, the host logic
of SVGPBase._device_loop (stream position, argument checks, what reaches the handle) and the data-parallel schedule of
dist.dp_svgp_adam over gloo."""
import os
import sys

import numpy as np
import pytest

from oracle import mfgp_oracle as onp
from tests import _minibatch_twin as twin

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("N", [1, 2, 3, 5, 64, 1164, 4095, 4096, 4097, 2**20 + 3])
def test_permutation_is_a_bijection(N):
    cases = [(0, 0), (2**63 + 5, 1)] if N > 10**5 else [(0, 0), (1, 0), (0, 1), (12345, 7), (2**64 - 1, 2**40)]
    for seed, e in cases:
        r = twin.permute(np.arange(N), N, seed, e)
        assert np.array_equal(np.sort(r), np.arange(N)), (N, seed, e)


@pytest.mark.parametrize("N", [64, 1164, 4097])
def test_epochs_and_seeds_give_different_orders(N):
    i = np.arange(N)
    orders = {tuple(twin.permute(i, N, s, e)) for s in (0, 1, 99) for e in (0, 1, 2)}
    assert len(orders) == 9
    assert not np.array_equal(twin.permute(i, N, 0, 0), i)


def test_small_data_sets_reach_every_order():
    for N, n_orders in ((2, 2), (3, 6)):
        orders = {tuple(twin.permute(np.arange(N), N, s, e)) for s in range(4) for e in range(20)}
        assert len(orders) == n_orders


@pytest.mark.parametrize("N,B", [(53, 16), (53, 53), (64, 8), (64, 24), (7, 3), (1, 1)])
def test_whole_epochs_hold_every_row_once(N, B):
    """Steps of B rows cross epoch boundaries; over any window of whole epochs every row appears once per epoch."""
    seed, epochs = 11, 5
    nsteps = -(-epochs * N // B) + 1
    for pos0 in (0, N, 3 * N + N // 2):
        stream = np.concatenate([twin.batch_rows(N, seed, pos0, t, B) for t in range(nsteps)])
        np.testing.assert_array_equal(stream, twin.rows(pos0 + np.arange(nsteps * B), N, seed))
        first = (-pos0) % N  # offset of the first epoch boundary in the window
        for e in range(epochs - 1):
            chunk = stream[first + e * N: first + (e + 1) * N]
            assert np.array_equal(np.sort(chunk), np.arange(N)), (pos0, e)
    # a shard [lo, lo + count) of a batch is the matching slice of the batch
    full = twin.batch_rows(N, seed, 5, 3, B)
    np.testing.assert_array_equal(twin.batch_rows(N, seed, 5, 3, B, lo=B // 2, count=B - B // 2), full[B // 2:])


# ---- _device_loop host logic with a recording handle --------------------------------------------------------------------
class _RecordingHandle:
    """Stand-in for _lib.Handle: records the loop calls and returns synthetic histories (no arithmetic claims)."""

    def __init__(self):
        self.calls = []

    def _hist(self, lr_t):
        n = len(lr_t)
        return np.arange(n, dtype=float), np.full(n, 0.5)

    def svgp_adam(self, X, Y, L, M, P, has_W, u, m, v, mask, lr_t, b1, b2, eps, scale=1.0, **kw):
        self.calls.append(dict(kind="full", rows=X.shape[0], nsteps=len(lr_t), scale=scale))
        return self._hist(lr_t)

    def svgp_adam_minibatch(self, X, Y, L, M, P, has_W, u, m, v, mask, lr_t, b1, b2, eps, batch_size=None, seed=0, pos0=0,
                            scale=1.0, **kw):
        self.calls.append(dict(kind="minibatch", rows=X.shape[0], nsteps=len(lr_t), B=batch_size, seed=seed, pos0=pos0,
                               scale=scale, kl_mult=kw["kl_mult"]))
        return self._hist(lr_t)


def _models(fh):
    from multi_fidelity_gpflow_b200.kernels import SquaredExponential
    from multi_fidelity_gpflow_b200.linear_svgp import LatentMFCoregionalizationSVGP
    from multi_fidelity_gpflow_b200.singlebin_svgp import SingleBinSVGP

    ds = onp.load_dataset("hbs")
    X, Y = ds["X"], np.ascontiguousarray(ds["Y"][:, :6])
    k = lambda: (SquaredExponential(lengthscales=np.ones(5)), SquaredExponential(lengthscales=np.ones(5)))
    lat = LatentMFCoregionalizationSVGP(X, Y, *k(), num_latents=3, num_inducing=8, num_outputs=6, handle=fh)
    sb = SingleBinSVGP(X, Y, *k(), 6, ds["Z_kmeans50"][:8], handle=fh)
    return X, Y, lat, sb


def test_minibatch_arguments_are_checked():
    fh = _RecordingHandle()
    X, Y, lat, sb = _models(fh)
    for bad in (0, -3, 54):
        with pytest.raises(ValueError, match="minibatch_size"):
            lat.optimize_on_device((X, Y), max_iters=3, initial_lr=0.01, minibatch_size=bad)
    with pytest.raises(ValueError, match="num_data"):  # scale 1 with B < N would silently bias the ELBO estimate
        sb.optimize_on_device((X, Y), max_iters=3, initial_lr=0.01, minibatch_size=16)
    assert fh.calls == []
    sb.optimize_on_device((X, Y), max_iters=3, initial_lr=0.01, minibatch_size=53)  # B = N: scale 1 is exact
    assert fh.calls[-1]["kind"] == "minibatch" and fh.calls[-1]["scale"] == 1.0


def test_stream_position_of_resumable_and_restarting_models():
    fh = _RecordingHandle()
    X, Y, lat, sb = _models(fh)
    lat.optimize_on_device((X, Y), max_iters=4, initial_lr=0.01, kl_multiplier=2.5, minibatch_size=16, seed=3)
    assert fh.calls[-1] == dict(kind="minibatch", rows=53, nsteps=4, B=16, seed=3, pos0=0, scale=53 / 16, kl_mult=2.5)
    assert lat.minibatch_position == 64
    lat.optimize_on_device((X, Y), max_iters=9, initial_lr=0.01, minibatch_size=10, seed=3)  # B changes: position in rows
    assert fh.calls[-1] == dict(kind="minibatch", rows=53, nsteps=5, B=10, seed=3, pos0=64, scale=5.3, kl_mult=1.0)
    assert lat.minibatch_position == 114 and len(lat.loss_history) == 9 and len(lat.kl_history) == 9
    lat.optimize_on_device((X, Y), max_iters=11, initial_lr=0.01)  # a full-batch call leaves the stream where it was
    assert fh.calls[-1] == dict(kind="full", rows=53, nsteps=2, scale=1.0)
    assert lat.minibatch_position == 114
    lat.optimize_on_device((X, Y), max_iters=11, initial_lr=0.01, minibatch_size=16)  # nothing left to run
    assert len(fh.calls) == 3 and lat.minibatch_position == 114
    sb.num_data = 53
    for max_iters in (3, 5):  # SingleBinSVGP restarts its loop, and the stream with it
        sb.optimize_on_device((X, Y), max_iters=max_iters, initial_lr=0.01, minibatch_size=16, seed=8)
        assert fh.calls[-1] == dict(kind="minibatch", rows=53, nsteps=max_iters, B=16, seed=8, pos0=0, scale=53 / 16,
                                    kl_mult=1.0)
        assert len(sb.loss_history) == max_iters
    assert not hasattr(sb, "minibatch_position")


# ---- data-parallel schedule over gloo ----------------------------------------------------------------------------------
def _schedule_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist

    from multi_fidelity_gpflow_b200.dist import dp_svgp_adam
    from multi_fidelity_gpflow_b200.optimizers import adam_step_factors
    from oracle import mfgp_oracle as onp
    from tests._helpers import OracleSvgpOps
    from tests._minibatch_twin import batch_rows

    class GatheringOps(OracleSvgpOps):
        """The oracle double plus the gather, computed by the twin from the step counter; records each rank's rows."""

        def __init__(self):
            super().__init__()
            self.rows = []

        def gather(self, X, Y, seed, pos0, step, B, lo, Xb, Yb):
            r = batch_rows(X.shape[0], seed, pos0, int(step[0]), B, lo, Xb.shape[0])
            self.rows.append(r)
            Xb.copy_(X[torch.from_numpy(r)])
            Yb.copy_(Y[torch.from_numpy(r)])

    torch.set_num_threads(1)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    ds = onp.load_dataset("hbs")
    X, Y = ds["X"], np.ascontiguousarray(ds["Y"][:, :6])
    rng = np.random.default_rng(1)
    M, L, P, d = 8, 3, 6, 5
    Z = X[rng.permutation(53)[:M]].copy()
    ths = np.tile(onp.default_theta(d), (L, 1))
    W = onp.initialize_W(P, L, 0.4, 0.2)
    u0 = np.concatenate([onp.softplus_inv(ths).ravel(), Z.ravel(), W.ravel(), 0.1 * rng.standard_normal(M * L),
                         np.tile(0.3 * np.eye(M), (L, 1, 1)).ravel(), onp.softplus_inv(np.array([0.8 - 1e-6]))])
    shape = dict(L=L, M=M, P=P, d=d, has_W=True, hetero=False, masked=False, lik_per_output=False, lik_lower=1e-6)
    lr_t, b1, b2 = adam_step_factors(0.05, 5, cosine_decay_steps=5)
    mb = (13, 21, 40)  # B = 13 splits 7 / 6; positions 40 ... 104 cross the epoch boundary at 53
    ops2 = GatheringOps()
    res2 = dp_svgp_adam(ops2, X, Y, shape, u0, None, lr_t, b1, b2, num_data=53, kl_mult=1.5, minibatch=mb)
    solo = dist.new_group([0])
    if rank == 0:
        ops1 = GatheringOps()
        res1 = dp_svgp_adam(ops1, X, Y, shape, u0, None, lr_t, b1, b2, num_data=53, kl_mult=1.5, minibatch=mb, group=solo)
        q.put(("rank0", ops2.rows, res2, ops1.rows, res1))
    else:
        q.put(("rank1", ops2.rows, res2))
    dist.destroy_process_group()


def test_two_rank_minibatch_schedule_matches_single_process():
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 27500 + os.getpid() % 2000
    procs = [ctx.Process(target=_schedule_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = {g[0]: g for g in (q.get(timeout=480), q.get(timeout=480))}
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    _, rows0, res2, rows_solo, res1 = got["rank0"]
    _, rows1, res2_rank1 = got["rank1"]
    assert len(rows0) == len(rows1) == len(rows_solo) == 5
    for t in range(5):
        want = twin.batch_rows(53, 21, 40, t, 13)
        np.testing.assert_array_equal(rows_solo[t], want)  # one rank draws the whole global batch
        assert len(rows0[t]) == 7 and len(rows1[t]) == 6 and not set(rows0[t]) & set(rows1[t])
        np.testing.assert_array_equal(np.concatenate([rows0[t], rows1[t]]), want)  # rank slices in order = the batch
    for a, b in zip(res2, res2_rank1):
        assert np.array_equal(a, b)  # both ranks end bit-identical
    np.testing.assert_allclose(res2[0], res1[0], rtol=1e-10, atol=1e-12)  # two ranks follow the one-rank trajectory
    np.testing.assert_allclose(res2[1], res1[1], rtol=1e-11)
    np.testing.assert_allclose(res2[2], res1[2], rtol=1e-11)
