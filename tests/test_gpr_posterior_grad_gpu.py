"""GPU tests of the input gradients of the cached exact-GP posterior (mfgp_gpr_posterior_predict_grad): both routes (fused
kernel for N <= 64, d <= 16, P <= 64; blocked otherwise) against the autograd oracle per problem (rtol 1e-7, atol 1e-7
max|ref|), mean and var against the library's own predict (rtol 1e-13), dead test rows, per-problem failure, pointer
kinds, other handles, split-independence and central differences of the library's predict."""
import numpy as np
import pytest

from oracle import mfgp_oracle as onp
from tests._grad_oracle import gpr_predict_grad_x

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def h():
    from multi_fidelity_gpflow_b200 import _lib

    return _lib.Handle(0)


def close(got, ref, rtol, atol_rel):
    ref = np.asarray(ref)
    np.testing.assert_allclose(got, ref, rtol=rtol, atol=atol_rel * max(np.abs(ref).max(), 1e-300))


def check_grad(post, X, Y, Xs, th, nz, P):
    """predict_grad against posterior.predict (mean, var) and the oracle per problem (all four)."""
    mean, var, dmean, dvar = post.predict_grad(Xs)
    B, Ns, d, ycols = th.shape[0], Xs.shape[0], Xs.shape[1] - 1, Y.shape[1]
    assert mean.shape == (B, Ns, P) and var.shape == (B, Ns) and dmean.shape == (B, Ns, P, d) and dvar.shape == (B, Ns, d)
    pm, pv = post.predict(Xs)
    close(mean, pm, 1e-13, 1e-14)
    close(var, pv, 1e-13, 1e-14)
    for b in range(B):
        c = (b * P) % ycols
        rm, rv, rdm, rdv = gpr_predict_grad_x(X, Y[:, c:c + P], Xs, th[b], nz[b])
        close(dmean[b], rdm[..., :-1], 1e-7, 1e-7)
        close(dvar[b], rdv[:, :-1], 1e-7, 1e-7)
    return mean, var, dmean, dvar


def hbs_perturbed(R=1, seed=0):
    ds = onp.load_dataset("hbs")
    B = 49 * R
    rng = np.random.default_rng(seed)
    th = np.tile(onp.default_theta(5), (B, 1)) * np.exp(0.3 * rng.standard_normal((B, 13)))
    nz = np.full(B, 1e-3) * np.exp(0.3 * rng.standard_normal(B))
    return ds, th, nz


def synthetic(rng, N, d, ycols, frac=0.4):
    X = np.hstack([rng.random((N, d)), (rng.random((N, 1)) < frac).astype(float)])
    return X, rng.standard_normal((N, ycols))


def test_hbs_all_bins_fused(h):
    ds, th, nz = hbs_perturbed()
    X, Y = ds["X"], ds["Y"]
    post = h.gpr_posterior(X, Y, th, nz)
    dead = np.repeat(X[:1], 3, axis=0)
    dead[:, -1] = [0.5, np.nextafter(1.0, 2.0), np.nan]
    Xs = np.vstack([ds["X_test"], X, dead])  # test inputs, the training inputs of both fidelities, dead rows
    _, _, dm, dv = check_grad(post, X, Y, Xs, th, nz, 1)
    assert np.all(dm[:, -3:] == 0.0) and np.all(dv[:, -3:] == 0.0)
    assert np.abs(dm).max() > 1e-3 and np.abs(dv).max() > 1e-6
    post.close()


@pytest.mark.parametrize("N,d,P,Ns", [
    (1, 1, 1, 5), (8, 5, 3, 9), (9, 16, 8, 9), (40, 1, 1, 17), (53, 5, 49, 7), (64, 16, 1, 9), (64, 5, 64, 8),
    (65, 5, 1, 7), (30, 17, 1, 9), (20, 5, 65, 8), (65, 17, 65, 9),
])
def test_sizes(h, N, d, P, Ns):
    """Fused route: N <= 64, d <= 16, P <= 64 (DFMA mean below P = 8, DMMA from 8); blocked for N = 65, d = 17, P = 65."""
    rng = np.random.default_rng(N * 1000 + d * 10 + P)
    B = 3
    X, Y = synthetic(rng, N, d, B * P)
    th = np.tile(onp.default_theta(d), (B, 1)) * np.exp(0.2 * rng.standard_normal((B, 2 * d + 3)))
    th[:, 1:1 + d] *= np.sqrt(d)
    th[:, 2 + d:2 + 2 * d] *= np.sqrt(d)
    th[:, 0] = 0.7
    nz = np.full(B, 1e-2)
    Xs = np.hstack([rng.random((Ns, d)), rng.integers(0, 2, (Ns, 1)).astype(float)])
    Xs[0] = X[0]  # a test point on a training point
    Xs[-1, -1] = 0.5  # a dead row
    _, _, dm, dv = check_grad(h.gpr_posterior(X, Y, th, nz, P=P), X, Y, Xs, th, nz, P)
    assert np.all(dm[:, -1] == 0.0) and np.all(dv[:, -1] == 0.0)


def test_goku_shared_and_per_bin_blocked(h):
    ds = onp.load_dataset("goku")
    X, Y, Xs = ds["X"], ds["Y"], ds["X_test"]
    th = onp.default_theta(10)
    check_grad(h.gpr_posterior(X, Y, th[None], np.array([1e-3]), P=64), X, Y, Xs, th[None], np.array([1e-3]), 64)
    rng = np.random.default_rng(5)
    ths = np.tile(th, (4, 1)) * np.exp(0.1 * rng.standard_normal((4, 23)))
    nz = np.full(4, 1e-3)
    Y4 = np.ascontiguousarray(Y[:, :4])
    check_grad(h.gpr_posterior(X, Y4, ths, nz), X, Y4, Xs, ths, nz, 1)


def test_model_level_predict_f_grad(h):
    from multi_fidelity_gpflow_b200.kernels import SquaredExponential
    from multi_fidelity_gpflow_b200.linear import MultiFidelityGPModel
    from multi_fidelity_gpflow_b200.multibin import MultiBinMFGP

    ds = onp.load_dataset("hbs")
    X, Y = ds["X"], ds["Y"]
    se = lambda: SquaredExponential(lengthscales=np.ones(5), variance=1.0)
    m = MultiFidelityGPModel(X, Y, se(), se(), handle=h)
    mean, var, dm, dv = m.posterior().predict_f_grad(ds["X_test"])
    th = m.kernel.theta(5)
    _, rv, rdm, rdv = gpr_predict_grad_x(X, Y, ds["X_test"], th, 1e-3)
    assert dm.shape == dv.shape == (10, 49, 6)
    close(dm, rdm, 1e-7, 1e-7)
    close(dv, np.repeat(rdv[:, None, :], 49, axis=1), 1e-7, 1e-7)
    mdl = MultiBinMFGP(X, Y, num_restarts=2, seed=2, handle=h)
    am, av, adm, adv = mdl.posterior("all").predict_f_grad(ds["X_test"])
    assert adm.shape == (2, 10, 49, 6)
    for r, p in [(0, 0), (1, 48)]:
        _, _, rdm, rdv = gpr_predict_grad_x(X, Y[:, p:p + 1], ds["X_test"], mdl.thetas[r, p], mdl.noise)
        close(adm[r, :, p], rdm[:, 0], 1e-7, 1e-7)
        close(adv[r, :, p], rdv, 1e-7, 1e-7)


@pytest.mark.parametrize("N", [53, 100])  # fused and blocked route
def test_non_pd_problem_is_nan_in_all_four(h, N):
    rng = np.random.default_rng(7)
    X, Y = synthetic(rng, N, 5, 4)
    th = np.tile(onp.default_theta(5), (4, 1))
    good = np.full(4, 1e-3)
    bad = good.copy()
    bad[2] = -5.0
    Xs = rng.random((17, 6))
    Xs[:, -1] = np.arange(17) % 2
    Xs[3, -1] = 0.5  # a dead row: still NaN in the failed problem
    ref = h.gpr_posterior(X, Y, th, good).predict_grad(Xs)
    info = np.zeros(4, dtype=np.int32)
    got = h.gpr_posterior(X, Y, th, bad, info=info).predict_grad(Xs)
    assert info[2] > 0 and np.all(info[[0, 1, 3]] == 0)
    for g, r in zip(got, ref):
        assert np.isnan(g[2]).all()
        np.testing.assert_array_equal(g[[0, 1, 3]], r[[0, 1, 3]])


@pytest.mark.parametrize("N", [53, 100])
def test_device_tensors_async_and_other_handle(h, N):
    import torch

    from multi_fidelity_gpflow_b200 import _lib

    rng = np.random.default_rng(8)
    X, Y = synthetic(rng, N, 5, 6)
    th = np.tile(onp.default_theta(5), (6, 1)) * np.exp(0.2 * rng.standard_normal((6, 13)))
    nz = np.full(6, 1e-3)
    Xs = np.hstack([rng.random((50, 5)), rng.integers(0, 2, (50, 1)).astype(float)])
    h1 = _lib.Handle(0)
    post = h1.gpr_posterior(X, Y, th, nz, P=2)
    ref = post.predict_grad(Xs)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    outs = [torch.empty(r.shape, dtype=torch.float64, device="cuda") for r in ref]
    post.handle = h  # a handle other than the creator, on the same device
    h.set_stream(torch.cuda.current_stream().cuda_stream)
    h.set_async(True)
    try:
        post.predict_grad(dev(Xs), *outs)
        assert h.sync() == 0
    finally:
        h.set_async(False)
        h.set_stream(None)
    for o, r in zip(outs, ref):
        np.testing.assert_array_equal(o.cpu().numpy(), r)
    post.close()
    h1.close()


def test_fused_route_is_independent_of_the_split(h):
    ds, th, nz = hbs_perturbed(seed=4)
    post = h.gpr_posterior(ds["X"], ds["Y"], th, nz)
    rng = np.random.default_rng(0)
    Xs = np.hstack([rng.random((5000, 5)), rng.integers(0, 2, (5000, 1)).astype(float)])
    full = post.predict_grad(Xs)
    for i in (0, 2500, 4999):
        one = post.predict_grad(Xs[i:i + 1])
        for a, b in zip(one, full):
            np.testing.assert_array_equal(a[:, 0], b[:, i])
    Y59 = np.ascontiguousarray(ds["Y"][:, 5:9])  # nor do the other problems of the call
    sub = h.gpr_posterior(ds["X"], Y59, th[5:9], nz[5:9]).predict_grad(Xs[:100])
    for a, b in zip(sub, full):
        np.testing.assert_array_equal(a, b[5:9, :100])


@pytest.mark.parametrize("N,P", [(53, 3), (100, 2)])
def test_central_differences_of_predict(h, N, P):
    """Independent of the oracle: the gradient against central differences of the library's own predict."""
    rng = np.random.default_rng(11)
    X, Y = synthetic(rng, N, 5, 2 * P)
    th = np.tile(onp.default_theta(5), (2, 1)) * np.exp(0.2 * rng.standard_normal((2, 13)))
    post = h.gpr_posterior(X, Y, th, np.full(2, 1e-2), P=P)
    Xs = np.hstack([rng.random((12, 5)), (np.arange(12) % 2)[:, None].astype(float)])
    _, _, dm, dv = post.predict_grad(Xs)
    eps = 1e-5
    for j in range(5):
        xp, xm = Xs.copy(), Xs.copy()
        xp[:, j] += eps
        xm[:, j] -= eps
        (mp, vp), (mm, vm) = post.predict(xp), post.predict(xm)
        close(dm[..., j], (mp - mm) / (2 * eps), 1e-5, 1e-5)
        close(dv[..., j], (vp - vm) / (2 * eps), 1e-5, 1e-5)
