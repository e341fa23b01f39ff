"""GPU tests of the joint posterior of the cached exact GPs (mfgp_gpr_posterior_predict_cov, mfgp_gpr_posterior_sample) on
both routes (one fused kernel for N <= 64, d <= 16, P <= 64 and Ns <= 64; the blocked route otherwise): the covariance
against the oracle, mean and diag(cov) bit for bit against predict, exact symmetry, the factor L through z = I, samples
against numpy's Cholesky of the library's own covariance, special rows, failures, independence of the other problems and
of the column split, pointer kinds, async mode and the model-level methods."""
import ctypes

import numpy as np
import pytest

from oracle import mfgp_oracle as onp
from tests._joint_oracle import gpr_predict_full_cov
from tests.test_gpr_posterior_gpu import hbs_perturbed, special_rows, synthetic

pytestmark = pytest.mark.gpu
JITTER = 1e-6


@pytest.fixture(scope="module")
def h():
    from multi_fidelity_gpflow_b200 import _lib

    return _lib.Handle(0)


def points(rng, n, d):
    return np.hstack([rng.random((n, d)), rng.integers(0, 2, (n, 1)).astype(float)])


def check_oracle(X, Y, Xs, th, nz, P, mean, cov, probs=None):
    ycols = Y.shape[1]
    for b in range(th.shape[0]) if probs is None else probs:
        c = (b * P) % ycols
        rm, rc = gpr_predict_full_cov(X, Y[:, c:c + P], Xs, th[b], nz[b])
        np.testing.assert_allclose(mean[b], rm, rtol=1e-8, atol=1e-8 * max(np.abs(rm).max(), 1e-300))
        kmax = max(onp.mf_K_diag(Xs, th[b]).max(), 1e-300)
        np.testing.assert_allclose(cov[b], rc, rtol=1e-8, atol=1e-8 * kmax)


def check_against_predict(post, Xs, mean, cov):
    pm, pv = post.predict(Xs)
    np.testing.assert_array_equal(mean, pm)
    np.testing.assert_array_equal(np.diagonal(cov, axis1=1, axis2=2), pv)
    np.testing.assert_array_equal(cov, np.swapaxes(cov, 1, 2))


def check_factor(post, Xs, mean, cov, jitter=JITTER):
    """z = I on the test-point axis (S = Ns): samples - mean is L for every column; L L^T = cov + jitter I."""
    B, Ns, P = mean.shape
    z = np.zeros((B, Ns, Ns, P))
    z[:, np.arange(Ns), np.arange(Ns), :] = 1.0
    s = post.sample(Xs, z, jitter=jitter)
    for b in range(B):
        for c in range(P):
            L = s[b, :, :, c] - mean[b, :, c][:, None]
            assert np.all(np.triu(L, 1) == 0.0)
            A = cov[b] + jitter * np.eye(Ns)
            # plus the rounding of (mean + L) - mean, which the extraction itself adds
            tol = 1e-13 * np.abs(np.diag(A)).max() + 4 * Ns * np.finfo(float).eps * np.abs(mean[b]).max() * np.abs(L).max()
            assert np.abs(L @ L.T - A).max() <= tol


def check_samples(post, Xs, mean, cov, S, seed, jitter=JITTER):
    B, Ns, P = mean.shape
    z = np.random.default_rng(seed).standard_normal((B, Ns, S, P))
    s = post.sample(Xs, z, jitter=jitter)
    for b in range(B):
        L = np.linalg.cholesky(cov[b] + jitter * np.eye(Ns))
        ref = mean[b][:, None, :] + np.einsum("ij,jkc->ikc", L, z[b])
        np.testing.assert_allclose(s[b], ref, rtol=1e-10, atol=1e-10 * np.abs(ref).max())
    return z, s


def test_hbs_all_bins_fused(h):
    ds, th, nz = hbs_perturbed(seed=11)
    X, Y = ds["X"], ds["Y"]
    post = h.gpr_posterior(X, Y, th, nz)
    rng = np.random.default_rng(0)
    Xs = np.vstack([ds["X_test"], points(rng, 54, 5)])  # Ns = 64: the largest fused size
    mean, cov = post.predict_cov(Xs)
    assert mean.shape == (49, 64, 1) and cov.shape == (49, 64, 64)
    check_oracle(X, Y, Xs, th, nz, 1, mean, cov)
    check_against_predict(post, Xs, mean, cov)
    check_factor(post, Xs, mean, cov)
    check_samples(post, Xs, mean, cov, 1000, 1)


def test_hbs_every_bin_and_restart(h):
    ds, th, nz = hbs_perturbed(R=64, seed=12)
    X, Y = ds["X"], ds["Y"]
    post = h.gpr_posterior(X, Y, th, nz)
    Xs = np.vstack([ds["X_test"], points(np.random.default_rng(1), 54, 5)])
    mean, cov = post.predict_cov(Xs)
    check_against_predict(post, Xs, mean, cov)
    sel = np.arange(0, 49 * 64, 97)
    check_oracle(X, Y, Xs, th, nz, 1, mean, cov, probs=sel)
    z = np.random.default_rng(2).standard_normal((49 * 64, 64, 16, 1))
    s = post.sample(Xs, z)
    for b in sel:
        L = np.linalg.cholesky(cov[b] + JITTER * np.eye(64))
        ref = mean[b][:, None, :] + np.einsum("ij,jkc->ikc", L, z[b])
        np.testing.assert_allclose(s[b], ref, rtol=1e-10, atol=1e-10 * np.abs(ref).max())


@pytest.mark.parametrize("N,d,P,Ns,S", [
    (1, 1, 1, 1, 3), (53, 5, 1, 7, 5), (64, 16, 3, 8, 7), (53, 5, 49, 9, 3), (64, 5, 64, 63, 1), (40, 1, 1, 64, 33),
    (53, 5, 1, 65, 7), (65, 5, 1, 9, 5), (130, 5, 3, 200, 3), (20, 17, 1, 8, 3), (20, 5, 65, 7, 1), (64, 16, 1, 200, 5),
])
def test_edge_sizes(h, N, d, P, Ns, S):
    """Fused: N <= 64, d <= 16, P <= 64, Ns <= 64; blocked: Ns = 65 / 200, N = 65 / 130, d = 17, P = 65.  S * P is odd in
    every case with odd P."""
    rng = np.random.default_rng(N * 1000 + d * 10 + P + Ns)
    B = 3
    X, Y = synthetic(rng, N, d, B * P)
    th = np.tile(onp.default_theta(d), (B, 1)) * np.exp(0.2 * rng.standard_normal((B, 2 * d + 3)))
    th[:, 1:1 + d] *= np.sqrt(d)
    th[:, 2 + d:2 + 2 * d] *= np.sqrt(d)
    nz = np.full(B, 1e-2)
    post = h.gpr_posterior(X, Y, th, nz, P=P)
    Xs = points(rng, Ns, d)
    mean, cov = post.predict_cov(Xs)
    check_oracle(X, Y, Xs, th, nz, P, mean, cov)
    check_against_predict(post, Xs, mean, cov)
    check_factor(post, Xs, mean, cov)
    check_samples(post, Xs, mean, cov, S, 3)


def test_fused_and_blocked_routes_agree(h):
    ds, th, nz = hbs_perturbed(seed=13)
    post = h.gpr_posterior(ds["X"], ds["Y"], th, nz)
    Xs = np.vstack([ds["X_test"], points(np.random.default_rng(4), 55, 5)])
    _, c64 = post.predict_cov(Xs[:64])
    _, c65 = post.predict_cov(Xs)
    kmax = np.abs(np.diagonal(c64, axis1=1, axis2=2)).max()
    assert np.abs(c65[:, :64, :64] - c64).max() <= 1e-12 * kmax


@pytest.mark.parametrize("Ns", [20, 70])  # fused and blocked
def test_special_rows_and_duplicates(h, Ns):
    from multi_fidelity_gpflow_b200 import _lib

    ds, th, nz = hbs_perturbed(seed=14)
    X = ds["X"]
    post = h.gpr_posterior(X, ds["Y"], th[:4], nz[:4])
    live = points(np.random.default_rng(5), Ns - 4, 5)
    Xs = np.vstack([live[:5], special_rows(X), live[5:], live[:1]])  # dead rows 5-7; the last row duplicates row 0
    dead = [5, 6, 7]
    mean, cov = post.predict_cov(Xs)
    assert np.all(mean[:, dead] == 0.0) and np.all(cov[:, dead, :] == 0.0) and np.all(cov[:, :, dead] == 0.0)
    check_against_predict(post, Xs, mean, cov)
    z = np.random.default_rng(6).standard_normal((4, Ns, 9, 1))
    s = post.sample(Xs, z)  # the duplicate makes Sigma singular: the jitter keeps it factorable
    assert np.isfinite(s).all()
    np.testing.assert_allclose(s[:, dead], np.sqrt(JITTER) * z[:, dead], rtol=4.5e-16, atol=0)
    info = np.zeros(4, dtype=np.int32)
    s0 = post.sample(Xs, z, jitter=0.0, info=info)
    np.testing.assert_array_equal(info, dead[0] + 1)  # a dead row without jitter is a failed pivot
    assert np.isnan(s0).all()
    with pytest.raises(_lib.NotPositiveDefiniteError):
        post.sample(Xs, z, jitter=0.0)


@pytest.mark.parametrize("N", [53, 100])  # fused and blocked
def test_failed_problem(h, N):
    from multi_fidelity_gpflow_b200 import _lib

    rng = np.random.default_rng(7)
    X, Y = synthetic(rng, N, 5, 4)
    th = np.tile(onp.default_theta(5), (4, 1))
    nz = np.full(4, 1e-3)
    nz[2] = -5.0
    cinfo = np.zeros(4, dtype=np.int32)
    post = h.gpr_posterior(X, Y, th, nz, info=cinfo)
    assert cinfo[2] > 0
    keep = [0, 1, 3]
    ref = h.gpr_posterior(X, Y, th, np.full(4, 1e-3))  # the same call without the failure
    Xs = points(rng, 17, 5)
    z = rng.standard_normal((4, 17, 5, 1))
    info = np.zeros(4, dtype=np.int32)
    s = post.sample(Xs, z, info=info)
    np.testing.assert_array_equal(info, [0, 0, 1, 0])
    assert np.isnan(s[2]).all()
    np.testing.assert_array_equal(s[keep], ref.sample(Xs, z)[keep])
    with pytest.raises(_lib.NotPositiveDefiniteError):
        post.sample(Xs, z)
    m, c = post.predict_cov(Xs)  # _predict_cov: NaN for the failed problem, as predict gives it, and no error
    assert np.isnan(m[2]).all() and np.isnan(c[2]).all()
    rm, rc = ref.predict_cov(Xs)
    np.testing.assert_array_equal(m[keep], rm[keep])
    np.testing.assert_array_equal(c[keep], rc[keep])


@pytest.mark.parametrize("Ns", [30, 90])  # fused and blocked
def test_independent_of_other_problems_and_of_the_column_split(h, Ns):
    ds, th, nz = hbs_perturbed(seed=15)
    X, Y = ds["X"], ds["Y"]
    post = h.gpr_posterior(X, Y, th, nz)
    th2 = th * np.exp(0.2 * np.random.default_rng(7).standard_normal(th.shape))
    th2[5:9] = th[5:9]
    other = h.gpr_posterior(X, Y, th2, nz)  # the same problems 5-8 among different neighbours
    Xs = points(np.random.default_rng(8), Ns, 5)
    m, c = post.predict_cov(Xs)
    mo, co = other.predict_cov(Xs)
    np.testing.assert_array_equal(mo[5:9], m[5:9])
    np.testing.assert_array_equal(co[5:9], c[5:9])
    z = np.random.default_rng(9).standard_normal((49, Ns, 1000, 1))
    s = post.sample(Xs, z)
    np.testing.assert_array_equal(other.sample(Xs, z)[5:9], s[5:9])
    s1 = post.sample(Xs, np.ascontiguousarray(z[:, :, :1]))
    np.testing.assert_array_equal(s1[:, :, 0], s[:, :, 0])
    s7 = post.sample(Xs, np.ascontiguousarray(z[:, :, 993:]))
    np.testing.assert_array_equal(s7, s[:, :, 993:])


@pytest.mark.parametrize("N", [53, 100])  # fused and blocked
def test_device_tensors_async_mode_and_status(h, N):
    import torch

    rng = np.random.default_rng(10)
    X, Y = synthetic(rng, N, 5, 6)
    th = np.tile(onp.default_theta(5), (3, 1)) * np.exp(0.2 * rng.standard_normal((3, 13)))
    nz = np.full(3, 1e-3)
    Xs = points(rng, 40, 5)
    z = rng.standard_normal((3, 40, 11, 2))
    post = h.gpr_posterior(X, Y, th, nz, P=2)
    ref_m, ref_c = post.predict_cov(Xs)
    ref_s = post.sample(Xs, z)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    f64 = dict(dtype=torch.float64, device="cuda")
    dm, dc, ds = torch.empty((3, 40, 2), **f64), torch.empty((3, 40, 40), **f64), torch.empty((3, 40, 11, 2), **f64)
    di = torch.zeros(3, dtype=torch.int32, device="cuda")
    h.set_stream(torch.cuda.current_stream().cuda_stream)
    h.set_async(True)
    try:
        post.predict_cov(dev(Xs), dm, dc)
        post.sample(dev(Xs), dev(z), samples=ds, info=di)
        assert h.sync() == 0
        Xd = Xs.copy()
        Xd[3, -1] = 0.5  # a dead row: with jitter 0 a failed pivot, reported through mfgp_sync
        post.sample(dev(Xd), dev(z), jitter=0.0, samples=torch.empty_like(ds), info=torch.zeros_like(di))
        assert h.sync() == 4
    finally:
        h.set_async(False)
        h.set_stream(None)
    np.testing.assert_array_equal(dm.cpu().numpy(), ref_m)
    np.testing.assert_array_equal(dc.cpu().numpy(), ref_c)
    np.testing.assert_array_equal(ds.cpu().numpy(), ref_s)
    assert not di.any()


def test_argument_checks_and_other_handles(h):
    from multi_fidelity_gpflow_b200 import _lib

    ds, th, nz = hbs_perturbed(seed=16)
    post = h.gpr_posterior(ds["X"], ds["Y"], th[:2], nz[:2])
    Xs = ds["X_test"]
    z = np.random.default_rng(11).standard_normal((2, 10, 4, 1))
    ref = post.sample(Xs, z)
    h2 = _lib.Handle(0)  # any handle on the posterior's device
    out2 = np.empty_like(z)
    assert _lib._lib.mfgp_gpr_posterior_sample(h2._h, post._p, _lib._ptr(Xs), 10, 4, JITTER, _lib._ptr(z), _lib._ptr(out2),
                                               None) == 0
    np.testing.assert_array_equal(out2, ref)
    for bad in (np.nan, np.inf, -1e-6):
        with pytest.raises(ValueError):
            post.sample(Xs, z, jitter=bad)
    L, p = _lib._lib, _lib._ptr
    out = np.empty_like(z)
    call = lambda *a: L.mfgp_gpr_posterior_sample(h._h, post._p, *a)
    assert call(p(Xs), 10, -1, 1e-6, p(z), p(out), None) == -1
    assert call(None, 10, 4, 1e-6, p(z), p(out), None) == -1
    assert call(p(Xs), 10, 4, 1e-6, None, p(out), None) == -1
    assert call(p(Xs), 10, 4, 1e-6, p(z), None, None) == -1
    assert call(p(Xs), 10, 4, 1e-6, p(z), ctypes.c_void_p(z.ctypes.data + 8), None) == -1  # z and samples overlap
    assert call(p(Xs), 0, 4, 1e-6, p(z), p(out), None) == 0
    assert call(p(Xs), 10, 0, 1e-6, p(z), p(out), None) == 0
    m, c = np.empty((2, 10, 1)), np.empty((2, 10, 10))
    assert L.mfgp_gpr_posterior_predict_cov(h._h, post._p, p(Xs), 10, None, p(c)) == -1
    assert L.mfgp_gpr_posterior_predict_cov(h._h, None, p(Xs), 10, p(m), p(c)) == -1
    assert L.mfgp_gpr_posterior_predict_cov(h._h, post._p, p(Xs), 0, p(m), p(c)) == 0


def test_goku_shared_blocked(h):
    ds = onp.load_dataset("goku")
    X, Y = ds["X"], ds["Y"]
    th = onp.default_theta(10)
    post = h.gpr_posterior(X, Y, th[None], np.array([1e-3]), P=64)
    Xs = points(np.random.default_rng(12), 256, 10)
    mean, cov = post.predict_cov(Xs)
    check_oracle(X, Y, Xs, th[None], [1e-3], 64, mean, cov)
    check_against_predict(post, Xs, mean, cov)
    check_samples(post, Xs, mean, cov, 3, 13)


def test_model_level(h):
    from multi_fidelity_gpflow_b200.kernels import SquaredExponential
    from multi_fidelity_gpflow_b200.linear import MultiFidelityGPModel
    from multi_fidelity_gpflow_b200.multibin import MultiBinMFGP

    ds = onp.load_dataset("hbs")
    X, Y = ds["X"], ds["Y"]
    Xs = np.vstack([ds["X_test"], X[X[:, -1] == 1.0]])
    Ns = Xs.shape[0]
    mdl = MultiBinMFGP(X, Y, num_restarts=2, seed=3, handle=h)
    post = mdl.posterior("all")
    mean, cov = post.predict_f_full_cov(Xs)
    assert mean.shape == (2, Ns, 49) and cov.shape == (2, 49, Ns, Ns)
    for r in range(2):
        for p in (0, 17, 48):
            rm, rc = gpr_predict_full_cov(X, Y[:, p:p + 1], Xs, mdl.thetas[r, p], mdl.noise)
            np.testing.assert_allclose(mean[r, :, p], rm[:, 0], rtol=1e-8, atol=1e-8 * np.abs(rm).max())
            np.testing.assert_allclose(cov[r, p], rc, rtol=1e-8, atol=1e-8 * onp.mf_K_diag(Xs, mdl.thetas[r, p]).max())
    f = post.predict_f_samples(Xs, num_samples=6, seed=4)
    assert f.shape == (2, 6, Ns, 49)
    z = np.random.default_rng(4).standard_normal((98, Ns, 6, 1))
    for r in range(2):
        for p in (0, 48):
            L = np.linalg.cholesky(cov[r, p] + JITTER * np.eye(Ns))
            ref = mean[r, :, p][:, None] + L @ z[r * 49 + p, :, :, 0]
            np.testing.assert_allclose(f[r, :, :, p], ref.T, rtol=1e-10, atol=1e-10 * np.abs(ref).max())
    best = mdl.predict_f_samples(Xs, seed=4)
    assert best.shape == (Ns, 49)
    np.testing.assert_array_equal(best, mdl.posterior("best").predict_f_samples(Xs, seed=4))

    se = lambda: SquaredExponential(lengthscales=np.ones(5), variance=1.0)
    m = MultiFidelityGPModel(X, Y, se(), se(), handle=h)
    mp = m.posterior()
    mm, mc = mp.predict_f_full_cov(Xs)
    assert mm.shape == (Ns, 49) and mc.shape == (49, Ns, Ns) and not mc.flags.writeable
    theta, noise = m._theta_noise()
    rm, rc = gpr_predict_full_cov(X, Y, Xs, theta, noise)
    np.testing.assert_allclose(mm, rm, rtol=1e-8, atol=1e-8 * np.abs(rm).max())
    np.testing.assert_allclose(mc[3], rc, rtol=1e-8, atol=1e-8 * onp.mf_K_diag(Xs, theta).max())
    pm, pv = mp.predict_f(Xs)
    np.testing.assert_array_equal(mm, pm)
    np.testing.assert_array_equal(np.diagonal(mc[0]), pv[:, 0])
    fs = mp.predict_f_samples(Xs, num_samples=4, seed=5)
    assert fs.shape == (4, Ns, 49)
    np.testing.assert_array_equal(m.predict_f_samples(Xs, num_samples=4, seed=5), fs)
    zz = np.random.default_rng(5).standard_normal((1, Ns, 4, 49))
    L = np.linalg.cholesky(mc[0] + JITTER * np.eye(Ns))
    ref = (mm[:, None, :] + np.einsum("ij,jkc->ikc", L, zz[0])).transpose(1, 0, 2)
    np.testing.assert_allclose(fs, ref, rtol=1e-10, atol=1e-10 * np.abs(ref).max())
    fd = mp.predict_f_samples(Xs, num_samples=4, full_cov=False, seed=5)
    np.testing.assert_allclose(fd, pm[None] + np.sqrt(pv)[None] * zz[0].transpose(1, 0, 2), rtol=1e-12)
