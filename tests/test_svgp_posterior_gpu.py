"""GPU tests of the cached SVGP posterior (mfgp_svgp_posterior_*): both predict routes (fused kernel for M <= 64, d <= 16;
blocked otherwise) against the oracle's SVGP.predict_f (1e-8 relative, atol 1e-8 max|ref|) and against svgp_predict,
dead test rows, per-latent failure, split independence, pointer kinds, lifetime and the model-level posterior()."""
import numpy as np
import pytest

from oracle import mfgp_oracle as onp

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def h():
    from multi_fidelity_gpflow_b200 import _lib

    return _lib.Handle(0)


def make_problem(rng, Z, L, d, P, mixing, perturb=True):
    """As tests/test_cuda_svgp.py builds its problems: default theta, q_mu, q_sqrt = 0.1 I, the band W, perturbed."""
    M = Z.shape[0]
    th = np.tile(onp.default_theta(d), (L, 1))
    q_mu = np.zeros((M, L))
    q_sqrt = np.tile(0.1 * np.eye(M), (L, 1, 1))
    W = onp.initialize_W(P, L, 0.4, 0.2) if mixing else None
    Zp = Z.copy()
    if perturb:
        th = th * np.exp(0.2 * rng.standard_normal(th.shape))
        q_mu = 0.3 * rng.standard_normal((M, L))
        q_sqrt = q_sqrt + 0.02 * np.tril(rng.standard_normal((L, M, M)))
        Zp[:, :-1] += 0.01 * rng.standard_normal((M, d))
        if mixing:
            W = W + 0.05 * rng.standard_normal(W.shape)
    return dict(Z=Zp, thetas=th, W=W, q_mu=q_mu, q_sqrt=q_sqrt)


def args(pr):
    return pr["Z"], pr["thetas"], pr["W"], pr["q_mu"], pr["q_sqrt"]


def close(got, ref, tol=1e-8):
    ref = np.asarray(ref)
    np.testing.assert_allclose(got, ref, rtol=tol, atol=tol * max(np.abs(ref).max(), 1e-300))


def check_oracle(pr, Xs, mean, var):
    rm, rv = onp.svgp_predict(Xs, pr["Z"], pr["thetas"], pr["q_mu"], pr["q_sqrt"], pr["W"])
    assert mean.shape == rm.shape and var.shape == rv.shape
    close(mean, rm)
    close(var, rv)


def random_points(rng, n, d):
    return np.hstack([rng.random((n, d)), rng.integers(0, 2, (n, 1)).astype(float)])


def special_rows(X):
    s = np.repeat(X[:1], 3, axis=0).copy()
    s[:, -1] = [0.5, np.nextafter(1.0, 2.0), np.nan]
    return s


@pytest.mark.parametrize("mixing", [False, True])  # single-bin L = 49, latent L = 10 with W
def test_hbs_fused(h, mixing):
    ds = onp.load_dataset("hbs")
    rng = np.random.default_rng(1 if not mixing else 2)
    pr = make_problem(rng, ds["Z_kmeans50"], 10 if mixing else 49, 5, 49, mixing)
    Xs = np.vstack([ds["X_test"], ds["X"], random_points(rng, 2000, 5)])
    post = h.svgp_posterior(*args(pr))
    mean, var = post.predict(Xs)
    assert mean.shape == var.shape == (Xs.shape[0], 49)
    check_oracle(pr, Xs, mean, var)
    sm, sv = h.svgp_predict(Xs, *args(pr))
    close(mean, sm)
    close(var, sv)
    m0, v0 = post.predict(special_rows(ds["X"]))  # fidelity 0.5 / 1 + 1 ulp / NaN: zero covariance, like the oracle
    assert np.all(m0 == 0.0) and np.all(v0 == 0.0)
    post.close()


@pytest.mark.parametrize("mixing", [False, True])  # single-bin 8-bin subset, latent L = 15
def test_goku_blocked(h, mixing):
    ds = onp.load_dataset("goku")
    Z = ds["Z_kmeans300"]
    assert np.any((Z[:, -1] != 0.0) & (Z[:, -1] != 1.0))  # quirk Q1: inducing points 1 ulp off fidelity 1 are dead
    rng = np.random.default_rng(3)
    L, P = (15, 64) if mixing else (8, 8)
    pr = make_problem(rng, Z, L, 10, P, mixing)
    Xs = np.vstack([ds["X_test"], special_rows(ds["X"])])
    post = h.svgp_posterior(*args(pr))
    mean, var = post.predict(Xs)
    check_oracle(pr, Xs, mean, var)
    assert np.all(mean[-3:] == 0.0) and np.all(var[-3:] == 0.0)
    sm, sv = h.svgp_predict(Xs, *args(pr))
    close(mean, sm, 1e-12)
    close(var, sv, 1e-12)


def synthetic(rng, M, d, L, mixing, P=3):
    Z = random_points(rng, M, d)
    th = np.tile(onp.default_theta(d), (L, 1)) * np.exp(0.2 * rng.standard_normal((L, 2 * d + 3)))
    th[:, 1:1 + d] *= np.sqrt(d)  # keep the covariance away from the identity in high d
    th[:, 2 + d:2 + 2 * d] *= np.sqrt(d)
    q_sqrt = np.tile(0.3 * np.eye(M), (L, 1, 1)) + 0.05 * rng.standard_normal((L, M, M))  # upper part is ignored
    W = rng.standard_normal((P, L)) if mixing else None
    return dict(Z=Z, thetas=th, W=W, q_mu=rng.standard_normal((M, L)), q_sqrt=q_sqrt)


@pytest.mark.parametrize("M,d,L,Ns,mixing", [
    (1, 1, 1, 1, False), (7, 5, 3, 7, False), (8, 1, 2, 9, True), (9, 16, 1, 2049, False), (63, 5, 4, 9, True),
    (64, 16, 3, 7, False), (64, 3, 1, 2049, True), (65, 5, 2, 9, False), (65, 16, 3, 7, True), (30, 17, 2, 9, False),
])
def test_edge_sizes(h, M, d, L, Ns, mixing):
    """Fused route: M <= 64, d <= 16; the blocked route for M = 65 and d = 17."""
    rng = np.random.default_rng(M * 1000 + d * 10 + L)
    pr = synthetic(rng, M, d, L, mixing)
    pr_ref = dict(pr, q_sqrt=np.tril(pr["q_sqrt"]))
    Xs = random_points(rng, Ns, d)
    mean, var = h.svgp_posterior(*args(pr)).predict(Xs)
    check_oracle(pr_ref, Xs, mean, var)


@pytest.mark.parametrize("M", [20, 70])  # fused and blocked route
@pytest.mark.parametrize("mixing", [False, True])
def test_failed_latent_is_its_own_status(h, M, mixing):
    from multi_fidelity_gpflow_b200 import _lib

    rng = np.random.default_rng(7)
    L, d = 4, 5
    pr = synthetic(rng, M, d, L, mixing, P=6)
    P = 6 if mixing else L
    Xs = random_points(rng, 33, d)
    ref_m, ref_v = h.svgp_posterior(*args(pr)).predict(Xs)
    bad = dict(pr, thetas=pr["thetas"].copy())
    bad["thetas"][2, 1 + d] = -1.0  # negative kernel variances: the first pivot of latent 2 is negative or NaN
    bad["thetas"][2, 2 + 2 * d] = -1.0
    info = np.zeros(L, dtype=np.int32)
    m, v = h.svgp_posterior(*args(bad), info=info).predict(Xs)
    assert info[2] > 0 and np.all(info[[0, 1, 3]] == 0)
    assert m.shape == v.shape == (33, P)
    if mixing:
        assert np.isnan(m).all() and np.isnan(v).all()  # NaN * 0 = NaN: every output mixes latent 2
    else:
        assert np.isnan(m[:, 2]).all() and np.isnan(v[:, 2]).all()
        keep = [0, 1, 3]
        np.testing.assert_array_equal(m[:, keep], ref_m[:, keep])
        np.testing.assert_array_equal(v[:, keep], ref_v[:, keep])
    with pytest.raises(_lib.NotPositiveDefiniteError):
        h.svgp_posterior(*args(bad))
    np.testing.assert_array_equal(h.svgp_posterior(*args(pr)).predict(Xs)[0], ref_m)  # the handle's status was cleared


@pytest.mark.parametrize("M,mixing", [(50, False), (50, True), (70, False), (70, True)])
def test_result_is_independent_of_the_split(h, M, mixing):
    rng = np.random.default_rng(9)
    pr = synthetic(rng, M, 5, 6, mixing, P=8)
    post = h.svgp_posterior(*args(pr))
    Xs = random_points(rng, 1001, 5)
    m, v = post.predict(Xs)
    for cut in (1, 333, 1000):
        m1, v1 = post.predict(Xs[:cut])
        m2, v2 = post.predict(Xs[cut:])
        np.testing.assert_array_equal(np.concatenate([m1, m2]), m)
        np.testing.assert_array_equal(np.concatenate([v1, v2]), v)


@pytest.mark.parametrize("M", [50, 70])
def test_device_tensors_and_async_mode(h, M):
    import torch

    rng = np.random.default_rng(8)
    pr = synthetic(rng, M, 5, 4, True, P=6)
    Xs = random_points(rng, 50, 5)
    ref_m, ref_v = h.svgp_posterior(*args(pr)).predict(Xs)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    post = h.svgp_posterior(dev(pr["Z"]), dev(pr["thetas"]), dev(pr["W"]), dev(pr["q_mu"]), dev(pr["q_sqrt"]))
    dm = torch.empty((50, 6), dtype=torch.float64, device="cuda")
    dv = torch.empty((50, 6), dtype=torch.float64, device="cuda")
    h.set_stream(torch.cuda.current_stream().cuda_stream)
    h.set_async(True)
    try:
        post.predict(dev(Xs), dm, dv)
        assert h.sync() == 0
    finally:
        h.set_async(False)
        h.set_stream(None)
    np.testing.assert_array_equal(dm.cpu().numpy(), ref_m)
    np.testing.assert_array_equal(dv.cpu().numpy(), ref_v)


def test_lifetime_and_other_handles(h):
    import ctypes

    from multi_fidelity_gpflow_b200 import _lib

    ds = onp.load_dataset("hbs")
    pr = make_problem(np.random.default_rng(5), ds["Z_kmeans50"], 10, 5, 49, True)
    h1 = _lib.Handle(0)
    post = h1.svgp_posterior(*args(pr))
    Xs = ds["X_test"]
    ref_m, ref_v = post.predict(Xs)
    m, v = np.empty_like(ref_m), np.empty_like(ref_v)
    rc = _lib._lib.mfgp_svgp_posterior_predict(h._h, post._p, _lib._ptr(Xs), 10, _lib._ptr(m), _lib._ptr(v))
    assert rc == 0  # any handle on the posterior's device may use it
    np.testing.assert_array_equal(m, ref_m)
    np.testing.assert_array_equal(v, ref_v)
    h1.close()
    m[:], v[:] = 0.0, 0.0
    rc = _lib._lib.mfgp_svgp_posterior_predict(h._h, post._p, _lib._ptr(Xs), 10, _lib._ptr(m), _lib._ptr(v))
    assert rc == 0  # and it outlives the handle that made it
    np.testing.assert_array_equal(m, ref_m)
    assert _lib._lib.mfgp_svgp_posterior_destroy(post._p) == 0
    post._p = None
    p2 = h.svgp_posterior(*args(pr))
    assert p2.predict(Xs[:0])[0].shape == (0, 49)  # Ns == 0
    p2.close()
    p2.close()  # idempotent
    assert _lib._lib.mfgp_svgp_posterior_destroy(ctypes.c_void_p()) == 0


def se(d):
    from multi_fidelity_gpflow_b200.kernels import SquaredExponential

    return SquaredExponential(lengthscales=np.ones(d), variance=1.0)


@pytest.mark.parametrize("latent", [False, True])
def test_model_posterior(h, latent):
    from multi_fidelity_gpflow_b200.linear_svgp import LatentMFCoregionalizationSVGP
    from multi_fidelity_gpflow_b200.singlebin_svgp import SingleBinSVGP

    ds = onp.load_dataset("hbs")
    X, Y = ds["X"], ds["Y"]
    if latent:
        m = LatentMFCoregionalizationSVGP(X, Y, se(5), se(5), 10, num_inducing=50, handle=h)
    else:
        m = SingleBinSVGP(X, Y, se(5), se(5), 49, ds["Z_kmeans50"], handle=h)
    rng = np.random.default_rng(11)
    M, L = m.q_mu.shape
    m.q_mu.assign(0.3 * rng.standard_normal((M, L)))
    m.q_sqrt.assign(m.q_sqrt.numpy() + 0.02 * np.tril(rng.standard_normal((L, M, M))))
    Xs = np.vstack([ds["X_test"], X])
    post = m.posterior()
    pm, pv = post.predict_f(Xs)
    mm, mv = m.predict_f(Xs)
    assert pm.shape == mm.shape == (63, 49) and pv.shape == mv.shape
    close(pm, mm)
    close(pv, mv)
    m.q_mu.assign(m.q_mu.numpy() + 1.0)
    m.kernel.kernels[0].kernel_L.variance.assign(2.5)
    am, av = post.predict_f(Xs)
    np.testing.assert_array_equal(am, pm)  # the posterior keeps the parameters it was made with
    np.testing.assert_array_equal(av, pv)
    assert not np.allclose(m.predict_f(Xs)[0], pm)
    with pytest.raises(NotImplementedError):
        post.predict_f(Xs, full_cov=True)
