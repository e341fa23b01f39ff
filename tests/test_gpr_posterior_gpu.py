"""GPU tests of the cached exact-GP posterior (mfgp_gpr_posterior_*): both predict routes (fused kernel for N <= 64,
d <= 16, P <= 64; blocked otherwise) against the oracle's GPR.predict_f per problem (1e-8 relative, atol 1e-8 max|ref|),
the model-level posteriors against today's predict_f, per-problem failure, reuse, chunking, pointer kinds and lifetime."""
import numpy as np
import pytest

from oracle import mfgp_oracle as onp

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def h():
    from multi_fidelity_gpflow_b200 import _lib

    return _lib.Handle(0)


def close(got, ref):
    ref = np.asarray(ref)
    np.testing.assert_allclose(got, ref, rtol=1e-8, atol=1e-8 * max(np.abs(ref).max(), 1e-300))


def check_all(X, Y, Xs, th, nz, P, mean, var):
    B, ycols = th.shape[0], Y.shape[1]
    assert mean.shape == (B, Xs.shape[0], P) and var.shape == (B, Xs.shape[0])
    for b in range(B):
        c = (b * P) % ycols
        rm, rv = onp.gpr_predict(X, Y[:, c:c + P], Xs, th[b], nz[b])
        close(mean[b], rm)
        close(var[b], rv)


def hbs_perturbed(R=1, seed=0):
    ds = onp.load_dataset("hbs")
    B = 49 * R
    rng = np.random.default_rng(seed)
    th = np.tile(onp.default_theta(5), (B, 1)) * np.exp(0.3 * rng.standard_normal((B, 13)))
    nz = np.full(B, 1e-3) * np.exp(0.3 * rng.standard_normal(B))
    return ds, th, nz


def special_rows(X):
    s = np.repeat(X[:1], 3, axis=0).copy()
    s[:, -1] = [0.5, np.nextafter(1.0, 2.0), np.nan]
    return s


def test_hbs_all_bins_fused(h):
    ds, th, nz = hbs_perturbed()
    X, Y = ds["X"], ds["Y"]
    post = h.gpr_posterior(X, Y, th, nz)
    Xs = np.vstack([ds["X_test"], X])  # test inputs and the training inputs of both fidelities
    mean, var = post.predict(Xs)
    check_all(X, Y, Xs, th, nz, 1, mean, var)
    m0, v0 = post.predict(special_rows(X))  # fidelity 0.5 / 1 + 1 ulp / NaN: zero covariance, like the oracle
    assert np.all(m0 == 0.0) and np.all(v0 == 0.0)
    post.close()


def synthetic(rng, N, d, ycols, frac=0.4):
    X = np.hstack([rng.random((N, d)), (rng.random((N, 1)) < frac).astype(float)])
    Y = rng.standard_normal((N, ycols))
    return X, Y


@pytest.mark.parametrize("N,d,P,Ns", [
    (1, 1, 1, 1), (2, 5, 1, 7), (63, 5, 1, 8), (64, 16, 1, 9), (64, 5, 3, 1000), (40, 1, 8, 9), (53, 5, 49, 7),
    (64, 3, 64, 8), (30, 17, 1, 9), (65, 5, 1, 7), (130, 5, 2, 1000), (20, 5, 65, 8),
])
def test_edge_sizes(h, N, d, P, Ns):
    """Fused route: N <= 64, d <= 16, P <= 64; the blocked route for d = 17, N = 65 / 130, P = 65."""
    rng = np.random.default_rng(N * 1000 + d * 10 + P)
    B = 3
    X, Y = synthetic(rng, N, d, B * P)
    th = np.tile(onp.default_theta(d), (B, 1)) * np.exp(0.2 * rng.standard_normal((B, 2 * d + 3)))
    th[:, 1:1 + d] *= np.sqrt(d)  # keep the covariance away from the identity in high d
    th[:, 2 + d:2 + 2 * d] *= np.sqrt(d)
    nz = np.full(B, 1e-2)
    Xs = np.hstack([rng.random((Ns, d)), rng.integers(0, 2, (Ns, 1)).astype(float)])
    mean, var = h.gpr_posterior(X, Y, th, nz, P=P).predict(Xs)
    check_all(X, Y, Xs, th, nz, P, mean, var)


def test_hbs_every_bin_and_restart_in_one_call(h):
    ds, th, nz = hbs_perturbed(R=64, seed=1)
    X, Y = ds["X"], ds["Y"]
    mean, var = h.gpr_posterior(X, Y, th, nz).predict(ds["X_test"])
    assert mean.shape == (49 * 64, 10, 1)
    check_all(X, Y, ds["X_test"], th, nz, 1, mean, var)


def se(d):
    from multi_fidelity_gpflow_b200.kernels import SquaredExponential

    return SquaredExponential(lengthscales=np.ones(d), variance=1.0)


def test_multi_output_model_posterior(h):
    from multi_fidelity_gpflow_b200.linear import MultiFidelityGPModel

    ds = onp.load_dataset("hbs")
    m = MultiFidelityGPModel(ds["X"], ds["Y"], se(5), se(5), handle=h)
    post = m.posterior()
    Xs = np.vstack([ds["X_test"], ds["X"]])
    pm, pv = post.predict_f(Xs)
    mm, mv = m.predict_f(Xs)
    assert pm.shape == mm.shape == (63, 49) and pv.shape == mv.shape
    close(pm, mm)
    close(pv, mv)
    ym, yv = post.predict_y(Xs)
    np.testing.assert_array_equal(ym, pm)
    np.testing.assert_allclose(yv, pv + 1e-3, rtol=1e-15)


def test_goku_shared_and_per_bin_blocked(h):
    ds = onp.load_dataset("goku")
    X, Y, Xs = ds["X"], ds["Y"], ds["X_test"]
    th = onp.default_theta(10)
    mean, var = h.gpr_posterior(X, Y, th[None], np.array([1e-3]), P=64).predict(Xs)
    rm, rv = onp.gpr_predict(X, Y, Xs, th, 1e-3)
    close(mean[0], rm)
    close(var[0], rv)
    rng = np.random.default_rng(5)
    ths = np.tile(th, (4, 1)) * np.exp(0.1 * rng.standard_normal((4, 23)))
    nz = np.full(4, 1e-3)
    Y4 = np.ascontiguousarray(Y[:, :4])
    mean, var = h.gpr_posterior(X, Y4, ths, nz).predict(Xs)
    check_all(X, Y4, Xs, ths, nz, 1, mean, var)


def test_multibin_posterior_best_and_all(h):
    from multi_fidelity_gpflow_b200.multibin import MultiBinMFGP

    ds = onp.load_dataset("hbs")
    X, Y = ds["X"], ds["Y"]
    mdl = MultiBinMFGP(X, Y, num_restarts=3, seed=2, handle=h).optimize(max_iters=20, learning_rate=0.02)
    Xs = np.vstack([ds["X_test"], X[X[:, -1] == 1.0]])
    bm, bv = mdl.posterior("best").predict_f(Xs)
    pm, pv = mdl.predict_f(Xs)
    close(bm, pm)
    close(bv, pv)
    post = mdl.posterior("all")
    am, av = post.predict_f(Xs)
    assert am.shape == (3, Xs.shape[0], 49) and not post.failed.any()
    th = mdl.thetas
    for r in range(3):
        for p in range(49):
            rm, rv = onp.gpr_predict(X, Y[:, p:p + 1], Xs, th[r, p], mdl.noise)
            close(am[r, :, p], rm[:, 0])
            close(av[r, :, p], rv)
    _, yv = post.predict_y(Xs)
    np.testing.assert_allclose(yv, av + mdl.noise, rtol=1e-15)


@pytest.mark.parametrize("N", [53, 100])  # fused and blocked route
def test_non_pd_problem_is_its_own_status(h, N):
    from multi_fidelity_gpflow_b200 import _lib

    rng = np.random.default_rng(7)
    X, Y = synthetic(rng, N, 5, 4)
    th = np.tile(onp.default_theta(5), (4, 1))
    good = np.full(4, 1e-3)
    bad = good.copy()
    bad[2] = -5.0
    Xs = rng.random((17, 6))
    Xs[:, -1] = np.arange(17) % 2
    ref_m, ref_v = h.gpr_posterior(X, Y, th, good).predict(Xs)
    info = np.zeros(4, dtype=np.int32)
    m, v = h.gpr_posterior(X, Y, th, bad, info=info).predict(Xs)
    assert info[2] > 0 and np.all(info[[0, 1, 3]] == 0)
    assert np.isnan(m[2]).all() and np.isnan(v[2]).all()
    keep = [0, 1, 3]
    np.testing.assert_array_equal(m[keep], ref_m[keep])
    np.testing.assert_array_equal(v[keep], ref_v[keep])
    with pytest.raises(_lib.NotPositiveDefiniteError):
        h.gpr_posterior(X, Y, th, bad)
    h.gpr_batched_nlml_grad(X, Y, th, good)  # the handle's status was cleared: the next call succeeds


def test_reuse_across_other_calls_and_workspace_modes(h):
    from multi_fidelity_gpflow_b200.optimizers import adam_step_factors

    ds, th, nz = hbs_perturbed(seed=3)
    X, Y = ds["X"], ds["Y"]
    posts = [h.gpr_posterior(X, Y, th, nz), h.gpr_posterior(X, np.ascontiguousarray(Y[:, :4]), th[:4], nz[:4], P=2)]
    Xs = np.vstack([ds["X_test"], X])
    first = [p.predict(Xs) for p in posts]
    h.gpr_batched_nlml_grad(X, Y, th, nz)
    u = onp.softplus_inv(th.copy())
    lr_t, b1, b2 = adam_step_factors(0.01, 5)
    h.gpr_batched_adam(X, Y, u, np.zeros_like(u), np.zeros_like(u), nz, lr_t, b1, b2)
    h.workspace(h.WS_MEASURE)
    h.gpr_batched_nlml_grad(X, Y, th, nz)
    h.workspace(h.WS_FIXED)
    mid = [p.predict(Xs) for p in posts]
    h.gpr_batched_nlml_grad(X, Y, th, nz)
    h.workspace(h.WS_POOL)
    last = [p.predict(Xs) for p in posts]
    for a, b, c in zip(first, mid, last):
        for k in range(2):
            np.testing.assert_array_equal(a[k], b[k])
            np.testing.assert_array_equal(a[k], c[k])


def test_fused_route_is_independent_of_the_split(h):
    ds, th, nz = hbs_perturbed(seed=4)
    post = h.gpr_posterior(ds["X"], ds["Y"], th, nz)
    rng = np.random.default_rng(0)
    Xs = np.hstack([rng.random((1001, 5)), rng.integers(0, 2, (1001, 1)).astype(float)])
    m, v = post.predict(Xs)
    for cut in (1, 333, 1000):
        m1, v1 = post.predict(Xs[:cut])
        m2, v2 = post.predict(Xs[cut:])
        np.testing.assert_array_equal(np.concatenate([m1, m2], axis=1), m)
        np.testing.assert_array_equal(np.concatenate([v1, v2], axis=1), v)
    Y59 = np.ascontiguousarray(ds["Y"][:, 5:9])  # nor do the other problems of the call
    ms, vs = h.gpr_posterior(ds["X"], Y59, th[5:9], nz[5:9]).predict(Xs)
    np.testing.assert_array_equal(ms, m[5:9])
    np.testing.assert_array_equal(vs, v[5:9])


@pytest.mark.parametrize("N", [53, 100])
def test_device_tensors_and_async_mode(h, N):
    import torch

    rng = np.random.default_rng(8)
    X, Y = synthetic(rng, N, 5, 6)
    th = np.tile(onp.default_theta(5), (6, 1)) * np.exp(0.2 * rng.standard_normal((6, 13)))
    nz = np.full(6, 1e-3)
    Xs = np.hstack([rng.random((50, 5)), rng.integers(0, 2, (50, 1)).astype(float)])
    ref_m, ref_v = h.gpr_posterior(X, Y, th, nz, P=2).predict(Xs)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    post = h.gpr_posterior(dev(X), dev(Y), dev(th), dev(nz), P=2)
    dm, dv = torch.empty((6, 50, 2), dtype=torch.float64, device="cuda"), torch.empty((6, 50), dtype=torch.float64, device="cuda")
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

    ds, th, nz = hbs_perturbed(seed=5)
    h1 = _lib.Handle(0)
    post = h1.gpr_posterior(ds["X"], ds["Y"], th, nz)
    ref_m, ref_v = post.predict(ds["X_test"])
    m, v = np.empty_like(ref_m), np.empty_like(ref_v)
    rc = _lib._lib.mfgp_gpr_posterior_predict(h._h, post._p, _lib._ptr(ds["X_test"]), 10, _lib._ptr(m), _lib._ptr(v))
    assert rc == 0  # any handle on the posterior's device may use it
    np.testing.assert_array_equal(m, ref_m)
    np.testing.assert_array_equal(v, ref_v)
    h1.close()
    assert _lib._lib.mfgp_gpr_posterior_destroy(post._p) == 0  # destroyed after its handle
    post._p = None
    p2 = h.gpr_posterior(ds["X"], ds["Y"], th, nz)
    p2.close()
    p2.close()  # idempotent
    assert _lib._lib.mfgp_gpr_posterior_destroy(ctypes.c_void_p()) == 0
