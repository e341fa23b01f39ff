"""GPU tests of mfgp_svgp_posterior_predict_grad: the input gradients of the cached SVGP posterior on both routes (fused
kernel for M <= 64, d <= 16; blocked otherwise) against the autograd oracle (1e-7 relative, atol 1e-7 max|ref|), mean and
var bitwise equal to predict, dead test rows, per-latent failure, split independence, pointer kinds, a second handle, the
model-level predict_f_grad and central differences of the library's own predict."""
import numpy as np
import pytest

from oracle import mfgp_oracle as onp
from tests._svgp_grad_oracle import svgp_predict_grad_x
from tests.test_svgp_posterior_gpu import args, make_problem, random_points, special_rows, synthetic

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def h():
    from multi_fidelity_gpflow_b200 import _lib

    return _lib.Handle(0)


def close(got, ref, tol=1e-7):
    ref = np.asarray(ref)
    np.testing.assert_allclose(got, ref, rtol=tol, atol=tol * max(np.abs(ref).max(), 1e-300))


def check(post, pr, Xs):
    """predict_grad against the oracle's gradients and against predict (bitwise); returns the four outputs."""
    mean, var, dm, dv = post.predict_grad(Xs)
    pm, pv = post.predict(Xs)
    np.testing.assert_array_equal(mean, pm)
    np.testing.assert_array_equal(var, pv)
    _, _, rdm, rdv = svgp_predict_grad_x(Xs, pr["Z"], pr["thetas"], pr["q_mu"], np.tril(pr["q_sqrt"]), pr["W"])
    assert dm.shape == rdm[..., :-1].shape and dv.shape == rdv[..., :-1].shape
    close(dm, rdm[..., :-1])
    close(dv, rdv[..., :-1])
    return mean, var, dm, dv


@pytest.mark.parametrize("mixing", [False, True])  # single-bin L = 49, latent L = 10 with W
def test_hbs_fused(h, mixing):
    ds = onp.load_dataset("hbs")
    rng = np.random.default_rng(21 if not mixing else 22)
    pr = make_problem(rng, ds["Z_kmeans50"], 10 if mixing else 49, 5, 49, mixing)
    Xs = np.vstack([ds["X_test"], ds["X"][::4], random_points(rng, 100, 5)])
    post = h.svgp_posterior(*args(pr))
    _, _, dm, dv = check(post, pr, Xs)
    assert dm.shape == dv.shape == (Xs.shape[0], 49, 5)
    _, _, dm0, dv0 = post.predict_grad(special_rows(ds["X"]))  # fidelity 0.5 / 1 + 1 ulp / NaN
    assert np.all(dm0 == 0.0) and np.all(dv0 == 0.0)


@pytest.mark.parametrize("mixing", [False, True])  # single-bin 8-bin subset, latent L = 15, P = 64
def test_goku_blocked(h, mixing):
    ds = onp.load_dataset("goku")
    Z = ds["Z_kmeans300"]
    assert np.any((Z[:, -1] != 0.0) & (Z[:, -1] != 1.0))  # quirk Q1: dead inducing points
    rng = np.random.default_rng(23)
    L, P = (15, 64) if mixing else (8, 8)
    pr = make_problem(rng, Z, L, 10, P, mixing)
    Xs = np.vstack([ds["X_test"], special_rows(ds["X"])])
    post = h.svgp_posterior(*args(pr))
    _, _, dm, dv = check(post, pr, Xs)
    assert dm.shape == (Xs.shape[0], P, 10)
    assert np.all(dm[-3:] == 0.0) and np.all(dv[-3:] == 0.0)


@pytest.mark.parametrize("M,d,L,P,Ns", [
    (1, 1, 1, 0, 1), (8, 1, 2, 5, 7), (9, 16, 1, 0, 7), (63, 5, 4, 2, 9), (64, 16, 3, 0, 7), (64, 3, 1, 4, 2049),
    (65, 5, 2, 0, 9), (65, 16, 3, 5, 7), (30, 17, 2, 0, 9), (9, 17, 4, 2, 2049),
])
def test_edge_sizes(h, M, d, L, P, Ns):
    """Fused route for M <= 64 and d <= 16, blocked otherwise; P = 0: no W, else W [P, L] with P > L or P < L."""
    rng = np.random.default_rng(M * 1000 + d * 10 + L)
    pr = synthetic(rng, M, d, L, P > 0, P=P)
    check(h.svgp_posterior(*args(pr)), pr, random_points(rng, Ns, d))


@pytest.mark.parametrize("M", [20, 70])  # fused and blocked route
@pytest.mark.parametrize("mixing", [False, True])
def test_failed_latent_gives_nan(h, M, mixing):
    rng = np.random.default_rng(27)
    L, d = 4, 5
    pr = synthetic(rng, M, d, L, mixing, P=6)
    Xs = random_points(rng, 33, d)
    ref = h.svgp_posterior(*args(pr)).predict_grad(Xs)
    bad = dict(pr, thetas=pr["thetas"].copy())
    bad["thetas"][2, 1 + d] = -1.0
    bad["thetas"][2, 2 + 2 * d] = -1.0
    info = np.zeros(L, dtype=np.int32)
    out = h.svgp_posterior(*args(bad), info=info).predict_grad(Xs)
    assert info[2] > 0
    for got, r in zip(out, ref):
        if mixing:
            assert np.isnan(got).all()
        else:
            assert np.isnan(got[:, 2]).all()
            np.testing.assert_array_equal(got[:, [0, 1, 3]], r[:, [0, 1, 3]])


@pytest.mark.parametrize("M,mixing", [(50, False), (50, True), (70, False), (70, True)])
def test_result_is_independent_of_the_split(h, M, mixing):
    rng = np.random.default_rng(29)
    pr = synthetic(rng, M, 5, 6, mixing, P=8)
    post = h.svgp_posterior(*args(pr))
    Xs = random_points(rng, 1001, 5)
    full = post.predict_grad(Xs)
    for s in (0, 7, 500, 1000):
        alone = post.predict_grad(Xs[s:s + 1])
        inner = post.predict_grad(Xs[s - 3 if s >= 3 else 0:])
        o = s - (s - 3 if s >= 3 else 0)
        for a, b, c in zip(full, alone, inner):
            np.testing.assert_array_equal(a[s], b[0])
            np.testing.assert_array_equal(a[s], c[o])


@pytest.mark.parametrize("M", [50, 70])
def test_device_tensors_async_and_second_handle(h, M):
    import torch

    from multi_fidelity_gpflow_b200 import _lib

    rng = np.random.default_rng(31)
    pr = synthetic(rng, M, 5, 4, True, P=6)
    Xs = random_points(rng, 50, 5)
    ref = h.svgp_posterior(*args(pr)).predict_grad(Xs)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    h2 = _lib.Handle(0)
    post = h2.svgp_posterior(dev(pr["Z"]), dev(pr["thetas"]), dev(pr["W"]), dev(pr["q_mu"]), dev(pr["q_sqrt"]))
    outs = [torch.empty(s, dtype=torch.float64, device="cuda") for s in ((50, 6), (50, 6), (50, 6, 5), (50, 6, 5))]
    h.set_stream(torch.cuda.current_stream().cuda_stream)
    h.set_async(True)
    try:
        rc = _lib._lib.mfgp_svgp_posterior_predict_grad(h._h, post._p, _lib._ptr(dev(Xs)), 50, *[_lib._ptr(o) for o in outs])
        assert rc == 0 and h.sync() == 0  # the posterior of handle h2 through handle h, on h's stream
    finally:
        h.set_async(False)
        h.set_stream(None)
    for o, r in zip(outs, ref):
        np.testing.assert_array_equal(o.cpu().numpy(), r)
    assert post.predict_grad(Xs[:0])[2].shape == (0, 6, 5)  # Ns == 0
    m = np.empty((50, 6))
    assert _lib._lib.mfgp_svgp_posterior_predict_grad(h._h, post._p, _lib._ptr(Xs), 50, _lib._ptr(m), _lib._ptr(m),
                                                      None, None) != 0  # dmean and dvar are required
    post.close()
    h2.close()


@pytest.mark.parametrize("M,d", [(40, 5), (80, 5), (30, 17)])
def test_central_differences_of_predict(h, M, d):
    rng = np.random.default_rng(37)
    pr = synthetic(rng, M, d, 3, True, P=4)
    post = h.svgp_posterior(*args(pr))
    Xs = random_points(rng, 20, d)
    _, _, dm, dv = post.predict_grad(Xs)
    step = 1e-5
    for j in range(d):
        xp, xm = Xs.copy(), Xs.copy()
        xp[:, j] += step
        xm[:, j] -= step
        (mp, vp), (mm, vm) = post.predict(xp), post.predict(xm)
        np.testing.assert_allclose(dm[:, :, j], (mp - mm) / (2 * step), rtol=1e-5, atol=1e-6 * np.abs(dm).max())
        np.testing.assert_allclose(dv[:, :, j], (vp - vm) / (2 * step), rtol=1e-5, atol=1e-6 * np.abs(dv).max())


def se(d):
    from multi_fidelity_gpflow_b200.kernels import SquaredExponential

    return SquaredExponential(lengthscales=np.ones(d), variance=1.0)


@pytest.mark.parametrize("latent", [False, True])
def test_model_predict_f_grad(h, latent):
    from multi_fidelity_gpflow_b200.linear_svgp import LatentMFCoregionalizationSVGP
    from multi_fidelity_gpflow_b200.singlebin_svgp import SingleBinSVGP

    ds = onp.load_dataset("hbs")
    X, Y = ds["X"], ds["Y"]
    if latent:
        m = LatentMFCoregionalizationSVGP(X, Y, se(5), se(5), 10, num_inducing=50, handle=h)
    else:
        m = SingleBinSVGP(X, Y, se(5), se(5), 49, ds["Z_kmeans50"], handle=h)
    rng = np.random.default_rng(41)
    M, L = m.q_mu.shape
    m.q_mu.assign(0.3 * rng.standard_normal((M, L)))
    post = m.posterior()
    mean, var, dm, dv = post.predict_f_grad(ds["X_test"])
    pm, pv = post.predict_f(ds["X_test"])
    np.testing.assert_array_equal(mean, pm)
    np.testing.assert_array_equal(var, pv)
    assert dm.shape == dv.shape == (10, 49, 6)
    assert np.all(dm[..., -1] == 0.0) and np.all(dv[..., -1] == 0.0)
    _, _, rdm, rdv = svgp_predict_grad_x(ds["X_test"], m.Z.numpy(), m._thetas(5), m.q_mu.numpy(), np.tril(m.q_sqrt.numpy()),
                                         m._W())
    close(dm, rdm)
    close(dv, rdv)
