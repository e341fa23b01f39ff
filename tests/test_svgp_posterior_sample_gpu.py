"""GPU tests of the joint posterior of the cached SVGP (mfgp_svgp_posterior_predict_cov, mfgp_svgp_posterior_sample) on
both routes (svgp_posterior_joint_kernel for M <= 64, d <= 16 and Ns <= 64; the blocked route otherwise): cov against the
oracle, mean and diag(cov) bit for bit against predict, exact symmetry, samples against numpy's Cholesky of the library's
own covariance, every switch and tile count of the fused kernel, special rows, failures, the S independence of a column,
pointer kinds, async mode, argument checks and the model-level methods."""
import ctypes

import numpy as np
import pytest

from oracle import mfgp_oracle as onp
from tests._svgp_joint_oracle import svgp_predict_full_cov
from tests.test_svgp_posterior_gpu import args, make_problem, random_points, special_rows, synthetic

pytestmark = pytest.mark.gpu
JITTER = 1e-6
ROUTE_TOL = 4e-12  # route differences relative to the output's scale (test_posterior_tile_sweep_gpu.py)


@pytest.fixture(scope="module")
def h():
    from multi_fidelity_gpflow_b200 import _lib

    return _lib.Handle(0)


def ref_of(pr):
    return dict(pr, q_sqrt=np.tril(pr["q_sqrt"]))


def check_oracle(pr, Xs, mean, cov):
    rm, rc = svgp_predict_full_cov(Xs, pr["Z"], pr["thetas"], pr["q_mu"], np.tril(pr["q_sqrt"]), pr["W"])
    assert mean.shape == rm.shape and cov.shape == rc.shape
    np.testing.assert_allclose(mean, rm, rtol=1e-8, atol=1e-8 * max(np.abs(rm).max(), 1e-300))
    kmax = max(max(onp.mf_K_diag(Xs, th).max() for th in pr["thetas"]), 1e-300)
    if pr["W"] is not None:
        kmax *= max((pr["W"] ** 2).sum(axis=1).max(), 1e-300)
    np.testing.assert_allclose(cov, rc, rtol=1e-8, atol=1e-8 * kmax)


def check_against_predict(post, Xs, mean, cov):
    pm, pv = post.predict(Xs)
    np.testing.assert_array_equal(mean, pm)
    np.testing.assert_array_equal(np.diagonal(cov, axis1=1, axis2=2).T, pv)
    np.testing.assert_array_equal(cov, np.swapaxes(cov, 1, 2))


def check_samples(post, Xs, mean, cov, S, seed, jitter=JITTER):
    P, Ns = cov.shape[0], cov.shape[1]
    z = np.random.default_rng(seed).standard_normal((P, Ns, S))
    s = post.sample(Xs, z, jitter=jitter)
    assert s.shape == (P, Ns, S)
    for p in range(P):
        Lc = np.linalg.cholesky(cov[p] + jitter * np.eye(Ns))
        ref = mean[:, p][:, None] + Lc @ z[p]
        np.testing.assert_allclose(s[p], ref, rtol=1e-10, atol=1e-10 * np.abs(ref).max())
    return z, s


def run_all(h, pr, Xs, S=16, seed=0):
    post = h.svgp_posterior(*args(pr))
    mean, cov = post.predict_cov(Xs)
    check_oracle(pr, Xs, mean, cov)
    check_against_predict(post, Xs, mean, cov)
    check_samples(post, Xs, mean, cov, S, seed)
    return post, mean, cov


@pytest.mark.parametrize("mixing", [False, True])  # single-bin L = P = 49, latent L = 10 with W [49, 10]
def test_hbs_fused(h, mixing):
    ds = onp.load_dataset("hbs")
    rng = np.random.default_rng(21 + mixing)
    pr = make_problem(rng, ds["Z_kmeans50"], 10 if mixing else 49, 5, 49, mixing)
    Xs = np.vstack([ds["X_test"], random_points(rng, 54, 5)])  # Ns = 64: the largest fused size
    run_all(h, pr, Xs, S=1024)


@pytest.mark.parametrize("Ns", [36, 256])
@pytest.mark.parametrize("mixing", [False, True])  # single-bin L = P = 64, latent L = 15 with W [64, 15]; M = 300
def test_goku_blocked(h, mixing, Ns):
    ds = onp.load_dataset("goku")
    rng = np.random.default_rng(31 + mixing + Ns)
    pr = make_problem(rng, ds["Z_kmeans300"], 15 if mixing else 64, 10, 64, mixing)
    Xs = np.vstack([ds["X_test"], ds["X"]])[:Ns]
    assert Xs.shape[0] == Ns
    run_all(h, pr, Xs, S=16)


@pytest.mark.parametrize("M,d,Ns", [(64, 5, 40), (65, 5, 40), (30, 16, 40), (30, 17, 40), (40, 5, 64), (40, 5, 65)])
@pytest.mark.parametrize("mix", ["none", "P>L", "P<L"])
def test_switches(h, M, d, Ns, mix):
    rng = np.random.default_rng(M * 100 + d * 10 + Ns)
    L, P = {"none": (4, 4), "P>L": (3, 7), "P<L": (6, 2)}[mix]
    pr = synthetic(rng, M, d, L, mix != "none", P=P)
    Xs = random_points(rng, Ns, d)
    run_all(h, pr, Xs, S=33, seed=M)


@pytest.mark.parametrize("mix", ["none", "P>L", "P<L"])
def test_fused_and_blocked_routes_agree(h, mix):
    """The first 64 points of an Ns = 65 call (blocked) match the Ns = 64 call (fused)."""
    rng = np.random.default_rng(41)
    L, P = {"none": (4, 4), "P>L": (3, 7), "P<L": (6, 2)}[mix]
    pr = synthetic(rng, 50, 5, L, mix != "none", P=P)
    Xs = random_points(rng, 65, 5)
    post = h.svgp_posterior(*args(pr))
    m64, c64 = post.predict_cov(Xs[:64])
    m65, c65 = post.predict_cov(Xs)
    np.testing.assert_array_equal(m65[:64], m64)  # predict's own route for both
    scale = np.abs(c64).max()
    assert np.abs(c65[:, :64, :64] - c64).max() <= ROUTE_TOL * scale


def tile_cases():
    cases = []
    for M in range(1, 65):
        NT = (M + 7) // 8
        Ns = 1 + (7 * M + 3 * NT) % 64  # walks through every NST = ceil(Ns / 8)
        cases.append((M, 1 if M % 2 else 16, Ns, ["none", "P>L", "P<L"][M % 3]))
    return cases


def test_tile_cases_cover_every_nt_and_nst():
    cs = tile_cases()
    assert {(M + 7) // 8 for M, _, _, _ in cs} == set(range(1, 9))
    assert {M % 8 for M, _, _, _ in cs} == set(range(8))
    assert {(Ns + 7) // 8 for _, _, Ns, _ in cs} == set(range(1, 9))
    assert {d for _, d, _, _ in cs} == {1, 16}


@pytest.mark.parametrize("M,d,Ns,mix", tile_cases())
def test_tile_sweep(h, M, d, Ns, mix):
    rng = np.random.default_rng(1000 + M)
    L, P = {"none": (2, 2), "P>L": (2, 3), "P<L": (3, 2)}[mix]
    pr = synthetic(rng, M, d, L, mix != "none", P=P)
    Xs = random_points(rng, Ns, d)
    post = h.svgp_posterior(*args(pr))
    mean, cov = post.predict_cov(Xs)
    check_oracle(pr, Xs, mean, cov)
    check_against_predict(post, Xs, mean, cov)


def test_special_rows(h):
    ds = onp.load_dataset("hbs")
    rng = np.random.default_rng(51)
    pr = make_problem(rng, ds["Z_kmeans50"], 10, 5, 49, True)
    post = h.svgp_posterior(*args(pr))
    sp = special_rows(ds["X"])  # fidelity 0.5 / 1 + 1 ulp / NaN: dead rows
    Z = pr["Z"]
    Xs = np.vstack([ds["X_test"], sp, Z[3:4]])  # and a test point on an inducing point
    mean, cov = post.predict_cov(Xs)
    check_against_predict(post, Xs, mean, cov)
    dead = np.arange(10, 13)
    assert np.all(mean[dead] == 0.0)
    assert np.all(cov[:, dead, :] == 0.0) and np.all(cov[:, :, dead] == 0.0)
    live = np.setdiff1d(np.arange(Xs.shape[0]), dead)
    check_oracle(pr, Xs[live], mean[live], cov[:, live][:, :, live])
    z = np.random.default_rng(2).standard_normal((49, Xs.shape[0], 8))
    s = post.sample(Xs, z)
    np.testing.assert_allclose(s[:, dead], np.sqrt(JITTER) * z[:, dead], rtol=1e-14, atol=0)
    info = np.zeros(49, dtype=np.int32)
    post.sample(Xs, z, jitter=0.0, info=info)
    assert np.all(info == 11)  # the first dead row is a zero pivot with jitter 0


def test_duplicate_points(h, record_property):
    """A duplicated test point makes Sigma_p singular: with the jitter every output factors; with jitter 0 an output either
    factors or reports a pivot at or after the duplicate, with NaN samples, and leaves the others bit for bit as a
    posterior of those latents alone gives them."""
    from multi_fidelity_gpflow_b200 import _lib

    ds = onp.load_dataset("hbs")
    rng = np.random.default_rng(61)
    pr = make_problem(rng, ds["Z_kmeans50"], 49, 5, 49, False)
    post = h.svgp_posterior(*args(pr))
    Xs = np.vstack([random_points(rng, 10, 5), np.zeros((1, 6))])
    Xs[10] = Xs[3]
    z = np.random.default_rng(3).standard_normal((49, 11, 4))
    assert np.isfinite(post.sample(Xs, z)).all()
    info = np.zeros(49, dtype=np.int32)
    s = post.sample(Xs, z, jitter=0.0, info=info)
    bad = info != 0
    record_property("failed_outputs", int(bad.sum()))
    assert np.all(info[bad] >= 11)
    assert np.isnan(s[bad]).all() and np.isfinite(s[~bad]).all()
    keep = np.flatnonzero(~bad)
    if keep.size:
        sub = dict(pr, thetas=pr["thetas"][keep], q_mu=np.ascontiguousarray(pr["q_mu"][:, keep]), q_sqrt=pr["q_sqrt"][keep])
        ref = h.svgp_posterior(*args(sub)).sample(Xs, np.ascontiguousarray(z[keep]), jitter=0.0)
        np.testing.assert_array_equal(s[keep], ref)
    if bad.any():
        with pytest.raises(_lib.NotPositiveDefiniteError):
            post.sample(Xs, z, jitter=0.0)


@pytest.mark.parametrize("M", [20, 70])  # fused and blocked route
@pytest.mark.parametrize("mixing", [False, True])
def test_failed_latent(h, M, mixing):
    rng = np.random.default_rng(71)
    L, d = 4, 5
    pr = synthetic(rng, M, d, L, mixing, P=6)
    P = 6 if mixing else L
    Xs = random_points(rng, 33, d)
    good = h.svgp_posterior(*args(pr))
    ref_m, ref_c = good.predict_cov(Xs)
    z = np.random.default_rng(4).standard_normal((P, 33, 5))
    ref_s = good.sample(Xs, z)
    bad = dict(pr, thetas=pr["thetas"].copy())
    bad["thetas"][2, 1 + d] = -1.0
    bad["thetas"][2, 2 + 2 * d] = -1.0
    info_c = np.zeros(L, dtype=np.int32)
    post = h.svgp_posterior(*args(bad), info=info_c)
    assert info_c[2] > 0
    mean, cov = post.predict_cov(Xs)  # returns 0
    info = np.zeros(P, dtype=np.int32)
    s = post.sample(Xs, z, info=info)
    hit = np.arange(P) == 2 if not mixing else np.ones(P, dtype=bool)  # NaN * 0 = NaN: with W every output
    assert np.all(info[hit] == 1) and np.all(info[~hit] == 0)
    assert np.isnan(s[hit]).all() and np.isnan(cov[hit]).all() and np.isnan(mean[:, hit]).all()
    np.testing.assert_array_equal(s[~hit], ref_s[~hit])
    np.testing.assert_array_equal(cov[~hit], ref_c[~hit])
    from multi_fidelity_gpflow_b200 import _lib

    with pytest.raises(_lib.NotPositiveDefiniteError):
        post.sample(Xs, z)


@pytest.mark.parametrize("Ns", [40, 100])
def test_column_does_not_depend_on_s(h, Ns):
    rng = np.random.default_rng(81)
    pr = synthetic(rng, 30, 5, 3, True, P=5)
    post = h.svgp_posterior(*args(pr))
    Xs = random_points(rng, Ns, 5)
    z = np.random.default_rng(5).standard_normal((5, Ns, 1000))
    big = post.sample(Xs, z)
    small = post.sample(Xs, np.ascontiguousarray(z[:, :, :7]))
    np.testing.assert_array_equal(big[:, :, :7], small)


@pytest.mark.parametrize("M", [50, 70])
def test_device_tensors_async_and_other_handle(h, M):
    import torch

    from multi_fidelity_gpflow_b200 import _lib

    rng = np.random.default_rng(91)
    pr = synthetic(rng, M, 5, 4, True, P=6)
    Xs = random_points(rng, 50, 5)
    post = h.svgp_posterior(*args(pr))
    ref_m, ref_c = post.predict_cov(Xs)
    z = np.random.default_rng(6).standard_normal((6, 50, 9))
    ref_s = post.sample(Xs, z)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    dm = torch.empty((50, 6), dtype=torch.float64, device="cuda")
    dc = torch.empty((6, 50, 50), dtype=torch.float64, device="cuda")
    ds = torch.empty((6, 50, 9), dtype=torch.float64, device="cuda")
    h.set_stream(torch.cuda.current_stream().cuda_stream)
    h.set_async(True)
    try:
        post.predict_cov(dev(Xs), dm, dc)
        post.sample(dev(Xs), dev(z), samples=ds)
        assert h.sync() == 0
    finally:
        h.set_async(False)
        h.set_stream(None)
    np.testing.assert_array_equal(dm.cpu().numpy(), ref_m)
    np.testing.assert_array_equal(dc.cpu().numpy(), ref_c)
    np.testing.assert_array_equal(ds.cpu().numpy(), ref_s)
    h2 = _lib.Handle(0)
    m2, c2 = np.empty_like(ref_m), np.empty_like(ref_c)
    assert _lib._lib.mfgp_svgp_posterior_predict_cov(h2._h, post._p, _lib._ptr(Xs), 50, _lib._ptr(m2), _lib._ptr(c2)) == 0
    np.testing.assert_array_equal(c2, ref_c)
    h2.close()


def test_argument_checks(h):
    from multi_fidelity_gpflow_b200 import _lib

    rng = np.random.default_rng(101)
    pr = synthetic(rng, 10, 3, 2, True, P=3)
    post = h.svgp_posterior(*args(pr))
    Xs = random_points(rng, 5, 3)
    buf = np.random.default_rng(7).standard_normal((3, 5, 4))
    f = _lib._lib.mfgp_svgp_posterior_sample
    P_ = _lib._ptr
    assert f(h._h, post._p, P_(Xs), 5, 4, 1e-6, P_(buf), P_(buf), None) == -1  # z overlaps samples
    out = np.empty_like(buf)
    assert f(h._h, post._p, P_(Xs), 5, 4, -1e-6, P_(buf), P_(out), None) == -1
    assert f(h._h, post._p, P_(Xs), 5, 4, float("nan"), P_(buf), P_(out), None) == -1
    assert f(h._h, post._p, P_(Xs), 5, -1, 1e-6, P_(buf), P_(out), None) == -1
    assert f(h._h, post._p, P_(Xs), 5, 0, 1e-6, P_(buf), P_(out), None) == 0
    assert f(h._h, post._p, P_(Xs), 0, 4, 1e-6, P_(buf), P_(out), None) == 0
    assert _lib._lib.mfgp_svgp_posterior_predict_cov(h._h, post._p, P_(Xs), 5, None, P_(out)) == -1
    # P > 65 535 outputs: _predict accepts them, the joint calls do not
    P = 65536
    W = np.full((P, 1), 0.5)
    big = h.svgp_posterior(pr["Z"], pr["thetas"][:1], W, pr["q_mu"][:, :1], pr["q_sqrt"][:1])
    pm, pv = big.predict(Xs)
    assert pm.shape == (5, P)
    m, c = np.empty((5, P)), np.empty((P, 5, 5))
    assert _lib._lib.mfgp_svgp_posterior_predict_cov(h._h, big._p, P_(Xs), 5, P_(m), P_(c)) == -1
    assert "65535" in _lib._lib.mfgp_last_error(h._h).decode()
    zb = np.zeros((P, 5, 1))
    sb = np.empty_like(zb)
    assert f(h._h, big._p, P_(Xs), 5, 1, 1e-6, P_(zb), P_(sb), None) == -1


def se(d):
    from multi_fidelity_gpflow_b200.kernels import SquaredExponential

    return SquaredExponential(lengthscales=np.ones(d), variance=1.0)


@pytest.mark.parametrize("latent", [False, True])
def test_model_level(h, latent):
    from multi_fidelity_gpflow_b200.linear_svgp import LatentMFCoregionalizationSVGP
    from multi_fidelity_gpflow_b200.singlebin_svgp import SingleBinSVGP

    ds = onp.load_dataset("hbs")
    X, Y = ds["X"], ds["Y"]
    if latent:
        m = LatentMFCoregionalizationSVGP(X, Y, se(5), se(5), 10, num_inducing=50, handle=h)
    else:
        m = SingleBinSVGP(X, Y, se(5), se(5), 49, ds["Z_kmeans50"], handle=h)
    rng = np.random.default_rng(111)
    M, L = m.q_mu.shape
    m.q_mu.assign(0.3 * rng.standard_normal((M, L)))
    m.q_sqrt.assign(m.q_sqrt.numpy() + 0.02 * np.tril(rng.standard_normal((L, M, M))))
    Xs = ds["X_test"]
    post = m.posterior()
    mean, cov = post.predict_f_full_cov(Xs)
    d = Xs.shape[1] - 1
    pr = dict(Z=m.Z.numpy(), thetas=m._thetas(d), W=m._W(), q_mu=m.q_mu.numpy(), q_sqrt=np.tril(m.q_sqrt.numpy()))
    check_oracle(pr, Xs, mean, cov)
    f = post.predict_f_samples(Xs, 64, seed=3)
    assert f.shape == (64, 10, 49)
    z = np.random.default_rng(3).standard_normal((49, 10, 64))
    for p in range(49):
        Lc = np.linalg.cholesky(cov[p] + JITTER * np.eye(10))
        ref = mean[:, p][:, None] + Lc @ z[p]
        np.testing.assert_allclose(f[:, :, p].T, ref, rtol=1e-10, atol=1e-10 * np.abs(ref).max())
    np.testing.assert_array_equal(m.predict_f_samples(Xs, 64, seed=3), f)
    with pytest.raises(NotImplementedError):
        post.predict_f(Xs, full_cov=True)
    post.close()
