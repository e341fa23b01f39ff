"""CPU tests of the natural-gradient step: the torch twin (tests/_natgrad_twin.py) against the closed form of
include/mfgp.h, against central differences of the oracle's loss in the expectation parameters, and, for a Gaussian
likelihood, against the conjugate optimum one step with gamma = 1 reaches; then the host logic of
optimize_on_device(natgrad_gamma=...) and NaturalGradient.minimize through a recording handle."""
import numpy as np
import pytest
import scipy.linalg as sla

from oracle import mfgp_oracle as onp
from oracle import mfgp_oracle_torch as oth
from tests import _natgrad_twin as twin


def _random_q(rng, M, L, negative=True):
    q_mu = rng.standard_normal((M, L))
    q_sqrt = np.tril(0.2 / np.sqrt(M) * rng.standard_normal((L, M, M)), -1)
    dg = rng.uniform(0.6, 1.4, (L, M))
    if negative:
        dg *= np.where(rng.random((L, M)) < 0.4, -1.0, 1.0)
    q_sqrt += dg[:, :, None] * np.eye(M)
    return q_mu, q_sqrt


@pytest.mark.parametrize("M", [1, 5, 12])
def test_twin_dL_deta_equals_closed_form(M):
    rng = np.random.default_rng(M)
    q_mu, q_sqrt = _random_q(rng, M, 3)
    gm, G = rng.standard_normal((M, 3)), np.tril(rng.standard_normal((3, M, M)))
    for l in range(3):
        d1, d2 = twin.dL_deta(q_mu[:, l], q_sqrt[l], gm[:, l], G[l])
        c1, c2 = twin.dL_deta_closed_form(q_mu[:, l], q_sqrt[l], gm[:, l], G[l])
        np.testing.assert_allclose(d1, c1, rtol=1e-11, atol=1e-12 * np.abs(c1).max())
        np.testing.assert_allclose(d2, c2, rtol=1e-11, atol=1e-12 * np.abs(c2).max())
        assert np.array_equal(d2, d2.T)


def _problem(W=True, hetero=False, masked=False, L=3):
    ds = onp.load_dataset("hbs")
    rng = np.random.default_rng(7)
    X, Y = ds["X"], ds["Y"][:, :6].copy()
    P, M, d = (6, 6, 5) if W else (L, 6, 5)
    Y = Y[:, :P]
    if hetero:
        Y = np.hstack([Y, 0.05 + 0.1 * rng.random(Y.shape)])
    if masked:
        Y[rng.random(Y.shape) < 0.3] = np.nan
    Z = X[rng.permutation(X.shape[0])[:M]].copy()
    ths = np.tile(onp.default_theta(d), (L, 1))
    Wm = onp.initialize_W(P, L, 0.4, 0.2) if W else None
    lik = np.full(P, 0.3) if masked else 0.3
    return X, np.ascontiguousarray(Y), Z, ths, Wm, lik


def test_twin_dL_deta_equals_central_differences_of_the_oracle_loss():
    X, Y, Z, ths, W, lik = _problem(W=True)
    rng = np.random.default_rng(2)
    M, L = Z.shape[0], ths.shape[0]
    q_mu, q_sqrt = _random_q(rng, M, L)
    kw = dict(W=W, num_data=200, kl_mult=2.5)
    r = oth.svgp_value_and_grad(X, Y, Z, ths, q_mu, q_sqrt, lik, **kw)

    def loss(qm, qs):
        elbo, kl = onp.svgp_elbo(X, Y, Z, ths, qm, qs, lik, W=W, num_data=200)
        return -elbo + 1.5 * kl

    for l in range(L):
        d1, d2 = twin.dL_deta(q_mu[:, l], q_sqrt[l], r["g_q_mu"][:, l], r["g_q_sqrt"][l])
        m, Lq = q_mu[:, l], np.tril(q_sqrt[l])
        e2 = Lq @ Lq.T + np.outer(m, m)
        signs = np.sign(np.diag(Lq))
        for _ in range(3):
            a = rng.standard_normal(M)
            B = rng.standard_normal((M, M))
            B = 0.5 * (B + B.T)
            h = 1e-5

            def at(t):
                e1t, e2t = m + t * a, e2 + t * B
                qm, qs = q_mu.copy(), q_sqrt.copy()
                qm[:, l] = e1t
                qs[l] = np.linalg.cholesky(e2t - np.outer(e1t, e1t)) * signs
                return loss(qm, qs)

            fd = (at(h) - at(-h)) / (2 * h)
            an = a @ d1 + np.sum(B * d2)
            assert abs(fd - an) < 1e-6 * max(1.0, abs(an)), (l, fd, an)


def _latent_A(X, Z, theta):
    M = Z.shape[0]
    Lm = np.linalg.cholesky(onp.mf_K(Z, None, theta) + onp.JITTER * np.eye(M))
    return sla.solve_triangular(Lm, onp.mf_K(Z, X, theta), lower=True)


@pytest.mark.parametrize("scale", [None, 140.0])
def test_one_step_with_gamma_one_reaches_the_conjugate_optimum(scale):
    X, Y, Z, ths, _, lik = _problem(W=False)
    rng = np.random.default_rng(4)
    M, L = Z.shape[0], ths.shape[0]
    q_mu, q_sqrt = _random_q(rng, M, L)
    r0 = oth.svgp_value_and_grad(X, Y, Z, ths, q_mu, q_sqrt, lik, num_data=scale)
    qm, qs, info = twin.natgrad_step(q_mu, q_sqrt, r0["g_q_mu"], r0["g_q_sqrt"], 1.0)
    assert not info.any()
    s = 1.0 if scale is None else scale / X.shape[0]
    for l in range(L):
        m_star, S_star = twin.conjugate_optimum(_latent_A(X, Z, ths[l]), Y[:, l], lik, s)
        np.testing.assert_allclose(qm[:, l], m_star, rtol=1e-9, atol=1e-10 * np.abs(m_star).max())
        np.testing.assert_allclose(qs[l] @ qs[l].T, S_star, rtol=1e-9, atol=1e-11)
    r1 = oth.svgp_value_and_grad(X, Y, Z, ths, qm, qs, lik, num_data=scale)
    assert np.abs(r1["g_q_mu"]).max() < 1e-9 * np.abs(r0["g_q_mu"]).max()
    assert np.abs(r1["g_q_sqrt"]).max() < 1e-9 * np.abs(r0["g_q_sqrt"]).max()


# ---- host logic with a recording handle ------------------------------------------------------------------------------
class _RecordingHandle:
    """Stand-in for _lib.Handle: records the natural-gradient calls; no arithmetic claims."""

    def __init__(self, fail=None):
        self.calls, self.fail = [], fail

    def svgp_natgrad_adam(self, X, Y, L, M, P, has_W, u, m, v, mask, lr_t, gamma_t, b1, b2, eps, batch_size=None, seed=0,
                          pos0=0, scale=1.0, info=None, **kw):
        self.calls.append(dict(rows=X.shape[0], nsteps=len(lr_t), gamma_t=np.array(gamma_t), B=batch_size, seed=seed,
                               pos0=pos0, scale=scale, mask=np.array(mask), kl_mult=kw["kl_mult"]))
        u += 1.0  # every entry moves, so that the write-back is visible
        if self.fail is not None:
            info[self.fail] = 3
        n = len(lr_t)
        return np.arange(n, dtype=float), np.full(n, 0.5)

    def svgp_natgrad(self, q_mu, q_sqrt, g_q_mu, g_q_sqrt, gamma, info=None):
        self.calls.append(dict(kind="natgrad", gamma=gamma, g_q_mu=np.array(g_q_mu), g_q_sqrt=np.array(g_q_sqrt)))
        q_mu -= gamma * g_q_mu
        q_sqrt -= gamma * np.tril(g_q_sqrt)
        if self.fail is not None:
            info[self.fail] = 2
        return info

    def svgp_adam_minibatch(self, X, Y, L, M, P, has_W, u, m, v, mask, lr_t, *a, **kw):
        self.calls.append(dict(kind="adam_minibatch", pos0=kw["pos0"], B=kw["batch_size"]))
        return np.zeros(len(lr_t)), np.zeros(len(lr_t))


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


def test_gamma_per_step_and_stream_positions():
    fh = _RecordingHandle()
    X, Y, lat, sb = _models(fh)
    lat.optimize_on_device((X, Y), max_iters=4, initial_lr=0.01, kl_multiplier=2.5, natgrad_gamma=0.3)
    c = fh.calls[-1]
    assert c["nsteps"] == 4 and c["B"] is None and c["rows"] == 53 and c["kl_mult"] == 2.5 and c["scale"] == 1.0
    np.testing.assert_array_equal(c["gamma_t"], np.full(4, 0.3))
    assert not hasattr(lat, "minibatch_position") and len(lat.kl_history) == 4
    gam = np.array([0.1, 0.2, 0.4])
    lat.optimize_on_device((X, Y), max_iters=7, initial_lr=0.01, minibatch_size=16, seed=5, natgrad_gamma=gam)
    c = fh.calls[-1]
    assert (c["nsteps"], c["B"], c["seed"], c["pos0"], c["scale"]) == (3, 16, 5, 0, 53 / 16)
    np.testing.assert_array_equal(c["gamma_t"], gam)
    assert lat.minibatch_position == 3 * 2 * 16  # two batches per step
    lat.optimize_on_device((X, Y), max_iters=9, initial_lr=0.01, minibatch_size=10, seed=5, natgrad_gamma=1.0)
    assert fh.calls[-1]["pos0"] == 96 and lat.minibatch_position == 96 + 2 * 2 * 10
    lat.optimize_on_device((X, Y), max_iters=10, initial_lr=0.01, minibatch_size=10, seed=5)  # Adam only: B per step
    assert lat.minibatch_position == 136 + 10
    with pytest.raises(ValueError):
        lat.optimize_on_device((X, Y), max_iters=12, initial_lr=0.01, natgrad_gamma=np.ones(3))  # 2 steps, 3 values
    sb.num_data = 53
    sb.optimize_on_device((X, Y), max_iters=3, initial_lr=0.01, minibatch_size=16, natgrad_gamma=0.5)
    assert fh.calls[-1]["pos0"] == 0 and fh.calls[-1]["nsteps"] == 3 and len(sb.loss_history) == 3


def test_the_mask_reaches_the_loop_unchanged_and_the_values_come_back():
    """The q blocks stay in the mask the loop receives (the loop itself keeps Adam off them: mfgp_svgp_natgrad_adam)."""
    fh = _RecordingHandle()
    X, Y, lat, _ = _models(fh)
    _, _, mask = lat._flat_pack(5)
    m0, z0 = lat.q_mu.numpy().copy(), lat.Z.numpy().copy()
    lat.optimize_on_device((X, Y), max_iters=2, initial_lr=0.01, natgrad_gamma=1.0)
    np.testing.assert_array_equal(fh.calls[-1]["mask"], mask)
    np.testing.assert_allclose(lat.q_mu.numpy(), m0 + 1.0, rtol=0, atol=1e-12)
    np.testing.assert_allclose(lat.Z.numpy(), z0 + 1.0, rtol=0, atol=1e-12)


def test_a_failed_latent_raises_after_the_write_back():
    from multi_fidelity_gpflow_b200._lib import NotPositiveDefiniteError

    fh = _RecordingHandle(fail=1)
    X, Y, lat, _ = _models(fh)
    m0 = lat.q_mu.numpy().copy()
    with pytest.raises(NotPositiveDefiniteError, match=r"\(1, 3\)"):
        lat.optimize_on_device((X, Y), max_iters=3, initial_lr=0.01, natgrad_gamma=1.0)
    assert len(lat.loss_history) == 3 and len(lat.kl_history) == 3
    np.testing.assert_allclose(lat.q_mu.numpy(), m0 + 1.0, rtol=0, atol=1e-12)


def test_natural_gradient_minimize_round_trips_through_the_handle():
    from multi_fidelity_gpflow_b200._lib import NotPositiveDefiniteError
    from multi_fidelity_gpflow_b200.optimizers import NaturalGradient

    fh = _RecordingHandle()
    X, Y, lat, _ = _models(fh)
    rng = np.random.default_rng(0)
    gm, gs = rng.standard_normal(lat.q_mu.shape), rng.standard_normal(lat.q_sqrt.shape)
    m0, s0 = lat.q_mu.numpy().copy(), lat.q_sqrt.numpy().copy()
    loss = NaturalGradient(0.25, handle=fh).minimize(lambda: (1.5, 0.2, [gm, gs]), var_list=[(lat.q_mu, lat.q_sqrt)])
    assert loss == 1.5 and fh.calls[-1]["gamma"] == 0.25
    np.testing.assert_array_equal(fh.calls[-1]["g_q_mu"], gm)
    np.testing.assert_array_equal(lat.q_mu.numpy(), m0 - 0.25 * gm)
    np.testing.assert_array_equal(lat.q_sqrt.numpy(), np.tril(s0) - 0.25 * np.tril(gs))
    with pytest.raises(ValueError):
        NaturalGradient(0.25, handle=fh).minimize(lambda: (1.5, [gm]), var_list=[(lat.q_mu, lat.q_sqrt)])
    fail = _RecordingHandle(fail=2)
    with pytest.raises(NotPositiveDefiniteError, match=r"\(0, 2, 2\)"):
        NaturalGradient(1.0, handle=fail).minimize(lambda: (1.0, [gm, gs]), var_list=[(lat.q_mu, lat.q_sqrt)])
