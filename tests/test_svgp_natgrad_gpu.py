"""GPU tests of the natural-gradient step (include/mfgp.h: mfgp_svgp_natgrad, mfgp_svgp_natgrad_adam): the step against the
torch twin (tests/_natgrad_twin.py) at the HBS shapes and on the GEMMs' 64-row tiles, the conjugate optimum one step with
gamma = 1 reaches, the per-latent failure rule, and the device loop against a host loop of value_and_grad,
NaturalGradient, value_and_grad and Adam.

Tolerance: 1e-9 relative to the largest entry of each output.  Every case asserts cond(Lam') <= 1e4 for the precision
the step factors (Lam' = Lam + 2 gamma g_S); a forward error of a few hundred ulps times that is well inside 1e-9."""
import copy
import ctypes

import numpy as np
import pytest

from oracle import mfgp_oracle as onp
from tests import _minibatch_twin as mbtwin
from tests import _natgrad_twin as twin

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def h():
    from multi_fidelity_gpflow_b200 import _lib

    hh = _lib.Handle(0)
    yield hh
    hh.close()


def _same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


def _rel(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b))) / max(np.max(np.abs(np.asarray(b))), 1e-300))


def _random_case(M, L, seed, gamma):
    """Lq with diagonal entries of both signs, and loss gradients G = tril(2 g_S Lq), gm of a known symmetric g_S small
    enough that Lam' stays well conditioned."""
    rng = np.random.default_rng(seed)
    q_mu = rng.standard_normal((M, L))
    q_sqrt = np.tril(0.2 / np.sqrt(M) * rng.standard_normal((L, M, M)), -1)
    dg = rng.uniform(0.6, 1.4, (L, M)) * np.where(rng.random((L, M)) < 0.4, -1.0, 1.0)
    q_sqrt += dg[:, :, None] * np.eye(M)
    gS = rng.standard_normal((L, M, M)) / np.sqrt(M)
    gS = 0.1 / gamma * (gS + gS.transpose(0, 2, 1))
    G = np.tril(2.0 * gS @ q_sqrt) + np.triu(rng.standard_normal((L, M, M)), 1)  # the upper part is never read
    q_sqrt = q_sqrt + np.triu(rng.standard_normal((L, M, M)), 1)
    return q_mu, q_sqrt, rng.standard_normal((M, L)), G


def _check_against_twin(h, q_mu, q_sqrt, gm, G, gamma):
    lam = twin.new_precision(q_sqrt, G, q_mu, gm, gamma)
    assert max(np.linalg.cond(x) for x in lam) <= 1e4
    want_m, want_s, want_info = twin.natgrad_step(q_mu, q_sqrt, gm, G, gamma)
    assert not want_info.any()
    m, s = q_mu.copy(), q_sqrt.copy()
    info = np.full(q_mu.shape[1], -1, dtype=np.int32)
    h.svgp_natgrad(m, s, gm, G, gamma, info=info)
    assert not info.any()
    assert _rel(m, want_m) < 1e-9 and _rel(s, want_s) < 1e-9
    assert not np.triu(s, 1).any()
    return m, s


def _hbs_case(kind, gamma):
    """q(u) and its loss gradients of the HBS models after a few Adam steps (so that q is not the prior)."""
    from multi_fidelity_gpflow_b200.kernels import SquaredExponential
    from multi_fidelity_gpflow_b200.linear_svgp import LatentMFCoregionalizationSVGP
    from multi_fidelity_gpflow_b200.singlebin_svgp import SingleBinSVGP

    ds = onp.load_dataset("hbs")
    X, Y = ds["X"], ds["Y"]
    k = lambda: (SquaredExponential(lengthscales=np.ones(5)), SquaredExponential(lengthscales=np.ones(5)))
    if kind == "singlebin":
        m = SingleBinSVGP(X, Y, *k(), Y.shape[1], ds["Z_kmeans50"])
    else:
        m = LatentMFCoregionalizationSVGP(X, Y, *k(), num_latents=8, num_inducing=30, num_outputs=49)
    m.optimize_on_device((X, Y), max_iters=5, initial_lr=0.01)
    _, _, (gm, gs) = m.value_and_grad((X, Y), [m.q_mu, m.q_sqrt])
    return m.q_mu.numpy().copy(), np.tril(m.q_sqrt.numpy()), gm, gs


@pytest.mark.parametrize("kind,gamma", [("singlebin", 0.1), ("latent", 0.1), ("latent", 1.0)])
def test_natgrad_matches_twin_at_hbs_shapes(h, kind, gamma):
    _check_against_twin(h, *_hbs_case(kind, gamma), gamma)


@pytest.mark.parametrize("M,L", [(300, 3), (1, 4), (127, 3), (129, 2)])
def test_natgrad_matches_twin_across_sizes(h, M, L):
    gamma = 0.5
    _check_against_twin(h, *_random_case(M, L, M, gamma), gamma)


def test_device_tensors_in_async_mode(h):
    import torch

    M, L, gamma = 129, 3, 0.5
    q_mu, q_sqrt, gm, G = _random_case(M, L, 11, gamma)
    m_host, s_host = q_mu.copy(), q_sqrt.copy()
    h.svgp_natgrad(m_host, s_host, gm, G, gamma)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    m, s, info = dev(q_mu), dev(q_sqrt), torch.full((L,), -1, dtype=torch.int32, device="cuda")
    h.set_async(True)
    try:
        h.svgp_natgrad(m, s, dev(gm), dev(G), gamma, info=info)
        assert h.sync() == 0
    finally:
        h.set_async(False)
    assert _same_bits(m.cpu().numpy(), m_host) and _same_bits(s.cpu().numpy(), s_host)
    assert not info.cpu().numpy().any()


def _A(X, Z, theta):
    import scipy.linalg as sla

    M = Z.shape[0]
    Lm = np.linalg.cholesky(onp.mf_K(Z, None, theta) + onp.JITTER * np.eye(M))
    return sla.solve_triangular(Lm, onp.mf_K(Z, X, theta), lower=True)


@pytest.mark.parametrize("lik", ["gaussian", "hetero", "masked"])
def test_one_step_reaches_the_conjugate_optimum(h, lik):
    ds = onp.load_dataset("hbs")
    rng = np.random.default_rng(12)
    X, P, M, d = ds["X"], 6, 20, 5
    Y = ds["Y"][:, :P].copy()
    hetero, masked = lik == "hetero", lik == "masked"
    if hetero:
        Y = np.hstack([Y, 0.05 + 0.2 * rng.random(Y.shape)])
    if masked:
        Y[rng.random(Y.shape) < 0.3] = np.nan
    Y = np.ascontiguousarray(Y)
    Z = X[rng.permutation(X.shape[0])[:M]].copy()
    ths = np.tile(onp.default_theta(d), (P, 1))
    ths[:, 1:1 + d] *= rng.uniform(0.7, 1.3, (P, d))
    lik_var = rng.uniform(0.2, 0.5, P) if masked else 0.3
    q_mu, q_sqrt = rng.standard_normal((M, P)), np.tile(0.7 * np.eye(M), (P, 1, 1))
    kw = dict(scale=2.5, hetero=hetero, masked=masked)
    r0 = h.svgp_elbo_grad(X, Y, Z, ths, None, q_mu, q_sqrt, lik_var, **kw)
    lam = twin.new_precision(q_sqrt, r0["g_q_sqrt"], q_mu, r0["g_q_mu"], 1.0)
    assert max(np.linalg.cond(x) for x in lam) <= 1e4
    h.svgp_natgrad(q_mu, q_sqrt, r0["g_q_mu"], r0["g_q_sqrt"], 1.0)
    r1 = h.svgp_elbo_grad(X, Y, Z, ths, None, q_mu, q_sqrt, lik_var, **kw)
    assert np.abs(r1["g_q_mu"]).max() < 1e-9 * np.abs(r0["g_q_mu"]).max()
    assert np.abs(r1["g_q_sqrt"]).max() < 1e-9 * np.abs(r0["g_q_sqrt"]).max()
    for l in range(P):
        nv = lik_var[l] if masked else (lik_var + Y[:, P + l] ** 2 if hetero else lik_var)
        m_star, S_star = twin.conjugate_optimum(_A(X, Z, ths[l]), Y[:, l], nv, 2.5)
        assert _rel(q_mu[:, l], m_star) < 1e-9
        assert _rel(q_sqrt[l] @ q_sqrt[l].T, S_star) < 1e-9


def test_a_failed_latent_keeps_its_values_and_leaves_the_others_alone(h):
    from multi_fidelity_gpflow_b200._lib import NotPositiveDefiniteError

    M, L, gamma = 40, 4, 0.5
    q_mu, q_sqrt, gm, G = _random_case(M, L, 3, gamma)
    bad = G.copy()
    bad[2] = np.tril(2.0 * (-10.0 / gamma) * q_sqrt[2])  # g_S = -10/gamma I: Lam' = Lam - 20 I is indefinite
    assert np.linalg.eigvalsh(twin.new_precision(q_sqrt, bad, q_mu, gm, gamma)[2]).min() < 0
    m_ok, s_ok = q_mu.copy(), q_sqrt.copy()
    h.svgp_natgrad(m_ok, s_ok, gm, G, gamma)
    m, s = q_mu.copy(), q_sqrt.copy()
    info = np.zeros(L, dtype=np.int32)
    h.svgp_natgrad(m, s, gm, bad, gamma, info=info)
    assert info[2] > 0 and not np.delete(info, 2).any()
    assert _same_bits(m[:, 2], q_mu[:, 2]) and _same_bits(s[2], q_sqrt[2])
    for l in (0, 1, 3):
        assert _same_bits(m[:, l], m_ok[:, l]) and _same_bits(s[l], s_ok[l])
    with pytest.raises(NotPositiveDefiniteError):
        h.svgp_natgrad(q_mu.copy(), q_sqrt.copy(), gm, bad, gamma)


def test_the_loop_never_moves_adam_state_of_the_q_blocks(h):
    ds = onp.load_dataset("hbs")
    X, Y = ds["X"], np.ascontiguousarray(ds["Y"][:, :6])
    L, M, P, d = 3, 8, 6, 5
    rng = np.random.default_rng(1)
    Z = X[rng.permutation(53)[:M]].copy()
    W = onp.initialize_W(P, L, 0.4, 0.2)
    u = np.concatenate([onp.softplus_inv(np.tile(onp.default_theta(d), (L, 1))).ravel(), Z.ravel(), W.ravel(),
                        0.1 * rng.standard_normal(M * L), np.tile(np.eye(M), (L, 1, 1)).ravel(),
                        onp.softplus_inv(np.array([0.3 - 1e-6]))])
    m, v = np.zeros_like(u), np.zeros_like(u)
    o_qm = L * (2 * d + 3) + M * (d + 1) + P * L
    o_lv = o_qm + M * L + L * M * M
    lr_t = np.full(12, 0.01)
    info = np.zeros(L, dtype=np.int32)
    h.svgp_natgrad_adam(X, Y, L, M, P, True, u, m, v, None, lr_t, np.full(12, 0.5), 0.9, 0.999, info=info)
    assert not info.any()
    assert not m[o_qm:o_lv].any() and not v[o_qm:o_lv].any()
    assert np.abs(m[:o_qm]).max() > 0 and np.abs(v[o_lv:]).max() > 0  # Adam did run on the other entries


def _kernels(d=5):
    from multi_fidelity_gpflow_b200.kernels import SquaredExponential

    return SquaredExponential(lengthscales=np.ones(d)), SquaredExponential(lengthscales=np.ones(d))


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


def _params(model):
    out = [model.q_mu.numpy(), np.tril(model.q_sqrt.numpy()), model.Z.numpy(), np.ravel(model.likelihood.variance.numpy())]
    W = getattr(model.kernel, "W", None)
    if W is not None:
        out.append(W.numpy())
    out.append(np.stack([k.theta(5) for k in model.kernel.kernels]))
    return out


def _host_natgrad_loop(model, X, Y, max_iters, lr, gamma, klm=1.0, B=None, seed=0):
    """GPflow's recipe: value_and_grad -> NaturalGradient on (q_mu, q_sqrt), value_and_grad -> Adam on the rest; with B
    the two evaluations of step t read the twin's stream positions 2 t B ... and (2 t + 1) B ...."""
    from multi_fidelity_gpflow_b200.optimizers import Adam, CosineDecay, NaturalGradient

    opt, ng = Adam(CosineDecay(lr, max_iters)), NaturalGradient(gamma)
    q = [model.q_mu, model.q_sqrt]
    others = [p for p in model.trainable_variables if p is not model.q_mu and p is not model.q_sqrt]
    batch = lambda k: (X, Y) if B is None else tuple(a[mbtwin.batch_rows(X.shape[0], seed, 0, k, B)] for a in (X, Y))
    losses, kls = [], []
    for t in range(max_iters):
        first = model.value_and_grad(batch(2 * t), q, klm)
        ng.minimize(lambda: first, [tuple(q)])
        _, _, grads = model.value_and_grad(batch(2 * t + 1), others, klm)
        opt.apply_gradients(zip(grads, others))
        losses.append(first[0])
        kls.append(first[1])
    return losses, kls


@pytest.mark.parametrize("kind,klm,B", [("latent", 1.0, None), ("latent", 2.5, None), ("singlebin", 1.0, None),
                                        ("hetero", 1.0, None), ("masked", 1.0, None), ("latent", 2.5, 16),
                                        ("singlebin", 1.0, 16), ("masked", 1.0, 16)])
def test_natgrad_device_loop_equals_host_loop(kind, klm, B):
    X, Y, a = _model(kind)
    b = copy.deepcopy(a)
    gamma = 0.1 if B else 0.5
    losses, kls = _host_natgrad_loop(a, X, Y, 11, 0.01, gamma, klm, B, seed=4)
    b.optimize_on_device((X, Y), max_iters=11, initial_lr=0.01, kl_multiplier=klm, minibatch_size=B, seed=4,
                         natgrad_gamma=gamma)
    np.testing.assert_allclose(b.loss_history, losses, rtol=1e-10)
    if kind != "singlebin":
        np.testing.assert_allclose(b.kl_history, kls, rtol=1e-10, atol=1e-12)
        if B:
            assert b.minibatch_position == 11 * 2 * B
    for pa, pb in zip(_params(a), _params(b)):
        np.testing.assert_allclose(pb, pa, rtol=1e-8, atol=1e-10)


def test_natgrad_loop_graph_owns_no_memory(h):
    rt = ctypes.CDLL("libcudart.so.12")
    val = ctypes.c_uint64(0)

    def reserved():
        assert rt.cudaDeviceGetGraphMemAttribute(0, 2, ctypes.byref(val)) == 0  # cudaGraphMemAttrReservedMemCurrent
        return val.value

    X, Y, m = _model("latent")
    m._handle = h
    m.optimize_on_device((X, Y), max_iters=3, initial_lr=0.01, minibatch_size=16, natgrad_gamma=0.1)  # warm the pool
    before = reserved()
    m.optimize_on_device((X, Y), max_iters=20, initial_lr=0.01, minibatch_size=16, natgrad_gamma=0.1)  # captured graph
    assert reserved() == before
    assert len(m.loss_history) == 20 and np.all(np.isfinite(m.loss_history))
