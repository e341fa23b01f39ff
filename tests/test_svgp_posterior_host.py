"""Host logic of SVGPBase.posterior() with a fake handle that predicts with the NumPy oracle: the arguments the model passes
(theta order, tril of q_sqrt, W orientation, jitter), output shapes of both SVGP models, snapshot semantics and the
full_cov raise.  No GPU."""
import numpy as np
import pytest

from oracle import mfgp_oracle as onp


class _FakeSvgpPosterior:
    def __init__(self, Z, thetas, W, q_mu, q_sqrt):
        self.args = [None if a is None else np.array(a, copy=True) for a in (Z, thetas, W, q_mu, q_sqrt)]

    def predict(self, Xs, mean=None, var=None):
        Z, thetas, W, q_mu, q_sqrt = self.args
        return onp.svgp_predict(Xs, Z, thetas, q_mu, q_sqrt, W)


class _OracleHandle:
    def __init__(self):
        self.created = []

    def svgp_posterior(self, Z, thetas, W, q_mu, q_sqrt, jitter=1e-6, info=None):
        self.created.append(dict(Z=Z, thetas=thetas, W=W, q_mu=q_mu, q_sqrt=q_sqrt, jitter=jitter))
        return _FakeSvgpPosterior(Z, thetas, W, q_mu, q_sqrt)

    def svgp_predict(self, Xs, Z, thetas, W, q_mu, q_sqrt, jitter=1e-6):
        assert jitter == onp.JITTER
        return onp.svgp_predict(Xs, Z, thetas, q_mu, q_sqrt, W)


def _data(rng, N=30, d=3, P=4):
    X = np.hstack([rng.random((N, d)), (np.arange(N) >= N - 8).astype(float)[:, None]])
    return X, rng.standard_normal((N, P))


def _kernels(d):
    from multi_fidelity_gpflow_b200.kernels import SquaredExponential

    return (SquaredExponential(lengthscales=np.ones(d), variance=1.0),
            SquaredExponential(lengthscales=np.ones(d), variance=1.0))


def _perturb(m, rng):
    M, L = m.q_mu.shape
    m.q_mu.assign(0.3 * rng.standard_normal((M, L)))
    m.q_sqrt.assign(m.q_sqrt.numpy() + 0.05 * rng.standard_normal((L, M, M)))  # upper part nonzero: must be dropped


def _singlebin(rng, fh, P=4, M=6):
    from multi_fidelity_gpflow_b200.singlebin_svgp import SingleBinSVGP

    X, Y = _data(rng, P=P)
    kL, kD = _kernels(3)
    m = SingleBinSVGP(X, Y, kL, kD, P, np.zeros((M, 4)), handle=fh)
    _perturb(m, rng)
    return m, X


def _latent(rng, fh, P=5, L=3, M=7):
    from multi_fidelity_gpflow_b200.linear_svgp import LatentMFCoregionalizationSVGP

    X, Y = _data(rng, P=P)
    kL, kD = _kernels(3)
    m = LatentMFCoregionalizationSVGP(X, Y, kL, kD, L, num_inducing=M, handle=fh)
    _perturb(m, rng)
    return m, X


def test_posterior_arguments():
    rng = np.random.default_rng(0)
    fh = _OracleHandle()
    for m, _ in (_singlebin(rng, fh), _latent(rng, fh)):
        m.posterior()
        a = fh.created[-1]
        Z = m.Z.numpy()
        d = Z.shape[1] - 1
        np.testing.assert_array_equal(a["Z"], Z)
        np.testing.assert_array_equal(a["thetas"], np.stack([k.theta(d) for k in m.kernel.kernels]))
        assert a["thetas"].shape == (m.q_mu.shape[1], 2 * d + 3)
        np.testing.assert_array_equal(a["q_mu"], m.q_mu.numpy())
        np.testing.assert_array_equal(a["q_sqrt"], np.tril(m.q_sqrt.numpy()))
        assert np.any(np.triu(m.q_sqrt.numpy(), 1) != 0) and np.all(np.triu(a["q_sqrt"], 1) == 0)
        assert a["jitter"] == onp.JITTER
        W = getattr(m.kernel, "W", None)
        if W is None:
            assert a["W"] is None
        else:
            assert a["W"].shape == (m.num_outputs, m.num_latents)  # [P, L], as svgp_predict takes it
            np.testing.assert_array_equal(a["W"], W.numpy())


def test_shapes_match_predict_f_for_both_models():
    rng = np.random.default_rng(1)
    fh = _OracleHandle()
    for m, X in (_singlebin(rng, fh, P=4), _latent(rng, fh, P=5, L=3)):
        Xs = X[:9]
        pm, pv = m.posterior().predict_f(Xs)
        mm, mv = m.predict_f(Xs)
        assert pm.shape == mm.shape == (9, m.num_outputs) and pv.shape == mv.shape == (9, m.num_outputs)
        np.testing.assert_allclose(pm, mm, rtol=1e-12, atol=1e-14)
        np.testing.assert_allclose(pv, mv, rtol=1e-12, atol=1e-14)


def test_posterior_is_a_snapshot():
    rng = np.random.default_rng(2)
    fh = _OracleHandle()
    for m, X in (_singlebin(rng, fh), _latent(rng, fh)):
        post = m.posterior()
        before = post.predict_f(X[:6])
        m.q_mu.assign(m.q_mu.numpy() + 1.0)
        m.kernel.kernels[0].kernel_L.variance.assign(3.0)
        after = post.predict_f(X[:6])
        np.testing.assert_array_equal(before[0], after[0])
        np.testing.assert_array_equal(before[1], after[1])
        assert not np.allclose(m.posterior().predict_f(X[:6])[0], before[0])


def test_full_cov_raises():
    rng = np.random.default_rng(3)
    m, X = _singlebin(rng, _OracleHandle())
    post = m.posterior()
    with pytest.raises(NotImplementedError):
        post.predict_f(X[:2], full_cov=True)
    with pytest.raises(NotImplementedError):
        post.predict_f(X[:2], full_output_cov=True)
