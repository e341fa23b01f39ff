"""Input gradients of the SVGP prediction without a GPU: the autograd oracle (tests/_svgp_grad_oracle.py: svgp_predict_grad_x)
against central finite differences of the NumPy svgp_predict, and the host logic of SVGPPosterior.predict_f_grad with a
fake handle that predicts with the oracle: shapes of both SVGP models, the zero fidelity column, snapshot semantics and a
closed posterior.  SvgpPosterior.predict_grad's column check runs before any library call."""
import numpy as np
import pytest

from oracle import mfgp_oracle as onp
from tests._svgp_grad_oracle import svgp_predict_grad_x
from tests.test_svgp_posterior_host import _FakeSvgpPosterior, _latent, _OracleHandle, _singlebin


def _fd(Xs, Z, th, q_mu, q_sqrt, W, h=1e-5):
    """Central differences of onp.svgp_predict: dmean, dvar [Ns, P, d]."""
    d = Xs.shape[1] - 1
    dm, dv = [], []
    for j in range(d):
        xp, xm = Xs.copy(), Xs.copy()
        xp[:, j] += h
        xm[:, j] -= h
        mp, vp = onp.svgp_predict(xp, Z, th, q_mu, q_sqrt, W)
        mm, vm = onp.svgp_predict(xm, Z, th, q_mu, q_sqrt, W)
        dm.append((mp - mm) / (2 * h))
        dv.append((vp - vm) / (2 * h))
    return np.stack(dm, axis=-1), np.stack(dv, axis=-1)


@pytest.mark.parametrize("d", [1, 5])
@pytest.mark.parametrize("mixing", [False, True])
def test_oracle_gradient_matches_finite_differences(d, mixing):
    rng = np.random.default_rng(10 * d + mixing)
    M, L, P = 9, 3, 4
    Z = np.hstack([rng.random((M, d)), (rng.random((M, 1)) < 0.4).astype(float)])
    Z[2, -1] = np.nextafter(1.0, 2.0)  # a dead inducing point (quirk Q1)
    th = np.tile(onp.default_theta(d), (L, 1)) * np.exp(0.2 * rng.standard_normal((L, 2 * d + 3)))
    th[:, 0] = 0.8
    q_mu = rng.standard_normal((M, L))
    q_sqrt = np.tril(np.tile(0.3 * np.eye(M), (L, 1, 1)) + 0.05 * rng.standard_normal((L, M, M)))
    W = rng.standard_normal((P, L)) if mixing else None
    Xs = np.hstack([rng.random((6, d)), np.array([0, 1, 0, 1, 0.5, 1.0])[:, None]])
    Xs[5] = Z[3]  # a test point on an inducing point
    mean, var, dmean, dvar = svgp_predict_grad_x(Xs, Z, th, q_mu, q_sqrt, W)
    rm, rv = onp.svgp_predict(Xs, Z, th, q_mu, q_sqrt, W)
    np.testing.assert_allclose(mean, rm, rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(var, rv, rtol=1e-10, atol=1e-12)
    Pout = P if mixing else L
    assert dmean.shape == dvar.shape == (6, Pout, d + 1)
    assert np.all(dmean[..., -1] == 0.0) and np.all(dvar[..., -1] == 0.0)  # the fidelity column
    assert np.all(dmean[4] == 0.0) and np.all(dvar[4] == 0.0)  # dead row (fidelity 0.5)
    fm, fv = _fd(Xs, Z, th, q_mu, q_sqrt, W)
    np.testing.assert_allclose(dmean[..., :-1], fm, rtol=1e-6, atol=1e-7 * np.abs(fm).max())
    np.testing.assert_allclose(dvar[..., :-1], fv, rtol=1e-6, atol=1e-7 * np.abs(fv).max())
    assert np.abs(fm).max() > 1e-3 and np.abs(fv).max() > 1e-4  # the check is not vacuous


class _GradSvgpPosterior(_FakeSvgpPosterior):
    def predict_grad(self, Xs):
        Z, thetas, W, q_mu, q_sqrt = self.args
        mean, var, dm, dv = svgp_predict_grad_x(Xs, Z, thetas, q_mu, q_sqrt, W)
        return mean, var, dm[..., :-1], dv[..., :-1]  # the C ABI's [Ns, P, d]


class _GradHandle(_OracleHandle):
    def svgp_posterior(self, Z, thetas, W, q_mu, q_sqrt, jitter=1e-6, info=None):
        super().svgp_posterior(Z, thetas, W, q_mu, q_sqrt, jitter, info)
        return _GradSvgpPosterior(Z, thetas, W, q_mu, q_sqrt)


def test_predict_f_grad_shapes_for_both_models():
    rng = np.random.default_rng(1)
    fh = _GradHandle()
    for m, X in (_singlebin(rng, fh, P=4), _latent(rng, fh, P=5, L=3)):
        Xs = X[:9]
        post = m.posterior()
        mean, var, dm, dv = post.predict_f_grad(Xs)
        P, d = m.num_outputs, X.shape[1] - 1
        assert mean.shape == var.shape == (9, P)
        assert dm.shape == dv.shape == (9, P, d + 1)
        assert np.all(dm[..., -1] == 0.0) and np.all(dv[..., -1] == 0.0)  # fidelity column, as tape.gradient gives it
        pm, pv = post.predict_f(Xs)
        np.testing.assert_allclose(mean, pm, rtol=1e-12, atol=1e-14)
        np.testing.assert_allclose(var, pv, rtol=1e-12, atol=1e-14)
        assert np.abs(dm).max() > 0 and np.abs(dv).max() > 0


def test_predict_f_grad_is_a_snapshot_and_close_raises():
    from multi_fidelity_gpflow_b200 import svgp_base

    rng = np.random.default_rng(2)
    fh = _GradHandle()
    for m, X in (_singlebin(rng, fh), _latent(rng, fh)):
        post = m.posterior()
        before = post.predict_f_grad(X[:6])
        m.q_mu.assign(m.q_mu.numpy() + 1.0)
        m.kernel.kernels[0].kernel_L.variance.assign(3.0)
        after = post.predict_f_grad(X[:6])
        for a, b in zip(before, after):
            np.testing.assert_array_equal(a, b)
        assert not np.allclose(m.posterior().predict_f_grad(X[:6])[2], before[2])

    class _Closed:
        def predict_grad(self, Xs):
            raise ValueError("SvgpPosterior is closed")

    with pytest.raises(ValueError, match="closed"):
        svgp_base.SVGPPosterior(_Closed()).predict_f_grad(X[:2])


def test_predict_grad_rejects_wrong_column_count():
    from multi_fidelity_gpflow_b200 import _lib

    post = _lib.SvgpPosterior.__new__(_lib.SvgpPosterior)
    post.handle, post._p, post.L, post.M, post.P, post.d = None, 1, 2, 3, 2, 4  # never reaches the library
    with pytest.raises(ValueError, match="5 columns"):
        post.predict_grad(np.zeros((3, 4)))
    post._p = None
    with pytest.raises(ValueError, match="closed"):
        post.predict_grad(np.zeros((3, 5)))
