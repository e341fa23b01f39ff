"""Host logic of the joint posterior of the SVGP models (predict_f_full_cov, predict_f_samples) with a fake handle backed
by the NumPy oracle, and the oracle itself: its diagonal and mean against onp.svgp_predict and its covariance against the
unwhitened algebra computed with plain solves.  No GPU."""
import numpy as np
import pytest

from oracle import mfgp_oracle as onp
from tests._svgp_joint_oracle import svgp_predict_full_cov
from tests.test_svgp_posterior_host import _FakeSvgpPosterior, _OracleHandle, _latent, _singlebin

JITTER = 1e-6


class _JointFakeSvgpPosterior(_FakeSvgpPosterior):
    """_FakeSvgpPosterior plus predict_cov / sample (the oracle's Sigma_p, numpy's Cholesky) and the library's draw_f."""

    def __init__(self, *a, failed=None):
        super().__init__(*a)
        self.d = self.args[0].shape[1] - 1
        self.P = self.args[1].shape[0] if self.args[2] is None else self.args[2].shape[0]
        self.failed = np.zeros(self.P, dtype=bool) if failed is None else failed
        self.closed = False

    def _xs(self, Xs):
        return np.asarray(Xs, dtype=np.float64)

    def predict_cov(self, Xs):
        Z, thetas, W, q_mu, q_sqrt = self.args
        mean, cov = svgp_predict_full_cov(Xs, Z, thetas, q_mu, q_sqrt, W)
        mean[:, self.failed], cov[self.failed] = np.nan, np.nan
        return mean, cov

    def sample(self, Xs, z, jitter=JITTER, info=None):
        mean, cov = self.predict_cov(Xs)
        out = np.empty_like(z)
        for p in range(self.P):
            if self.failed[p]:
                if info is None:
                    from multi_fidelity_gpflow_b200._lib import NotPositiveDefiniteError

                    raise NotPositiveDefiniteError("not positive definite")
                info[p], out[p] = 1, np.nan
                continue
            Lc = np.linalg.cholesky(cov[p] + jitter * np.eye(cov.shape[1]))
            out[p] = mean[:, p][:, None] + Lc @ z[p]
        return out

    def close(self):
        self.closed = True

    from multi_fidelity_gpflow_b200._lib import SvgpPosterior as _S
    draw_f = _S.draw_f


class _JointHandle(_OracleHandle):
    fail_outputs = None

    def svgp_posterior(self, Z, thetas, W, q_mu, q_sqrt, jitter=1e-6, info=None):
        super().svgp_posterior(Z, thetas, W, q_mu, q_sqrt, jitter, info)
        self.last = _JointFakeSvgpPosterior(Z, thetas, W, q_mu, q_sqrt, failed=self.fail_outputs)
        return self.last


def _problem(rng, M, d, L, P, mixing):
    Z = np.hstack([rng.random((M, d)), (np.arange(M) % 3 == 0).astype(float)[:, None]])
    th = np.tile(onp.default_theta(d), (L, 1)) * np.exp(0.2 * rng.standard_normal((L, 2 * d + 3)))
    q_sqrt = np.tile(0.3 * np.eye(M), (L, 1, 1)) + 0.05 * np.tril(rng.standard_normal((L, M, M)))
    W = rng.standard_normal((P, L)) if mixing else None
    return Z, th, W, rng.standard_normal((M, L)), q_sqrt


@pytest.mark.parametrize("L,P,mixing", [(4, 4, False), (3, 7, True), (6, 2, True)])  # no W, P > L, P < L
def test_oracle_against_marginals_and_unwhitened_form(L, P, mixing):
    rng = np.random.default_rng(L * 10 + P)
    M, d = 9, 3
    Z, th, W, q_mu, q_sqrt = _problem(rng, M, d, L, P, mixing)
    Xs = np.hstack([rng.random((12, d)), rng.integers(0, 2, (12, 1)).astype(float)])
    mean, cov = svgp_predict_full_cov(Xs, Z, th, q_mu, q_sqrt, W)
    assert mean.shape == (12, P) and cov.shape == (P, 12, 12)
    rm, rv = onp.svgp_predict(Xs, Z, th, q_mu, q_sqrt, W)
    np.testing.assert_allclose(mean, rm, rtol=1e-14, atol=1e-14 * np.abs(rm).max())
    np.testing.assert_allclose(np.diagonal(cov, axis1=1, axis2=2).T, rv, rtol=1e-14, atol=1e-14 * np.abs(rv).max())
    # unwhitened: K_ss - K_sm K_mm^-1 K_ms + K_sm Lm^-T Lq Lq^T Lm^-1 K_ms, with plain solves
    lat = []
    for l in range(L):
        Kmm = onp.mf_K(Z, None, th[l]) + onp.JITTER * np.eye(M)
        Kms = onp.mf_K(Z, Xs, th[l])
        Lm = np.linalg.cholesky(Kmm)
        B = np.linalg.solve(Lm.T, np.tril(q_sqrt[l]))  # Lm^-T Lq
        lat.append(onp.mf_K(Xs, None, th[l]) - Kms.T @ np.linalg.solve(Kmm, Kms) + (Kms.T @ B) @ (B.T @ Kms))
    lat = np.stack(lat)
    ref = lat if W is None else np.einsum("pl,lij->pij", W * W, lat)
    np.testing.assert_allclose(cov, ref, rtol=1e-9, atol=1e-9 * np.abs(ref).max())


@pytest.mark.parametrize("latent", [False, True])
def test_axes_shapes_seed_and_branches(latent):
    rng = np.random.default_rng(3)
    fh = _JointHandle()
    m, X = (_latent if latent else _singlebin)(rng, fh)
    P = m.q_mu.shape[1] if not latent else 5
    Xs = X[:7]
    post = m.posterior()
    mean, cov = post.predict_f_full_cov(Xs)
    assert mean.shape == (7, P) and cov.shape == (P, 7, 7)
    pm, pv = post.predict_f(Xs)
    np.testing.assert_allclose(mean, pm, rtol=1e-13)
    np.testing.assert_allclose(np.diagonal(cov, axis1=1, axis2=2).T, pv, rtol=1e-12, atol=1e-14)
    f = post.predict_f_samples(Xs, 5, seed=4)
    assert f.shape == (5, 7, P)
    z = np.random.default_rng(4).standard_normal((P, 7, 5))
    for p in range(P):
        Lc = np.linalg.cholesky(cov[p] + JITTER * np.eye(7))
        np.testing.assert_allclose(f[:, :, p], (mean[:, p][:, None] + Lc @ z[p]).T, rtol=1e-12, atol=1e-12)
    np.testing.assert_array_equal(post.predict_f_samples(Xs, 5, seed=4), f)  # seed reproducibility
    assert not np.array_equal(post.predict_f_samples(Xs, 5, seed=5), f)
    one = post.predict_f_samples(Xs, seed=4)
    assert one.shape == (7, P)
    np.testing.assert_array_equal(one, post.predict_f_samples(Xs, 1, seed=4)[0])
    # full_cov=False: independent per point, from predict_f's marginals
    g = post.predict_f_samples(Xs, 3, full_cov=False, seed=6)
    zz = np.random.default_rng(6).standard_normal((P, 7, 3))
    np.testing.assert_allclose(g, np.transpose(pm.T[:, :, None] + np.sqrt(pv).T[:, :, None] * zz, (2, 1, 0)), rtol=1e-14)
    with pytest.raises(NotImplementedError):
        post.predict_f_samples(Xs, 2, full_output_cov=True)
    with pytest.raises(NotImplementedError):
        post.predict_f(Xs, full_cov=True)  # predict_f keeps its marginal-only contract
    with pytest.raises(NotImplementedError):
        m.predict_f(Xs, full_cov=True)
    # the model-level call makes a posterior and frees it
    fm = m.predict_f_samples(Xs, 5, seed=4)
    np.testing.assert_allclose(fm, f, rtol=1e-12, atol=1e-12)
    assert fh.last is not post.post and fh.last.closed


def test_failed_output_is_nan_with_info_and_raises_without():
    from multi_fidelity_gpflow_b200._lib import NotPositiveDefiniteError

    rng = np.random.default_rng(5)
    fh = _JointHandle()
    m, X = _singlebin(rng, fh)
    P = m.q_mu.shape[1]
    fh.fail_outputs = np.arange(P) == 1
    post = m.posterior()
    info = np.zeros(P, dtype=np.int32)
    s = post.post.draw_f(X[:6], 4, seed=1, info=info)
    assert s.shape == (P, 6, 4)
    assert info[1] == 1 and np.all(info[np.arange(P) != 1] == 0)
    assert np.isnan(s[1]).all() and np.isfinite(s[np.arange(P) != 1]).all()
    with pytest.raises(NotPositiveDefiniteError):
        post.predict_f_samples(X[:6], 4, seed=1)
