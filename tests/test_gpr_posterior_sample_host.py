"""Host logic of the joint posterior of the exact GPs (predict_f_full_cov, predict_f_samples) with a fake handle that
computes every problem with the NumPy oracle: the oracle's joint covariance itself, shapes and axis moves for "best",
"all" and the single model, seed reproducibility, the full_cov=False branch, the full_output_cov raise, NaN for a failed
restart and snapshot semantics.  No GPU."""
import numpy as np
import pytest
import scipy.linalg as sla

from oracle import mfgp_oracle as onp
from tests._joint_oracle import gpr_predict_full_cov
from tests.test_gpr_posterior_host import _FakePosterior, _OracleHandle, _problem

JITTER = 1e-6


class _JointFakePosterior(_FakePosterior):
    """_FakePosterior plus predict_cov / sample (the oracle's Sigma, numpy's Cholesky) and the library's draw_f."""

    def __init__(self, *a):
        super().__init__(*a)
        self.B, self.d = self.thetas.shape[0], self.X.shape[1] - 1

    def _xs(self, Xs):
        return np.asarray(Xs, dtype=np.float64)

    def predict_cov(self, Xs):
        B, ycols, Ns = self.B, self.Y.shape[1], Xs.shape[0]
        mean, cov = np.empty((B, Ns, self.P)), np.empty((B, Ns, Ns))
        for b in range(B):
            c = (b * self.P) % ycols
            if self.failed[b]:
                mean[b], cov[b] = np.nan, np.nan
            else:
                mean[b], cov[b] = gpr_predict_full_cov(self.X, self.Y[:, c:c + self.P], Xs, self.thetas[b], self.noises[b])
        return mean, cov

    def sample(self, Xs, z, jitter=JITTER, info=None):
        mean, cov = self.predict_cov(Xs)
        out = np.empty_like(z)
        for b in range(self.B):
            if self.failed[b]:
                if info is None:
                    raise np.linalg.LinAlgError("not positive definite")
                info[b], out[b] = 1, np.nan
                continue
            L = np.linalg.cholesky(cov[b] + jitter * np.eye(cov.shape[1]))
            out[b] = mean[b][:, None, :] + np.einsum("ij,jkc->ikc", L, z[b])
        return out

    from multi_fidelity_gpflow_b200._lib import GprPosterior as _G
    draw_f = _G.draw_f


class _JointHandle(_OracleHandle):
    def gpr_posterior(self, X, Y, thetas, noises, P=1, info=None):
        bad = self._failed(thetas.shape[0])
        if bad.any():
            if info is None:
                raise np.linalg.LinAlgError("not positive definite")
            info[bad] = 1
        self.created.append((thetas.copy(), noises.copy(), P))
        return _JointFakePosterior(np.asarray(X), np.asarray(Y), np.asarray(thetas), np.asarray(noises), P, bad)


def test_oracle_joint_covariance():
    rng = np.random.default_rng(0)
    X, Y = _problem(rng, N=20, d=3, P=2)
    th = np.exp(0.2 * rng.standard_normal(9))
    Xs = np.vstack([rng.random((7, 4)), X[:3]])
    Xs[:7, -1] = [0, 1, 0, 1, 0.5, 1, 0]
    mean, cov = gpr_predict_full_cov(X, Y, Xs, th, 1e-3)
    m, v = onp.gpr_predict(X, Y, Xs, th, 1e-3)
    np.testing.assert_allclose(np.diag(cov), v, rtol=1e-10, atol=1e-14)
    np.testing.assert_allclose(mean, m, rtol=1e-10, atol=1e-12)
    K = onp.mf_K(X, None, th) + 1e-3 * np.eye(20)
    Ks = onp.mf_K(X, Xs, th)
    alt = onp.mf_K(Xs, None, th) - Ks.T @ sla.solve(K, Ks, assume_a="pos")
    np.testing.assert_allclose(cov, alt, rtol=1e-8, atol=1e-10)
    assert np.all(cov[4] == 0.0) and np.all(cov[:, 4] == 0.0)  # fidelity 0.5: no covariance


def _multibin(R=3, seed=2):
    from multi_fidelity_gpflow_b200.multibin import MultiBinMFGP

    rng = np.random.default_rng(seed)
    X, Y = _problem(rng)
    fh = _JointHandle()
    mdl = MultiBinMFGP(X, Y, num_restarts=R, seed=seed, handle=fh)
    Xs = np.vstack([rng.random((5, 4)), X[:2]])
    Xs[:5, -1] = [0, 1, 0, 1, 1]
    return X, Y, fh, mdl, Xs


def test_multibin_full_cov_and_samples_shapes_and_axes():
    X, Y, fh, mdl, Xs = _multibin()
    P, Ns = 4, Xs.shape[0]
    post = mdl.posterior("all")
    mean, cov = post.predict_f_full_cov(Xs)
    assert mean.shape == (3, Ns, P) and cov.shape == (3, P, Ns, Ns)
    for r in range(3):
        for p in range(P):
            rm, rc = gpr_predict_full_cov(X, Y[:, p:p + 1], Xs, mdl.thetas[r, p], mdl.noise)
            np.testing.assert_allclose(mean[r, :, p], rm[:, 0], rtol=1e-12)
            np.testing.assert_allclose(cov[r, p], rc, rtol=1e-12)
    m2, v2 = post.predict_f(Xs)
    np.testing.assert_allclose(np.diagonal(cov, axis1=2, axis2=3).transpose(0, 2, 1), v2, rtol=1e-9, atol=1e-14)

    f = post.predict_f_samples(Xs, num_samples=5, seed=7)
    assert f.shape == (3, 5, Ns, P)
    z = np.random.default_rng(7).standard_normal((3 * P, Ns, 5, 1))  # the documented draw order
    for r in range(3):
        for p in range(P):
            L = np.linalg.cholesky(cov[r, p] + JITTER * np.eye(Ns))
            ref = mean[r, :, p][:, None] + L @ z[r * P + p, :, :, 0]
            np.testing.assert_allclose(f[r, :, :, p], ref.T, rtol=1e-12)
    np.testing.assert_array_equal(post.predict_f_samples(Xs, num_samples=5, seed=7), f)  # reproducible
    assert not np.array_equal(post.predict_f_samples(Xs, num_samples=5, seed=8), f)
    one = post.predict_f_samples(Xs, seed=7)
    assert one.shape == (3, Ns, P)
    z1 = np.random.default_rng(7).standard_normal((3 * P, Ns, 1, 1))
    for r in range(3):
        for p in range(P):
            L = np.linalg.cholesky(cov[r, p] + JITTER * np.eye(Ns))
            np.testing.assert_allclose(one[r, :, p], mean[r, :, p] + L @ z1[r * P + p, :, 0, 0], rtol=1e-12)

    diag = post.predict_f_samples(Xs, num_samples=5, full_cov=False, seed=7)
    ref = m2[:, None] + np.sqrt(v2)[:, None] * z[..., 0].reshape(3, P, Ns, 5).transpose(0, 3, 2, 1)
    np.testing.assert_allclose(diag, ref, rtol=1e-12)
    with pytest.raises(NotImplementedError):
        post.predict_f_samples(Xs, full_output_cov=True)

    best = mdl.posterior("best")
    mb, cb = best.predict_f_full_cov(Xs)
    assert mb.shape == (Ns, P) and cb.shape == (P, Ns, Ns)
    fb = best.predict_f_samples(Xs, num_samples=2, seed=1)
    assert fb.shape == (2, Ns, P)
    np.testing.assert_array_equal(mdl.predict_f_samples(Xs, num_samples=2, seed=1), fb)  # model-level shim
    assert best.predict_f_samples(Xs, seed=1).shape == (Ns, P)


def test_multibin_failed_restart_is_nan_and_best_raises():
    X, Y, fh, mdl, Xs = _multibin()
    fh.fail = {2 * 4 + 1}  # restart 2 of bin 1
    post = mdl.posterior("all")
    f = post.predict_f_samples(Xs, num_samples=3, seed=0)
    assert np.isnan(f[2, :, :, 1]).all()
    keep = np.ones((3, 4), dtype=bool)
    keep[2, 1] = False
    assert np.isfinite(f.transpose(0, 3, 1, 2)[keep]).all()
    _, cov = post.predict_f_full_cov(Xs)
    assert np.isnan(cov[2, 1]).all()
    best = _JointFakePosterior(X, Y, mdl.thetas[0], np.full(4, 1e-3), 1, np.array([False, True, False, False]))
    from multi_fidelity_gpflow_b200.multibin import MultiBinPosterior

    with pytest.raises(np.linalg.LinAlgError):
        MultiBinPosterior(best, np.full(4, 1e-3), None).predict_f_samples(Xs)


def test_single_model_full_cov_samples_and_snapshot():
    from multi_fidelity_gpflow_b200.kernels import SquaredExponential
    from multi_fidelity_gpflow_b200.linear import MultiFidelityGPModel

    rng = np.random.default_rng(4)
    X, Y = _problem(rng)
    fh = _JointHandle()
    se = lambda: SquaredExponential(lengthscales=np.ones(3), variance=1.0)
    m = MultiFidelityGPModel(X, Y, se(), se(), handle=fh)
    mp = m.posterior()
    Xs = X[:6]
    mean, cov = mp.predict_f_full_cov(Xs)
    th, nz, _ = fh.created[-1]
    rm, rc = gpr_predict_full_cov(X, Y, Xs, th[0], nz[0])
    assert mean.shape == (6, 4) and cov.shape == (4, 6, 6)
    np.testing.assert_allclose(mean, rm, rtol=1e-12)
    for p in range(4):
        np.testing.assert_array_equal(cov[p], cov[0])
    np.testing.assert_allclose(cov[0], rc, rtol=1e-12)
    assert not cov.flags.writeable  # one matrix broadcast over the P outputs
    f = mp.predict_f_samples(Xs, num_samples=3, seed=5)
    assert f.shape == (3, 6, 4)
    z = np.random.default_rng(5).standard_normal((1, 6, 3, 4))
    L = np.linalg.cholesky(rc + JITTER * np.eye(6))
    np.testing.assert_allclose(f, (rm[:, None, :] + np.einsum("ij,jkc->ikc", L, z[0])).transpose(1, 0, 2), rtol=1e-12)
    assert mp.predict_f_samples(Xs, seed=5).shape == (6, 4)
    np.testing.assert_array_equal(m.predict_f_samples(Xs, num_samples=3, seed=5), f)
    with pytest.raises(NotImplementedError):
        mp.predict_f_samples(Xs, full_output_cov=True)
    with pytest.raises(NotImplementedError):
        mp.predict_f(Xs, full_cov=True)  # predict_f keeps its marginal-only contract
    m.kernel.kernel_L.variance.assign(2.0)
    np.testing.assert_array_equal(mp.predict_f_samples(Xs, num_samples=3, seed=5), f)  # snapshot
    assert not np.allclose(m.predict_f_samples(Xs, num_samples=3, seed=5), f)
