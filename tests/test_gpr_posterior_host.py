"""Host logic of the cached posteriors (MultiBinMFGP.posterior, MultiFidelityGPModel.posterior) with a fake handle that
computes every problem with the NumPy oracle: problem ordering b = r * P + p, the "best" / "all" reshapes, NaN for failed
restarts, predict_y adding each problem's noise, and snapshot semantics.  No GPU."""
import numpy as np
import pytest

from oracle import mfgp_oracle as onp


class _FakePosterior:
    def __init__(self, X, Y, thetas, noises, P, failed):
        self.X, self.Y, self.P = X.copy(), Y.copy(), P
        self.thetas, self.noises, self.failed = thetas.copy(), noises.copy(), failed
        self.closed = False

    def predict(self, Xs, mean=None, var=None):
        B, ycols = self.thetas.shape[0], self.Y.shape[1]
        mean, var = np.empty((B, Xs.shape[0], self.P)), np.empty((B, Xs.shape[0]))
        for b in range(B):
            c = (b * self.P) % ycols
            if self.failed[b]:
                mean[b], var[b] = np.nan, np.nan
            else:
                mean[b], var[b] = onp.gpr_predict(self.X, self.Y[:, c:c + self.P], Xs, self.thetas[b], self.noises[b])
        return mean, var

    def close(self):
        self.closed = True


class _OracleHandle:
    """Stand-in for _lib.Handle: the oracle per problem; problems listed in `fail` are not positive definite."""

    def __init__(self):
        self.fail = set()
        self.created = []

    def _failed(self, B):
        return np.array([b in self.fail for b in range(B)])

    def gpr_batched_nlml_grad(self, X, Y, thetas, noises, want_grad=True, info=None, **kw):
        B = thetas.shape[0]
        nlml = np.array([-onp.gpr_lml(X, Y[:, b % Y.shape[1]:b % Y.shape[1] + 1], thetas[b], noises[b]) for b in range(B)])
        bad = self._failed(B)
        if info is not None:
            info[bad] = 1
        return np.where(bad, np.nan, nlml), None

    def gpr_predict(self, X, y, Xnew, theta, noise):
        return onp.gpr_predict(X, y, Xnew, theta, noise)

    def gpr_posterior(self, X, Y, thetas, noises, P=1, info=None):
        bad = self._failed(thetas.shape[0])
        if bad.any():
            if info is None:
                raise np.linalg.LinAlgError("not positive definite")
            info[bad] = 1
        self.created.append((thetas.copy(), noises.copy(), P))
        return _FakePosterior(np.asarray(X), np.asarray(Y), np.asarray(thetas), np.asarray(noises), P, bad)


def _problem(rng, N=20, d=3, P=4):
    X = np.hstack([rng.random((N, d)), (np.arange(N) >= N - 5).astype(float)[:, None]])
    return X, rng.standard_normal((N, P))


def test_multibin_posterior_ordering_reshapes_and_failed_restarts():
    from multi_fidelity_gpflow_b200.multibin import MultiBinMFGP

    rng = np.random.default_rng(1)
    X, Y = _problem(rng)
    fh = _OracleHandle()
    mdl = MultiBinMFGP(X, Y, num_restarts=3, seed=2, handle=fh)
    Xs = np.vstack([rng.random((6, 4)), X[:2]])
    Xs[:6, -1] = np.array([0, 1, 0, 1, 0.5, 1])

    post = mdl.posterior("all")
    th, nz, P = fh.created[-1]
    assert P == 1 and th.shape == (12, 9) and nz.shape == (12,)
    for r in range(3):
        for p in range(4):
            np.testing.assert_array_equal(th[r * 4 + p], mdl.thetas[r, p])  # problem b = r * P + p
    mean, var = post.predict_f(Xs)
    assert mean.shape == (3, 8, 4) and var.shape == (3, 8, 4)
    for r in range(3):
        for p in range(4):
            m, v = onp.gpr_predict(X, Y[:, p:p + 1], Xs, mdl.thetas[r, p], mdl.noise)
            np.testing.assert_allclose(mean[r, :, p], m[:, 0], rtol=1e-12)
            np.testing.assert_allclose(var[r, :, p], v, rtol=1e-12)

    best = mdl.posterior("best")
    mb, vb = best.predict_f(Xs)
    mp, vp = mdl.predict_f(Xs)
    assert mb.shape == (8, 4) and vb.shape == (8, 4)
    np.testing.assert_allclose(mb, mp, rtol=1e-12)
    np.testing.assert_allclose(vb, vp, rtol=1e-12)

    fh.fail = {2 * 4 + 1}  # restart 2 of bin 1
    post = mdl.posterior("all")
    assert post.failed[2, 1] == 1 and np.count_nonzero(post.failed) == 1
    mean2, var2 = post.predict_f(Xs)
    assert np.isnan(mean2[2, :, 1]).all() and np.isnan(var2[2, :, 1]).all()
    keep = np.ones((3, 4), dtype=bool)
    keep[2, 1] = False
    np.testing.assert_array_equal(mean2.transpose(0, 2, 1)[keep], mean.transpose(0, 2, 1)[keep])
    with pytest.raises(ValueError):
        mdl.posterior("some")


def test_predict_y_adds_each_problems_noise():
    from multi_fidelity_gpflow_b200.multibin import MultiBinPosterior

    rng = np.random.default_rng(3)
    X, Y = _problem(rng, P=2)
    fh = _OracleHandle()
    th = np.exp(0.2 * rng.standard_normal((6, 9)))
    noises = np.array([1e-3, 2e-3, 3e-3, 4e-3, 5e-3, 6e-3])
    post = MultiBinPosterior(fh.gpr_posterior(X, Y, th, noises), noises.reshape(3, 2), np.zeros((3, 2), dtype=np.int32))
    Xs = X[:5]
    mf, vf = post.predict_f(Xs)
    my, vy = post.predict_y(Xs)
    np.testing.assert_array_equal(my, mf)
    np.testing.assert_allclose(vy - vf, np.broadcast_to(noises.reshape(3, 1, 2), vf.shape), rtol=1e-9)
    best = MultiBinPosterior(fh.gpr_posterior(X, Y, th[:2], noises[:2]), noises[:2], None)
    _, vf = best.predict_f(Xs)
    _, vy = best.predict_y(Xs)
    np.testing.assert_allclose(vy - vf, np.broadcast_to(noises[:2], vf.shape), rtol=1e-9)


def test_posteriors_are_snapshots():
    from multi_fidelity_gpflow_b200.kernels import SquaredExponential
    from multi_fidelity_gpflow_b200.linear import MultiFidelityGPModel
    from multi_fidelity_gpflow_b200.multibin import MultiBinMFGP

    rng = np.random.default_rng(4)
    X, Y = _problem(rng)
    fh = _OracleHandle()
    mdl = MultiBinMFGP(X, Y, num_restarts=2, seed=1, handle=fh)
    post = mdl.posterior("all")
    before = post.predict_f(X[:4])
    mdl.u += 0.3  # "training" after the posterior was taken
    after = post.predict_f(X[:4])
    np.testing.assert_array_equal(before[0], after[0])
    np.testing.assert_array_equal(before[1], after[1])
    assert not np.allclose(mdl.posterior("all").predict_f(X[:4])[0], before[0])

    se = lambda: SquaredExponential(lengthscales=np.ones(3), variance=1.0)
    m = MultiFidelityGPModel(X, Y, se(), se(), handle=fh)
    mp = m.posterior()
    th, nz, P = fh.created[-1]
    assert th.shape == (1, 9) and P == 4 and nz[0] == pytest.approx(1e-3)
    mean, var = mp.predict_f(X[:4])
    ref_m, ref_v = onp.gpr_predict(X, Y, X[:4], th[0], nz[0])
    assert mean.shape == (4, 4) and var.shape == (4, 4)
    np.testing.assert_allclose(mean, ref_m, rtol=1e-12)
    np.testing.assert_allclose(var, np.tile(ref_v[:, None], (1, 4)), rtol=1e-12)
    np.testing.assert_allclose(mp.predict_y(X[:4])[1] - var, nz[0])
    with pytest.raises(NotImplementedError):
        mp.predict_f(X[:4], full_cov=True)
    m.kernel.kernel_L.variance.assign(2.0)
    np.testing.assert_array_equal(mp.predict_f(X[:4])[0], mean)  # the posterior keeps the parameters it was made with
