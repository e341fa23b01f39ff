"""Input gradients of the exact-GP prediction without a GPU: the autograd oracle (tests/_grad_oracle.py:
gpr_predict_grad_x) against central finite differences of the NumPy predict_f, and the host logic of
MultiBinPosterior.predict_f_grad / MultiFidelityGPPosterior.predict_f_grad with a fake handle that computes every problem
with the oracle: the "best" / "all" reshapes, the tiling of var, the zero fidelity column, NaN for failed restarts and
snapshot semantics."""
import numpy as np
import pytest

from oracle import mfgp_oracle as onp
from tests._grad_oracle import gpr_predict_grad_x
from tests.test_gpr_posterior_host import _FakePosterior, _OracleHandle, _problem


def _close(got, ref):
    np.testing.assert_allclose(got, ref, rtol=1e-10, atol=1e-12 * max(np.nanmax(np.abs(ref)), 1e-300))


def _fd(X, Y, Xs, th, noise, h=1e-5):
    """Central differences of onp.gpr_predict: dmean [Ns, P, d], dvar [Ns, d]."""
    Ns, d = Xs.shape[0], Xs.shape[1] - 1
    dm, dv = np.empty((Ns, Y.shape[1], d)), np.empty((Ns, d))
    for j in range(d):
        xp, xm = Xs.copy(), Xs.copy()
        xp[:, j] += h
        xm[:, j] -= h
        mp, vp = onp.gpr_predict(X, Y, xp, th, noise)
        mm, vm = onp.gpr_predict(X, Y, xm, th, noise)
        dm[:, :, j] = (mp - mm) / (2 * h)
        dv[:, j] = (vp - vm) / (2 * h)
    return dm, dv


@pytest.mark.parametrize("d,P", [(1, 1), (1, 3), (5, 1), (5, 3)])
def test_oracle_gradient_matches_finite_differences(d, P):
    rng = np.random.default_rng(10 * d + P)
    N = 15
    X = np.hstack([rng.random((N, d)), (rng.random((N, 1)) < 0.4).astype(float)])
    Y = rng.standard_normal((N, P))
    th = onp.default_theta(d) * np.exp(0.2 * rng.standard_normal(2 * d + 3))
    th[0] = 0.8
    noise = 1e-2
    Xs = np.hstack([rng.random((6, d)), np.array([0, 1, 0, 1, 0.5, 1.0])[:, None]])
    Xs[5] = X[3]  # a test point equal to a training point (its own fidelity)
    mean, var, dmean, dvar = gpr_predict_grad_x(X, Y, Xs, th, noise)
    rm, rv = onp.gpr_predict(X, Y, Xs, th, noise)
    np.testing.assert_allclose(mean, rm, rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(var, rv, rtol=1e-10, atol=1e-12)
    assert dmean.shape == (6, P, d + 1) and dvar.shape == (6, d + 1)
    assert np.all(dmean[..., -1] == 0.0) and np.all(dvar[:, -1] == 0.0)  # the fidelity column
    assert np.all(dmean[4] == 0.0) and np.all(dvar[4] == 0.0)  # dead row (fidelity 0.5)
    fm, fv = _fd(X, Y, Xs, th, noise)
    np.testing.assert_allclose(dmean[..., :-1], fm, rtol=1e-6, atol=1e-7 * np.abs(fm).max())
    np.testing.assert_allclose(dvar[:, :-1], fv, rtol=1e-6, atol=1e-7 * np.abs(fv).max())
    assert np.abs(fm).max() > 1e-3 and np.abs(fv).max() > 1e-4  # the check is not vacuous


class _GradPosterior(_FakePosterior):
    def predict_grad(self, Xs):
        B, ycols = self.thetas.shape[0], self.Y.shape[1]
        Ns, d = Xs.shape[0], Xs.shape[1] - 1
        out = (np.empty((B, Ns, self.P)), np.empty((B, Ns)), np.empty((B, Ns, self.P, d)), np.empty((B, Ns, d)))
        for b in range(B):
            c = (b * self.P) % ycols
            if self.failed[b]:
                for o in out:
                    o[b] = np.nan
                continue
            m, v, dm, dv = gpr_predict_grad_x(self.X, self.Y[:, c:c + self.P], Xs, self.thetas[b], self.noises[b])
            out[0][b], out[1][b], out[2][b], out[3][b] = m, v, dm[..., :-1], dv[:, :-1]
        return out


class _GradHandle(_OracleHandle):
    def gpr_posterior(self, X, Y, thetas, noises, P=1, info=None):
        fp = super().gpr_posterior(X, Y, thetas, noises, P=P, info=info)
        return _GradPosterior(fp.X, fp.Y, fp.thetas, fp.noises, fp.P, fp.failed)


def test_multibin_predict_f_grad_reshapes_and_failed_restarts():
    from multi_fidelity_gpflow_b200.multibin import MultiBinMFGP

    rng = np.random.default_rng(1)
    X, Y = _problem(rng)
    fh = _GradHandle()
    mdl = MultiBinMFGP(X, Y, num_restarts=3, seed=2, handle=fh)
    Xs = np.vstack([rng.random((6, 4)), X[:2]])
    Xs[:6, -1] = np.array([0, 1, 0, 1, 0.5, 1])

    fh.fail = {2 * 4 + 1}  # restart 2 of bin 1
    post = mdl.posterior("all")
    mean, var, dm, dv = post.predict_f_grad(Xs)
    assert mean.shape == var.shape == (3, 8, 4) and dm.shape == dv.shape == (3, 8, 4, 4)
    m0, v0 = post.predict_f(Xs)
    _close(mean, m0)
    _close(var, v0)
    for r in range(3):
        for p in range(4):
            if (r, p) == (2, 1):
                assert np.isnan(mean[2, :, 1]).all() and np.isnan(var[2, :, 1]).all()
                assert np.isnan(dm[2, :, 1, :-1]).all() and np.isnan(dv[2, :, 1, :-1]).all()
                assert np.all(dm[2, :, 1, -1] == 0.0) and np.all(dv[2, :, 1, -1] == 0.0)
                continue
            _, _, rdm, rdv = gpr_predict_grad_x(X, Y[:, p:p + 1], Xs, mdl.thetas[r, p], mdl.noise)
            _close(dm[r, :, p], rdm[:, 0])
            _close(dv[r, :, p], rdv)
            assert np.all(dm[r, :, p, -1] == 0.0) and np.all(dv[r, :, p, -1] == 0.0)
            assert np.all(dm[r, 4, p] == 0.0) and np.all(dv[r, 4, p] == 0.0)  # dead test row

    fh.fail = set()
    best = mdl.posterior("best")
    bm, bv, bdm, bdv = best.predict_f_grad(Xs)
    assert bm.shape == bv.shape == (8, 4) and bdm.shape == bdv.shape == (8, 4, 4)
    r = mdl.best_restart()
    _close(bm, mdl.predict_f(Xs)[0])
    for p in range(4):
        _, _, rdm, rdv = gpr_predict_grad_x(X, Y[:, p:p + 1], Xs, mdl.thetas[r[p], p], mdl.noise)
        _close(bdm[:, p], rdm[:, 0])
        _close(bdv[:, p], rdv)


def test_model_predict_f_grad_tiling_and_snapshot():
    from multi_fidelity_gpflow_b200.kernels import SquaredExponential
    from multi_fidelity_gpflow_b200.linear import MultiFidelityGPModel
    from multi_fidelity_gpflow_b200.multibin import MultiBinMFGP

    rng = np.random.default_rng(4)
    X, Y = _problem(rng)
    fh = _GradHandle()
    se = lambda: SquaredExponential(lengthscales=np.ones(3), variance=1.0)
    m = MultiFidelityGPModel(X, Y, se(), se(), handle=fh)
    mp = m.posterior()
    th, nz, _ = fh.created[-1]
    Xs = X[:4]
    mean, var, dm, dv = mp.predict_f_grad(Xs)
    rm, rv, rdm, rdv = gpr_predict_grad_x(X, Y, Xs, th[0], nz[0])
    assert mean.shape == var.shape == (4, 4) and dm.shape == dv.shape == (4, 4, 4)
    _close(mean, rm)
    _close(var, np.tile(rv[:, None], (1, 4)))
    _close(dm, rdm)
    for p in range(4):  # the variance and its gradient are the same in every output column
        np.testing.assert_array_equal(dv[:, p], dv[:, 0])
    _close(dv[:, 0], rdv)
    assert np.all(dm[..., -1] == 0.0) and np.all(dv[..., -1] == 0.0)
    m.kernel.kernel_L.variance.assign(2.0)
    np.testing.assert_array_equal(mp.predict_f_grad(Xs)[2], dm)  # the posterior keeps the parameters it was made with

    mdl = MultiBinMFGP(X, Y, num_restarts=2, seed=1, handle=fh)
    post = mdl.posterior("all")
    before = post.predict_f_grad(X[:4])
    mdl.u += 0.3
    after = post.predict_f_grad(X[:4])
    for a, b in zip(before, after):
        np.testing.assert_array_equal(a, b)
    assert not np.allclose(mdl.posterior("all").predict_f_grad(X[:4])[2], before[2])
