"""The NumPy twin of the device L-BFGS (tests/_lbfgs_twin.py) against SciPy, and the host logic of
MultiBinMFGP.optimize_lbfgs with a fake handle that runs the twin on the NumPy/torch oracle.  No GPU.

- The dcsrch / dcstep port against scipy.optimize._dcsrch.DCSRCH, call by call, on the same (f, g) sequences: every
  state variable and every returned step bitwise equal.
- The twin against scipy.optimize.minimize(method="L-BFGS-B") on Rosenbrock and on the oracle NLML of the reference's
  test_scipy sine data, the Forrester data and HBS bin 17.
- The one deliberate deviation (a failed trial point restarts the search short of it) on an objective that is NaN
  beyond a radius, where SciPy's behaviour is not defined."""
import numpy as np
import pytest
import scipy.optimize as so
from scipy.optimize._dcsrch import DCSRCH

from oracle import mfgp_oracle as onp
from oracle import mfgp_oracle_torch as otc
from tests import _lbfgs_twin as twin
from tests.test_gpr_posterior_host import _OracleHandle, _problem

_STATE = ("stx", "fx", "gx", "sty", "fy", "gy", "stmin", "stmax", "width", "width1", "brackt", "stage", "finit",
          "ginit", "gtest")


def _rosen(x):
    return so.rosen(x), so.rosen_der(x)


@pytest.mark.parametrize("case", range(6))
def test_dcsrch_port_matches_scipy_stage_by_stage(case):
    """Both line searches see the same phi(stp), phi'(stp) along Rosenbrock directions; after every call all state and
    the next step agree bit for bit, through bracketing, the modified-function stage and the final task."""
    rng = np.random.default_rng(case)
    n = 2 + case
    x = rng.uniform(-1.5, 1.5, n)
    d = -so.rosen_der(x) * (1.0 if case % 2 else rng.uniform(0.5, 50.0))
    phi = lambda a: (so.rosen(x + a * d), so.rosen_der(x + a * d) @ d)
    f0, g0 = phi(0.0)
    stp0 = [1.0, 1e-3, 0.3, 5.0, 1.0 / np.linalg.norm(d), 2.0][case]
    ref = DCSRCH(None, None, 1e-3, 0.9, 0.1, 0.0, 1e10)
    mine = twin.Dcsrch()
    stp_r, _, _, task_r = ref._iterate(stp0, f0, g0, b"START")
    stp_m, task_m = mine.start(stp0, f0, g0)
    calls = 0
    while True:
        assert stp_m == stp_r and task_m == task_r.decode()[:len(task_m)]
        for k in _STATE:
            assert getattr(mine, k) == getattr(ref, k), (calls, k)
        if task_m != "FG":
            break
        f, g = phi(stp_m)
        stp_r, _, _, task_r = ref._iterate(stp_r, f, g, task_r)
        stp_m, task_m = mine.step(stp_m, f, g)
        calls += 1
        assert calls < 60
    assert task_m in ("CONV", "WARN")


def _scipy_iterates(fg, x0, **options):
    xs = [np.array(x0, dtype=np.float64)]
    res = so.minimize(fg, x0, jac=True, method="L-BFGS-B", options=options, callback=lambda xk: xs.append(xk.copy()))
    return res, xs


_REASON = {"CONVERGENCE: NORM OF PROJECTED GRADIENT <= PGTOL": "pgtol",
           "CONVERGENCE: RELATIVE REDUCTION OF F <= FACTR*EPSMCH": "ftol",
           "STOP: TOTAL NO. OF ITERATIONS REACHED LIMIT": "maxiter",
           "STOP: TOTAL NO. OF F,G EVALUATIONS EXCEEDS LIMIT": "maxfun",
           "ABNORMAL: ": "abnormal"}


def _reason(res):
    return next(v for k, v in _REASON.items() if res.message.startswith(k))


@pytest.mark.parametrize("n,seed,xtol", [(2, 0, 1e-12), (5, 1, 1e-12), (13, 7, 2e-12)])
def test_twin_reproduces_scipy_on_rosenbrock(n, seed, xtol):
    """Identical nit, nfev and termination reason, and the final x.  At n = 13 the last iterates along the valley differ
    from SciPy's by the rounding of its BLAS dot products (1.7e-12 observed)."""
    x0 = 0.5 * np.random.default_rng(seed).standard_normal(n)
    res, _ = _scipy_iterates(_rosen, x0)
    out = twin.minimize(_rosen, x0)
    assert (out["nit"], out["nfev"], out["status"]) == (res.nit, res.nfev, _reason(res))
    np.testing.assert_allclose(out["x"], res.x, rtol=0, atol=xtol)
    assert abs(out["f"] - res.fun) <= 1e-12 * max(1.0, abs(res.fun))


@pytest.mark.parametrize("n", [3, 10, 20, 35])
def test_twin_first_iterates_match_scipy(n):
    x0 = 0.5 * np.random.default_rng(n).standard_normal(n)
    _, xs = _scipy_iterates(_rosen, x0)
    out = twin.minimize(_rosen, x0)
    for a, b in zip(out["iterates"][:11], xs[:11]):
        np.testing.assert_allclose(a, b, rtol=0, atol=1e-12)


def test_twin_termination_order_is_scipys():
    """SciPy tests maxiter and maxfun before pgtol / ftol: a limit equal to what convergence needs reports the limit."""
    x0 = np.array([-1.2, 1.0])
    res, _ = _scipy_iterates(_rosen, x0)
    for opts in (dict(maxiter=res.nit), dict(maxfun=res.nfev - 1), dict(maxiter=7), dict(maxfun=9)):
        r, _ = _scipy_iterates(_rosen, x0, **opts)
        out = twin.minimize(_rosen, x0, **opts)
        assert (out["nit"], out["nfev"], out["status"]) == (r.nit, r.nfev, _reason(r))
        np.testing.assert_allclose(out["x"], r.x, rtol=0, atol=1e-12)


def _sine_data():
    """tests/test_scipy.py of the reference (as test_models_gpu.test_scipy_lbfgs_path_like_reference_test_scipy)."""
    rng = np.random.default_rng(0)
    xl, xh = np.linspace(0, 1, 10)[:, None], np.linspace(0, 1, 5)[:, None]
    yl = np.sin(2 * np.pi * xl) + 0.1 * rng.standard_normal(xl.shape)
    yh = 1.5 * np.sin(2 * np.pi * xh) + 0.2 + 0.05 * rng.standard_normal(xh.shape)
    X = np.vstack([np.hstack([xl, np.zeros_like(xl)]), np.hstack([xh, np.ones_like(xh)])])
    return X, np.vstack([yl, yh])


def _gp_data(name):
    if name == "sine":
        return _sine_data()
    if name == "forrester":
        ds = onp.forrester_dataset()
        return ds["X"], ds["Y"]
    ds = onp.load_dataset("hbs")
    return ds["X"], np.ascontiguousarray(ds["Y"][:, 17:18])


def oracle_objective(X, y, noise=1e-3):
    """u-space NLML and gradient with theta = softplus(u), the objective of the device loop's phase 1."""
    nth = 2 * (X.shape[1] - 1) + 3

    def fg(u):
        th = onp.softplus(u)
        try:
            lml, g, _ = otc.gpr_lml_value_and_grad(X, y, th, noise)
        except Exception:  # a covariance that is not positive definite: a failed point
            return np.nan, np.full(nth, np.nan)
        return -lml, -np.asarray(g[:nth]) * (1.0 - np.exp(-th))

    return fg


@pytest.mark.parametrize("name", ["sine", "forrester", "hbs17"])
def test_twin_matches_scipy_on_the_oracle_nlml(name):
    """First 10 iterates to 1e-9 (observed <= 1.5e-12) and final f to 1e-6 relative (observed <= 3e-8)."""
    X, y = _gp_data(name)
    fg = oracle_objective(X, y)
    u0 = onp.softplus_inv(np.ones(2 * (X.shape[1] - 1) + 3))
    res, xs = _scipy_iterates(fg, u0, maxiter=1000)
    out = twin.minimize(fg, u0, maxiter=1000)
    assert out["status"] in ("pgtol", "ftol") and _reason(res) in ("pgtol", "ftol")
    for a, b in zip(out["iterates"][:11], xs[:11]):
        np.testing.assert_allclose(a, b, rtol=0, atol=1e-9 * max(1.0, np.abs(b).max()))
    assert abs(out["f"] - res.fun) <= 1e-6 * abs(res.fun)


@pytest.mark.parametrize("seed", [0, 2, 3])
def test_failed_trial_restarts_short_of_it_and_converges(seed):
    """NaN beyond |x| = 1.42 (the minimum (1, 1) is at 1.414): after a failed trial its search never again goes beyond
    0.5 x the failed step, and the problem still converges to the minimum."""
    R = 1.42

    def fg(x):
        if np.linalg.norm(x) > R:
            return np.nan, np.full_like(x, np.nan)
        return _rosen(x)

    x0 = np.random.default_rng(seed).uniform(-1.0, 1.0, 2)
    trace = []
    out = twin.minimize(fg, x0, trace=trace)
    failed = [i for i, (x, _, _) in enumerate(trace) if np.linalg.norm(x) > R]
    assert failed and out["status"] in ("pgtol", "ftol")
    np.testing.assert_allclose(out["x"], [1.0, 1.0], atol=1e-4)
    for i in failed:
        bad = trace[i][1]
        nxt = trace[i + 1]
        assert nxt[2] == 0.5 * bad and nxt[1] == 0.1 * bad  # the restarted search: stpmax and first step
        for _, stp, stpmax in trace[i + 1:]:
            if stpmax != nxt[2]:
                break  # the next search
            assert stp <= 0.5 * bad
    assert out["nfev"] == len(trace) + 1


def test_start_point_failure_and_abnormal_line_search():
    nan = lambda x: (np.nan, np.full_like(x, np.nan))
    out = twin.minimize(nan, np.zeros(3))
    assert out["status"] == "not_pd" and out["nfev"] == 1 and out["nit"] == 0 and np.isnan(out["f"])
    # finite only at the start point: every trial fails, maxls runs out with an empty memory
    x0 = np.array([0.3, -0.2])
    fg = lambda x: _rosen(x) if np.array_equal(x, x0) else nan(x)
    out = twin.minimize(fg, x0, maxls=5)
    assert out["status"] == "abnormal" and out["nfev"] == 6 and out["nit"] == 1
    np.testing.assert_array_equal(out["x"], x0)


# ---- MultiBinMFGP.optimize_lbfgs with a fake handle --------------------------------------------------------------
class _LbfgsHandle(_OracleHandle):
    """gpr_batched_lbfgs runs the twin per problem on the oracle objective, with the device call's variable layout."""

    def __init__(self):
        super().__init__()
        self.lbfgs_calls = []

    def gpr_batched_lbfgs(self, X, Y, u, noises, fix_rho=False, train_noise=False, maxiter=15000, info=None, **kw):
        self.lbfgs_calls.append(dict(train_noise=train_noise, fix_rho=fix_rho, maxiter=maxiter, noises=noises.copy()))
        B, nth = u.shape
        f, nit, nfev, status = np.empty(B), np.empty(B, np.int32), np.empty(B, np.int32), np.empty(B, np.int32)
        codes = {v: k for k, v in enumerate(twin.STATUS, start=1)}
        for b in range(B):
            y = Y[:, b % Y.shape[1]:b % Y.shape[1] + 1]
            lo = 1 if fix_rho else 0

            def fg(x, b=b, y=y):
                uu = u[b].copy()
                uu[lo:] = x[:nth - lo]
                th = onp.softplus(uu)
                nz = 1e-6 + onp.softplus(x[-1]) if train_noise else noises[b]
                if b in self.fail:
                    return np.nan, np.full(x.shape, np.nan)
                lml, g, gn = otc.gpr_lml_value_and_grad(X, y, th, nz)
                gu = -np.asarray(g[lo:nth]) * (1.0 - np.exp(-th[lo:]))
                if train_noise:
                    gu = np.append(gu, -gn * (1.0 - np.exp(-(nz - 1e-6))))
                return -lml, gu

            x0 = u[b, lo:].copy()
            if train_noise:
                x0 = np.append(x0, onp.softplus_inv(noises[b] - 1e-6))
            out = twin.minimize(fg, x0, maxiter=maxiter)
            f[b], nit[b], nfev[b], status[b] = out["f"], out["nit"], out["nfev"], codes[out["status"]]
            if out["status"] == "not_pd":
                if info is None:
                    raise np.linalg.LinAlgError("not positive definite")
                info[b] = 1
                continue
            u[b, lo:] = out["x"][:nth - lo]
            if train_noise:
                noises[b] = 1e-6 + onp.softplus(out["x"][-1])
        return f, nit, nfev, status


def test_optimize_lbfgs_phases_noises_result_and_failed():
    from multi_fidelity_gpflow_b200.multibin import MultiBinMFGP

    rng = np.random.default_rng(5)
    X, Y = _problem(rng, N=16, d=2, P=3)
    fh = _LbfgsHandle()
    mdl = MultiBinMFGP(X, Y, num_restarts=2, seed=1, handle=fh, use_rho=False)
    fh.fail = {1 * 3 + 2}  # restart 1 of bin 2
    u0, m0, v0 = mdl.u.copy(), mdl.m.copy(), mdl.v.copy()
    loss0 = mdl.training_loss()
    mdl.optimize_lbfgs(max_iters=50)

    assert [c["train_noise"] for c in fh.lbfgs_calls] == [False, True]
    assert all(c["fix_rho"] and c["maxiter"] == 50 for c in fh.lbfgs_calls)
    np.testing.assert_array_equal(fh.lbfgs_calls[0]["noises"], np.full(6, 1e-3))  # phase 1: the noise as passed
    ph1, ph2 = mdl.lbfgs_result
    assert (ph1["train_noise"], ph2["train_noise"]) == (False, True)
    for ph in (ph1, ph2):
        assert ph["status"].shape == ph["nit"].shape == ph["nfev"].shape == ph["f"].shape == (2, 3)
        assert ph["status"][1, 2] == "not_pd" and np.isnan(ph["f"][1, 2])
        keep = np.ones((2, 3), dtype=bool)
        keep[1, 2] = False
        assert set(ph["status"][keep]) <= {"pgtol", "ftol", "maxiter"}
    # phase 2 started from phase 1's noise and moved every healthy problem's noise
    np.testing.assert_array_equal(fh.lbfgs_calls[1]["noises"], np.full(6, 1e-3))
    assert mdl.noises.shape == (2, 3) and mdl.noises[1, 2] == 1e-3
    assert np.all(mdl.noises[keep] != 1e-3) and np.all(mdl.noises[keep] >= 1e-6)
    # rho stays, the failed restart's u stays, the Adam state is untouched
    np.testing.assert_array_equal(mdl.u[:, 0], u0[:, 0])
    np.testing.assert_array_equal(mdl.u[5], u0[5])
    np.testing.assert_array_equal(mdl.m, m0)
    np.testing.assert_array_equal(mdl.v, v0)
    assert mdl.iterations == 0 and mdl.loss_history.shape == (0, 2, 3)
    assert mdl.failed[1, 2] == 1 and mdl.failed.sum() == 1
    # the model's losses use the trained per-problem noises and went down
    loss = mdl.training_loss()
    np.testing.assert_allclose(loss[keep], ph2["f"][keep], rtol=1e-9)
    assert np.all(loss[keep] < loss0[keep])
    r = mdl.best_restart()
    th, nz = mdl._best()
    np.testing.assert_array_equal(nz, mdl.noises[r, np.arange(3)])
    post = mdl.posterior("all")
    np.testing.assert_array_equal(fh.created[-1][1], mdl.noises.reshape(6))
    np.testing.assert_array_equal(post.noises, mdl.noises)
    mdl.posterior("best")
    np.testing.assert_array_equal(fh.created[-1][1], nz)


def test_optimize_lbfgs_noise_only_phase():
    from multi_fidelity_gpflow_b200.multibin import MultiBinMFGP

    rng = np.random.default_rng(6)
    X, Y = _problem(rng, N=14, d=2, P=2)
    fh = _LbfgsHandle()
    mdl = MultiBinMFGP(X, Y, num_restarts=1, handle=fh)
    mdl.optimize_lbfgs(max_iters=20, fix_noise_first=False)
    assert [c["train_noise"] for c in fh.lbfgs_calls] == [True]
    assert len(mdl.lbfgs_result) == 1 and mdl.lbfgs_result[0]["train_noise"]
