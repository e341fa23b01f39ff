"""One linear multi-fidelity GPR per output bin, many hyper-parameter restarts per bin, trained together on the device.

This is BASELINE config 2 ("Ho-Bird-Shelton 2021 50LF-3HF multi-bin: one linear MF GPR per k-bin, batched"), the
"many single-output GP" design announced in reference `mfgpflow/gpemulator_singlebin.py:1-14`, driven by the Adam branch of
`MultiFidelityGPModel.optimize` (`mfgpflow/linear.py:190-221`: loss = -log_marginal_likelihood, gradient w.r.t. the
unconstrained variables, Keras Adam with float32-stored hyper-parameters, likelihood noise fixed at 1e-3 -- quirk Q3).
Every bin p and restart r is an independent problem b = r * P + p of `mfgp_gpr_batched_adam` (SURVEY 8(f) rank 1): the whole
loop -- softplus, K6 NLML + gradient, chain rule, Adam -- runs on the GPU; the host only supplies the per-step factors
lr(step) * sqrt(1 - beta2^t) / (1 - beta1^t).  No CPU fallback: every number comes from libmfgp.so.
"""
from __future__ import annotations

import numpy as np

from . import _lib
from .base import positive
from .optimizers import adam_step_factors


class MultiBinMFGP:
    def __init__(self, X, Y, num_restarts=1, noise=1e-3, seed=0, spread=0.3, use_rho=True, handle=None):
        """X [N, d+1] with the fidelity column last, Y [N, P] (one column per bin), N <= 64.  Restart 0 starts at the
        reference's initial values (rho = 1, lengthscales = 1, variances = 1: linear.py:42-52 with gpflow defaults);
        restarts r > 0 at log-normal perturbations of them (sigma = `spread`, seeded)."""
        self.X = np.ascontiguousarray(X, dtype=np.float64)
        self.Y = np.ascontiguousarray(Y, dtype=np.float64)
        self.N, self.d = self.X.shape[0], self.X.shape[1] - 1
        self.P, self.R = self.Y.shape[1], int(num_restarts)
        if self.N > 64:
            raise ValueError("MultiBinMFGP runs the small-matrix kernel (N <= 64); use MultiFidelityGPModel for larger problems")
        self.handle = handle if handle is not None else _lib.default_handle()
        self.noise = float(noise)
        self.noises = np.full((self.R, self.P), self.noise)  # likelihood variance of every (restart, bin)
        self.use_rho = bool(use_rho)
        self._tf = positive()
        np_ = 2 * self.d + 3
        rng = np.random.default_rng(seed)
        theta0 = np.ones((self.R, self.P, np_))
        if self.R > 1:
            theta0[1:] *= np.exp(spread * rng.standard_normal((self.R - 1, self.P, np_)))
        self.u = np.ascontiguousarray(self._tf.inverse(theta0).reshape(self.R * self.P, np_))
        self.m = np.zeros_like(self.u)
        self.v = np.zeros_like(self.u)
        self.iterations = 0
        self.loss_history = np.zeros((0, self.R, self.P))
        self.failed = np.zeros((self.R, self.P), dtype=np.int32)  # first failing Cholesky pivot per (restart, bin), 0 = healthy
        self.lbfgs_result = []  # per phase of the last optimize_lbfgs call

    # ---- parameters --------------------------------------------------------------------------------
    @property
    def thetas(self):
        """Constrained hyper-parameters [R, P, 2d+3] = [rho, ls_L (d), var_L, ls_delta (d), var_delta]."""
        return self._tf.forward(self.u).reshape(self.R, self.P, -1)

    def training_loss(self):
        """NLML of every (restart, bin): [R, P]; NaN where that problem's covariance is not positive definite."""
        B = self.R * self.P
        info = np.zeros(B, dtype=np.int32)
        nlml, _ = self.handle.gpr_batched_nlml_grad(self.X, self.Y, self.thetas.reshape(B, -1), self.noises.reshape(B),
                                                    info=info, want_grad=False)
        return np.where(info == 0, nlml, np.nan).reshape(self.R, self.P)

    def log_marginal_likelihood(self):
        return -self.training_loss()

    # ---- training ------------------------------------------------------------------------------------
    def optimize(self, max_iters=1000, learning_rate=0.01, use_cosine_decay=False, beta_1=0.9, beta_2=0.999, epsilon=1e-7):
        """max_iters Adam steps for all R * P problems on the device.  A restart whose covariance stops being positive
        definite is that restart's failure only: `failed[r, p]` records the 1-based pivot of its first failure, its later
        losses are NaN (so best_restart() skips it) and the remaining restarts train on -- the step counter and
        loss_history advance for everyone, so the bias correction / schedule stay right on the next call."""
        lr_t, b1, b2 = adam_step_factors(learning_rate, max_iters, first_step=self.iterations,
                                         cosine_decay_steps=max_iters if use_cosine_decay else None, beta_1=beta_1, beta_2=beta_2)
        B = self.R * self.P
        hist = np.empty((max_iters, B))
        info = np.zeros(B, dtype=np.int32)
        self.handle.gpr_batched_adam(self.X, self.Y, self.u, self.m, self.v, self.noises.reshape(B), lr_t, b1, b2, epsilon,
                                     fix_rho=not self.use_rho, loss_hist=hist, info=info)
        self.iterations += max_iters
        self.loss_history = np.concatenate([self.loss_history, hist.reshape(max_iters, self.R, self.P)])
        new = info.reshape(self.R, self.P)
        self.failed = np.where(self.failed != 0, self.failed, new)
        return self

    def optimize_lbfgs(self, max_iters=1000, fix_noise_first=True):
        """The SciPy L-BFGS-B branch of the reference's optimize (linear.py:222-234, MultiFidelityGPModel.optimize with
        use_adam=False) for all R * P problems in one device loop (Handle.gpr_batched_lbfgs, SciPy's default options):
        phase 1 with every problem's noise fixed, then phase 2 with the noise trained as well (noise = 1e-6 +
        softplus(v), gpflow Gaussian's bound), maxiter=max_iters each.  fix_noise_first=False runs phase 2 only.
        Updates u and `noises`; `lbfgs_result` holds one dict per phase (train_noise, f, nit, nfev, status [R, P], status
        names from _lib.LBFGS_STATUS).  A restart whose start point is not positive definite stops with status "not_pd"
        and is recorded in `failed` as optimize does; the others run on.  L-BFGS leaves the Adam state alone: the moments
        m and v, `iterations` and `loss_history` are not touched."""
        B = self.R * self.P
        self.lbfgs_result = []
        for train_noise in ((False, True) if fix_noise_first else (True,)):
            noises = np.ascontiguousarray(self.noises.reshape(B))
            info = np.zeros(B, dtype=np.int32)
            f, nit, nfev, status = self.handle.gpr_batched_lbfgs(self.X, self.Y, self.u, noises, fix_rho=not self.use_rho,
                                                                 train_noise=train_noise, maxiter=max_iters, info=info)
            self.noises = noises.reshape(self.R, self.P)
            shape = (self.R, self.P)
            self.lbfgs_result.append(dict(train_noise=train_noise, f=np.asarray(f).reshape(shape),
                                          nit=np.asarray(nit).reshape(shape), nfev=np.asarray(nfev).reshape(shape),
                                          status=np.vectorize(_lib.LBFGS_STATUS.get)(np.asarray(status).reshape(shape))))
            new = info.reshape(shape)
            self.failed = np.where(self.failed != 0, self.failed, new)
        return self

    # ---- model selection and prediction ----------------------------------------------------------------
    def best_restart(self):
        """Per bin, the restart with the lowest NLML at the current hyper-parameters: [P]."""
        loss = self.training_loss()
        return np.argmin(np.where(np.isfinite(loss), loss, np.inf), axis=0)

    def best_thetas(self):
        return self._best()[0]

    def _best(self):
        """(thetas [P, 2d+3], noises [P]) of every bin at its best restart."""
        r = self.best_restart()
        return self.thetas[r, np.arange(self.P)], self.noises[r, np.arange(self.P)]

    def predict_f(self, Xnew):
        """Posterior mean / variance [N*, P] of every bin at its best restart (GPR.predict_f per bin)."""
        Xnew = np.ascontiguousarray(Xnew, dtype=np.float64)
        th, nz = self._best()
        mean, var = np.empty((Xnew.shape[0], self.P)), np.empty((Xnew.shape[0], self.P))
        for p in range(self.P):
            mu, s2 = self.handle.gpr_predict(self.X, np.ascontiguousarray(self.Y[:, p:p + 1]), Xnew, th[p], nz[p])
            mean[:, p], var[:, p] = mu[:, 0], s2
        return mean, var

    def predict_f_samples(self, Xnew, num_samples=None, full_cov=True, full_output_cov=False, seed=None):
        """GPflow's GPModel.predict_f_samples for every bin at its best restart: [S, N*, P] ([N*, P] when num_samples is
        None), from a cached posterior made and freed by this call (MultiBinPosterior.predict_f_samples)."""
        post = self.posterior("best")
        try:
            return post.predict_f_samples(Xnew, num_samples, full_cov, full_output_cov, seed)
        finally:
            post.close()

    def posterior(self, restarts="best"):
        """Cached posterior of the bins at the current hyper-parameters (a snapshot: later training does not change it).
        restarts="best": each bin at its best restart, predict_f(Xnew) -> [N*, P] (equal to predict_f);
        "all": every (restart, bin), predict_f -> [R, N*, P], NaN for a restart whose covariance is not positive
        definite.  One cached factorisation per problem b = r * P + p; every prediction is one library call."""
        if restarts == "best":
            th, nz = self._best()
            post = self.handle.gpr_posterior(self.X, self.Y, np.ascontiguousarray(th), np.ascontiguousarray(nz))
            return MultiBinPosterior(post, nz, None)
        if restarts == "all":
            B = self.R * self.P
            info = np.zeros(B, dtype=np.int32)
            post = self.handle.gpr_posterior(self.X, self.Y, np.ascontiguousarray(self.thetas.reshape(B, -1)),
                                             np.ascontiguousarray(self.noises.reshape(B)), info=info)
            return MultiBinPosterior(post, self.noises.copy(), info.reshape(self.R, self.P))
        raise ValueError('restarts must be "best" or "all"')


class MultiBinPosterior:
    """What MultiBinMFGP.posterior returns: predictions of every bin (and restart) from factors kept on the device."""

    def __init__(self, post, noises, failed):
        self._post = post
        self.noises = noises  # [P] ("best") or [R, P] ("all")
        self.failed = failed  # [R, P] first failing pivot per (restart, bin) at creation, 0 = ok; None for "best"

    def predict_f(self, Xnew):
        """Mean and variance [N*, P] ("best") or [R, N*, P] ("all")."""
        mean, var = self._post.predict(np.ascontiguousarray(Xnew, dtype=np.float64))  # [B, N*, 1], [B, N*]
        P = self.noises.shape[-1]
        mean = mean[:, :, 0].reshape(-1, P, mean.shape[1])
        var = var.reshape(-1, P, var.shape[1])
        mean, var = np.swapaxes(mean, 1, 2), np.swapaxes(var, 1, 2)  # [R, N*, P]
        if self.noises.ndim == 1:
            return np.ascontiguousarray(mean[0]), np.ascontiguousarray(var[0])
        return mean, var

    def predict_f_grad(self, Xnew):
        """predict_f and its gradient with respect to Xnew: mean, var [N*, P] and dmean_dx, dvar_dx [N*, P, d+1] ("best"),
        or the same with a leading restart axis R ("all"; NaN for a failed restart).  The last (fidelity) column of the
        gradients is exactly 0, as tape.gradient gives it in the reference."""
        mean, var, dmean, dvar = self._post.predict_grad(np.ascontiguousarray(Xnew, dtype=np.float64))
        P = self.noises.shape[-1]
        B, Ns, _, d = dmean.shape
        pad = lambda g: np.concatenate([g, np.zeros(g.shape[:-1] + (1,))], axis=-1)
        mean = np.swapaxes(mean[:, :, 0].reshape(-1, P, Ns), 1, 2)  # [R, N*, P], problem b = r * P + p
        var = np.swapaxes(var.reshape(-1, P, Ns), 1, 2)
        dmean = pad(np.swapaxes(dmean[:, :, 0, :].reshape(-1, P, Ns, d), 1, 2))  # [R, N*, P, d+1]
        dvar = pad(np.swapaxes(dvar.reshape(-1, P, Ns, d), 1, 2))
        out = (mean, var, dmean, dvar)
        if self.noises.ndim == 1:
            return tuple(np.ascontiguousarray(a[0]) for a in out)
        return tuple(np.ascontiguousarray(a) for a in out)

    def predict_f_full_cov(self, Xnew):
        """GPflow's predict_f(Xnew, full_cov=True): mean [N*, P] and the joint covariance [P, N*, N*] of each bin ("best"),
        or the same with a leading restart axis R ("all"; NaN for a failed restart)."""
        mean, cov = self._post.predict_cov(np.ascontiguousarray(Xnew, dtype=np.float64))  # [B, N*, 1], [B, N*, N*]
        P, Ns = self.noises.shape[-1], mean.shape[1]
        mean = np.swapaxes(mean[:, :, 0].reshape(-1, P, Ns), 1, 2)  # [R, N*, P], problem b = r * P + p
        cov = cov.reshape(-1, P, Ns, Ns)
        if self.noises.ndim == 1:
            return np.ascontiguousarray(mean[0]), cov[0]
        return np.ascontiguousarray(mean), cov

    def predict_f_samples(self, Xnew, num_samples=None, full_cov=True, full_output_cov=False, seed=None):
        """GPflow's predict_f_samples: draws [S, N*, P] of every bin ([N*, P] when num_samples is None), with a leading
        restart axis R for "all" (NaN for a restart whose joint covariance cannot be factored; "best" raises
        NotPositiveDefiniteError instead).  full_cov=True draws jointly over the N* points with jitter 1e-6, full_cov=False
        independently per point.  The normals are np.random.default_rng(seed).standard_normal((R * P, N*, S, 1))."""
        info = None if self.failed is None else np.zeros(self.failed.size, dtype=np.int32)
        f = self._post.draw_f(np.ascontiguousarray(Xnew, dtype=np.float64), num_samples, full_cov, full_output_cov, seed,
                              info)  # [B, N*, S, 1]
        P, Ns, S = self.noises.shape[-1], f.shape[1], f.shape[2]
        f = f[..., 0].reshape(-1, P, Ns, S).transpose(0, 3, 2, 1)  # [R, S, N*, P]
        if num_samples is None:
            f = f[:, 0]
        return np.ascontiguousarray(f[0] if self.noises.ndim == 1 else f)

    def predict_y(self, Xnew):
        """predict_f plus each problem's likelihood noise on the variance."""
        mean, var = self.predict_f(Xnew)
        return mean, var + (self.noises if self.noises.ndim == 1 else self.noises[:, None, :])

    def close(self):
        self._post.close()
