"""MultiFidelityGPModel -- host-side mirror of the reference's exact-GP model
(mfgpflow/linear.py:138-234): same constructor, attributes, `log_marginal_likelihood`,
`training_loss`, `predict_f`, `trainable_variables` and `optimize` (Adam | SciPy L-BFGS-B)
semantics, including its quirks (SURVEY App. C: Q2 only rho[0] is used, Q3 "unfix noise" is a
no-op under Adam).  Objective, analytic gradient and prediction run in libmfgp.so."""
from __future__ import annotations

import numpy as np

from . import _lib
from .base import set_trainable
from .kernels import LinearMultiFidelityKernel
from .likelihoods import Gaussian
from .optimizers import Adam, Scipy


class MultiFidelityGPModel:
    _param_order = ("kernel", "likelihood")

    def __init__(self, X, Y, kernel_L, kernel_delta, handle=None):
        X = np.ascontiguousarray(X, dtype=np.float64)
        Y = np.ascontiguousarray(Y, dtype=np.float64)
        num_output_dims = Y.shape[1]
        self._handle = handle
        self.kernel = LinearMultiFidelityKernel(kernel_L, kernel_delta, num_output_dims, handle=handle)
        self.likelihood = Gaussian(variance=1e-3)  # linear.py:151
        set_trainable(self.likelihood.variance, False)  # linear.py:154
        self.data = (X, Y)
        self.num_output_dims = num_output_dims
        self.loss_history = []

    @property
    def handle(self):
        return self._handle or _lib.default_handle()

    # ---- objective ---------------------------------------------------------------------------
    def _theta_noise(self):
        X, _ = self.data
        return self.kernel.theta(X.shape[1] - 1), float(self.likelihood.variance.numpy())

    def log_marginal_likelihood(self):
        X, Y = self.data
        theta, noise = self._theta_noise()
        return -self.handle.gpr_nlml(X, Y, theta, noise)

    def training_loss(self):
        return -self.log_marginal_likelihood()

    @property
    def trainable_variables(self):
        vs = self.kernel.trainable_parameters()
        if self.likelihood.variance.trainable:
            vs.append(self.likelihood.variance)
        return vs

    def value_and_grad(self, variables=None):
        """(loss = -LML, [d loss / d unconstrained variable]) for `variables` (default: trainable_variables)."""
        variables = self.trainable_variables if variables is None else variables
        X, Y = self.data
        d = X.shape[1] - 1
        theta, noise = self._theta_noise()
        nlml, g = self.handle.gpr_nlml_grad(X, Y, theta, noise)
        by_param = {id(p): gu for p, gu in self.kernel.scatter_theta_grad(g[: 2 * d + 3], d)}
        by_param[id(self.likelihood.variance)] = self.likelihood.variance.grad_to_unconstrained(g[2 * d + 3])
        return nlml, [by_param[id(p)] for p in variables]

    # ---- prediction --------------------------------------------------------------------------
    def predict_f(self, Xnew, full_cov=False, full_output_cov=False):
        if full_cov or full_output_cov:
            raise NotImplementedError("the reference only calls predict_f(Xnew) (marginal variances)")
        X, Y = self.data
        theta, noise = self._theta_noise()
        mean, var = self.handle.gpr_predict(X, Y, np.asarray(Xnew, dtype=np.float64), theta, noise)
        return mean, np.tile(var[:, None], (1, Y.shape[1]))  # same variance in every output column

    def predict_y(self, Xnew):
        mean, var = self.predict_f(Xnew)
        return mean, var + float(self.likelihood.variance.numpy())

    def posterior(self):
        """Cached posterior at the current parameters (GPflow's model.posterior(), PrecomputeCacheType.TENSOR): the
        factorisation is done once here and reused by every predict_f / predict_y of the returned object; later training
        does not change it.  predict_f keeps the reference's behaviour of factoring on every call."""
        X, Y = self.data
        theta, noise = self._theta_noise()
        post = self.handle.gpr_posterior(X, Y, np.ascontiguousarray(theta)[None, :], np.array([noise]), P=Y.shape[1])
        return MultiFidelityGPPosterior(post, noise)

    def predict_f_samples(self, Xnew, num_samples=None, full_cov=True, full_output_cov=False, seed=None):
        """GPflow's GPModel.predict_f_samples: [S, N*, P] ([N*, P] when num_samples is None), from a cached posterior made
        and freed by this call (MultiFidelityGPPosterior.predict_f_samples)."""
        post = self.posterior()
        try:
            return post.predict_f_samples(Xnew, num_samples, full_cov, full_output_cov, seed)
        finally:
            post.close()

    # ---- training loops (linear.py:190-234) ----------------------------------------------------
    def optimize(self, max_iters=1000, learning_rate=0.01, use_adam=True, unfix_noise_after=500, verbose=True):
        self.loss_history = []
        if use_adam:
            optimizer = Adam(learning_rate)
            traced = self.trainable_variables  # the reference's tf.function captures this list once (quirk Q3)
            if verbose:
                print("Optimizing with Adam...")
            for i in range(max_iters):
                loss, grads = self.value_and_grad(traced)
                optimizer.apply_gradients(zip(grads, traced))
                self.loss_history.append(loss)
                if i == unfix_noise_after:
                    if verbose:
                        print(f"Unfixing noise at iteration {i}")
                    set_trainable(self.likelihood.variance, True)  # no effect on `traced`
                if verbose and i % 100 == 0:
                    print(f"Iteration {i}: Loss = {-loss}")
        else:
            if verbose:
                print("Optimizing with L-BFGS (Scipy)...")
            opt = Scipy()
            vs = self.trainable_variables
            opt.minimize(lambda: self.value_and_grad(vs), vs, options={"maxiter": max_iters})
            set_trainable(self.likelihood.variance, True)
            vs = self.trainable_variables
            opt.minimize(lambda: self.value_and_grad(vs), vs, options={"maxiter": max_iters})
        return self


class MultiFidelityGPPosterior:
    """What MultiFidelityGPModel.posterior returns: predict_f / predict_y with the model's shapes, from cached factors."""

    def __init__(self, post, noise):
        self._post = post
        self.noise = float(noise)

    def predict_f(self, Xnew, full_cov=False, full_output_cov=False):
        if full_cov or full_output_cov:
            raise NotImplementedError("the reference only calls predict_f(Xnew) (marginal variances)")
        mean, var = self._post.predict(np.ascontiguousarray(Xnew, dtype=np.float64))
        return mean[0], np.tile(var[0][:, None], (1, mean.shape[2]))  # same variance in every output column

    def predict_y(self, Xnew):
        mean, var = self.predict_f(Xnew)
        return mean, var + self.noise

    def predict_f_full_cov(self, Xnew):
        """GPflow's predict_f(Xnew, full_cov=True): mean [N*, P] and cov [P, N*, N*], the P slices one read-only matrix
        (every output column shares the kernel)."""
        mean, cov = self._post.predict_cov(np.ascontiguousarray(Xnew, dtype=np.float64))
        return mean[0], np.broadcast_to(cov[0], (mean.shape[2],) + cov.shape[1:])

    def predict_f_samples(self, Xnew, num_samples=None, full_cov=True, full_output_cov=False, seed=None):
        """GPflow's predict_f_samples: [S, N*, P] ([N*, P] when num_samples is None).  full_cov=True draws jointly over
        the N* points with jitter 1e-6, full_cov=False independently per point.  The normals are
        np.random.default_rng(seed).standard_normal((1, N*, S, P))."""
        f = self._post.draw_f(np.ascontiguousarray(Xnew, dtype=np.float64), num_samples, full_cov, full_output_cov, seed)
        f = np.swapaxes(f[0], 0, 1)  # [S, N*, P]
        return np.ascontiguousarray(f[0] if num_samples is None else f)

    def predict_f_grad(self, Xnew):
        """predict_f and its gradient with respect to Xnew: mean [N*, P], var [N*, P], dmean_dx [N*, P, d+1] and
        dvar_dx [N*, P, d+1] (d value[s, p] / d Xnew[s, j]).  The last (fidelity) column is exactly 0, as
        tape.gradient gives it in the reference; predict_y has the same gradient."""
        mean, var, dmean, dvar = self._post.predict_grad(np.ascontiguousarray(Xnew, dtype=np.float64))
        P = mean.shape[2]
        dm = np.zeros(dmean.shape[1:3] + (dmean.shape[3] + 1,))
        dm[..., :-1] = dmean[0]
        dv = np.zeros_like(dm)
        dv[..., :-1] = dvar[0][:, None, :]
        return mean[0], np.tile(var[0][:, None], (1, P)), dm, dv

    def close(self):
        self._post.close()
