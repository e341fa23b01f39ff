"""Shared machinery of the two SVGP models: gpflow.models.SVGP surface (elbo, prior_kl, predict_f,
q_mu, q_sqrt, inducing_variable, kernel, likelihood, trainable_variables) over mfgp_svgp_*."""
from __future__ import annotations

import pickle

import numpy as np

from . import _lib
from .base import Parameter, multiple_assign, parameter_dict


class InducingPoints:
    _param_order = ("Z",)

    def __init__(self, Z):
        self.Z = Parameter(np.asarray(Z, dtype=np.float64))


class SharedIndependentInducingVariables:
    _param_order = ("inducing_variable",)

    def __init__(self, inducing_variable):
        self.inducing_variable = inducing_variable


def kmeans_inducing_points(X, num_inducing, random_state=42):
    """KMeans on X INCLUDING the fidelity column, like the reference (singlebin_svgp.py:50-51; quirk Q1)."""
    from sklearn.cluster import KMeans

    return KMeans(n_clusters=num_inducing, random_state=random_state).fit(X).cluster_centers_


class SVGPBase:
    _param_order = ("kernel", "likelihood", "inducing_variable", "q_mu", "q_sqrt")
    whiten = True

    def _init_svgp(self, kernel, likelihood, Z, num_latent_gps, q_mu=None, q_sqrt=None, num_data=None, handle=None):
        self._handle = handle
        self.kernel = kernel
        self.likelihood = likelihood
        self.inducing_variable = SharedIndependentInducingVariables(InducingPoints(Z))
        M = Z.shape[0]
        self.num_latent_gps = num_latent_gps
        self.num_data = num_data
        self.q_mu = Parameter(np.zeros((M, num_latent_gps)) if q_mu is None else q_mu)
        self.q_sqrt = Parameter(np.tile(np.eye(M), (num_latent_gps, 1, 1)) if q_sqrt is None else q_sqrt)
        self.loss_history = []

    @property
    def handle(self):
        return self._handle or _lib.default_handle()

    @property
    def Z(self):
        return self.inducing_variable.inducing_variable.Z

    # ---- parameter views -----------------------------------------------------------------------
    def _thetas(self, d):
        return np.stack([k.theta(d) for k in self.kernel.kernels])

    def _W(self):
        W = getattr(self.kernel, "W", None)
        return None if W is None else W.numpy()

    def _lik_var(self):
        """Scalar, or the [P] vector of a per-output likelihood (MaskedGaussian)."""
        v = np.ravel(self.likelihood.variance.numpy())
        return float(v[0]) if v.size == 1 else v

    @property
    def trainable_variables(self):
        """GPflow order seen in the reference notebooks: q_mu, q_sqrt, Z, [W], kernels..., likelihood.variance."""
        vs = [self.q_mu, self.q_sqrt, self.Z]
        W = getattr(self.kernel, "W", None)
        if W is not None:
            vs.append(W)
        for k in self.kernel.kernels:
            vs.extend([k.rho, k.kernel_L.lengthscales, k.kernel_L.variance, k.kernel_delta.lengthscales, k.kernel_delta.variance])
        vs.append(self.likelihood.variance)
        return [p for p in vs if p.trainable]

    # ---- objective -----------------------------------------------------------------------------
    def _call(self, data, want_grad, kl_multiplier=1.0):
        X, Y = data
        X = np.ascontiguousarray(X, dtype=np.float64)
        Y = np.ascontiguousarray(Y, dtype=np.float64)
        d = X.shape[1] - 1
        scale = 1.0 if self.num_data is None else float(self.num_data) / X.shape[0]
        return self.handle.svgp_elbo_grad(
            X, Y, self.Z.numpy(), self._thetas(d), self._W(), self.q_mu.numpy(), np.tril(self.q_sqrt.numpy()),
            self._lik_var(), scale=scale, kl_mult=kl_multiplier, hetero=self.likelihood.heteroscedastic, want_grad=want_grad,
            masked=self.likelihood.masked,
        ), d

    def elbo(self, data):
        return self._call(data, False)[0]["elbo"]

    def prior_kl(self):
        M, L = self.q_mu.shape
        q_mu, Lq = self.q_mu.numpy(), np.tril(self.q_sqrt.numpy())
        dg = np.diagonal(Lq, axis1=-2, axis2=-1)
        return 0.5 * float(np.sum(q_mu * q_mu) - M * L - np.sum(np.log(dg * dg)) + np.sum(Lq * Lq))

    def training_loss(self, data):
        return -self.elbo(data)

    def value_and_grad(self, data, variables=None, kl_multiplier=1.0):
        """loss = -ELBO + (kl_multiplier - 1) KL; gradients w.r.t. the UNCONSTRAINED `variables`."""
        variables = self.trainable_variables if variables is None else variables
        r, d = self._call(data, True, kl_multiplier)
        by = {id(self.q_mu): r["g_q_mu"], id(self.q_sqrt): r["g_q_sqrt"], id(self.Z): r["g_Z"]}
        W = getattr(self.kernel, "W", None)
        if W is not None:
            by[id(W)] = r["g_W"]
        for l, k in enumerate(self.kernel.kernels):
            for p, gu in k.scatter_theta_grad(r["g_thetas"][l], d):
                by[id(p)] = gu
        lv = self.likelihood.variance
        g_lv = r["g_lik_var"]
        by[id(lv)] = lv.grad_to_unconstrained(g_lv if np.ndim(g_lv) else (np.full(lv.shape, g_lv) if lv.shape else g_lv))
        loss = -r["elbo"] + (kl_multiplier - 1.0) * r["kl"]
        return loss, r["kl"], [np.asarray(by[id(p)], dtype=np.float64).reshape(p.shape) for p in variables]

    # ---- device-resident training loop (SURVEY 8(f) rank 1) --------------------------------------------
    def _flat_parameters(self, d):
        """(list of (Parameter, flat slice, per-entry source index or None), n): the flat layout of mfgp_svgp_adam."""
        W = getattr(self.kernel, "W", None)
        items, o = [], 0
        for k in self.kernel.kernels:
            for par, cnt in ((k.rho, 1), (k.kernel_L.lengthscales, d), (k.kernel_L.variance, 1), (k.kernel_delta.lengthscales, d),
                             (k.kernel_delta.variance, 1)):
                if int(np.size(par.unconstrained)) != cnt:
                    raise NotImplementedError("the device loop needs one rho per kernel and ARD lengthscales of shape (d,); "
                                              "use optimize() (host loop) for shared lengthscales")
                items.append((par, slice(o, o + cnt)))
                o += cnt
        for par in [self.Z] + ([W] if W is not None else []) + [self.q_mu, self.q_sqrt, self.likelihood.variance]:
            cnt = int(np.size(par.unconstrained))
            items.append((par, slice(o, o + cnt)))
            o += cnt
        return items, o

    def _flat_pack(self, d):
        items, n = self._flat_parameters(d)
        u, mask = np.empty(n), np.zeros(n, dtype=np.uint8)
        for par, sl in items:
            vals = np.ravel(par.unconstrained)
            if par is self.q_sqrt:
                vals = np.ravel(np.tril(par.unconstrained))
            u[sl] = vals
            mask[sl] = 1 if par.trainable else 0
        return items, u, mask

    def _device_loop(self, data, max_iters, initial_lr, kl_multiplier, run, minibatch_size=None, seed=0, batches_per_step=1):
        """Shared by optimize_on_device / optimize_data_parallel: history semantics of the reference loops, flat packing,
        per-step factors, the minibatch stream position; `run(X, Y, shape, u, mask, lr_t, b1, b2, batch)` -> (u_final,
        loss_hist, kl_hist), with batch None (full batch) or (minibatch_size, seed, pos0).  Each step draws
        batches_per_step minibatches from the stream."""
        from .optimizers import adam_step_factors

        X, Y = data
        X = np.ascontiguousarray(X, dtype=np.float64)
        Y = np.ascontiguousarray(Y, dtype=np.float64)
        d = X.shape[1] - 1
        if minibatch_size is not None:
            N, B = X.shape[0], int(minibatch_size)
            if not 1 <= B <= N:
                raise ValueError(f"minibatch_size must be in [1, {N}] (the number of rows), got {minibatch_size}")
            if self.num_data is None and B < N:
                raise ValueError("minibatches need the model's num_data (the ELBO scale num_data / minibatch_size): this "
                                 "model has num_data=None, which scales the ELBO by 1 and would bias the estimate; set "
                                 "model.num_data = N")
        resumable = hasattr(self, "kl_history")
        if not resumable:
            self.loss_history = []
        nsteps = int(max_iters) - (len(self.loss_history) if resumable else 0)
        if nsteps <= 0:
            return self
        batch = None
        if minibatch_size is not None:
            # a resumable model continues the stream where its last minibatch call stopped (counted in rows, so that the
            # batch size may change between calls); a model that restarts its loop restarts the stream too
            batch = (B, int(seed), getattr(self, "minibatch_position", 0) if resumable else 0)
        items, u, mask = self._flat_pack(d)
        lr_t, b1, b2 = adam_step_factors(initial_lr, nsteps, cosine_decay_steps=int(max_iters))
        M, L = self.q_mu.shape
        W = getattr(self.kernel, "W", None)
        lik = self.likelihood
        shape = dict(L=L, M=M, P=L if W is None else W.shape[0], d=d, has_W=W is not None, hetero=lik.heteroscedastic,
                     masked=lik.masked, lik_per_output=int(np.size(lik.variance.unconstrained)) > 1,
                     lik_lower=lik.variance.transform.lower)
        u, loss, kl = run(X, Y, shape, u, mask, lr_t, b1, b2, batch)
        for par, sl in items:
            par.unconstrained = u[sl].reshape(np.shape(par.unconstrained)).copy()
        self.loss_history = list(self.loss_history) + list(loss)
        if resumable:
            self.kl_history = list(self.kl_history) + list(kl)
            if batch is not None:
                self.minibatch_position = batch[2] + nsteps * batches_per_step * batch[0]
        return self

    def optimize_on_device(self, data, max_iters, initial_lr, kl_multiplier=1.0, minibatch_size=None, seed=0,
                           natgrad_gamma=None):
        """The model's optimize() loop -- full-batch Adam with CosineDecay(initial_lr, max_iters) on the unconstrained
        trainable variables, loss = -ELBO + (kl_multiplier - 1) KL -- run by mfgp_svgp_adam without a host round trip per
        step.  Same trajectory and the same history semantics as the model's optimize() (tests/test_svgp_device_loop.py):
        a model with a `kl_history` (LatentMFCoregionalizationSVGP, linear_svgp.py:194) runs the REMAINING steps
        range(len(loss_history), max_iters) and appends; SingleBinSVGP (singlebin_svgp.py:79) resets loss_history and runs
        max_iters steps.  Like the reference, every call starts a fresh optimizer (Adam moments zero, iteration 0).

        minibatch_size=B trains on shuffled minibatches instead (GPflow's Dataset.shuffle(N).repeat().batch(B) feeding
        training_loss): step t uses the B rows at positions pos0 + t B ... of the stream of shuffled epochs over the N rows
        of `data` drawn with `seed` (include/mfgp.h: minibatch stream), gathered on the GPU inside the captured step by
        mfgp_svgp_adam_minibatch, with ELBO scale num_data / B.  loss_history receives each step's minibatch estimate.  A
        resumable model continues the stream at `minibatch_position` (rows drawn so far); SingleBinSVGP starts at 0.
        A model with num_data=None (SingleBinSVGP's default) accepts only B = N: set num_data to train on minibatches.

        natgrad_gamma (a float, or one value per step this call runs) trains q_mu and q_sqrt with natural gradients
        instead, as GPflow's natural-gradient recipe does: every step is NaturalGradient(gamma).minimize on
        [(q_mu, q_sqrt)] and then Adam on the other trainable variables, each on a fresh evaluation of the loss
        (mfgp_svgp_natgrad_adam).  loss_history receives the loss before the natural-gradient step.  With minibatch_size
        each of the two evaluations draws its own batch, so minibatch_position advances 2 B per step.  A latent whose
        natural-gradient step fails keeps its q(u); the parameters and histories are written back and then
        NotPositiveDefiniteError names the latents."""
        failed = []

        def run(X, Y, shape, u, mask, lr_t, b1, b2, batch):
            m, v = np.zeros_like(u), np.zeros_like(u)
            kw = dict(kl_mult=kl_multiplier, hetero=shape["hetero"], lik_lower=shape["lik_lower"], masked=shape["masked"],
                      lik_per_output=shape["lik_per_output"])
            args = (X, Y, shape["L"], shape["M"], shape["P"], shape["has_W"], u, m, v, mask, lr_t, b1, b2, 1e-7)
            if natgrad_gamma is not None:
                n = len(lr_t)
                gamma_t = np.ascontiguousarray(np.broadcast_to(np.asarray(natgrad_gamma, dtype=np.float64), (n,)))
                info = np.zeros(shape["L"], dtype=np.int32)
                gkw = dict(scale=1.0 if self.num_data is None else float(self.num_data) / X.shape[0])
                if batch is not None:
                    B, seed_, pos0 = batch
                    gkw = dict(batch_size=B, seed=seed_, pos0=pos0,
                               scale=float(X.shape[0] if self.num_data is None else self.num_data) / B)
                args = args[:11] + (gamma_t,) + args[11:]
                loss, kl = self.handle.svgp_natgrad_adam(*args, info=info, **gkw, **kw)
                failed.extend((int(l), int(info[l])) for l in np.flatnonzero(info))
                return u, loss, kl
            if batch is None:
                scale = 1.0 if self.num_data is None else float(self.num_data) / X.shape[0]
                loss, kl = self.handle.svgp_adam(*args, scale=scale, **kw)
            else:
                B, seed_, pos0 = batch
                scale = float(X.shape[0] if self.num_data is None else self.num_data) / B
                loss, kl = self.handle.svgp_adam_minibatch(*args, batch_size=B, seed=seed_, pos0=pos0, scale=scale, **kw)
            return u, loss, kl

        if natgrad_gamma is not None and np.ndim(natgrad_gamma) not in (0, 1):
            raise ValueError("natgrad_gamma must be a float or one value per step")
        self._device_loop(data, max_iters, initial_lr, kl_multiplier, run, minibatch_size, seed,
                          batches_per_step=1 if natgrad_gamma is None else 2)
        if failed:
            raise _lib.NotPositiveDefiniteError(
                "natural-gradient step: Cholesky decomposition was not successful for (latent, pivot) " + str(failed)
                + "; those latents kept their q(u), the other parameters and the histories were written back")
        return self

    def optimize_data_parallel(self, data, max_iters, initial_lr, kl_multiplier=1.0, group=None, timing=None,
                               minibatch_size=None, seed=0):
        """optimize_on_device across the ranks of a torch.distributed group (one process per GPU, NCCL): the rows of the
        batch shard across ranks, one in-place all-reduce of the flat device gradient per step (dist.dp_svgp_adam); every
        rank ends with the same parameters and histories.  With minibatch_size=B every rank holds the whole data set and
        draws its shard_range slice of each global batch of B rows of optimize_on_device's stream inside the captured
        step, so the run follows the single-GPU minibatch trajectory (ELBO scale num_data / B)."""
        from .dist import dp_svgp_adam

        def run(X, Y, shape, u, mask, lr_t, b1, b2, batch):
            num_data = self.num_data if batch is None or self.num_data is not None else X.shape[0]
            return dp_svgp_adam(self.handle, X, Y, shape, u, mask, lr_t, b1, b2, 1e-7, num_data=num_data,
                                kl_mult=kl_multiplier, group=group, timing=timing, minibatch=batch)

        return self._device_loop(data, max_iters, initial_lr, kl_multiplier, run, minibatch_size, seed)

    def predict_f(self, Xnew, full_cov=False, full_output_cov=False):
        if full_cov or full_output_cov:
            raise NotImplementedError("the reference only calls predict_f(Xnew) (marginal variances)")
        Xnew = np.ascontiguousarray(Xnew, dtype=np.float64)
        d = Xnew.shape[1] - 1
        return self.handle.svgp_predict(Xnew, self.Z.numpy(), self._thetas(d), self._W(), self.q_mu.numpy(),
                                        np.tril(self.q_sqrt.numpy()))

    def posterior(self):
        """SVGPPosterior: the inducing covariances factored once at the current parameters (a snapshot of Z, the
        kernels, W, q_mu and tril(q_sqrt)); its predict_f gives what predict_f gives, without factoring on every call."""
        Z = self.Z.numpy()
        d = Z.shape[1] - 1
        return SVGPPosterior(self.handle.svgp_posterior(Z, self._thetas(d), self._W(), self.q_mu.numpy(),
                                                        np.tril(self.q_sqrt.numpy())))

    def predict_f_samples(self, Xnew, num_samples=None, full_cov=True, full_output_cov=False, seed=None):
        """GPflow's GPModel.predict_f_samples: [S, N*, P] ([N*, P] when num_samples is None), from a cached posterior made
        and freed by this call (SVGPPosterior.predict_f_samples)."""
        post = self.posterior()
        try:
            return post.predict_f_samples(Xnew, num_samples, full_cov, full_output_cov, seed)
        finally:
            post.close()

    # ---- checkpoint (pickle of gpflow.utilities.parameter_dict-style names) ------------------------
    def save_model(self, filename):
        with open(filename, "wb") as f:
            pickle.dump(parameter_dict(self), f)

    def _load_params(self, filename):
        with open(filename, "rb") as f:
            multiple_assign(self, pickle.load(f))
        return self


class SVGPPosterior:
    """What SVGPBase.posterior() returns: predict_f(Xnew) -> mean, var [N*, P] from the cached factors,
    predict_f_grad(Xnew) with their input gradients, and the joint posterior over the N* points, predict_f_full_cov and
    predict_f_samples."""

    def __init__(self, post):
        self.post = post

    def predict_f(self, Xnew, full_cov=False, full_output_cov=False):
        if full_cov or full_output_cov:
            raise NotImplementedError("the reference only calls predict_f(Xnew) (marginal variances)")
        return self.post.predict(_lib.as_f64(Xnew))

    def predict_f_full_cov(self, Xnew):
        """SVGP.predict_f(Xnew, full_cov=True): mean [N*, P] and each output's covariance over the N* points, cov
        [P, N*, N*].  mean and the diagonals are predict_f's, bit for bit."""
        return self.post.predict_cov(_lib.as_f64(Xnew))

    def predict_f_samples(self, Xnew, num_samples=None, full_cov=True, full_output_cov=False, seed=None):
        """GPflow's predict_f_samples with full_output_cov=False: [S, N*, P] ([N*, P] when num_samples is None), each
        output drawn on its own.  full_cov=True draws jointly over the N* points with jitter 1e-6, full_cov=False
        independently per point.  The normals are np.random.default_rng(seed).standard_normal((P, N*, S))."""
        f = self.post.draw_f(_lib.as_f64(Xnew), num_samples, full_cov, full_output_cov, seed)
        f = np.transpose(f, (2, 1, 0))  # [S, N*, P]
        return np.ascontiguousarray(f[0] if num_samples is None else f)

    def close(self):
        self.post.close()

    def predict_f_grad(self, Xnew):
        """predict_f and its gradient with respect to Xnew: mean, var [N*, P] and dmean_dx, dvar_dx [N*, P, d+1]
        (d value[s, p] / d Xnew[s, j]).  The last (fidelity) column is exactly 0, as tape.gradient gives it in the
        reference."""
        mean, var, dmean, dvar = self.post.predict_grad(_lib.as_f64(Xnew))
        pad = lambda g: np.concatenate([g, np.zeros(g.shape[:-1] + (1,))], axis=-1)
        return mean, var, pad(dmean), pad(dvar)
