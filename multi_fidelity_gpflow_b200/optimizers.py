"""Optimisers as the reference's training loops drive them (linear.py:201-234,
singlebin_svgp.py:77, linear_svgp.py:169): tf.optimizers.Adam with optional
tf.keras CosineDecay, gpflow.optimizers.Scipy (L-BFGS-B) and gpflow.optimizers.NaturalGradient."""
from __future__ import annotations

import math

import numpy as np


class CosineDecay:
    """tf.keras.optimizers.schedules.CosineDecay(initial_lr, decay_steps), evaluated in float32 like TF."""

    def __init__(self, initial_learning_rate, decay_steps, alpha=0.0):
        self.lr0 = np.float32(initial_learning_rate)
        self.decay_steps = int(decay_steps)
        self.alpha = np.float32(alpha)

    def __call__(self, step):
        s = np.float32(min(int(step), self.decay_steps))
        frac = s / np.float32(self.decay_steps)
        cosd = np.float32(0.5) * (np.float32(1.0) + np.cos(np.float32(math.pi) * frac, dtype=np.float32))
        dec = (np.float32(1.0) - self.alpha) * cosd + self.alpha
        return float(np.float32(self.lr0 * dec))


def adam_step_factors(learning_rate, num_steps, first_step=0, cosine_decay_steps=None, beta_1=0.9, beta_2=0.999):
    """Per-step factors lr(step) * sqrt(1 - beta2^t) / (1 - beta1^t), t = step + 1, that the device-resident loops
    (mfgp_gpr_batched_adam, mfgp_svgp_adam) consume: Keras Adam with float32-stored hyper-parameters (quirk Q8) and the
    optional CosineDecay(learning_rate, cosine_decay_steps) schedule, evaluated exactly like `Adam.apply_gradients` below.
    Returns (factors [num_steps], beta1, beta2) with the float32-rounded betas."""
    b1, b2 = float(np.float32(beta_1)), float(np.float32(beta_2))
    sched = CosineDecay(learning_rate, cosine_decay_steps) if cosine_decay_steps else None
    out = np.empty(int(num_steps))
    for s in range(int(num_steps)):
        step = first_step + s
        lr = sched(step) if sched else float(np.float32(learning_rate))
        t = float(step + 1)
        out[s] = lr * math.sqrt(1.0 - b2**t) / (1.0 - b1**t)
    return out, b1, b2


class Adam:
    """Keras-2.10 Adam (ResourceApplyAdam): float32-stored lr/beta hypers cast to float64, eps=1e-7,
    zero gradient => zero update (SURVEY App. A.8, quirk Q8)."""

    def __init__(self, learning_rate=0.001, beta_1=0.9, beta_2=0.999, epsilon=1e-7):
        self.schedule = learning_rate if callable(learning_rate) else None
        self.lr = None if self.schedule else float(np.float32(learning_rate))
        self.b1 = float(np.float32(beta_1))
        self.b2 = float(np.float32(beta_2))
        self.eps = float(epsilon)
        self.iterations = 0
        self._slots = {}

    def apply_gradients(self, grads_and_params):
        lr = self.schedule(self.iterations) if self.schedule else self.lr
        self.iterations += 1
        t = float(self.iterations)
        lr_t = lr * math.sqrt(1.0 - self.b2**t) / (1.0 - self.b1**t)
        for g, p in grads_and_params:
            if g is None:
                continue
            slot = self._slots.get(id(p))
            if slot is None:
                slot = self._slots[id(p)] = (np.zeros_like(p.unconstrained), np.zeros_like(p.unconstrained))
            m, v = slot
            m += (g - m) * (1.0 - self.b1)
            v += (g * g - v) * (1.0 - self.b2)
            p.unconstrained = p.unconstrained - lr_t * m / (np.sqrt(v) + self.eps)


class Scipy:
    """gpflow.optimizers.Scipy().minimize(closure, variables, options=...): packs the UNCONSTRAINED
    variables into one float64 vector (in the given order) and runs scipy L-BFGS-B with jac=True."""

    def minimize(self, value_and_grad, variables, method="L-BFGS-B", options=None):
        import scipy.optimize

        shapes = [p.shape for p in variables]
        sizes = [int(np.prod(s)) if s else 1 for s in shapes]

        def unpack(x):
            o = 0
            for p, s, n in zip(variables, shapes, sizes):
                p.unconstrained = np.array(x[o:o + n], dtype=np.float64).reshape(s)
                o += n

        def fun(x):
            unpack(x)
            loss, grads = value_and_grad()
            return float(loss), np.concatenate([np.ravel(g) for g in grads]) if grads else np.zeros(0)

        x0 = np.concatenate([np.ravel(p.unconstrained) for p in variables]) if variables else np.zeros(0)
        res = scipy.optimize.minimize(fun, x0, jac=True, method=method, options=options or {})
        unpack(res.x)
        return res


class NaturalGradient:
    """gpflow.optimizers.NaturalGradient(gamma) with its default XiNat: minimize(value_and_grad, var_list=[(q_mu, q_sqrt)])
    takes one natural-gradient step on each (q_mu, q_sqrt) pair.  value_and_grad() returns the loss and, LAST, the list of
    loss gradients of the pairs' parameters in var_list order ([g_q_mu, g_q_sqrt, ...]), for example
    ``lambda: model.value_and_grad(data, [model.q_mu, model.q_sqrt])``.  The step runs on the GPU
    (Handle.svgp_natgrad, include/mfgp.h: mfgp_svgp_natgrad).  Unlike GPflow, a latent whose Cholesky factorisation fails
    does not abort the others: they are updated, it keeps its values, and NotPositiveDefiniteError names it afterwards."""

    def __init__(self, gamma, handle=None):
        self.gamma = float(gamma)
        self.handle = handle

    def minimize(self, value_and_grad, var_list):
        from . import _lib

        h = self.handle or _lib.default_handle()
        out = value_and_grad()
        loss, grads = out[0], out[-1]
        if len(grads) != 2 * len(var_list):
            raise ValueError(f"value_and_grad returned {len(grads)} gradients for {len(var_list)} (q_mu, q_sqrt) pairs")
        failed = []
        for k, (q_mu, q_sqrt) in enumerate(var_list):
            m = np.array(q_mu.unconstrained, dtype=np.float64, order="C")
            S = np.ascontiguousarray(np.tril(q_sqrt.unconstrained), dtype=np.float64)
            info = np.zeros(m.shape[1], dtype=np.int32)
            h.svgp_natgrad(m, S, grads[2 * k], grads[2 * k + 1], self.gamma, info=info)
            q_mu.unconstrained = m
            q_sqrt.unconstrained = S
            failed += [(k, int(l), int(info[l])) for l in np.flatnonzero(info)]
        if failed:
            raise _lib.NotPositiveDefiniteError(
                "natural-gradient step: Cholesky decomposition was not successful for (pair, latent, pivot) " + str(failed))
        return loss
