"""Torch-fp64 twin of the natural-gradient step of include/mfgp.h (mfgp_svgp_natgrad): GPflow 2.9's NaturalGradient with
the default XiNat, written along GPflow's code path for each latent:

    eta1, eta2 = meanvarsqrt_to_expectation(m, Lq)
    dL/deta    = autograd through expectation_to_meanvarsqrt(eta1, eta2) with output gradients (g_m, G)
    nat1, nat2 = meanvarsqrt_to_natural(m, Lq)
    m', Lq'    = natural_to_meanvarsqrt(nat1 - gamma dL/deta1, nat2 - gamma dL/deta2)

One point differs from a literal transcription: expectation_to_meanvarsqrt factors eta2 - eta1 eta1^T with the signs of
Lq's diagonal (chol(S) D, D = diag(sign(Lq_ii))), so that the output gradient G, taken at Lq, is applied at the factor it
was taken at.  With a positive diagonal that is GPflow's factor; q_sqrt has no positivity, and with negative diagonal
entries GPflow's positive factor would apply G at another matrix.  TF's Cholesky gradient is symmetric; the twin
symmetrises torch's the same way.  A failed Cholesky (torch.linalg.cholesky_ex) leaves the latent as it was, with the
1-based pivot in info (R first), as the library does."""
import numpy as np
import torch

DT = torch.float64


def _t(x):
    return torch.as_tensor(np.asarray(x, dtype=np.float64))


def meanvarsqrt_to_expectation(m, Lq):
    return m, Lq @ Lq.T + torch.outer(m, m)


def expectation_to_meanvarsqrt(eta1, eta2, signs):
    S = eta2 - torch.outer(eta1, eta1)
    return eta1, torch.linalg.cholesky(S) * signs


def meanvarsqrt_to_natural(m, Lq):
    Wq = torch.linalg.solve_triangular(Lq, torch.eye(Lq.shape[0], dtype=DT), upper=False)
    Lam = Wq.T @ Wq
    return Lam @ m, -0.5 * Lam


def natural_to_meanvarsqrt(nat1, nat2):
    """(m, Lq, info): info is the 1-based pivot of the first failed Cholesky (R first), 0 when both succeed."""
    R, info = torch.linalg.cholesky_ex(-2.0 * nat2)
    if int(info):
        return None, None, int(info)
    Rinv = torch.linalg.solve_triangular(R, torch.eye(R.shape[0], dtype=DT), upper=False)
    S = Rinv.T @ Rinv
    Lq, info = torch.linalg.cholesky_ex(S)
    if int(info):
        return None, None, int(info)
    return S @ nat1, Lq, 0


def dL_deta(m, Lq, g_m, G):
    """(dL/deta1, dL/deta2) of one latent by autograd through expectation_to_meanvarsqrt."""
    m, Lq, g_m, G = _t(m), torch.tril(_t(Lq)), _t(g_m), torch.tril(_t(G))
    e1, e2 = meanvarsqrt_to_expectation(m, Lq)
    e1, e2 = e1.clone().requires_grad_(True), e2.clone().requires_grad_(True)
    signs = torch.sign(torch.diagonal(Lq))
    mo, Lo = expectation_to_meanvarsqrt(e1, e2, signs)
    d1, d2 = torch.autograd.grad([mo, Lo], [e1, e2], grad_outputs=[g_m, G])
    return d1.numpy().copy(), (0.5 * (d2 + d2.T)).numpy().copy()


def dL_deta_closed_form(m, Lq, g_m, G):
    """The closed form of include/mfgp.h: g_S = sym(Lq^-T Phi(Lq^T G) Lq^-1), dL/deta1 = g_m - 2 g_S m."""
    Lq, G = np.tril(Lq), np.tril(G)
    Wq = np.linalg.inv(Lq)
    T = Lq.T @ G
    Phi = np.tril(T) - 0.5 * np.diag(np.diag(T))
    X = Wq.T @ Phi @ Wq
    gS = 0.5 * (X + X.T)
    return g_m - 2.0 * gS @ m, gS


def natgrad_step(q_mu, q_sqrt, g_q_mu, g_q_sqrt, gamma):
    """q_mu [M, L], q_sqrt [L, M, M] -> (q_mu', q_sqrt' (upper part zero), info [L]); failed latents keep their values."""
    q_mu, q_sqrt = np.array(q_mu, dtype=np.float64), np.array(q_sqrt, dtype=np.float64)
    M, L = q_mu.shape
    info = np.zeros(L, dtype=np.int32)
    for l in range(L):
        m, Lq = _t(q_mu[:, l]), torch.tril(_t(q_sqrt[l]))
        d1, d2 = dL_deta(q_mu[:, l], q_sqrt[l], g_q_mu[:, l], g_q_sqrt[l])
        n1, n2 = meanvarsqrt_to_natural(m, Lq)
        mn, Lqn, info[l] = natural_to_meanvarsqrt(n1 - gamma * _t(d1), n2 - gamma * _t(d2))
        if not info[l]:
            q_mu[:, l] = mn.numpy()
            q_sqrt[l] = Lqn.numpy()
    return q_mu, q_sqrt, info


def new_precision(q_sqrt, g_q_sqrt, q_mu, g_q_mu, gamma):
    """Lam' = S^-1 + 2 gamma g_S per latent [L, M, M] (the matrix R factors): its condition number bounds the step's error."""
    out = []
    for l in range(q_mu.shape[1]):
        _, gS = dL_deta_closed_form(q_mu[:, l], q_sqrt[l], g_q_mu[:, l], g_q_sqrt[l])
        Wq = np.linalg.inv(np.tril(q_sqrt[l]))
        out.append(Wq.T @ Wq + 2.0 * gamma * gS)
    return np.stack(out)


def conjugate_optimum(A, y, noise_var, scale):
    """Optimal whitened q(u) of one latent under a Gaussian likelihood with per-row variances noise_var (rows where y is
    NaN dropped) and ELBO scale s: S* = (I + s A diag(1/noise_var) A^T)^-1, m* = S* s A (y / noise_var).  A = Lm^-1 Kmn."""
    keep = ~np.isnan(y)
    A, y, nv = A[:, keep], y[keep], np.broadcast_to(noise_var, keep.shape)[keep]
    S = np.linalg.inv(np.eye(A.shape[0]) + scale * (A / nv) @ A.T)
    return S @ (scale * A @ (y / nv)), S
