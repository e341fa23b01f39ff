"""Oracle for the joint posterior of the whitened SVGP (SVGP.predict_f(full_cov=True), full_output_cov=False), built from
the oracle's mf_K the way onp.svgp_latent_conditional builds the marginals, then mixed with W^2 as
gpflow.conditionals.util.mix_latent_gp does with full_cov=True."""
import numpy as np
import scipy.linalg as sla

from oracle import mfgp_oracle as onp


def svgp_latent_full_cov(Xs, Z, theta, q_mu_l, q_sqrt_l):
    """(mean [Ns], Sigma [Ns, Ns]) of one latent: Sigma = K_ss - A^T A + (Lq^T A)^T (Lq^T A), A = Lm^-1 K_ms."""
    M = Z.shape[0]
    Lm = np.linalg.cholesky(onp.mf_K(Z, None, theta) + onp.JITTER * np.eye(M))
    A = sla.solve_triangular(Lm, onp.mf_K(Z, Xs, theta), lower=True)
    LTA = np.tril(q_sqrt_l).T @ A
    return A.T @ q_mu_l, onp.mf_K(Xs, None, theta) - A.T @ A + LTA.T @ LTA


def svgp_predict_full_cov(Xs, Z, thetas, q_mu, q_sqrt, W=None):
    """(mean [Ns, P], cov [P, Ns, Ns]): per output sum_l W_pl^2 Sigma_l, or the output's own latent without W."""
    L = thetas.shape[0]
    parts = [svgp_latent_full_cov(Xs, Z, thetas[l], q_mu[:, l], q_sqrt[l]) for l in range(L)]
    g_mean = np.stack([p[0] for p in parts], axis=1)
    g_cov = np.stack([p[1] for p in parts])
    if W is None:
        return g_mean, g_cov
    return g_mean @ W.T, np.einsum("pl,lij->pij", W * W, g_cov)
