"""Oracle for the joint posterior of the exact GP (GPR.predict_f(full_cov=True)), built from the oracle's mf_K the way
onp.gpr_predict builds the marginal one."""
import numpy as np
import scipy.linalg as sla

from oracle import mfgp_oracle as onp


def gpr_predict_full_cov(X, Y, Xs, theta, noise):
    """(mean [N*, P], cov [N*, N*]) with cov = K_ss - A^T A, A = L^-1 K_s, L L^T = K + noise I."""
    X = np.asarray(X, dtype=np.float64)
    Lm = np.linalg.cholesky(onp.mf_K(X, None, theta) + noise * np.eye(X.shape[0]))
    A = sla.solve_triangular(Lm, onp.mf_K(X, Xs, theta), lower=True)
    cov = onp.mf_K(Xs, None, theta) - A.T @ A
    mean = sla.solve_triangular(Lm.T, A, lower=False).T @ np.asarray(Y, dtype=np.float64)
    return mean, cov
