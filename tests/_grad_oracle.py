"""Autograd oracle of the input gradient of GPR.predict_f, for the tests of the posterior input gradients and for
scripts/posterior_grad_bench.py.  TEST INFRASTRUCTURE ONLY: built on the torch twins of the reference kernel in
oracle/mfgp_oracle_torch.py (mf_K, mf_K_diag), never imported by the product."""
import torch

from oracle.mfgp_oracle_torch import DT, _t, mf_K, mf_K_diag


def gpr_predict_grad_x(X, Y, Xnew, theta, noise):
    """GPR.predict_f(Xnew) (base_conditional, white=False) and its gradient with respect to Xnew by autograd, as
    tape.gradient(predict_f(Xnew), Xnew) gives it.  Returns mean [Ns, P], var [Ns], dmean [Ns, P, d+1], dvar [Ns, d+1];
    a test point's outputs depend on its own row only, so the gradient of a column sum is the per-point gradient."""
    X, Y = _t(X), _t(Y)
    th = _t(theta)
    Xs = _t(Xnew).clone().requires_grad_(True)
    N, P = X.shape[0], Y.shape[1]
    Lm = torch.linalg.cholesky(mf_K(X, None, th) + float(noise) * torch.eye(N, dtype=DT))
    A = torch.linalg.solve_triangular(Lm, mf_K(X, Xs, th), upper=False)
    var = mf_K_diag(Xs, th) - (A * A).sum(0)
    mean = torch.linalg.solve_triangular(Lm.T, A, upper=True).T @ Y
    dvar = torch.autograd.grad(var.sum(), Xs, retain_graph=True)[0]
    dmean = torch.stack([torch.autograd.grad(mean[:, p].sum(), Xs, retain_graph=True)[0] for p in range(P)], dim=1)
    return mean.detach().numpy(), var.detach().numpy(), dmean.numpy(), dvar.numpy()
