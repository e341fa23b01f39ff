"""Autograd oracle of the input gradient of SVGP.predict_f, for the tests of the SVGP posterior input gradients and for
scripts/svgp_posterior_grad_bench.py.  TEST INFRASTRUCTURE ONLY: built on the torch twin of the reference in
oracle/mfgp_oracle_torch.py (svgp_predict), never imported by the product."""
import torch

from oracle.mfgp_oracle_torch import _t, svgp_predict


def svgp_predict_grad_x(Xnew, Z, thetas, q_mu, q_sqrt, W=None):
    """SVGP.predict_f(Xnew) (whitened, marginal variances, mixed by W when given) and its gradient with respect to Xnew by
    autograd through oracle/mfgp_oracle_torch.svgp_predict, one backward per output column.  Returns mean [Ns, P],
    var [Ns, P], dmean [Ns, P, d+1], dvar [Ns, P, d+1]; a point's outputs depend on its own row only, so the gradient of
    a column sum is the per-point gradient."""
    Xs = _t(Xnew).clone().requires_grad_(True)
    mean, var = svgp_predict(Xs, _t(Z), _t(thetas), _t(q_mu), _t(q_sqrt), None if W is None else _t(W))
    P = mean.shape[1]
    col = lambda f, p: torch.autograd.grad(f[:, p].sum(), Xs, retain_graph=True)[0]
    dmean = torch.stack([col(mean, p) for p in range(P)], dim=1)
    dvar = torch.stack([col(var, p) for p in range(P)], dim=1)
    return mean.detach().numpy(), var.detach().numpy(), dmean.numpy(), dvar.numpy()
