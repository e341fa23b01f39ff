"""GPU parity tests of the graph-structured multi-fidelity kernel and its exact-GP objective (reference mfgpflow/graph.py;
SURVEY 8(f) rank 3) through the C-ABI (mfgp_graph_cov / _cov_diag / _gpr_nlml_grad) and the host model.  No reference
artefact pins this model (the reference has neither a test nor a notebook for it): the oracle restates graph.py block by
block and is checked by finite differences in tests/test_graph_oracle.py."""
import numpy as np
import pytest

from oracle import mfgp_oracle as onp
from oracle import mfgp_oracle_torch as otc
from tests.test_graph_oracle import graph_problem

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def h():
    from multi_fidelity_gpflow_b200 import _lib

    return _lib.Handle(0)


@pytest.mark.parametrize("m,d,N", [(1, 2, 30), (2, 3, 40), (3, 5, 150), (2, 10, 333), (2, 32, 70)])
def test_graph_cov_and_diag(h, m, d, N):
    rng = np.random.default_rng(m * 100 + d)
    X, _, gth = graph_problem(rng, N=N, d=d, m=m)
    X[1, -1] = m + 1.0  # dead rows (graph.py:54): not a fidelity level / NaN
    X[2, -1] = np.nan
    K = h.graph_cov(X, m, gth)
    ref = onp.graph_K(X, gth, m)
    np.testing.assert_allclose(K, ref, rtol=1e-12, atol=1e-14)
    assert np.all(K[1, [0, 2, 3]] == 0) and K[1, 1] == 1e-6 and K[2, 2] == 1e-6
    np.testing.assert_allclose(h.graph_cov_diag(X, m, gth), onp.graph_K_diag(X, gth, m), rtol=1e-14)


@pytest.mark.parametrize("m,d,N,P", [(1, 2, 30, 1), (2, 3, 40, 2), (3, 5, 150, 4), (2, 6, 300, 1), (2, 32, 80, 2)])
def test_graph_gpr_nlml_grad(h, m, d, N, P):
    """Value 1e-9, gradient 1e-7 (north-star tolerances) against the torch oracle, which follows TensorFlow's semantics
    for the (asymmetric) graph covariance: lower-triangle Cholesky, symmetrised sensitivity, all N^2 entries."""
    rng = np.random.default_rng(m * 1000 + N)
    X, Y, gth = graph_problem(rng, N=N, d=d, m=m, P=P)
    nlml, g = h.graph_gpr_nlml_grad(X, Y, m, gth, 1e-3)
    lml, gth_ref, gnz = otc.graph_gpr_lml_value_and_grad(X, Y, gth, m, 1e-3)
    assert abs(nlml + lml) < 1e-9 * abs(lml), (nlml, lml)
    ref = -np.concatenate([gth_ref, [gnz]])
    np.testing.assert_allclose(g, ref, rtol=1e-7, atol=1e-7 * np.abs(ref).max())
    for i in range(m):
        assert g[m + i * m + i] == 0.0  # rho_LF diagonal is never read (graph.py:62)
    v_only, none = h.graph_gpr_nlml_grad(X, Y, m, gth, 1e-3, want_grad=False)
    assert none is None and v_only == nlml


def test_graph_model_matches_linear_model_for_one_source(h):
    """num_LF = 1: f_H = rho f_L + delta is the linear multi-fidelity model; the graph kernel only adds its 1e-6 jitter."""
    from multi_fidelity_gpflow_b200.graph import GraphMultiFidelityGPModel
    from multi_fidelity_gpflow_b200.kernels import SquaredExponential
    from multi_fidelity_gpflow_b200.linear import MultiFidelityGPModel

    ds = onp.forrester_dataset()
    X, Y = ds["X"], ds["Y"]
    se = lambda: SquaredExponential(lengthscales=np.ones(1))
    gm = GraphMultiFidelityGPModel(X, Y, [se()], se(), handle=h)
    lm = MultiFidelityGPModel(X, Y, se(), se(), handle=h)
    lm.likelihood.variance.assign(1e-3 + 1e-6)
    assert abs(gm.log_marginal_likelihood() - lm.log_marginal_likelihood()) < 1e-9 * abs(lm.log_marginal_likelihood())
    assert [p.shape for p in gm.trainable_variables] == [(1, 1), (1, 1), (1,), (), (1,), ()]
    with pytest.raises(NotImplementedError):
        gm.predict_f(ds["X_plot_H"])


def test_graph_model_adam_follows_the_reference_loop(h):
    """graph.py:144-170 (Adam on the unconstrained variables, noise fixed): trajectory against the oracle's TF-Adam."""
    from multi_fidelity_gpflow_b200.graph import GraphMultiFidelityGPModel
    from multi_fidelity_gpflow_b200.kernels import SquaredExponential

    rng = np.random.default_rng(9)
    m, d = 2, 3
    X, Y, gth = graph_problem(rng, N=60, d=d, m=m, P=2)
    rho, rho_LF, kL, kD = onp.graph_unpack(gth, m, d)
    mk = lambda k: SquaredExponential(variance=k[1], lengthscales=k[0])
    mdl = GraphMultiFidelityGPModel(X, Y, [mk(k) for k in kL], mk(kD), handle=h)
    mdl.kernel.rho.assign(np.tile(rho[:, None], (1, 2)))
    mdl.kernel.rho_LF.assign(rho_LF)
    steps = 15
    mdl.optimize(max_iters=steps, learning_rate=0.01, verbose=False)
    # oracle loop: unconstrained vector = [softplus^-1(rho), logit(rho_LF), softplus^-1(kernel parameters)]
    sig = lambda u: 1.0 / (1.0 + np.exp(-u))
    n = gth.size
    is_sig = np.zeros(n, dtype=bool)
    is_sig[m:m + m * m] = True
    u = np.where(is_sig, np.log(gth) - np.log1p(-gth), onp.softplus_inv(gth))
    opt = onp.TFAdam(lr=0.01)
    hist = []
    for _ in range(steps):
        th = np.where(is_sig, sig(u), onp.softplus(u))
        lml, g, _ = otc.graph_gpr_lml_value_and_grad(X, Y, th, m, 1e-3)
        hist.append(-lml)
        du = np.where(is_sig, th * (1.0 - th), 1.0 - np.exp(-th))
        gu = -g * du
        gu[[m + i * m + i for i in range(m)]] = 0.0
        opt.step([u], [gu])
    np.testing.assert_allclose(mdl.loss_history, hist, rtol=1e-8)
    assert mdl.loss_history[-1] < mdl.loss_history[0]


def test_graph_edge_cases(h):
    """No high-fidelity rows (graph.py:69,82 skip the LF-HF / HF-HF blocks), a single point, all rows dead."""
    rng = np.random.default_rng(3)
    m, d = 2, 3
    gth = onp.graph_pack([1.0, 0.8], [[0.5, 0.05], [0.07, 0.5]], [(np.full(d, 0.4), 1.0), (np.full(d, 0.5), 0.9)], (np.full(d, 0.3), 0.7))
    X = np.hstack([rng.random((25, d)), rng.integers(0, m, size=(25, 1)).astype(float)])  # LF sources only
    np.testing.assert_allclose(h.graph_cov(X, m, gth), onp.graph_K(X, gth, m), rtol=1e-12, atol=1e-14)
    Y = rng.standard_normal((25, 1))
    nlml, g = h.graph_gpr_nlml_grad(X, Y, m, gth, 1e-2)
    lml, gr, gn = otc.graph_gpr_lml_value_and_grad(X, Y, gth, m, 1e-2)
    assert abs(nlml + lml) < 1e-9 * abs(lml)
    ref = -np.concatenate([gr, [gn]])
    np.testing.assert_allclose(g, ref, rtol=1e-7, atol=1e-7 * np.abs(ref).max())
    assert g[0] == 0.0 and g[1] == 0.0  # rho never enters without high-fidelity rows; neither does the delta kernel
    assert np.all(g[m + m * m + 2 * (d + 1):m + m * m + 3 * (d + 1)] == 0.0)
    # a single point
    X1 = np.array([[0.3, 0.2, 0.9, 2.0]])
    assert h.graph_cov(X1, m, gth).shape == (1, 1)
    v1, _ = h.graph_gpr_nlml_grad(X1, np.array([[0.5]]), m, gth, 1e-3)
    assert abs(v1 + otc.graph_gpr_lml_value_and_grad(X1, np.array([[0.5]]), gth, m, 1e-3)[0]) < 1e-12
    # every row dead (fidelity not in {0, 1, 2}): K = 1e-6 I, the objective is that of white noise
    Xd = np.hstack([rng.random((6, d)), np.full((6, 1), 5.0)])
    K = h.graph_cov(Xd, m, gth)
    assert np.array_equal(K, 1e-6 * np.eye(6))
    vd, gd = h.graph_gpr_nlml_grad(Xd, np.ones((6, 1)), m, gth, 1e-3)
    s2 = 1e-3 + 1e-6
    assert abs(vd - (0.5 * 6 / s2 + 3 * np.log(s2) + 3 * np.log(2 * np.pi))) < 1e-9 * abs(vd)
    assert np.all(gd[:-1] == 0.0)
