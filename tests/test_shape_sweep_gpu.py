"""Training objectives and building blocks at the shapes the datasets do not reach, against the oracle: the SVGP ELBO
gradient (K7) on 128-row GEMM tiles and at the potrf block edges, inputs up to d = 32 (MFGP_MAX_D), the blocked batched
exact-GP route with restarts, a wide Y buffer and its chunk boundary, the shared-small / blocked switch of mfgp_gpr_nlml,
and the "lower triangle only" contracts of potrf and q_sqrt.  North-star tolerances: values 1e-9, gradients 1e-7,
predictions 1e-8; the inputs are chosen so that the conditioning keeps them meaningful."""
import numpy as np
import pytest

from oracle import mfgp_oracle as onp
from oracle import mfgp_oracle_torch as otc
from tests.test_cuda_kernels import rand_theta, rand_X
from tests.test_cuda_svgp import compare, make_problem
from tests.test_svgp_posterior_gpu import random_points, synthetic

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def h():
    from multi_fidelity_gpflow_b200 import _lib

    return _lib.Handle(0)


# ------------------------------------------------------------------------------------ A. K7 shape sweep
# M: inducing points, L: latents, B: data rows, P: outputs (None: no mixing matrix, P = L), lik: "per_output" gives every
# output its own likelihood variance (scalar otherwise), plus the hetero likelihood, num_data scaling and kl_mult.
K7_CASES = [
    dict(M=1, d=1, L=1, B=1),
    dict(M=7, d=5, L=2, B=9, P=3, num_data=40),
    dict(M=64, d=7, L=3, B=33, kl_mult=2.5),
    dict(M=65, d=10, L=4, B=65, P=2, lik="per_output"),
    dict(M=127, d=16, L=2, B=51, hetero=True, lik="per_output"),
    dict(M=128, d=17, L=2, B=130, P=5, hetero=True, num_data=1000),
    dict(M=129, d=32, L=2, B=97, num_data=500, kl_mult=0.5),
    dict(M=129, d=1, L=3, B=1, P=2),
    dict(M=257, d=5, L=1, B=300, P=2, lik="per_output"),
    dict(M=64, d=32, L=2, B=7, P=1),
    dict(M=256, d=5, L=40, B=200, lik="per_output", num_data=2000),  # every product on 128x64 tiles
    dict(M=256, d=10, L=24, B=600, P=30, hetero=True, lik="per_output", kl_mult=1.5),  # M x B on 128x64, M x M on 64x64
]


def case_id(c):
    return "M{M}-d{d}-L{L}-B{B}".format(**c) + ("-P%d" % c["P"] if c.get("P") else "")


def gemm_tile_rows(m, n, batch):
    """The tile rule of launch_gemm (csrc/gemm.cu) for an m x n output in `batch` batches: 128-row tiles once the grid has
    two CTAs per SM of a 148-SM B200 and 128-row tiles do not pad m by > 12 % more than 64-row tiles."""
    ctas = -(-m // 128) * -(-n // 64) * batch
    pad128, pad64 = -(-m // 128) * 128 / m, -(-m // 64) * 64 / m
    return 64 if ctas < 2 * 148 or pad128 > 1.12 * pad64 else 128


def k7_tile_rows(c):
    """Tile rows of the K7 products: M x M (S1, S2, T1, T2, T3) and M x B (A, C, Abar, Kmnbar), all batched over L."""
    return {gemm_tile_rows(c["M"], c["M"], c["L"]), gemm_tile_rows(c["M"], c["B"], c["L"])}


def test_k7_cases_cover_both_tile_configs():
    """If the tile rule changes, the sweep must still run every K7 product on 128-row tiles in one case and mix the two
    configurations in another (the k-range and skip arithmetic differs on BM != BN tiles)."""
    tiles = [k7_tile_rows(c) for c in K7_CASES]
    assert {128} in tiles
    assert {64, 128} in tiles


def k7_problem(rng, M, d, L, B, P=None, hetero=False, **_):
    """synthetic() inducing points and parameters with the length-scales shortened as M grows (and the first coordinate of
    Z stratified), so that K(Z,Z) stays well conditioned at M = 257: cond(K_l(Z,Z) + jitter I) <= 1e6 for every latent."""
    pr = synthetic(rng, M, d, L, P is not None, P=P or L)
    Z, th = pr["Z"], pr["thetas"]
    Z[:, 0] = (rng.permutation(M) + 0.2 + 0.6 * rng.random(M)) / M
    s = min(1.0, 0.5 * M ** (-1.0 / d))
    th[:, 1:1 + d] *= s
    th[:, 2 + d:2 + 2 * d] *= s
    for t in th:
        assert np.linalg.cond(onp.mf_K(Z, None, t) + 1e-6 * np.eye(M)) <= 1e6
    X = random_points(rng, B, d)
    Y = rng.standard_normal((B, P or L))
    if hetero:
        Y = np.hstack([Y, 0.1 + 0.2 * rng.random(Y.shape)])
    return dict(pr, X=X, Y=Y)


@gpu
@pytest.mark.parametrize("c", K7_CASES, ids=case_id)
def test_k7_shape_sweep(h, c):
    rng = np.random.default_rng(c["M"] * 1000 + c["d"] * 10 + c["L"])
    pr = k7_problem(rng, **c)
    P = c.get("P") or c["L"]
    lik = 0.3 + rng.random(P) if c.get("lik") == "per_output" else 0.7
    compare(h, pr, lik, num_data=c.get("num_data"), kl_mult=c.get("kl_mult", 1.0), hetero=c.get("hetero", False))


# ------------------------------------------------------------------------------------ B. exact GP at d = 17 and 32
@gpu
@pytest.mark.parametrize("N", [40, 200])
@pytest.mark.parametrize("d", [17, 32])
def test_gpr_objective_and_predict_high_d(h, d, N):
    """d > 16 takes the blocked route at every N, with the run-time-d K1, K5 and prediction kernels."""
    rng = np.random.default_rng(d * 1000 + N)
    X, th = rand_X(rng, N, d), rand_theta(rng, d)
    th[1:1 + d] *= np.sqrt(d) / 2  # keep the covariance away from the identity in high d
    th[2 + d:2 + 2 * d] *= np.sqrt(d) / 2
    Y = rng.standard_normal((N, 2))
    v = h.gpr_nlml(X, Y, th, 1e-2)
    nlml, g = h.gpr_nlml_grad(X, Y, th, 1e-2)
    lml, gth, gnz = otc.gpr_lml_value_and_grad(X, Y, th, 1e-2)
    assert abs(v + lml) < 1e-9 * abs(lml), (v, lml)
    assert abs(nlml + lml) < 1e-9 * abs(lml), (nlml, lml)
    ref = -np.concatenate([gth, [gnz]])
    np.testing.assert_allclose(g, ref, rtol=1e-7, atol=1e-7 * np.abs(ref).max())
    Xs = np.vstack([rand_X(rng, 50, d), X[:3]])
    mean, var = h.gpr_predict(X, Y, Xs, th, 1e-2)
    rm, rv = onp.gpr_predict(X, Y, Xs, th, 1e-2)
    np.testing.assert_allclose(mean, rm, rtol=1e-8, atol=1e-8 * np.abs(rm).max())
    np.testing.assert_allclose(var, rv, rtol=1e-8, atol=1e-8 * np.abs(rv).max())


# ------------------------------------------------------------------------------------ C. batched exact GP
def batched_raw(h, X, Ybuf, ycols, thetas, noises, info=None):
    """mfgp_gpr_batched_nlml_grad with an explicit ldy (the row pitch of Ybuf) and ycols <= ldy."""
    from multi_fidelity_gpflow_b200 import _lib

    N, d = X.shape[0], X.shape[1] - 1
    B = thetas.shape[0]
    nlml, grad = np.full(B, -1.0), np.full((B, 2 * d + 4), -1.0)
    rc = _lib._lib.mfgp_gpr_batched_nlml_grad(h._h, _lib._ptr(X), N, d, _lib._ptr(Ybuf), Ybuf.shape[1], ycols, B,
                                             _lib._ptr(thetas), _lib._ptr(noises), _lib._ptr(nlml), _lib._ptr(grad),
                                             _lib._ptr(info))
    assert rc == 0 or (rc > 0 and info is not None), _lib._lib.mfgp_last_error(h._h)
    return nlml, grad


def check_batched(X, Y, ycols, th, nz, nlml, grad, problems):
    """Problems b against the oracle; problem b uses column b % ycols."""
    cols = [b % ycols for b in problems]
    vals, grads = otc.gpr_batched_value_and_grad(X, Y[:, cols], th[problems], nz[problems])
    np.testing.assert_allclose(nlml[problems], -vals, rtol=1e-9, atol=1e-10)
    for i, b in enumerate(problems):
        np.testing.assert_allclose(grad[b], -grads[i], rtol=1e-7, atol=1e-7 * max(1.0, np.abs(grads[i]).max()))


@gpu
@pytest.mark.parametrize("N,d", [(65, 3), (40, 17), (53, 5)])  # blocked (N > 64), blocked (d > 16), K6
def test_batched_restarts_and_wide_y(h, N, d):
    """B = 8 problems on ycols = 3 columns (restarts: problem b uses column b % 3) of a Y buffer with ldy = 5 whose
    two extra columns hold NaN: they must never be read."""
    rng = np.random.default_rng(N + d)
    X = rand_X(rng, N, d)
    ycols, ldy, B = 3, 5, 8
    Ybuf = np.full((N, ldy), np.nan)
    Ybuf[:, :ycols] = rng.standard_normal((N, ycols))
    th = np.stack([rand_theta(rng, d) for _ in range(B)])
    nz = rng.uniform(1e-3, 1e-1, B)
    nlml, grad = batched_raw(h, X, Ybuf, ycols, th, nz)
    check_batched(X, Ybuf, ycols, th, nz, nlml, grad, list(range(B)))
    n2, g2 = h.gpr_batched_nlml_grad(X, np.ascontiguousarray(Ybuf[:, :ycols]), th, nz)  # ldy is only the row pitch
    np.testing.assert_array_equal(n2, nlml)
    np.testing.assert_array_equal(g2, grad)


@gpu
def test_batched_blocked_chunk_boundary(h):
    """16 384 + 11 problems at N = 65 (blocked route, chunked over B by free memory, at most 16 384 per chunk; ~3.9 GB):
    theta and noise repeat with period 6 and Y has 3 columns, so every result repeats bit for bit with period 6, across
    whatever chunk boundaries the free memory gives.  Two non-positive-definite problems, one on each side of 16 384,
    are their own info[b] and NaN; sampled problems around 16 384 and the last one match the oracle."""
    rng = np.random.default_rng(16395)
    N, d, ycols, B = 65, 2, 3, 16384 + 11
    X = rand_X(rng, N, d)
    X[5] = X[4]  # a duplicate point: K + noise I is singular for a negative noise
    Y = rng.standard_normal((N, ycols))
    th = np.tile(np.stack([rand_theta(rng, d) for _ in range(6)]), (-(-B // 6), 1))[:B].copy()
    nz = np.tile(rng.uniform(1e-3, 1e-1, 6), -(-B // 6))[:B].copy()
    bad = [7, 16389]
    nz[bad] = -1e-3
    info = np.full(B, -7, dtype=np.int32)
    nlml, grad = batched_raw(h, X, Y, ycols, th, nz, info=info)
    assert np.all(info[bad] > 0)
    good = np.setdiff1d(np.arange(B), bad)
    assert np.all(info[good] == 0)
    assert np.isnan(nlml[bad]).all() and np.isnan(grad[bad]).all()
    assert np.isfinite(nlml[good]).all() and np.isfinite(grad[good]).all()
    rep = good[np.arange(B)[good] % 6]  # the first problem of each residue class (0..5, all good)
    np.testing.assert_array_equal(nlml[good], nlml[rep])
    np.testing.assert_array_equal(grad[good], grad[rep])
    check_batched(X, Y, ycols, th, nz, nlml, grad, [0, 1, 2, 3, 4, 5, 16380, 16383, 16384, 16385, 16390, B - 1])


@gpu
@pytest.mark.parametrize("P", [8192, 8193])
def test_gpr_nlml_shared_small_route_boundary(h, P):
    """N = 20, d = 3: P <= 8192 output columns run as P K6 problems reduced in index order, P = 8193 takes the blocked route."""
    rng = np.random.default_rng(P)
    X, th = rand_X(rng, 20, 3), rand_theta(rng, 3)
    Y = rng.standard_normal((20, P))
    v = h.gpr_nlml(X, Y, th, 1e-2)
    nlml, g = h.gpr_nlml_grad(X, Y, th, 1e-2)
    lml, gth, gnz = otc.gpr_lml_value_and_grad(X, Y, th, 1e-2)
    assert abs(v + lml) < 1e-9 * abs(lml), (v, lml)
    assert abs(nlml + lml) < 1e-9 * abs(lml), (nlml, lml)
    ref = -np.concatenate([gth, [gnz]])
    np.testing.assert_allclose(g, ref, rtol=1e-7, atol=1e-7 * np.abs(ref).max())


# ------------------------------------------------------------------------------------ D. lower-triangle contracts
def junk_upper(A, n):
    """A copy of A whose strictly upper n x n part cycles through quiet NaN, +Inf and -Inf."""
    A = A.copy()
    i, j = np.triu_indices(n, 1)
    A[i, j] = np.array([np.nan, np.inf, -np.inf])[np.arange(i.size) % 3]
    return A


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


@gpu
@pytest.mark.parametrize("N", [1, 5, 127, 128, 129, 300, 1164, 4097])
def test_potrf_reads_only_the_lower_triangle(h, N):
    """mfgp_potrf references only the lower triangle (include/mfgp.h): NaN / Inf above the diagonal change nothing in L or
    W = L^-1; the strict upper part of every 128 x 128 diagonal block of L is zeroed, the upper off-diagonal blocks are
    left as they were, and W is zero above the diagonal."""
    rng = np.random.default_rng(N)
    d = 4
    X, th = rand_X(rng, N, d), rand_theta(rng, d)
    lda = N + (N & 1)
    A0 = np.zeros((N, lda))
    A0[:, :N] = np.tril(onp.mf_K(X, None, th) + 1e-2 * np.eye(N))
    A1 = junk_upper(A0, N)
    L0, W0 = h.potrf(A0, want_inverse=True)
    L1, W1 = h.potrf(A1, want_inverse=True)
    L0, W0, L1, W1, A1 = L0[:, :N], W0[:, :N], L1[:, :N], W1[:, :N], A1[:, :N]
    bi, bj = np.indices((N, N)) // 128
    i, j = np.indices((N, N))
    upper_blocks = bj > bi
    assert np.array_equal(bits(L1)[~upper_blocks], bits(L0)[~upper_blocks])
    assert np.all(L1[(j > i) & (bi == bj)] == 0.0)
    assert np.array_equal(bits(L1)[upper_blocks], bits(A1)[upper_blocks])
    assert np.array_equal(bits(W1), bits(W0))
    assert np.all(W1[j > i] == 0.0)
    assert np.isfinite(np.tril(L1)).all() and np.isfinite(W1).all()


def nan_problem(which):
    if which == 0:
        ds = onp.load_dataset("hbs")
        return make_problem(np.random.default_rng(21), ds["X"], ds["Y"], ds["Z_kmeans50"], 10, 5, True), ds["X_test"]
    rng = np.random.default_rng(22)
    return k7_problem(rng, 129, 5, 3, 70, P=4), random_points(rng, 40, 5)


@gpu
@pytest.mark.parametrize("which", [0, 1])  # HBS latent (M = 50, W); M = 129 (blocked potrf / trtri), W with P > L
def test_svgp_reads_only_tril_q_sqrt(h, which):
    """K7 and mfgp_svgp_predict read only tril(q_sqrt): NaN / Inf above the diagonal give exactly what tril(q_sqrt) gives."""
    pr, Xs = nan_problem(which)
    M = pr["Z"].shape[0]
    lo = dict(pr, q_sqrt=np.tril(pr["q_sqrt"]))
    junk = dict(pr, q_sqrt=np.stack([junk_upper(q, M) for q in lo["q_sqrt"]]))
    run = lambda p: h.svgp_elbo_grad(p["X"], p["Y"], p["Z"], p["thetas"], p["W"], p["q_mu"], p["q_sqrt"], 0.6, scale=3.0)
    a, b = run(lo), run(junk)
    assert np.isfinite(a["elbo"]) and a["elbo"] == b["elbo"] and a["kl"] == b["kl"] and a["g_lik_var"] == b["g_lik_var"]
    for k in ("g_thetas", "g_W", "g_q_mu", "g_q_sqrt"):
        np.testing.assert_array_equal(b[k], a[k], err_msg=k)
    # g_Z is summed over the rows of K(Z,Z) and K(Z,X) with atomics (CovGradArgs::rowgrad), so its last bits vary from run
    # to run even for equal inputs
    assert np.isfinite(b["g_Z"]).all()
    np.testing.assert_allclose(b["g_Z"], a["g_Z"], rtol=1e-12, atol=1e-12 * np.abs(a["g_Z"]).max())
    pa = h.svgp_predict(Xs, lo["Z"], lo["thetas"], lo["W"], lo["q_mu"], lo["q_sqrt"])
    pb = h.svgp_predict(Xs, junk["Z"], junk["thetas"], junk["W"], junk["q_mu"], junk["q_sqrt"])
    assert np.isfinite(pa[1]).all()
    np.testing.assert_array_equal(pb[0], pa[0])
    np.testing.assert_array_equal(pb[1], pa[1])
