"""Every tile-count instantiation of the five fused posterior kernels (csrc/posterior.cu) against the oracle, and problem
batches past the 65 535 grid-y limit.

The fused kernels are templates on NT = ceil(N / 8) (M for the SVGP kernels), and `with_nt` compiles NT = 1 ... 8, each
with its own unrolled fragment loops, lower-tile loops and padding of the last 8-row tile.  The case tables below sweep N
over every value 1 ... 64, so every NT and every fill of the last tile runs, and vary the other dimensions with N:
d = 1 and d = 16 at every NT, both sides of the P = 8 DFMA / DMMA switch of the mean at every NT, every NST = ceil(Ns / 8)
of the joint kernel at every NT, sample columns split over several CTAs, more than one 8-point group per CTA, the SVGP
kernels with and without W, kernel variance and Y scaled by 10^k for k = -3 ... 3, and the special inputs: a training
(inducing) row of fidelity 0.5, a test point on a training point, a dead test row and test points so far away that every
exponent is clamped by fexp512 (mean ~1e-300, var = k_ss).  test_tables_cover_every_instantiation (CPU) keeps the tables
honest.

Each case is checked against the existing oracles (predict 1e-8, gradients 1e-7, joint as test_gpr_posterior_sample_gpu)
and against a second device route that shares no code with the fused kernels, at 4e-12 of the output's scale: the
blocked route of the exact GP (P = 65, or Ns = 65 for the joint) and K8 (mfgp_svgp_predict) for the SVGP.

for_batch_slices splits a call into grid-y slices of 65 535 problems and offsets every input and output by the slice's
first problem: test_gpr_batch_past_the_grid_y_limit runs 65 538 problems whose inputs repeat with period 65 535 except
at one second-slice problem, so that a wrong output offset breaks the repetition and a dropped input offset gives that
problem the wrong values."""
import os
import re

import numpy as np
import pytest

from oracle import mfgp_oracle as onp
from tests._grad_oracle import gpr_predict_grad_x
from tests._svgp_grad_oracle import svgp_predict_grad_x
from tests.test_gpr_posterior_sample_gpu import check_against_predict, check_factor, check_oracle, check_samples

gpu = pytest.mark.gpu
CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "multi_fidelity_gpflow_b200", "csrc")


@pytest.fixture(scope="module")
def h():
    from multi_fidelity_gpflow_b200 import _lib

    return _lib.Handle(0)


# ------------------------------------------------------------------------------------ case tables
PS = (1, 3, 7, 8, 9, 33, 63, 64)  # exact-GP outputs; the mean contraction is DFMA below P = 8, DMMA from 8
FAR = 1e3  # far test points sit at +-FAR in every coordinate: every exponent is far below -745


def nt(n):
    return -(-n // 8)


def fill(n):
    """Rows of the last 8-row tile, 1 ... 8."""
    return n - 8 * (nt(n) - 1)


def sweep_d(n):
    """d = 1 in the first and d = 16 in the last fill of every NT, 2 ... 15 in between."""
    f = fill(n)
    return 1 if f == 1 else 16 if f == 8 else 2 + (5 * n) % 14


def common(n):
    """What every table shares: B (or L) >= 3, the 10^k scale, a dead training (inducing) row in every third case, far
    test points in every second one."""
    return dict(d=sweep_d(n), B=3 + (n // 3) % 3, k=n % 7 - 3, dead_train=n % 3 == 1 and n >= 2, far=n % 2 == 0)


def gpr_case(n):
    """Exact-GP predict and predict_grad: every P at every NT (so both mean paths at every NT and P = 64 at NT = 8)."""
    Ns = {21: 4001, 46: 2053}.get(n, 5 + (11 * n) % 53)
    return dict(common(n), N=n, P=PS[(fill(n) - 1 + nt(n)) % 8], Ns=Ns)


def joint_case(n):
    """Joint covariance and samples: every NST at every NT, Ns from 1 to 64; S * P > 256 (JOINT_MIN_COLS) splits the
    sample columns over several CTAs."""
    NST = (fill(n) - 1 + 3 * nt(n)) % 8 + 1
    return dict(common(n), N=n, P=PS[(fill(n) - 1 + nt(n)) % 8], Ns=8 * (NST - 1) + 1 + (3 * n) % 8, S=3 + 2 * (n % 4))


def svgp_case(n):
    """SVGP predict and predict_grad over M: L latents, no W (P = 0), or W with P > L or P < L."""
    c = common(n)
    L = c.pop("B")
    P = (0, L + 3, L - 2)[n % 3]
    Ns = {18: 4001, 43: 2051}.get(n, 5 + (13 * n) % 47)
    return dict(c, M=n, L=L, P=P, Ns=Ns)


GPR_CASES = [gpr_case(n) for n in range(1, 65)]
JOINT_CASES = [joint_case(n) for n in range(1, 65)]
SVGP_CASES = [svgp_case(n) for n in range(1, 65)]


def gpr_id(c):
    return "N{N}-NT{nt}-d{d}-P{P}-Ns{Ns}".format(nt=nt(c["N"]), **c) + ("-S%d" % c["S"] if "S" in c else "")


def svgp_id(c):
    return "M{M}-NT{nt}-d{d}-L{L}-P{P}-Ns{Ns}".format(nt=nt(c["M"]), **c)


def csrc_constants():
    """The limits the tables are built against, read from the sources."""
    small = open(os.path.join(CSRC, "gpr_small.cuh")).read()
    post = open(os.path.join(CSRC, "posterior.cu")).read()
    get = lambda src, pat: int(re.search(pat, src).group(1))
    return dict(max_n=get(small, r"#define MFGP_SMALL_MAX_N (\d+)"), max_d=get(small, r"#define MFGP_SMALL_MAX_D (\d+)"),
                max_p=get(post, r"constexpr int MAX_P = (\d+);"), max_ns=get(post, r"constexpr int JOINT_MAX_NS = (\d+);"),
                min_cols=get(post, r"constexpr long JOINT_MIN_COLS = (\d+);"), dmma_p=get(post, r"if \(P >= (\d+)\) \{"))


def groups_per_cta(Ns, batch, sms=148):
    """csrc/posterior.cu's groups_per_cta on a 148-SM B200: 8-point groups per CTA along grid x."""
    G = -(-Ns // 8)
    return max(1, min(256, G, -(-G * batch // (sms * 8))))


def test_tables_cover_every_instantiation():
    """Per kernel: every NT and every last-tile fill (N = 1 ... 64 each once, so dropping any case fails here), d = 1 and
    d = 16 at every NT, both mean paths at every NT, every NST at every NT, the grid-x splits and the special inputs."""
    k = csrc_constants()
    for cases, key in ((GPR_CASES, "N"), (JOINT_CASES, "N"), (SVGP_CASES, "M")):
        assert sorted(c[key] for c in cases) == list(range(1, k["max_n"] + 1))
        assert {c["d"] for c in cases} == set(range(1, k["max_d"] + 1))
        for t in range(1, nt(k["max_n"]) + 1):
            at = [c for c in cases if nt(c[key]) == t]
            assert {1, k["max_d"]} <= {c["d"] for c in at}, t
        assert min(c.get("B", c.get("L")) for c in cases) >= 3
        assert {c["k"] for c in cases} == set(range(-3, 4))
        assert sum(c["Ns"] % 8 != 0 for c in cases) > len(cases) // 2
        assert any(c["dead_train"] for c in cases) and any(c["far"] and c["Ns"] >= 4 for c in cases)
    for cases in (GPR_CASES, JOINT_CASES):
        assert {c["P"] for c in cases} <= set(PS) and max(c["P"] for c in cases) == k["max_p"]
        for t in range(1, 9):
            ps = {c["P"] for c in cases if nt(c["N"]) == t}
            assert min(ps) < k["dmma_p"] <= max(ps), t
        assert k["max_p"] in {c["P"] for c in cases if nt(c["N"]) == 8}
    for cases in (GPR_CASES, SVGP_CASES):
        assert max(c["Ns"] for c in cases) > 2048
        assert any(groups_per_cta(c["Ns"], c.get("B", c.get("L"))) > 1 for c in cases)
    assert {(nt(c["N"]), nt(c["Ns"])) for c in JOINT_CASES} == {(a, b) for a in range(1, 9) for b in range(1, 9)}
    assert {c["Ns"] for c in JOINT_CASES} == set(range(1, k["max_ns"] + 1))
    assert any(c["S"] * c["P"] > k["min_cols"] for c in JOINT_CASES)
    assert {0} < {c["P"] for c in SVGP_CASES}
    assert any(0 < c["P"] < c["L"] for c in SVGP_CASES) and any(c["P"] > c["L"] for c in SVGP_CASES)


# ------------------------------------------------------------------------------------ problems
def points(rng, n, d):
    return np.hstack([rng.random((n, d)), rng.integers(0, 2, (n, 1)).astype(float)])


def query_points(rng, c, train):
    """Ns points: row 0 on training row 0, rows 1-2 far away (c["far"], Ns >= 4), the last row dead (Ns >= 2)."""
    Ns, d = c["Ns"], c["d"]
    Xs = points(rng, Ns, d)
    Xs[0] = train[0]
    far = []
    if c["far"] and Ns >= 4:
        far = [1, 2]
        Xs[1, :-1], Xs[2, :-1] = FAR, -FAR
    if Ns >= 2:
        Xs[-1, -1] = 0.5
    return Xs, far, [Ns - 1] if Ns >= 2 else []


def gpr_problem(c):
    """Problem b reads Y[:, bP : (b+1)P]; kernel variances, Y and the noise scaled by 10^k (noise >= 1e-4)."""
    rng = np.random.default_rng(1000 * c["N"] + 10 * c["d"] + c["P"])
    N, d, P, B = c["N"], c["d"], c["P"], c["B"]
    s = 10.0 ** c["k"]
    X = points(rng, N, d)
    if c["dead_train"]:
        X[-1, -1] = 0.5
    Y = s * rng.standard_normal((N, B * P))
    th = np.tile(onp.default_theta(d), (B, 1)) * np.exp(0.2 * rng.standard_normal((B, 2 * d + 3)))
    th[:, 1:1 + d] *= np.sqrt(d)  # keep the covariance away from the identity in high d
    th[:, 2 + d:2 + 2 * d] *= np.sqrt(d)
    th[:, [1 + d, 2 + 2 * d]] *= s
    nz = max(1e-2 * s, 1e-4) * (1.0 + rng.random(B))
    Xs, far, dead = query_points(rng, c, X)
    return dict(X=X, Y=Y, th=th, nz=nz, Xs=Xs, far=far, dead=dead, s=s, rng=rng)


def svgp_problem(c):
    """Z with its first coordinate stratified and length-scales shortened as M grows (as tests/test_shape_sweep_gpu.py's
    k7_problem), so that cond(K_l(Z,Z) + jitter I) <= 1e6 over the live inducing points of every latent; the upper
    triangle of q_sqrt is noise that must not be read."""
    rng = np.random.default_rng(1000 * c["M"] + 10 * c["d"] + c["L"])
    M, d, L, P = c["M"], c["d"], c["L"], c["P"]
    s = 10.0 ** c["k"]
    Z = points(rng, M, d)
    Z[:, 0] = (rng.permutation(M) + 0.2 + 0.6 * rng.random(M)) / M
    if c["dead_train"]:
        Z[-1, -1] = 0.5
    th = np.tile(onp.default_theta(d), (L, 1)) * np.exp(0.2 * rng.standard_normal((L, 2 * d + 3)))
    ls = np.sqrt(d) * min(1.0, 0.5 * M ** (-1.0 / d))
    th[:, 1:1 + d] *= ls
    th[:, 2 + d:2 + 2 * d] *= ls
    th[:, [1 + d, 2 + 2 * d]] *= s
    live = np.flatnonzero((Z[:, -1] == 0) | (Z[:, -1] == 1))
    for t in th:
        K = onp.mf_K(Z[live], None, t) + onp.JITTER * np.eye(live.size)
        assert np.linalg.cond(K) <= 1e6
    q_sqrt = np.tile(0.3 * np.eye(M), (L, 1, 1)) + 0.05 * rng.standard_normal((L, M, M))
    W = rng.standard_normal((P, L)) if P else None
    Xs, far, dead = query_points(rng, c, Z)
    return dict(Z=Z, thetas=th, W=W, q_mu=s * rng.standard_normal((M, L)), q_sqrt=q_sqrt, Xs=Xs, far=far, dead=dead)


def svgp_args(pr):
    return pr["Z"], pr["thetas"], pr["W"], pr["q_mu"], pr["q_sqrt"]


def close(got, ref, tol):
    ref = np.asarray(ref)
    np.testing.assert_allclose(got, ref, rtol=tol, atol=tol * max(np.abs(ref).max(), 1e-300))


def route_close(record_property, name, got, ref, scale, tol=4e-12):
    """The second device route: |got - ref| <= tol * scale, the ratio recorded as a test property.  Two kinds of case
    reach 1e-12: d = 1 with length-scales near 0.01 (the expanded square |x/l|^2 + |z/l|^2 - 2 x.z / l^2 of every kernel
    entry, GPflow's form, carries ~eps |x/l|^2 of rounding, and the two routes round it differently), and means that are
    sums of much larger terms of both signs (a = L^-1 y is large where K + noise I is ill-conditioned).  The largest
    seen is 2.3e-12; a dropped tile, k-step or padding term is many orders larger."""
    err = np.abs(np.asarray(got) - np.asarray(ref)).max(initial=0.0) / scale
    record_property(name, float(err))
    assert err <= tol, (name, err, tol)


def k_ss_max(Xs, thetas):
    return max(max(onp.mf_K_diag(Xs, t).max() for t in thetas), 1e-300)


# ------------------------------------------------------------------------------------ exact GP: predict
def blocked_y(pr, P):
    """A Y with 65 columns per problem whose first P are problem b's: P = 65 runs the blocked route."""
    Y, B = pr["Y"], pr["th"].shape[0]
    extra = pr["rng"].standard_normal((Y.shape[0], B, 65 - P))
    return np.concatenate([Y.reshape(Y.shape[0], B, P), extra], axis=2).reshape(Y.shape[0], B * 65)


@gpu
@pytest.mark.parametrize("c", GPR_CASES, ids=gpr_id)
def test_gpr_predict(h, c, record_property):
    pr = gpr_problem(c)
    X, Y, th, nz, Xs, P = pr["X"], pr["Y"], pr["th"], pr["nz"], pr["Xs"], c["P"]
    mean, var = h.gpr_posterior(X, Y, th, nz, P=P).predict(Xs)
    for b in range(c["B"]):
        rm, rv = onp.gpr_predict(X, Y[:, b * P:(b + 1) * P], Xs, th[b], nz[b])
        close(mean[b], rm, 1e-8)
        close(var[b], rv, 1e-8)
    assert np.all(mean[:, pr["dead"]] == 0.0) and np.all(var[:, pr["dead"]] == 0.0)
    for i in pr["far"]:
        assert np.abs(mean[:, i]).max() <= 1e-290
        np.testing.assert_allclose(var[:, i], [onp.mf_K_diag(Xs[i:i + 1], t)[0] for t in th], rtol=1e-14)
    bm, bv = h.gpr_posterior(X, blocked_y(pr, P), th, nz, P=65).predict(Xs)
    route_close(record_property, "route_mean", mean, bm[..., :P], np.abs(bm[..., :P]).max())
    route_close(record_property, "route_var", var, bv, k_ss_max(Xs, th))


# ------------------------------------------------------------------------------------ exact GP: predict_grad
@gpu
@pytest.mark.parametrize("c", GPR_CASES, ids=gpr_id)
def test_gpr_predict_grad(h, c, record_property):
    pr = gpr_problem(c)
    X, Y, th, nz, Xs, P = pr["X"], pr["Y"], pr["th"], pr["nz"], pr["Xs"], c["P"]
    post = h.gpr_posterior(X, Y, th, nz, P=P)
    mean, var, dm, dv = post.predict_grad(Xs)
    pm, pv = post.predict(Xs)
    np.testing.assert_allclose(mean, pm, rtol=1e-13, atol=1e-14 * max(np.abs(pm).max(), 1e-300))
    np.testing.assert_allclose(var, pv, rtol=1e-13, atol=1e-14 * max(np.abs(pv).max(), 1e-300))
    for b in range(c["B"]):
        _, _, rdm, rdv = gpr_predict_grad_x(X, Y[:, b * P:(b + 1) * P], Xs, th[b], nz[b])
        assert np.all(rdm[..., -1] == 0.0) and np.all(rdv[:, -1] == 0.0)  # the fidelity column, which is not returned
        close(dm[b], rdm[..., :-1], 1e-7)
        close(dv[b], rdv[:, :-1], 1e-7)
    assert np.all(dm[:, pr["dead"]] == 0.0) and np.all(dv[:, pr["dead"]] == 0.0)
    if pr["far"]:
        assert np.abs(dm[:, pr["far"]]).max() <= 1e-290 and np.abs(dv[:, pr["far"]]).max() <= 1e-290
    _, _, bdm, bdv = h.gpr_posterior(X, blocked_y(pr, P), th, nz, P=65).predict_grad(Xs)
    route_close(record_property, "route_dmean", dm, bdm[:, :, :P], np.abs(bdm[:, :, :P]).max())
    route_close(record_property, "route_dvar", dv, bdv, np.abs(bdv).max())


# ------------------------------------------------------------------------------------ exact GP: joint
@gpu
@pytest.mark.parametrize("c", JOINT_CASES, ids=gpr_id)
def test_gpr_joint(h, c, record_property):
    pr = gpr_problem(c)
    X, Y, th, nz, Xs, P, Ns = pr["X"], pr["Y"], pr["th"], pr["nz"], pr["Xs"], c["P"], c["Ns"]
    post = h.gpr_posterior(X, Y, th, nz, P=P)
    mean, cov = post.predict_cov(Xs)
    check_oracle(X, Y, Xs, th, nz, P, mean, cov)
    check_against_predict(post, Xs, mean, cov)
    jitter = 1e-6 * pr["s"]  # GPflow's 1e-6 at the scale of the kernel
    check_factor(post, Xs, mean, cov, jitter=jitter)
    check_samples(post, Xs, mean, cov, c["S"], c["N"], jitter=jitter)
    assert np.all(cov[:, pr["dead"], :] == 0.0) and np.all(cov[:, :, pr["dead"]] == 0.0)
    # the blocked route: Ns = 65, whose leading Ns x Ns block is this covariance
    Xb = np.vstack([Xs, points(pr["rng"], 65 - Ns, c["d"])])
    _, c65 = post.predict_cov(Xb)
    route_close(record_property, "route_cov", cov, c65[:, :Ns, :Ns], k_ss_max(Xs, th))


# ------------------------------------------------------------------------------------ SVGP
@gpu
@pytest.mark.parametrize("c", SVGP_CASES, ids=svgp_id)
def test_svgp_predict(h, c, record_property):
    pr = svgp_problem(c)
    Xs = pr["Xs"]
    mean, var = h.svgp_posterior(*svgp_args(pr)).predict(Xs)
    rm, rv = onp.svgp_predict(Xs, pr["Z"], pr["thetas"], pr["q_mu"], np.tril(pr["q_sqrt"]), pr["W"])
    assert mean.shape == rm.shape and var.shape == rv.shape
    close(mean, rm, 1e-8)
    close(var, rv, 1e-8)
    assert np.all(mean[pr["dead"]] == 0.0) and np.all(var[pr["dead"]] == 0.0)
    for i in pr["far"]:
        kss = np.array([onp.mf_K_diag(Xs[i:i + 1], t)[0] for t in pr["thetas"]])
        assert np.abs(mean[i]).max() <= 1e-290
        np.testing.assert_allclose(var[i], kss if pr["W"] is None else (pr["W"] ** 2) @ kss, rtol=1e-14)
    km, kv = h.svgp_predict(Xs, *svgp_args(pr))  # K8: factors on every call and shares no code with the fused kernel
    route_close(record_property, "route_mean", mean, km, np.abs(km).max())
    route_close(record_property, "route_var", var, kv, np.abs(kv).max())


@gpu
@pytest.mark.parametrize("c", SVGP_CASES, ids=svgp_id)
def test_svgp_predict_grad(h, c):
    pr = svgp_problem(c)
    Xs = pr["Xs"]
    post = h.svgp_posterior(*svgp_args(pr))
    mean, var, dm, dv = post.predict_grad(Xs)
    pm, pv = post.predict(Xs)
    np.testing.assert_array_equal(mean, pm)
    np.testing.assert_array_equal(var, pv)
    _, _, rdm, rdv = svgp_predict_grad_x(Xs, pr["Z"], pr["thetas"], pr["q_mu"], np.tril(pr["q_sqrt"]), pr["W"])
    assert np.all(rdm[..., -1] == 0.0) and np.all(rdv[..., -1] == 0.0)  # the fidelity column, which is not returned
    close(dm, rdm[..., :-1], 1e-7)
    close(dv, rdv[..., :-1], 1e-7)
    assert np.all(dm[pr["dead"]] == 0.0) and np.all(dv[pr["dead"]] == 0.0)
    if pr["far"]:
        assert np.abs(dm[pr["far"]]).max() <= 1e-290 and np.abs(dv[pr["far"]]).max() <= 1e-290


# ------------------------------------------------------------------------------------ past the grid-y limit
@gpu
def test_gpr_batch_past_the_grid_y_limit(h):
    """65 538 problems at the HBS shape (N = 53, d = 5: NT = 7) run as two grid-y slices, 0 ... 65 534 and 65 535 ...
    65 537, and the create call factors them in chunks of at most 16 384.  theta, the noise and z repeat with period
    65 535 and Y has 257 columns (257 divides 65 535), except at problem 65 536, whose theta, noise and z are its own.
    Problems 65 535 and 65 537 are then problems 0 and 2 again: every output and both info arrays must repeat bit for
    bit, which checks the output offsets of the second slice.  Problem 65 536 differs from problem 1, so a second slice
    that read the first slice's theta, W, a or z (an input offset dropped) gives problem 1's values there, and the
    oracle and the small call below fail.  (The fused kernels do not read the noise: it is inside W and a.)  Problem 2
    (and so 65 537) has a negative noise: its info is its pivot and its outputs NaN on both sides.  Problems on both
    sides of the split match the oracle and, bit for bit, a call with only their theta.  That call has 1 024 problems:
    K1 builds the covariances of a call with fewer than 1 024 one-tile problems with its tile kernel, which rounds
    differently from its streaming kernel.  W takes 65 538 x 53 x 54 doubles, about 1.5 GB."""
    MAX_GRID_Y = 65535
    B, N, d, ycols, Ns, S = MAX_GRID_Y + 3, 53, 5, 257, 7, 3
    own = MAX_GRID_Y + 1  # the one second-slice problem that is not a copy of a first-slice problem
    rng = np.random.default_rng(65538)
    X = points(rng, N, d)
    Y = rng.standard_normal((N, ycols))
    per = np.arange(B) % MAX_GRID_Y
    th = np.tile(onp.default_theta(d), (MAX_GRID_Y, 1)) * np.exp(0.3 * rng.standard_normal((MAX_GRID_Y, 2 * d + 3)))
    th = th[per]
    nz = (1e-3 * np.exp(0.3 * rng.standard_normal(MAX_GRID_Y)))[per]
    nz[per == 2] = -5.0
    th[own] *= np.exp(0.3 * rng.standard_normal(2 * d + 3))
    nz[own] *= 2.0
    info = np.full(B, -7, dtype=np.int32)
    post = h.gpr_posterior(X, Y, th, nz, info=info)
    assert np.all(info[[2, B - 1]] > 0) and np.count_nonzero(info) == 2
    Xs = points(rng, Ns, d)
    z = rng.standard_normal((MAX_GRID_Y, Ns, S, 1))[per]
    z[own] = rng.standard_normal((Ns, S, 1))
    sinfo = np.full(B, -7, dtype=np.int32)
    outs = list(post.predict(Xs)) + list(post.predict_grad(Xs)) + list(post.predict_cov(Xs))
    outs += [post.sample(Xs, z, info=sinfo), info, sinfo]
    np.testing.assert_array_equal(sinfo[[2, B - 1]], 1)
    assert np.count_nonzero(sinfo) == 2
    bits = lambda a: np.ascontiguousarray(a).view(np.uint64 if a.dtype == np.float64 else np.uint32)
    for a in outs:  # second slice against the first, NaN bits included
        assert np.array_equal(bits(a[[MAX_GRID_Y, B - 1]]), bits(a[[0, 2]]))
    assert np.isnan(outs[0][[2, B - 1]]).all() and np.isfinite(outs[0][[0, 1, MAX_GRID_Y - 1, own]]).all()
    for a in outs[:7]:  # problem 65 536 is not problem 1: the checks below see a dropped input offset
        assert not np.array_equal(a[own], a[1])

    probs = [0, MAX_GRID_Y - 1, MAX_GRID_Y, own]
    mean, var, _, _, dm, dv, cmean, cov = outs[:8]
    for b in probs:
        rm, rv, rdm, rdv = gpr_predict_grad_x(X, Y[:, b % ycols:b % ycols + 1], Xs, th[b], nz[b])
        close(mean[b], rm, 1e-8)
        close(var[b], rv, 1e-8)
        close(dm[b], rdm[..., :-1], 1e-7)
        close(dv[b], rdv[:, :-1], 1e-7)
    check_oracle(X, Y, Xs, th, nz, 1, cmean, cov, probs=probs)
    samples = outs[8]
    for b in probs:
        ref = cmean[b][:, None, :] + np.einsum("ij,jkc->ikc", np.linalg.cholesky(cov[b] + 1e-6 * np.eye(Ns)), z[b])
        np.testing.assert_allclose(samples[b], ref, rtol=1e-10, atol=1e-10 * np.abs(ref).max())
    # the same four problems, repeated to 1 024 so that the factorisation's K1 takes the same (streaming) kernel as above
    rep = np.tile(probs, 256)
    small = h.gpr_posterior(X, np.ascontiguousarray(Y[:, [b % ycols for b in probs]]), th[rep], nz[rep])
    souts = list(small.predict(Xs)) + list(small.predict_grad(Xs)) + list(small.predict_cov(Xs))
    souts.append(small.sample(Xs, np.ascontiguousarray(z[rep])))
    for a, sa in zip(outs, souts):
        assert np.array_equal(bits(a[probs]), bits(sa[:4])) and np.array_equal(bits(sa[:4]), bits(sa[-4:]))


@gpu
def test_svgp_largest_fused_latent_count(h):
    """L = 65 535 latents (the most the fused route and the factorisation's grid y / z take) at M = 8: a few latents on
    both ends against the oracle; L = 65 536 is a bad argument."""
    L, M, d = 65535, 8, 2
    rng = np.random.default_rng(L)
    Z = points(rng, M, d)
    th = np.tile(onp.default_theta(d), (L, 1)) * np.exp(0.3 * rng.standard_normal((L, 2 * d + 3)))
    q_mu = rng.standard_normal((M, L))
    q_sqrt = np.tile(0.3 * np.eye(M), (L, 1, 1)) + 0.05 * np.tril(rng.standard_normal((L, M, M)))
    Xs = points(rng, 9, d)
    post = h.svgp_posterior(Z, th, None, q_mu, q_sqrt)
    mean, var, dm, dv = post.predict_grad(Xs)
    assert mean.shape == (9, L)
    ls = [0, 1, 2, L // 2, L - 2, L - 1]
    rm, rv, rdm, rdv = svgp_predict_grad_x(Xs, Z, th[ls], q_mu[:, ls], q_sqrt[ls])
    close(mean[:, ls], rm, 1e-8)
    close(var[:, ls], rv, 1e-8)
    close(dm[:, ls], rdm[..., :-1], 1e-7)
    close(dv[:, ls], rdv[..., :-1], 1e-7)
    post.close()
    # one more latent: refused by an argument check before anything is launched
    with pytest.raises(ValueError, match="at most 65535"):
        h.svgp_posterior(Z, np.vstack([th, th[:1]]), None, np.hstack([q_mu, q_mu[:, :1]]),
                         np.concatenate([q_sqrt, q_sqrt[:1]]))
