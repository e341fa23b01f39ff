"""Joint covariance and posterior samples of the cached exact-GP posterior (mfgp_gpr_posterior_predict_cov,
mfgp_gpr_posterior_sample).  Prints one JSON document.

  a  HBS, 49 bins at the best restart, Ns = 10 (the test set), S = 1000, host buffers: wall time of
     MultiBinPosterior.predict_f_samples against what a user writes without it (three Handle.cov calls per bin, then
     numpy: Cholesky of K + noise I, a triangular solve, Sigma, its Cholesky and mean + L z)
  b  HBS, 49 bins x 64 restarts, Ns = 64, S = 1024, device buffers: kernel time (CUDA events) of _sample, _predict_cov and
     _predict in the same run, alternating.  Bytes (z in, samples out, factors) over 6 547.8 GB/s; FP64 work
     (V = W K_s: Ns N^2, Sigma: Ns^2 N, its factor: Ns^3 / 3, L z: Ns^2 S P) over the live DMMA peak.  The rebuild share
     is the time of _sample with S = 1 (each CTA's Sigma and L and one column) over the time at S = 1024
  c  blocked route: Ns = 65 against Ns = 64 (the route boundary) at HBS size (49 bins, S = 1024, device buffers), and Goku
     shared (B = 1, N = 1164, P = 64) at Ns = 256, S = 16: wall time of _sample and _predict_cov
Every leg asserts a parity sample against the oracle's joint covariance (rtol 1e-8) and the samples against numpy's
Cholesky of the library's covariance (rtol 1e-10).  Usage: python scripts/posterior_sample_bench.py [--out FILE]"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from multi_fidelity_gpflow_b200 import _lib  # noqa: E402
from multi_fidelity_gpflow_b200.multibin import MultiBinMFGP  # noqa: E402
from oracle import mfgp_oracle as onp  # noqa: E402
from tests._joint_oracle import gpr_predict_full_cov  # noqa: E402
from posterior_bench import HBM_GBS, gpu_info, load, wall  # noqa: E402

JITTER = 1e-6


def close_cov(mean, cov, X, y, Xs, th, noise):
    rm, rc = gpr_predict_full_cov(X, y, Xs, th, noise)
    np.testing.assert_allclose(mean, rm, rtol=1e-8, atol=1e-8 * np.abs(rm).max())
    np.testing.assert_allclose(cov, rc, rtol=1e-8, atol=1e-8 * onp.mf_K_diag(Xs, th).max())


def close_samples(s, mean, cov, z):
    """s [Ns, S, P] against mean [Ns, P] + chol(cov + jitter I) z [Ns, S, P]."""
    L = np.linalg.cholesky(cov + JITTER * np.eye(cov.shape[0]))
    ref = mean[:, None, :] + np.einsum("ij,jkc->ikc", L, z)
    np.testing.assert_allclose(s, ref, rtol=1e-10, atol=1e-10 * np.abs(ref).max())


def points(rng, n, d):
    return np.hstack([rng.random((n, d)), rng.integers(0, 2, (n, 1)).astype(float)])


def leg_a(h):
    X, Y, Xt = load("hbs")
    mdl = MultiBinMFGP(X, Y, num_restarts=4, seed=0, handle=h).optimize(max_iters=200, learning_rate=0.02)
    post = mdl.posterior("best")
    Xs = np.ascontiguousarray(Xt[:10])
    r, th, S, P = mdl.best_restart(), mdl.best_thetas(), 1000, 49
    mean, cov = post.predict_f_full_cov(Xs)
    f = post.predict_f_samples(Xs, num_samples=S, seed=0)
    z = np.random.default_rng(0).standard_normal((P, 10, S, 1))
    for p in (0, 24, 48):
        close_cov(mean[:, p], cov[p], X, Y[:, p], Xs, mdl.thetas[r[p], p], mdl.noise)
        close_samples(f[:, :, p].T[:, :, None], mean[:, p:p + 1], cov[p], z[p])

    def by_hand():
        out = np.empty((S, 10, P))
        for p in range(P):
            K = h.cov(X, None, th[p]) + mdl.noise * np.eye(X.shape[0])
            Ks, Kss = h.cov(X, Xs, th[p]), h.cov(Xs, None, th[p])
            L = np.linalg.cholesky(K)
            A = np.linalg.solve(L, Ks)  # numpy has no triangular solve; a user without scipy writes this
            m = A.T @ np.linalg.solve(L, Y[:, p])
            Ls = np.linalg.cholesky(Kss - A.T @ A + JITTER * np.eye(10))
            out[:, :, p] = (m[:, None] + Ls @ z[p, :, :, 0]).T
        return out

    hand = by_hand()
    np.testing.assert_allclose(hand, f, rtol=1e-6, atol=1e-6 * np.abs(f).max())
    lib = wall(lambda: post.predict_f_samples(Xs, num_samples=S, seed=0), n=50)
    user = wall(by_hand, n=10)
    cov_t = wall(lambda: post.predict_f_full_cov(Xs), n=100)
    return {"Ns": 10, "S": S, "P": P, "predict_f_samples_s": lib, "predict_f_full_cov_s": cov_t,
            "by_hand_three_cov_calls_per_bin_plus_numpy_s": user, "by_hand_over_predict_f_samples": user[0] / lib[0]}


def kernel_times(h, calls, reps=10, rounds=5):
    import torch

    stream = torch.cuda.current_stream()
    times = {k: [] for k in calls}
    for fn in calls.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    for _ in range(rounds):
        for k, fn in calls.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(reps):
                fn()
            e1.record(stream)
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1) / 1e3 / reps)
    return {k: (float(np.median(v)), v) for k, v in times.items()}


def device_calls(h, post, Xs, S):
    import torch

    B, Ns, P = post.B, Xs.shape[0], post.P
    f64 = dict(dtype=torch.float64, device="cuda")
    dXs = torch.from_numpy(Xs).cuda()
    z = torch.randn((B, Ns, S, P), generator=torch.Generator(device="cuda").manual_seed(0), **f64)
    z1 = z[:, :, :1].contiguous()
    out, out1 = torch.empty_like(z), torch.empty_like(z1)
    info = torch.zeros(B, dtype=torch.int32, device="cuda")
    dm, dc, dv = torch.empty((B, Ns, P), **f64), torch.empty((B, Ns, Ns), **f64), torch.empty((B, Ns), **f64)
    calls = {"sample": lambda: post.sample(dXs, z, samples=out, info=info),
             "sample_S1": lambda: post.sample(dXs, z1, samples=out1, info=info),
             "predict_cov": lambda: post.predict_cov(dXs, dm, dc),
             "predict": lambda: post.predict(dXs, dm, dv)}
    return calls, z, out, info, dm, dc


def leg_b(h, peak):
    import torch

    X, Y, _ = load("hbs")
    R, P, N, d, Ns, S = 64, 49, X.shape[0], 5, 64, 1024
    B = R * P
    rng = np.random.default_rng(0)
    th = np.exp(0.3 * rng.standard_normal((B, 2 * d + 3)))
    nz = np.full(B, 1e-3)
    post = h.gpr_posterior(X, Y, th, nz)
    Xs = points(rng, Ns, d)
    calls, z, out, info, dm, dc = device_calls(h, post, Xs, S)
    h.set_stream(torch.cuda.current_stream().cuda_stream)
    h.set_async(True)
    try:
        t = kernel_times(h, calls)
        calls["predict_cov"]()
        calls["sample"]()
        assert h.sync() == 0 and not info.any()
    finally:
        h.set_async(False)
        h.set_stream(None)
    m, c, s, zz = dm.cpu().numpy(), dc.cpu().numpy(), out.cpu().numpy(), z.cpu().numpy()
    for b in (0, 17, 48, 49 * 31 + 5, B - 1):
        close_cov(m[b], c[b], X, Y[:, b % P:b % P + 1], Xs, th[b], nz[b])
        close_samples(s[b], m[b], c[b], zz[b])
    ts = t["sample"][0]
    flop = B * (Ns * N * N + Ns * Ns * N + Ns ** 3 / 3 + Ns * Ns * S)
    nbytes = 8 * (2 * B * Ns * S + B * (N * (N + 1) // 2 + N) + Ns * (d + 1))
    t_flop, t_mem = flop / peak, nbytes / (HBM_GBS * 1e9)
    res = {"B": B, "N": N, "d": d, "P": 1, "Ns": Ns, "S": S}
    for k, (med, runs) in t.items():
        res[f"{k}_kernel_s"], res[f"{k}_kernel_s_runs"] = med, runs
    res.update({"samples_per_s": B * Ns * S / ts, "rebuild_share_S1_over_S1024": t["sample_S1"][0] / ts,
                "predict_cov_over_predict": t["predict_cov"][0] / t["predict"][0], "flop": flop, "flop_per_s": flop / ts,
                "fp64_peak_flop_per_s": peak, "share_of_fp64_peak": t_flop / ts, "bytes": nbytes,
                "bytes_per_s": nbytes / ts, "share_of_hbm": t_mem / ts,
                "bound": "FP64 (flop / peak > bytes / bandwidth)" if t_flop > t_mem else "HBM (bytes / bandwidth > flop / peak)"})
    return res


def leg_c(h):
    import torch

    X, Y, _ = load("hbs")
    d = X.shape[1] - 1
    rng = np.random.default_rng(1)
    th = np.exp(0.3 * rng.standard_normal((49, 2 * d + 3)))
    nz = np.full(49, 1e-3)
    post = h.gpr_posterior(X, Y, th, nz)
    Xs65 = points(rng, 65, d)
    out = {}
    for ns in (64, 65):
        Xs = np.ascontiguousarray(Xs65[:ns])
        calls, z, s, info, dm, dc = device_calls(h, post, Xs, 1024)
        h.set_stream(torch.cuda.current_stream().cuda_stream)
        h.set_async(True)
        try:
            t = kernel_times(h, {k: calls[k] for k in ("sample", "predict_cov")})
            calls["predict_cov"]()
            calls["sample"]()
            assert h.sync() == 0
        finally:
            h.set_async(False)
            h.set_stream(None)
        m, c = dm.cpu().numpy(), dc.cpu().numpy()
        for b in (0, 48):
            close_cov(m[b], c[b], X, Y[:, b:b + 1], Xs, th[b], nz[b])
            close_samples(s[b].cpu().numpy(), m[b], c[b], z[b].cpu().numpy())
        out[f"hbs49_Ns{ns}"] = {"route": "fused" if ns <= 64 else "blocked", "sample_S1024_s": t["sample"][0],
                                "predict_cov_s": t["predict_cov"][0]}
    out["blocked_over_fused_sample"] = out["hbs49_Ns65"]["sample_S1024_s"] / out["hbs49_Ns64"]["sample_S1024_s"]

    X, Y, _ = load("goku")
    d = X.shape[1] - 1
    th = np.ones(2 * d + 3)
    post = h.gpr_posterior(X, Y, th[None], np.array([1e-3]), P=64)
    Xs = points(rng, 256, d)
    mean, cov = post.predict_cov(Xs)
    close_cov(mean[0], cov[0], X, Y, Xs, th, 1e-3)
    z = rng.standard_normal((1, 256, 16, 64))
    s = post.sample(Xs, z)
    close_samples(s[0], mean[0], cov[0], z[0])
    out["goku_shared_Ns256_S16"] = {"sample_s": wall(lambda: post.sample(Xs, z), n=50),
                                    "predict_cov_s": wall(lambda: post.predict_cov(Xs), n=50),
                                    "predict_s": wall(lambda: post.predict(Xs), n=50)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON document to this file")
    args = ap.parse_args()
    h = _lib.Handle(0)
    peak = h.fp64_peak(1)
    res = {"gpu": gpu_info(), "gpu_fields": "name, power.limit, clocks.max.sm", "fp64_dmma_peak_flop_per_s": peak,
           "timing": "wall: median, p10, p90 of the calls (s); kernel: median of 5 rounds of 10 launches (s)"}
    res["a_hbs_best"] = leg_a(h)
    res["b_hbs_all_restarts"] = leg_b(h, peak)
    res["c_blocked"] = leg_c(h)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
