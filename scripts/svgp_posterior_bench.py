"""Cached SVGP posterior (mfgp_svgp_posterior_*) against today's per-call prediction (mfgp_svgp_predict, which factors the
inducing covariances on every call).  Prints one JSON document.

  a  HBS single-bin (L = 49) and latent (L = 10, W [49, 10]) models, M = 50, Ns = 1 and 10, host buffers: wall time of
     posterior().predict_f against model.predict_f, and the creation time of posterior()
  b  HBS single-bin at Ns = 262 144, device buffers: kernel time of the fused route (CUDA events) against
     mfgp_svgp_predict at the same size in the same run, alternating; (latent, point) pairs/s and the share of the live
     DMMA peak on 2M(M+1) + 6M flop per pair (V = Wm K_s, U = Lq^T V, three reductions; assembly / exp not counted)
  c  Goku single-bin (L = 64) and latent (L = 15, W [64, 15]), M = 300, Ns = 36 and 4096, host buffers: blocked route
     against mfgp_svgp_predict, and whether the two agree bitwise
Every leg asserts parity of a sample against the oracle (1e-8 relative, atol 1e-8 max|ref|).  Wall times are medians of
>= 200 calls after a warm-up.  Usage: python scripts/svgp_posterior_bench.py [--out profiles/r05_svgp_posterior.json]"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from multi_fidelity_gpflow_b200 import _lib  # noqa: E402
from multi_fidelity_gpflow_b200.kernels import SquaredExponential  # noqa: E402
from multi_fidelity_gpflow_b200.linear_svgp import LatentMFCoregionalizationSVGP  # noqa: E402
from multi_fidelity_gpflow_b200.singlebin_svgp import SingleBinSVGP  # noqa: E402
from oracle import mfgp_oracle as onp  # noqa: E402


def close(got, ref):
    np.testing.assert_allclose(got, ref, rtol=1e-8, atol=1e-8 * np.abs(ref).max())


def check_oracle(Xs, Z, th, W, q_mu, q_sqrt, mean, var):
    rm, rv = onp.svgp_predict(Xs, Z, th, q_mu, q_sqrt, W)
    close(mean, rm)
    close(var, rv)


def wall(fn, n=200, warm=5):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(n):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), float(np.percentile(ts, 10)), float(np.percentile(ts, 90))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def se(d):
    return SquaredExponential(lengthscales=np.ones(d), variance=1.0)


def perturbed(rng, Z, L, d, P, mixing):
    """Trained-looking parameters: theta, q_mu, q_sqrt and W moved off their initial values (tests/test_cuda_svgp.py)."""
    M = Z.shape[0]
    th = np.tile(onp.default_theta(d), (L, 1)) * np.exp(0.2 * rng.standard_normal((L, 2 * d + 3)))
    q_mu = 0.3 * rng.standard_normal((M, L))
    q_sqrt = np.tile(0.1 * np.eye(M), (L, 1, 1)) + 0.02 * np.tril(rng.standard_normal((L, M, M)))
    W = onp.initialize_W(P, L, 0.4, 0.2) + 0.05 * rng.standard_normal((P, L)) if mixing else None
    return th, W, q_mu, q_sqrt


def leg_a(h):
    ds = onp.load_dataset("hbs")
    X, Y, Xt = ds["X"], ds["Y"], ds["X_test"]
    rng = np.random.default_rng(0)
    out = {}
    for name, mdl in (("singlebin_L49", SingleBinSVGP(X, Y, se(5), se(5), 49, ds["Z_kmeans50"], handle=h)),
                      ("latent_L10", LatentMFCoregionalizationSVGP(X, Y, se(5), se(5), 10, num_inducing=50, handle=h))):
        M, L = mdl.q_mu.shape
        mdl.q_mu.assign(0.3 * rng.standard_normal((M, L)))
        mdl.q_sqrt.assign(mdl.q_sqrt.numpy() + 0.02 * np.tril(rng.standard_normal((L, M, M))))
        res = {"create_s": wall(lambda: mdl.posterior().post.close(), n=200)[0]}
        post = mdl.posterior()
        for ns in (1, 10):
            Xs = np.ascontiguousarray(Xt[:ns])
            pm, pv = post.predict_f(Xs)
            rm, rv = mdl.predict_f(Xs)
            close(pm, rm)
            close(pv, rv)
            d = X.shape[1] - 1
            check_oracle(Xs, mdl.Z.numpy(), mdl._thetas(d), mdl._W(), mdl.q_mu.numpy(), mdl.q_sqrt.numpy(), pm, pv)
            cached = wall(lambda: post.predict_f(Xs))
            today = wall(lambda: mdl.predict_f(Xs))
            res[f"Ns{ns}"] = {"posterior_predict_f_s": cached, "model_predict_f_s": today, "speedup": today[0] / cached[0]}
        out[name] = res
    return out


def svgp_predict_device(h, cfg, Xs, Ns, Z, th, W, q_mu, q_sqrt, mean, var):
    P = _lib._ptr
    h._check(_lib._lib.mfgp_svgp_predict(h._h, ctypes.byref(cfg), P(Xs), Ns, P(Z), P(th), P(W), P(q_mu), P(q_sqrt), P(mean),
                                         P(var)), "mfgp_svgp_predict")


def leg_b(h, peak):
    import torch

    ds = onp.load_dataset("hbs")
    Z = ds["Z_kmeans50"]
    L, M, d, Ns = 49, Z.shape[0], 5, 262144
    rng = np.random.default_rng(1)
    th, W, q_mu, q_sqrt = perturbed(rng, Z, L, d, L, False)
    t0 = time.perf_counter()
    post = h.svgp_posterior(Z, th, W, q_mu, q_sqrt)
    create_s = time.perf_counter() - t0
    Xs = np.hstack([rng.random((Ns, d)), rng.integers(0, 2, (Ns, 1)).astype(float)])
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    dXs, dZ, dth, dqm, dqs = dev(Xs), dev(Z), dev(th), dev(q_mu), dev(q_sqrt)
    cfg = _lib.SvgpCfg(L, M, L, Ns, d, 0, 1.0, 1.0, 1e-6, 0.0, 0, 0)
    pm, pv = (torch.empty((Ns, L), dtype=torch.float64, device="cuda") for _ in range(2))
    sm, sv = (torch.empty((Ns, L), dtype=torch.float64, device="cuda") for _ in range(2))
    stream = torch.cuda.current_stream()
    h.set_stream(stream.cuda_stream)
    h.set_async(True)
    cached_fn = lambda: post.predict(dXs, pm, pv)
    today_fn = lambda: svgp_predict_device(h, cfg, dXs, Ns, dZ, dth, None, dqm, dqs, sm, sv)

    def timed(fn, reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1) / 1e3 / reps

    try:
        for _ in range(3):
            cached_fn()
            today_fn()
        torch.cuda.synchronize()
        cached, today = [], []
        for _ in range(5):  # alternating: both see the same clocks and neighbours
            cached.append(timed(cached_fn, 20))
            today.append(timed(today_fn, 5))
        assert h.sync() == 0
    finally:
        h.set_async(False)
        h.set_stream(None)
    t, t0_ = float(np.median(cached)), float(np.median(today))
    m, v = pm.cpu().numpy(), pv.cpu().numpy()
    check_oracle(Xs[:256], Z, th, None, q_mu, q_sqrt, m[:256], v[:256])
    close(m, sm.cpu().numpy())
    close(v, sv.cpu().numpy())
    pairs = L * Ns
    flop = pairs * (2 * M * (M + 1) + 6 * M)
    return {"L": L, "M": M, "Ns": Ns, "create_s": create_s, "fused_kernel_s": t, "fused_kernel_s_runs": cached,
            "svgp_predict_s": t0_, "svgp_predict_s_runs": today, "speedup": t0_ / t, "pairs_per_s": pairs / t,
            "flop": flop, "flop_per_s": flop / t, "fp64_peak_flop_per_s": peak, "share_of_fp64_peak": flop / peak / t}


def leg_c(h):
    ds = onp.load_dataset("goku")
    Z, Xt = ds["Z_kmeans300"], ds["X_test"]
    d = Z.shape[1] - 1
    rng = np.random.default_rng(2)
    out = {}
    for name, L, mixing in (("singlebin_L64", 64, False), ("latent_L15", 15, True)):
        th, W, q_mu, q_sqrt = perturbed(rng, Z, L, d, 64, mixing)
        t0 = time.perf_counter()
        post = h.svgp_posterior(Z, th, W, q_mu, q_sqrt)
        res = {"create_s": time.perf_counter() - t0}
        for ns in (36, 4096):
            Xs = Xt if ns == 36 else np.hstack([rng.random((ns, d)), rng.integers(0, 2, (ns, 1)).astype(float)])
            pm, pv = post.predict(Xs)
            sm, sv = h.svgp_predict(Xs, Z, th, W, q_mu, q_sqrt)
            check_oracle(Xs[:256], Z, th, W, q_mu, q_sqrt, pm[:256], pv[:256])
            close(pm, sm)
            close(pv, sv)
            cached = wall(lambda: post.predict(Xs))
            today = wall(lambda: h.svgp_predict(Xs, Z, th, W, q_mu, q_sqrt))
            res[f"Ns{ns}"] = {"posterior_predict_s": cached, "svgp_predict_s": today, "speedup": today[0] / cached[0],
                              "bitwise_equal_to_svgp_predict": bool(np.array_equal(pm, sm) and np.array_equal(pv, sv))}
        out[name] = res
        post.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON document to this file")
    args = ap.parse_args()
    h = _lib.Handle(0)
    peak = h.fp64_peak(1)
    res = {"gpu": gpu_info(), "fp64_dmma_peak_flop_per_s": peak, "timing": "wall: median, p10, p90 of 200 calls (s)"}
    res["a_hbs"] = leg_a(h)
    res["b_hbs_singlebin_large_ns"] = leg_b(h, peak)
    res["c_goku_blocked"] = leg_c(h)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
