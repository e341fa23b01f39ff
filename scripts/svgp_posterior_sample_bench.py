"""Joint predictive covariance and posterior samples of the cached SVGP posterior (profiles/r13_svgp_posterior_sample.json).

    python scripts/svgp_posterior_sample_bench.py [--out PATH]

Legs (B200 numbers need the card's name, power limit and max SM clock, recorded under "gpu" in the same run):
  (a) HBS single-bin and latent models, host buffers, Ns = 10, S = 1 000: posterior().predict_f_samples and
      predict_f_full_cov, against the same draws built on the host from the oracle's covariance and numpy's Cholesky;
  (b) HBS single-bin, device buffers, Ns = 64, S = 1 024: _predict_cov and _sample (CUDA events over back-to-back calls),
      bytes over the measured 6 547.8 GB/s, and each kernel's share of _sample from a separate torch.profiler run;
  (c) Goku single-bin (L = P = 64) and latent (L = 15, P = 64), M = 300, on the blocked route: Ns = 36 / 256 and
      S = 16 / 1 024, device buffers.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from multi_fidelity_gpflow_b200 import _lib  # noqa: E402
from multi_fidelity_gpflow_b200.kernels import SquaredExponential  # noqa: E402
from multi_fidelity_gpflow_b200.linear_svgp import LatentMFCoregionalizationSVGP  # noqa: E402
from multi_fidelity_gpflow_b200.singlebin_svgp import SingleBinSVGP  # noqa: E402
from oracle import mfgp_oracle as onp  # noqa: E402
from tests._svgp_joint_oracle import svgp_predict_full_cov  # noqa: E402

HBM_GBS = 6547.8  # measured copy bandwidth of the card (profiles/README.md)


def gpu_info():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,driver_version", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()


def se(d):
    return SquaredExponential(lengthscales=np.ones(d), variance=1.0)


def wall(fn, reps):
    fn()
    t = time.perf_counter()
    for _ in range(reps):
        fn()
    return (time.perf_counter() - t) / reps * 1e3


def events(fn, reps=50):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def hbs_model(h, latent):
    ds = onp.load_dataset("hbs")
    X, Y = ds["X"], ds["Y"]
    if latent:
        m = LatentMFCoregionalizationSVGP(X, Y, se(5), se(5), 10, num_inducing=50, handle=h)
    else:
        m = SingleBinSVGP(X, Y, se(5), se(5), 49, ds["Z_kmeans50"], handle=h)
    rng = np.random.default_rng(1)
    M, L = m.q_mu.shape
    m.q_mu.assign(0.3 * rng.standard_normal((M, L)))
    m.q_sqrt.assign(m.q_sqrt.numpy() + 0.02 * np.tril(rng.standard_normal((L, M, M))))
    return m, ds


def leg_a(h):
    out = {}
    for latent in (False, True):
        m, ds = hbs_model(h, latent)
        Xs = ds["X_test"]
        d = Xs.shape[1] - 1
        post = m.posterior()
        Z, th, W, qm, qs = m.Z.numpy(), m._thetas(d), m._W(), m.q_mu.numpy(), np.tril(m.q_sqrt.numpy())

        def host():
            mean, cov = svgp_predict_full_cov(Xs, Z, th, qm, qs, W)
            z = np.random.default_rng(0).standard_normal((cov.shape[0], Xs.shape[0], 1000))
            f = np.stack([mean[:, p][:, None] + np.linalg.cholesky(cov[p] + 1e-6 * np.eye(Xs.shape[0])) @ z[p]
                          for p in range(cov.shape[0])])
            return np.transpose(f, (2, 1, 0))

        out["latent" if latent else "single_bin"] = {
            "Ns": 10, "S": 1000,
            "predict_f_full_cov_ms": wall(lambda: post.predict_f_full_cov(Xs), 20),
            "predict_f_samples_ms": wall(lambda: post.predict_f_samples(Xs, 1000, seed=0), 20),
            "host_oracle_numpy_samples_ms": wall(host, 3),
        }
        post.close()
    return out


def device_post(h, pr):
    dev = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return h.svgp_posterior(dev(pr["Z"]), dev(pr["thetas"]), dev(pr["W"]), dev(pr["q_mu"]), dev(pr["q_sqrt"]))


def time_joint(h, post, Xs, S):
    P, Ns = post.P, Xs.shape[0]
    dX = torch.from_numpy(Xs).cuda()
    dm = torch.empty((Ns, P), dtype=torch.float64, device="cuda")
    dc = torch.empty((P, Ns, Ns), dtype=torch.float64, device="cuda")
    z = torch.randn((P, Ns, S), dtype=torch.float64, device="cuda")
    ds = torch.empty_like(z)
    h.set_stream(torch.cuda.current_stream().cuda_stream)
    h.set_async(True)
    try:
        t_cov = events(lambda: post.predict_cov(dX, dm, dc))
        t_smp = events(lambda: post.sample(dX, z, samples=ds))
        assert h.sync() == 0
    finally:
        h.set_async(False)
        h.set_stream(None)
    return t_cov, t_smp, (dX, z, ds)


def leg_b(h):
    m, ds = hbs_model(h, False)
    d = 5
    pr = dict(Z=m.Z.numpy(), thetas=m._thetas(d), W=m._W(), q_mu=m.q_mu.numpy(), q_sqrt=np.tril(m.q_sqrt.numpy()))
    post = device_post(h, pr)
    rng = np.random.default_rng(2)
    Xs = np.vstack([ds["X_test"], np.hstack([rng.random((54, d)), rng.integers(0, 2, (54, 1)).astype(float)])])
    Ns, S, P, M, L = 64, 1024, 49, 50, 49
    t_cov, t_smp, (dX, z, dsm) = time_joint(h, post, Xs, S)
    cov_bytes = 8 * (L * M * M * 2 + Ns * P + P * Ns * Ns)
    smp_bytes = 8 * (L * M * M * 2 + 2 * P * Ns * S + 3 * P * Ns * Ns)
    res = {"Ns": Ns, "S": S, "P": P, "predict_cov_ms": t_cov, "sample_ms": t_smp,
           "sample_bytes": smp_bytes, "sample_bytes_over_hbm_ms": smp_bytes / (HBM_GBS * 1e9) * 1e3,
           "sample_share_of_hbm_bound": smp_bytes / (HBM_GBS * 1e9) * 1e3 / t_smp,
           "predict_cov_bytes": cov_bytes}
    h.set_stream(torch.cuda.current_stream().cuda_stream)
    h.set_async(True)
    try:
        for _ in range(3):
            post.sample(dX, z, samples=dsm)
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(20):
                post.sample(dX, z, samples=dsm)
            torch.cuda.synchronize()
        h.sync()
    finally:
        h.set_async(False)
        h.set_stream(None)
    kt = {}
    for e in prof.key_averages():
        if e.device_type == torch.autograd.DeviceType.CUDA and getattr(e, "device_time_total", 0) > 0:
            kt[e.key[:120]] = e.device_time_total / 20 / 1e3
    tot = sum(kt.values())
    res["sample_kernels_ms_per_call"] = dict(sorted(kt.items(), key=lambda kv: -kv[1]))
    res["sample_kernel_share"] = {k: v / tot for k, v in res["sample_kernels_ms_per_call"].items()}
    return res


def leg_c(h):
    ds = onp.load_dataset("goku")
    Xall = np.vstack([ds["X_test"], ds["X"]])
    out = {}
    for latent in (False, True):
        rng = np.random.default_rng(3)
        L, P, M, d = (15, 64, 300, 10) if latent else (64, 64, 300, 10)
        th = np.tile(onp.default_theta(d), (L, 1)) * np.exp(0.2 * rng.standard_normal((L, 2 * d + 3)))
        pr = dict(Z=ds["Z_kmeans300"], thetas=th, W=onp.initialize_W(P, L, 0.4, 0.2) if latent else None,
                  q_mu=0.3 * rng.standard_normal((M, L)),
                  q_sqrt=np.tile(0.1 * np.eye(M), (L, 1, 1)) + 0.02 * np.tril(rng.standard_normal((L, M, M))))
        post = device_post(h, pr)
        rows = []
        for Ns in (36, 256):
            for S in (16, 1024):
                t_cov, t_smp, _ = time_joint(h, post, Xall[:Ns], S)
                rows.append({"Ns": Ns, "S": S, "predict_cov_ms": t_cov, "sample_ms": t_smp})
        out["latent" if latent else "single_bin"] = {"L": L, "P": P, "M": M, "rows": rows}
        post.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r13_svgp_posterior_sample.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: nothing measured")
    h = _lib.Handle(0)
    res = {"gpu": gpu_info(), "torch": torch.__version__}
    res["a_hbs_host"] = leg_a(h)
    res["b_hbs_single_bin_device"] = leg_b(h)
    res["c_goku_blocked_device"] = leg_c(h)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
