"""Input gradients of the cached exact-GP posterior (mfgp_gpr_posterior_predict_grad) against prediction alone and against
the central differences a user needs without them.  Prints one JSON document.

  a  HBS, 49 bins at the best restart, Ns = 1 and 10, host buffers: wall time of MultiBinPosterior.predict_f_grad against
     predict_f and against the 2d + 1 predict_f calls of central differences
  b  HBS, 49 bins x 64 restarts, Ns = 16 384, device buffers: kernel time (CUDA events) of the grad launch and of the
     predict launch in the same run, alternating; (problem, point) pairs/s; counted FP64 work per pair
     2N(N+1) (V, beta) + 2N(P+1) (mean, var) + 4N d (P+1) (the two derivative contractions), exps and differences not
     counted, over the live DMMA peak; bytes (factors + inputs + outputs) over 6 547.8 GB/s
  c  Goku shared (B = 1, N = 1164, P = 64, Ns = 36 and 4096) and per-bin (B = 64, P = 1, Ns = 36), blocked route: wall
     time of predict_grad against predict
Every leg asserts a parity sample against the autograd oracle (rtol 1e-7, atol 1e-7 max|ref|).  Wall times are medians
of >= 200 calls after a warm-up.  Usage: python scripts/posterior_grad_bench.py [--out profiles/r04_gpr_posterior_grad.json]"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from multi_fidelity_gpflow_b200 import _lib  # noqa: E402
from multi_fidelity_gpflow_b200.multibin import MultiBinMFGP  # noqa: E402
from tests._grad_oracle import gpr_predict_grad_x  # noqa: E402
from posterior_bench import HBM_GBS, gpu_info, load, wall  # noqa: E402


def close(got, ref):
    ref = np.asarray(ref)
    np.testing.assert_allclose(got, ref, rtol=1e-7, atol=1e-7 * np.abs(ref).max())


def leg_a(h):
    X, Y, Xt = load("hbs")
    d = X.shape[1] - 1
    mdl = MultiBinMFGP(X, Y, num_restarts=4, seed=0, handle=h).optimize(max_iters=200, learning_rate=0.02)
    post = mdl.posterior("best")
    r = mdl.best_restart()
    out = {}
    for ns in (1, 10):
        Xs = np.ascontiguousarray(Xt[:ns])
        _, _, dm, dv = post.predict_f_grad(Xs)
        for p in (0, 24, 48):
            _, _, rdm, rdv = gpr_predict_grad_x(X, Y[:, p:p + 1], Xs, mdl.thetas[r[p], p], mdl.noise)
            close(dm[:, p], rdm[:, 0])
            close(dv[:, p], rdv)

        def central():
            post.predict_f(Xs)
            for j in range(d):
                for s in (1e-5, -1e-5):
                    x = Xs.copy()
                    x[:, j] += s
                    post.predict_f(x)

        grad = wall(lambda: post.predict_f_grad(Xs))
        pred = wall(lambda: post.predict_f(Xs))
        fd = wall(central)
        out[f"Ns{ns}"] = {"predict_f_grad_s": grad, "predict_f_s": pred, "central_differences_2d_plus_1_predict_f_s": fd,
                          "grad_over_predict": grad[0] / pred[0], "central_differences_over_grad": fd[0] / grad[0]}
    return out


def leg_b(h, peak):
    import torch

    X, Y, _ = load("hbs")
    R, P, N, d, Ns = 64, 49, X.shape[0], 5, 16384
    B = R * P
    rng = np.random.default_rng(0)
    th = np.exp(0.3 * rng.standard_normal((B, 2 * d + 3)))
    nz = np.full(B, 1e-3)
    post = h.gpr_posterior(X, Y, th, nz)
    Xs = np.hstack([rng.random((Ns, d)), rng.integers(0, 2, (Ns, 1)).astype(float)])
    dXs = torch.from_numpy(Xs).cuda()
    f64 = dict(dtype=torch.float64, device="cuda")
    dm, dv = torch.empty((B, Ns, 1), **f64), torch.empty((B, Ns), **f64)
    gdm, gdv = torch.empty((B, Ns, 1, d), **f64), torch.empty((B, Ns, d), **f64)
    stream = torch.cuda.current_stream()
    h.set_stream(stream.cuda_stream)
    h.set_async(True)
    calls = {"grad": lambda: post.predict_grad(dXs, dm, dv, gdm, gdv), "predict": lambda: post.predict(dXs, dm, dv)}
    times = {k: [] for k in calls}
    try:
        for fn in calls.values():
            for _ in range(3):
                fn()
        torch.cuda.synchronize()
        reps = 10
        for _ in range(5):
            for k, fn in calls.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(reps):
                    fn()
                e1.record(stream)
                e1.synchronize()
                times[k].append(e0.elapsed_time(e1) / 1e3 / reps)
        post.predict_grad(dXs, dm, dv, gdm, gdv)
        assert h.sync() == 0
    finally:
        h.set_async(False)
        h.set_stream(None)
    t, tp = float(np.median(times["grad"])), float(np.median(times["predict"]))
    m, v, gm, gv = (a.cpu().numpy() for a in (dm, dv, gdm, gdv))
    for b in (0, 17, 48, 49 * 31 + 5, B - 1):
        rm, rv, rdm, rdv = gpr_predict_grad_x(X, Y[:, b % P:b % P + 1], Xs[:256], th[b], nz[b])
        close(m[b, :256], rm)
        close(v[b, :256], rv)
        close(gm[b, :256], rdm[..., :-1])
        close(gv[b, :256], rdv[:, :-1])
    pairs = B * Ns
    flop = pairs * (2 * N * (N + 1) + 2 * N * (1 + 1) + 4 * N * d * (1 + 1))
    nbytes = 8 * (B * (N * (N + 1) // 2 + N) + Ns * (d + 1) + pairs * (1 + 1) * (1 + d))
    t_flop, t_mem = flop / peak, nbytes / (HBM_GBS * 1e9)
    return {"B": B, "N": N, "d": d, "P": 1, "Ns": Ns, "grad_kernel_s": t, "grad_kernel_s_runs": times["grad"],
            "predict_kernel_s": tp, "predict_kernel_s_runs": times["predict"], "grad_over_predict": t / tp,
            "pairs_per_s": pairs / t, "flop": flop, "flop_per_s": flop / t, "fp64_peak_flop_per_s": peak,
            "share_of_fp64_peak": t_flop / t, "bytes": nbytes, "share_of_hbm": t_mem / t,
            "bound": "FP64 (flop / peak > bytes / bandwidth)" if t_flop > t_mem else "HBM"}


def leg_c(h):
    X, Y, Xt = load("goku")
    d = X.shape[1] - 1
    th = np.ones(2 * d + 3)
    out = {}
    post = h.gpr_posterior(X, Y, th[None], np.array([1e-3]), P=64)
    rng = np.random.default_rng(1)
    for ns in (36, 4096):
        Xs = Xt if ns == 36 else np.hstack([rng.random((ns, d)), rng.integers(0, 2, (ns, 1)).astype(float)])
        _, _, dm, dv = post.predict_grad(Xs)
        _, _, rdm, rdv = gpr_predict_grad_x(X, Y[:, :8], Xs[:36], th, 1e-3)
        close(dm[0, :36, :8], rdm[..., :-1])
        close(dv[0, :36], rdv[:, :-1])
        grad = wall(lambda: post.predict_grad(Xs), n=100)
        pred = wall(lambda: post.predict(Xs), n=100)
        out[f"shared_Ns{ns}"] = {"predict_grad_s": grad, "predict_s": pred, "grad_over_predict": grad[0] / pred[0]}
    ths = np.tile(th, (64, 1)) * np.exp(0.1 * rng.standard_normal((64, 2 * d + 3)))
    post = h.gpr_posterior(X, Y, ths, np.full(64, 1e-3))
    _, _, dm, dv = post.predict_grad(Xt)
    for p in (0, 63):
        _, _, rdm, rdv = gpr_predict_grad_x(X, Y[:, p:p + 1], Xt, ths[p], 1e-3)
        close(dm[p], rdm[..., :-1])
        close(dv[p], rdv[:, :-1])
    grad = wall(lambda: post.predict_grad(Xt), n=100)
    pred = wall(lambda: post.predict(Xt), n=100)
    out["per_bin_Ns36"] = {"predict_grad_s": grad, "predict_s": pred, "grad_over_predict": grad[0] / pred[0]}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON document to this file")
    args = ap.parse_args()
    h = _lib.Handle(0)
    peak = h.fp64_peak(1)
    res = {"gpu": gpu_info(), "gpu_fields": "name, power.limit, clocks.max.sm", "fp64_dmma_peak_flop_per_s": peak,
           "timing": "wall: median, p10, p90 of the calls (s)"}
    res["a_hbs_best"] = leg_a(h)
    res["b_hbs_all_restarts"] = leg_b(h, peak)
    res["c_goku"] = leg_c(h)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
