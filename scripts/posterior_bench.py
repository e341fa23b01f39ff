"""Cached exact-GP posterior (mfgp_gpr_posterior_*) against today's per-call prediction.  Writes one JSON document.

  a  HBS, 49 bins at the best restart, Ns = 1 and 10, host buffers: wall time per predict call and creation time,
     against MultiBinMFGP.predict_f (one mfgp_gpr_predict per bin, each factoring again)
  b  HBS, 49 bins x 64 restarts, Ns = 16 384, device buffers: kernel time of the fused route (CUDA events), (problem,
     point) pairs/s, FP64 work N(N+1) + 2N(P+1) flop per pair (assembly / exp not counted) over the live DMMA peak, bytes
     (factors + inputs + outputs) over 6 547.8 GB/s
  c  Goku shared (B = 1, N = 1164, P = 64, Ns = 36 and 4096) and per-bin (B = 64, P = 1, Ns = 36), blocked route, against
     mfgp_gpr_predict (a loop over the bins for the per-bin case)
Every leg asserts parity of a sample against mfgp_gpr_predict (1e-8 relative).  Wall times are medians of >= 200 calls
after a warm-up.  Usage: python scripts/posterior_bench.py [--out profiles/r03_gpr_posterior.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from multi_fidelity_gpflow_b200 import _lib  # noqa: E402
from multi_fidelity_gpflow_b200.data import PowerSpecs  # noqa: E402
from multi_fidelity_gpflow_b200.multibin import MultiBinMFGP  # noqa: E402

HBM_GBS = 6547.8


def load(name):
    ps = PowerSpecs().read_from_npz(os.path.join(ROOT, "tests", "golden", f"{name}.npz"))
    X, Y = ps.training_arrays()
    return X, Y, ps.test_arrays()[0]


def close(got, ref):
    np.testing.assert_allclose(got, ref, rtol=1e-8, atol=1e-8 * np.abs(ref).max())


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


def leg_a(h):
    X, Y, Xt = load("hbs")
    mdl = MultiBinMFGP(X, Y, num_restarts=4, seed=0, handle=h).optimize(max_iters=200, learning_rate=0.02)
    out = {"create_s": wall(lambda: mdl.posterior("best").close(), n=50)[0]}
    post = mdl.posterior("best")
    for ns in (1, 10):
        Xs = np.ascontiguousarray(Xt[:ns])
        pm, pv = post.predict_f(Xs)
        rm, rv = mdl.predict_f(Xs)
        close(pm, rm)
        close(pv, rv)
        cached = wall(lambda: post.predict_f(Xs))
        today = wall(lambda: mdl.predict_f(Xs))
        out[f"Ns{ns}"] = {"posterior_predict_s": cached, "multibin_predict_f_s": today, "speedup": today[0] / cached[0]}
    return out


def leg_b(h, peak):
    import torch

    X, Y, _ = load("hbs")
    R, P, N, d, Ns = 64, 49, X.shape[0], 5, 16384
    B = R * P
    rng = np.random.default_rng(0)
    th = np.exp(0.3 * rng.standard_normal((B, 2 * d + 3)))
    nz = np.full(B, 1e-3)
    t0 = time.perf_counter()
    post = h.gpr_posterior(X, Y, th, nz)
    create_s = time.perf_counter() - t0
    Xs = np.hstack([rng.random((Ns, d)), rng.integers(0, 2, (Ns, 1)).astype(float)])
    dXs = torch.from_numpy(Xs).cuda()
    dm = torch.empty((B, Ns, 1), dtype=torch.float64, device="cuda")
    dv = torch.empty((B, Ns), dtype=torch.float64, device="cuda")
    stream = torch.cuda.current_stream()
    h.set_stream(stream.cuda_stream)
    h.set_async(True)
    try:
        for _ in range(3):
            post.predict(dXs, dm, dv)
        torch.cuda.synchronize()
        reps = 20
        times = []
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(reps):
                post.predict(dXs, dm, dv)
            e1.record(stream)
            e1.synchronize()
            times.append(e0.elapsed_time(e1) / 1e3 / reps)
        assert h.sync() == 0
    finally:
        h.set_async(False)
        h.set_stream(None)
    t = float(np.median(times))
    m, v = dm.cpu().numpy(), dv.cpu().numpy()
    for b in (0, 17, 48, 49 * 31 + 5, B - 1):
        rm, rv = h.gpr_predict(X, np.ascontiguousarray(Y[:, b % P:b % P + 1]), Xs[:256], th[b], nz[b])
        close(m[b, :256], rm)
        close(v[b, :256], rv)
    pairs = B * Ns
    flop = pairs * (N * (N + 1) + 2 * N * (1 + 1))
    nbytes = 8 * (B * (N * (N + 1) // 2 + N) + Ns * (d + 1) + pairs * 2)
    t_flop, t_mem = flop / peak, nbytes / (HBM_GBS * 1e9)
    return {"B": B, "N": N, "P": 1, "Ns": Ns, "create_s": create_s, "kernel_s": t, "kernel_s_runs": times,
            "pairs_per_s": pairs / t, "flop": flop, "flop_per_s": flop / t, "fp64_peak_flop_per_s": peak,
            "share_of_fp64_peak": t_flop / t, "bytes": nbytes, "share_of_hbm": t_mem / t,
            "bound": "FP64 (flop / peak > bytes / bandwidth)" if t_flop > t_mem else "HBM"}


def leg_c(h):
    X, Y, Xt = load("goku")
    d = X.shape[1] - 1
    th = np.ones(2 * d + 3)
    out = {}
    t0 = time.perf_counter()
    post = h.gpr_posterior(X, Y, th[None], np.array([1e-3]), P=64)
    out["shared_create_s"] = time.perf_counter() - t0
    rng = np.random.default_rng(1)
    for ns in (36, 4096):
        Xs = Xt if ns == 36 else np.hstack([rng.random((ns, d)), rng.integers(0, 2, (ns, 1)).astype(float)])
        pm, pv = post.predict(Xs)
        rm, rv = h.gpr_predict(X, Y, Xs, th, 1e-3)
        close(pm[0], rm)
        close(pv[0], rv)
        cached = wall(lambda: post.predict(Xs))
        today = wall(lambda: h.gpr_predict(X, Y, Xs, th, 1e-3))
        out[f"shared_Ns{ns}"] = {"posterior_predict_s": cached, "gpr_predict_s": today, "speedup": today[0] / cached[0]}
    ths = np.tile(th, (64, 1)) * np.exp(0.1 * rng.standard_normal((64, 2 * d + 3)))
    nz = np.full(64, 1e-3)
    t0 = time.perf_counter()
    post = h.gpr_posterior(X, Y, ths, nz)
    out["per_bin_create_s"] = time.perf_counter() - t0
    cols = [np.ascontiguousarray(Y[:, p:p + 1]) for p in range(64)]

    def loop():
        return [h.gpr_predict(X, cols[p], Xt, ths[p], 1e-3) for p in range(64)]

    pm, pv = post.predict(Xt)
    for p, (rm, rv) in enumerate(loop()):
        close(pm[p], rm)
        close(pv[p], rv)
    cached = wall(lambda: post.predict(Xt))
    today = wall(loop, n=200, warm=2)
    out["per_bin_Ns36"] = {"posterior_predict_s": cached, "gpr_predict_loop_s": today, "speedup": today[0] / cached[0]}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON document to this file")
    args = ap.parse_args()
    h = _lib.Handle(0)
    peak = h.fp64_peak(1)
    res = {"gpu": gpu_info(), "fp64_dmma_peak_flop_per_s": peak, "timing": "wall: median, p10, p90 of 200 calls (s)"}
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
