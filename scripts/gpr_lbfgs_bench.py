"""Device-resident multi-start L-BFGS of the per-bin exact GPs (mfgp_gpr_batched_lbfgs, MultiBinMFGP.optimize_lbfgs) on
HBS, 49 bins x R restarts, R in {1, 8, 64}.  Prints one JSON document (and writes it to --out).

Per R and phase (1: noise fixed, 2: noise trained), with SciPy's default options and maxiter = 1000 as the reference
drives it:
  - wall time of the call (it always synchronises; median of 3 after one warm-up call of the same shape);
  - rounds (lbfgs_step_kernel launches, from torch.profiler in a separate run), the K6 and step-kernel time per round and
    the step kernel's share of a round, and the fraction of K6 work spent on problems that had already finished
    (1 - sum nfev / (B * rounds));
  - nfev / nit percentiles and the status histogram.
Against: 1000 device Adam steps (lr 0.01, MultiBinMFGP.optimize) and their wall time; the final loss per bin at the best
restart of both; the host SciPy loop (MultiFidelityGPModel(X, Y[:, p]).optimize(use_adam=False)) timed on the bins listed
in HOST_BINS and extrapolated to 49 x R.  Usage: python scripts/gpr_lbfgs_bench.py [--out FILE]"""
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
from oracle import mfgp_oracle as onp  # noqa: E402
from posterior_bench import gpu_info  # noqa: E402

# SciPy's loop aborts on some bins when a trial point is not positive definite (GPflow's closure raises); such bins are
# recorded with their error and left out of the extrapolation
HOST_BINS = (1, 17, 30)
MAX_ITERS = 1000


def phase_call(h, X, Y, u, noise, train_noise):
    u, noise = u.copy(), noise.copy()
    info = np.zeros(u.shape[0], dtype=np.int32)
    t0 = time.perf_counter()
    f, nit, nfev, status = h.gpr_batched_lbfgs(X, Y, u, noise, train_noise=train_noise, maxiter=MAX_ITERS, info=info)
    return time.perf_counter() - t0, dict(u=u, noise=noise, f=f, nit=nit, nfev=nfev, status=status, info=info)


def profile_call(h, X, Y, u, noise, train_noise):
    """Kernel count and time by name for one call (torch.profiler, CUDA activities)."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        phase_call(h, X, Y, u, noise, train_noise)
        torch.cuda.synchronize()
    out = {}
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        key = "k6" if "gpr_small_v4_kernel" in ev.name else ("step" if "lbfgs_step_kernel" in ev.name else None)
        if key:
            c, t = out.get(key, (0, 0.0))
            out[key] = (c + 1, t + ev.device_time * 1e-6)
    return out


def stats(r, rounds):
    B = r["nfev"].size
    names = [_lib.LBFGS_STATUS[int(s)] for s in r["status"]]
    pct = lambda a: {f"p{q}": float(np.percentile(a, q)) for q in (0, 50, 90, 100)}
    return {"nfev": pct(r["nfev"]), "nit": pct(r["nit"]), "status": {k: names.count(k) for k in sorted(set(names))},
            "finished_work_fraction": 1.0 - float(r["nfev"].sum()) / (B * rounds)}


def bench_R(h, X, Y, R):
    mdl = MultiBinMFGP(X, Y, num_restarts=R, seed=0, handle=h)
    B = R * 49
    u0, nz0 = mdl.u.copy(), np.full(B, mdl.noise)
    out = {"B": B}
    u, nz = u0, nz0
    for phase, train_noise in ((1, False), (2, True)):
        phase_call(h, X, Y, u, nz, train_noise)  # warm-up of this shape
        ts = []
        for _ in range(3):
            t, r = phase_call(h, X, Y, u, nz, train_noise)
            ts.append(t)
        prof = profile_call(h, X, Y, u, nz, train_noise)
        rounds, k6_s = prof["k6"]
        _, step_s = prof["step"]
        out[f"phase{phase}"] = {"wall_s": float(np.median(ts)), "wall_s_runs": ts, "rounds": rounds,
                                "k6_s_per_round": k6_s / rounds, "step_s_per_round": step_s / rounds,
                                "step_share_of_round": step_s / (k6_s + step_s), **stats(r, rounds)}
        u, nz = r["u"], r["noise"]
    loss = r["f"].reshape(R, 49)
    out["lbfgs_best_loss_per_bin"] = np.nanmin(np.where(np.isfinite(loss), loss, np.nan), axis=0).tolist()
    # the same problems under 1000 device Adam steps (lr 0.01), noise fixed as in phase 1
    adam = MultiBinMFGP(X, Y, num_restarts=R, seed=0, handle=h)
    adam.optimize(max_iters=10, learning_rate=0.01)  # warm-up
    adam = MultiBinMFGP(X, Y, num_restarts=R, seed=0, handle=h)
    t0 = time.perf_counter()
    adam.optimize(max_iters=1000, learning_rate=0.01)
    out["adam_1000_wall_s"] = time.perf_counter() - t0
    al = adam.training_loss()
    out["adam_best_loss_per_bin"] = np.nanmin(np.where(np.isfinite(al), al, np.nan), axis=0).tolist()
    return out


def phase1_best(h, X, Y, R):
    """Best-restart loss per bin after phase 1 only (the objective Adam optimises)."""
    mdl = MultiBinMFGP(X, Y, num_restarts=R, seed=0, handle=h)
    _, r = phase_call(h, X, Y, mdl.u, np.full(R * 49, mdl.noise), False)
    loss = r["f"].reshape(R, 49)
    return np.nanmin(np.where(np.isfinite(loss), loss, np.nan), axis=0)


def host_scipy(X, Y):
    from multi_fidelity_gpflow_b200.kernels import SquaredExponential
    from multi_fidelity_gpflow_b200.linear import MultiFidelityGPModel

    se = lambda: SquaredExponential(lengthscales=np.ones(5), variance=1.0)
    out = {}
    for p in HOST_BINS:
        m = MultiFidelityGPModel(X, np.ascontiguousarray(Y[:, p:p + 1]), se(), se())
        t0 = time.perf_counter()
        try:
            m.optimize(max_iters=MAX_ITERS, use_adam=False, verbose=False)
            out[str(p)] = {"wall_s": time.perf_counter() - t0, "loss": m.training_loss()}
        except np.linalg.LinAlgError as e:
            out[str(p)] = {"wall_s": time.perf_counter() - t0, "error": str(e)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    args = ap.parse_args()
    h = _lib.default_handle()
    ds = onp.load_dataset("hbs")
    X, Y = ds["X"], np.ascontiguousarray(ds["Y"])
    doc = {"gpu": gpu_info(), "workload": "HBS 50LF-3HF, N = 53, d = 5, 49 bins x R restarts, maxiter = 1000 per phase",
           "host_bins": list(HOST_BINS)}
    host = host_scipy(X, Y)
    ok = [v["wall_s"] for v in host.values() if "error" not in v]
    doc["host_scipy"] = host
    for R in (1, 8, 64):
        res = bench_R(h, X, Y, R)
        res["lbfgs_phase1_best_loss_per_bin"] = phase1_best(h, X, Y, R).tolist()
        res["host_scipy_extrapolated_s"] = float(np.mean(ok)) * 49 * R if ok else None
        doc[f"R{R}"] = res
        print(json.dumps({f"R{R}": {k: res[k] for k in ("B", "phase1", "phase2", "adam_1000_wall_s")}}), flush=True)
    text = json.dumps(doc, indent=1)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
