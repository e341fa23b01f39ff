"""Natural-gradient steps for the SVGP variational distributions (profiles/r12_svgp_natgrad.json).

    python scripts/svgp_natgrad_bench.py [--out PATH] [--steps N]

Legs (B200 numbers need the card's name, power limit and max SM clock, recorded under "gpu" in the same run):
  * one mfgp_svgp_natgrad call (device tensors, CUDA events over back-to-back calls) at the Goku single-bin
    (L = 64, M = 300), Goku latent (L = 15, M = 300) and HBS single-bin (L = 49, M = 50) shapes;
  * steady-state ms per replayed step, (t(120) - t(20)) / 100 with t(n) the wall time of one optimize_on_device call of n
    steps, of the natgrad + Adam loop against the Adam-only loop, full batch and B = 256;
  * for Goku single-bin and latent: loss against step and against wall time (ms per step x step) for Adam only and for
    natgrad + Adam with gamma = 1 and 0.1, at the learning rate of the minibatch bench (0.005), full batch and B = 256.
"""
import argparse
import copy
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from multi_fidelity_gpflow_b200 import _lib  # noqa: E402
from multi_fidelity_gpflow_b200.kernels import SquaredExponential  # noqa: E402
from multi_fidelity_gpflow_b200.linear_svgp import LatentMFCoregionalizationSVGP  # noqa: E402
from multi_fidelity_gpflow_b200.singlebin_svgp import SingleBinSVGP  # noqa: E402
from oracle import mfgp_oracle as onp  # noqa: E402

LR = 0.005


def gpu_info():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,driver_version", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()


def kern(d):
    return SquaredExponential(lengthscales=np.ones(d)), SquaredExponential(lengthscales=np.ones(d))


def natgrad_call_ms(h, L, M, reps=50):
    """Mean ms of one mfgp_svgp_natgrad on device tensors; the gradients are those of a known small g_S (well posed)."""
    rng = np.random.default_rng(0)
    q_sqrt = np.tril(0.2 / np.sqrt(M) * rng.standard_normal((L, M, M)), -1) + np.eye(M)
    gS = rng.standard_normal((L, M, M)) / np.sqrt(M)
    gS = 0.05 * (gS + gS.transpose(0, 2, 1))
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    qm0, qs0 = dev(rng.standard_normal((M, L))), dev(q_sqrt)
    gm, gs = dev(rng.standard_normal((M, L))), dev(np.tril(2.0 * gS @ q_sqrt))
    info = torch.zeros(L, dtype=torch.int32, device="cuda")
    qm, qs = qm0.clone(), qs0.clone()
    h.set_async(True)
    try:
        for _ in range(3):
            qm.copy_(qm0), qs.copy_(qs0)
            h.svgp_natgrad(qm, qs, gm, gs, 1.0, info=info)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ms = 0.0
        for _ in range(reps):  # the step is in place: restore q (not timed) before every call
            qm.copy_(qm0), qs.copy_(qs0)
            e0.record()
            h.svgp_natgrad(qm, qs, gm, gs, 1.0, info=info)
            e1.record()
            torch.cuda.synchronize()
            ms += e0.elapsed_time(e1)
        h.sync()
    finally:
        h.set_async(False)
    return ms / reps, int(info.cpu().sum())


def run_seconds(model, data, n, B, gamma, reps=3):
    ts, last = [], None
    for _ in range(reps):
        m = copy.deepcopy(model)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        try:
            m.optimize_on_device(data, max_iters=n, initial_lr=LR, minibatch_size=B, natgrad_gamma=gamma)
        except _lib.NotPositiveDefiniteError as e:  # reported with the curve: the step failed for some latents
            m.natgrad_failure = str(e)
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
        last = m
    return min(ts), last


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r12_svgp_natgrad.json"))
    ap.add_argument("--steps", type=int, default=400)
    args = ap.parse_args()
    h = _lib.Handle(0)
    out = {"gpu": gpu_info(), "lr": LR}
    out["natgrad_call_ms"] = {}
    for name, L, M in (("goku_singlebin", 64, 300), ("goku_latent", 15, 300), ("hbs_singlebin", 49, 50)):
        ms, fails = natgrad_call_ms(h, L, M)
        out["natgrad_call_ms"][name] = dict(L=L, M=M, ms=ms, failed_latents=fails)
        print(name, L, M, f"{ms:.3f} ms", flush=True)

    ds = onp.load_dataset("goku")
    X, Y = ds["X"], ds["Y"]
    P = Y.shape[1]
    models = {
        "latent": LatentMFCoregionalizationSVGP(X, Y, *kern(10), num_latents=15, num_inducing=300, num_outputs=P, handle=h),
        "singlebin": SingleBinSVGP(X, Y, *kern(10), P, ds["Z_kmeans300"], handle=h),
    }
    models["singlebin"].num_data = X.shape[0]
    out["step_ms"], out["curves"] = {}, {}
    for name, model in models.items():
        for B in (None, 256):
            for gamma in (None, 1.0, 0.1):
                key = f"{name}/B={B or 'full'}/gamma={gamma}"
                t20, _ = run_seconds(model, (X, Y), 20, B, gamma)
                t120, _ = run_seconds(model, (X, Y), 120, B, gamma)
                ms = (t120 - t20) / 100 * 1e3
                if gamma != 0.1:
                    out["step_ms"][key] = ms
                _, m = run_seconds(model, (X, Y), args.steps, B, gamma, reps=1)
                loss = np.asarray(m.loss_history, dtype=float)
                out["curves"][key] = dict(ms_per_step=ms, loss=loss.tolist(),
                                          wall_s=(np.arange(1, loss.size + 1) * ms * 1e-3).tolist(),
                                          final_loss=float(loss[-1]), min_loss=float(np.nanmin(loss)),
                                          natgrad_failure=getattr(m, "natgrad_failure", None))
                print(key, f"{ms:.3f} ms/step", "final loss", loss[-1], flush=True)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    h.close()


if __name__ == "__main__":
    main()
