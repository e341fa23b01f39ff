"""Minibatch SVGP training in the device loops (profiles/r11_svgp_minibatch.json).

    python scripts/svgp_minibatch_bench.py [--out PATH] [--no-dp]

Legs (B200 numbers need the card's name, power limit and max SM clock, recorded under "gpu"):
  * steady-state ms per replayed step, (t(220) - t(20)) / 200 with t(n) the wall time of one optimize_on_device call of n
    steps (DESIGN §5), for the Goku latent (L = 15, M = 300, P = 64) and Goku single-bin (L = P = 64, num_data set) models at
    B = 1164 (the full-batch loop, and the minibatch loop with B = N), 512, 256 and 64; plus the step's temporaries (the
    arena the captured step takes, measured with mfgp_workspace around one evaluation of B rows);
  * minibatch_gather_kernel alone: CUDA events around back-to-back launches, and its kernel time from torch.profiler;
  * the Goku latent shape on N = 2^20 synthetic rows at B = 1024 (a full-batch loop cannot hold Kuf at this N);
  * the data-parallel minibatch step (dist.dp_svgp_adam, timing['ms_per_step'] of the replayed steps, max over ranks) on
    1, 2 and 8 GPUs, as many as the machine has.
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


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,driver_version", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q


def kern(d):
    return SquaredExponential(lengthscales=np.ones(d)), SquaredExponential(lengthscales=np.ones(d))


def goku_models(X, Y, h):
    ds = onp.load_dataset("goku")
    P = Y.shape[1]
    lat = LatentMFCoregionalizationSVGP(X, Y, *kern(10), num_latents=15, num_inducing=300, num_outputs=P, handle=h)
    sb = SingleBinSVGP(X, Y, *kern(10), P, ds["Z_kmeans300"], handle=h)
    sb.num_data = X.shape[0]
    return {"latent": lat, "singlebin": sb}


def call_seconds(model, data, n, B, reps=3):
    ts = []
    for _ in range(reps):
        m = copy.deepcopy(model)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        m.optimize_on_device(data, max_iters=n, initial_lr=0.005, minibatch_size=B)
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts))


def steady_ms(model, data, B):
    model = copy.deepcopy(model)
    model.optimize_on_device(data, max_iters=3, initial_lr=0.005, minibatch_size=B)  # warm-up: pool, attributes
    model.loss_history, model.kl_history = [], []
    fresh = copy.deepcopy(model)
    t20, t220 = call_seconds(fresh, data, 20, B), call_seconds(fresh, data, 220, B)
    return {"ms_per_step": (t220 - t20) / 200 * 1e3, "t20_s": t20, "t220_s": t220}


def step_bytes(h, model, X, Y, B):
    """Temporaries of one evaluation of B rows: what the captured step's arena holds."""
    d = X.shape[1] - 1
    h.workspace(h.WS_MEASURE)
    try:
        h.svgp_elbo_grad(X[:B], Y[:B], model.Z.numpy(), model._thetas(d), model._W(), model.q_mu.numpy(),
                         np.tril(model.q_sqrt.numpy()), model._lik_var(), scale=1.0)
    finally:
        need = h.workspace(h.WS_POOL)
    return need


def gather_leg(h, N, xcols, ycols, B, launches=2000):
    rng = np.random.default_rng(0)
    X = torch.from_numpy(rng.random((N, xcols))).cuda()
    Y = torch.from_numpy(rng.random((N, ycols))).cuda()
    Xb = torch.empty((B, xcols), dtype=torch.float64, device="cuda")
    Yb = torch.empty((B, ycols), dtype=torch.float64, device="cuda")
    step = torch.zeros(1, dtype=torch.int32, device="cuda")
    h.set_stream(torch.cuda.current_stream().cuda_stream)
    h.set_async(True)
    try:
        for _ in range(50):
            h.minibatch_gather(X, Y, 1, 12345, B, step=step, Xb=Xb, Yb=Yb)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(launches):
            h.minibatch_gather(X, Y, 1, 12345, B, step=step, Xb=Xb, Yb=Yb)
        e1.record()
        torch.cuda.synchronize()
        ev_us = e0.elapsed_time(e1) / launches * 1e3
        from torch.profiler import ProfilerActivity, profile

        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(200):
                h.minibatch_gather(X, Y, 1, 12345, B, step=step, Xb=Xb, Yb=Yb)
            torch.cuda.synchronize()
        kus = [e for e in prof.key_averages() if "minibatch_gather_kernel" in e.key]
        k_us = (kus[0].self_device_time_total / kus[0].count) if kus else None
    finally:
        h.set_async(False)
        h.set_stream(None)
    bytes_moved = 2 * B * (xcols + ycols) * 8  # each gathered double is read once and written once
    return {"N": N, "B": B, "xcols": xcols, "ycols": ycols, "events_us_per_launch": ev_us, "kernel_us": k_us,
            "bytes_read_and_written": bytes_moved,
            "kernel_GB_per_s": (bytes_moved / (k_us * 1e-6) / 1e9) if k_us else None}


DP_WORKER = r'''
import json, os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, %r)
from multi_fidelity_gpflow_b200 import _lib
from multi_fidelity_gpflow_b200.kernels import SquaredExponential
from multi_fidelity_gpflow_b200.linear_svgp import LatentMFCoregionalizationSVGP
from oracle import mfgp_oracle as onp
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
h = _lib.Handle(rank)
ds = onp.load_dataset("goku")
X, Y = ds["X"], ds["Y"]
k = lambda: SquaredExponential(lengthscales=np.ones(10))
res = {}
for B in (1164, 512, 256):
    m = LatentMFCoregionalizationSVGP(X, Y, k(), k(), num_latents=15, num_inducing=300, num_outputs=64, handle=h)
    m.optimize_data_parallel((X, Y), max_iters=5, initial_lr=0.005, minibatch_size=B)
    t = {}
    m.optimize_data_parallel((X, Y), max_iters=225, initial_lr=0.005, minibatch_size=B, timing=t)
    v = torch.tensor([t["ms_per_step"]], dtype=torch.float64, device="cuda")
    dist.all_reduce(v, op=dist.ReduceOp.MAX)
    res[B] = float(v.item())
if rank == 0:
    print("RESULT " + json.dumps(res))
dist.destroy_process_group()
''' % ROOT


def dp_leg(world):
    path = os.path.join(os.environ.get("TMPDIR", "/tmp"), f"svgp_mb_dp_{os.getpid()}.py")
    with open(path, "w") as f:
        f.write(DP_WORKER)
    res = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
                          "--master-addr", "127.0.0.1", "--master-port", str(29650 + world), path],
                         capture_output=True, text=True, timeout=1200)
    os.unlink(path)
    line = [l for l in res.stdout.splitlines() if l.startswith("RESULT ")]
    if res.returncode or not line:
        return {"error": res.stderr[-1500:]}
    return {f"B{k}_ms_per_step": v for k, v in json.loads(line[0][7:]).items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11_svgp_minibatch.json"))
    ap.add_argument("--no-dp", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU and has no CPU mode")
    h = _lib.Handle(0)
    out = {"gpu": gpu_info(), "gpu_fields": "name, power.limit, clocks.max.sm, driver_version",
           "method": "ms_per_step = (t(220) - t(20)) / 200, t(n) = median of 3 wall times of an optimize_on_device call of n "
                     "steps (ends in a device synchronise); step_bytes = mfgp_workspace MEASURE around one evaluation"}
    ds = onp.load_dataset("goku")
    X, Y = ds["X"], ds["Y"]
    models = goku_models(X, Y, h)
    for name, mdl in models.items():
        leg = {}
        base = copy.deepcopy(mdl)
        # the full-batch loop (minibatch_size=None), then the minibatch loop at each B
        for B in (None, 1164, 512, 256, 64):
            r = steady_ms(base, (X, Y), B)
            r["step_bytes"] = step_bytes(h, base, X, Y, B or X.shape[0])
            leg["full_batch_loop" if B is None else f"B{B}"] = r
            print(name, B, r, flush=True)
        out[f"goku_{name}"] = leg
    out["gather"] = [gather_leg(h, 1164, 11, 64, 256), gather_leg(h, 1164, 11, 64, 1164), gather_leg(h, 2**20, 11, 64, 1024)]
    print("gather", out["gather"], flush=True)
    # N = 2^20 synthetic rows in the Goku latent shape; inducing points from KMeans on a 4096-row subsample
    rng = np.random.default_rng(7)
    N = 2**20
    Xs = np.hstack([rng.random((N, 10)), (rng.random((N, 1)) < 0.2).astype(float)])
    Ys = np.sin(3 * Xs[:, :1] + np.linspace(0, 2, 64)[None, :]) + 0.1 * Xs[:, -1:] + 0.01 * rng.standard_normal((N, 64))
    big = LatentMFCoregionalizationSVGP(Xs[:4096], Ys[:4096], *kern(10), num_latents=15, num_inducing=300, num_outputs=64,
                                        handle=h)
    big.num_data = N
    r = steady_ms(big, (Xs, Ys), 1024)
    r["step_bytes"] = step_bytes(h, big, Xs, Ys, 1024)
    r["N"] = N
    r["full_batch_Kuf_bytes"] = 15 * 300 * N * 8
    out["synthetic_2p20_latent_B1024"] = r
    print("2^20", r, flush=True)
    if not a.no_dp:
        n = torch.cuda.device_count()
        out["data_parallel_goku_latent"] = {f"{w}_gpus": (dp_leg(w) if w <= n else "not measured: fewer GPUs")
                                            for w in (1, 2, 8)}
        print("dp", out["data_parallel_goku_latent"], flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
