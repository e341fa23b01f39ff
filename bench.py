#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (contract in the task statement).

Workload (BASELINE.json configs[1]): Ho-Bird-Shelton 2021 50LF-3HF multi-bin -- one linear
multi-fidelity GPR per k-bin (49 bins, N = 53, d = 5), NLML + analytic gradient, batched:
one STEP evaluates R independent hyper-parameter sets (restarts, seeded log-normal around the
reference's initial values) for all 49 bins in one launch of the K6 kernel.
metric = "NLML+grad evals/sec across bins", one eval = one full 49-bin NLML+gradient.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

--dump-outputs DIR writes the last timed step's nlml and gradient (rank 0) as DIR/nlml.npy and DIR/grad.npy, so that two
builds can be compared output for output: the inputs depend only on the arguments.

N > 1 (torchrun, one rank per GPU): bins/restarts shard across ranks with no data-path
collective; every rank runs the same per-GPU batch (weak scaling); value = all ranks' evals /
max-over-ranks device time.

Besides the headline line the run measures -- and VERIFIES, every timed result is checked in the
same run -- the other halves of BASELINE's metric and the two communicating multi-GPU paths
(reported under `config`, `roofline_extra` and `multi_gpu`):
  * fp64 Cholesky at N = 16 384 (residual |L L^T - A| / |A| asserted), K(X, X) assembly at N = 32 768;
  * the 32 768-point two-fidelity exact GP (BASELINE config 5): NLML and NLML+gradient, on one GPU
    (world 1) or through the 2-D block-cyclic distributed Cholesky (world > 1, asserted against the
    single-GPU value computed by rank 0 in the same run);
  * one data-parallel SVGP training step on the Goku latent configuration (BASELINE config 4:
    L = 15, M = 300, batch 1164 and 256), rows sharded across ranks, one in-place NCCL all-reduce of the
    flat device gradient (asserted against the one-rank trajectory).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NBINS, NPTS, DIM = 49, 53, 5
METRIC = "NLML+grad evals/sec across bins"
UNIT = "evals/s"
ALG_FLOPS_PER_BIN = NPTS**3 + 4 * NPTS**2  # SURVEY 8(d): gpr_nlml_grad(N, P=1) = N^3 + 4 N^2 P
DATA = "synthetic restarts on the in-repo HBS2021 arrays"


def load_hbs():
    from multi_fidelity_gpflow_b200.data import PowerSpecs

    ps = PowerSpecs().read_from_npz(os.path.join(ROOT, "tests", "golden", "hbs.npz"))
    return ps.training_arrays()


def make_thetas(R, seed):
    rng = np.random.default_rng(seed)
    th = np.exp(0.3 * rng.standard_normal((R * NBINS, 2 * DIM + 3)))
    return np.ascontiguousarray(th), np.full(R * NBINS, 1e-3)


DUMP_ROWS = 1 << 18  # problems kept by --dump-outputs: nlml + grad of 2^18 problems are 31.5 MB of float64


def dump_outputs(out_dir, nlml, grad):
    """nlml [nprob] and grad [nprob, 2d+4] (float64 tensors, as gpr_batched_nlml_grad returns them) -> out_dir/nlml.npy and
    out_dir/grad.npy.  A step of more than DUMP_ROWS problems is cut to a seeded sample of DUMP_ROWS problems in increasing
    order, the same on every run with the same --restarts."""
    import torch

    n = nlml.shape[0]
    if n > DUMP_ROWS:
        idx = np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))
        idx = torch.from_numpy(idx).to(nlml.device)
        nlml, grad = nlml[idx], grad[idx]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "nlml.npy"), nlml.cpu().numpy())
    np.save(os.path.join(out_dir, "grad.npy"), grad.cpu().numpy())


def config(R, extra=None):
    c = {
        "workload": "HBS2021 50LF-3HF multi-bin: 49 per-k-bin linear MF GPRs (N=53, d=5), NLML+grad, "
                    f"R={R} hyper-parameter sets per step in one launch",
        "bins": NBINS, "N": NPTS, "d": DIM, "restarts_per_step": R,
        "l2_policy": "per-step inputs+outputs (theta, noise, nlml, grad) exceed the 126 MB L2",
    }
    if extra:
        c.update(extra)
    return c


# ---------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the CPU oracle (GPflow-equivalent restatement) on all host cores
# ---------------------------------------------------------------------------------------------
def _cpu_worker(args):
    import torch

    torch.set_num_threads(1)
    from oracle import mfgp_oracle_torch as otc

    X, Y, th, nz, lo, hi = args
    acc = 0.0
    for p in range(lo, hi):
        b = p % NBINS
        v, g, gn = otc.gpr_lml_value_and_grad(X, Y[:, b:b + 1], th[p], nz[p])
        acc += v + g.sum() + gn
    return acc


def cpu_evals_per_sec(sample_evals, steps, warmup):
    """Times `steps` passes over a bounded sample of `sample_evals` 49-bin evaluations."""
    import multiprocessing as mp

    X, Y = load_hbs()
    th, nz = make_thetas(sample_evals, 0)
    cores = os.cpu_count() or 1
    nprob = sample_evals * NBINS
    chunks = [(X, Y, th, nz, i * nprob // cores, (i + 1) * nprob // cores) for i in range(cores)]
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        pool.map(_cpu_worker, [(X, Y, th, nz, 0, 1)] * cores)  # import / first-call warm-up in every worker
        for _ in range(warmup):
            pool.map(_cpu_worker, chunks)
        t0 = time.perf_counter()
        for _ in range(steps):
            pool.map(_cpu_worker, chunks)
        dt = time.perf_counter() - t0
    return sample_evals * steps / dt, dt / steps, cores


def cpu_dpotrf_gflops(n=8192):
    """LAPACK dpotrf on the host cores (SciPy), the CPU line for the Cholesky half of the metric (bounded sample: N = 8192)."""
    import scipy.linalg as sla

    rng = np.random.default_rng(0)
    x = rng.standard_normal((n, 64))
    a = x @ x.T
    a[np.diag_indices(n)] += n
    t0 = time.perf_counter()
    sla.cholesky(a, lower=True, overwrite_a=True, check_finite=False)
    return n**3 / 3 / (time.perf_counter() - t0) / 1e9


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample = args.sample_evals
    v, sec, cores = cpu_evals_per_sec(sample, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": DATA,
        "config": config(args.restarts, {
            "cpu_sample_evals_per_step": sample,
            "note": "same workload and per-evaluation metric as the GPU arm; each CPU step is a bounded sample of "
                    f"{sample} of the step's {args.restarts} hyper-parameter sets (x 49 bins), evals/s is a rate so the arms compare"}),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{sample} evals x 49 bins per step, torch-fp64 autograd oracle, one process per core; "
                                   "GPflow/TensorFlow are not installable here, the oracle reproduces their recorded outputs G1-G7"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if args.cpu_potrf:
        line["cpu_baseline"]["dpotrf_n8192_gflops"] = cpu_dpotrf_gflops()
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in ln.split(",")]))

    def mark(self, which):
        setattr(self, which, time.perf_counter())

    def stop(self):
        if self.proc:
            self.proc.terminate()
        # samples taken inside the timed region [t0, t1] (nvidia-smi started before the warm-up so it is already streaming)
        rows = [r for t, r in self.rows if self.t0 is None or (self.t0 <= t <= (self.t1 or t))]
        num = lambda s: s.replace(".", "").isdigit()
        sm = [float(r[0]) for r in rows if r and num(r[0])]
        mx = [float(r[1]) for r in self.rows_all() if len(r) > 1 and num(r[1])]
        pw = [float(r[2]) for r in rows if len(r) > 2 and num(r[2])]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_median": float(np.median(pw)) if pw else None, "reasons": reasons, "samples": len(sm)}

    def rows_all(self):
        return [r for _, r in self.rows]


class Ctx:
    """Per-rank state shared by the measurement legs."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist

        from multi_fidelity_gpflow_b200 import _lib

        self.torch, self.dist, self._lib, self.args = torch, dist, _lib, args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
        torch.cuda.set_device(self.local)
        torch.manual_seed(self.rank)  # the potrf / covariance legs draw their inputs from torch: the same on every run
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.stream = torch.cuda.Stream()
        torch.cuda.set_stream(self.stream)
        self.h = _lib.Handle(self.local)
        self.h.set_stream(self.stream.cuda_stream)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.world == 1:
            return float(x)
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def events(self):
        return self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)

    def raw_gemm(self, ta, tb, m, n, k, alpha, A, B, beta, C):
        L, p = self._lib._lib, self._lib._ptr
        rc = L.mfgp_gemm(self.h._h, b"T" if ta else b"N", b"T" if tb else b"N", m, n, k, float(alpha), p(A), A.stride(0), p(B),
                         B.stride(0), float(beta), p(C), C.stride(0))
        assert rc == 0, L.mfgp_last_error(self.h._h)


# ---------------------------------------------------------------------------------------------
def leg_potrf(cx, peak):
    """Second half of BASELINE's metric: fp64 Cholesky TFLOP/s at N = 16 384, with the factor verified in the run."""
    torch, h = cx.torch, cx.h
    n = 16384
    x = torch.randn(n, 64, dtype=torch.float64, device=cx.dev)
    a = x @ x.T
    a.diagonal().add_(float(n))
    w = torch.empty_like(a)
    h.set_async(True)
    e0, e1 = cx.events()
    best = 1e30
    for rep in range(4):
        w.copy_(a)
        e0.record(cx.stream)
        h.potrf_device(w, n, n)
        e1.record(cx.stream)
        torch.cuda.synchronize()
        if rep:
            best = min(best, e0.elapsed_time(e1) * 1e-3)
    assert h.sync() == 0
    # verify what was timed: relative residual of the factor (the library's own DMMA GEMM forms L L^T - A)
    w.tril_()
    norm_a = float(torch.linalg.matrix_norm(a))
    cx.raw_gemm(False, True, n, n, n, 1.0, w, w, -1.0, a)
    assert h.sync() == 0
    resid = float(torch.linalg.matrix_norm(a)) / norm_a
    assert resid < 1e-13, f"potrf N={n}: |L L^T - A| / |A| = {resid}"
    tf = n**3 / 3 / best / 1e12
    del a, w, x
    return {"kernel": "potrf (diag/panel chain + DMMA trailing updates)", "bound": "tensor", "achieved": tf, "peak": peak / 1e12,
            "unit": "TFLOP/s", "frac": tf * 1e12 / peak, "N": n, "ms": best * 1e3, "residual_rel": resid, "alg_flops": n**3 / 3}


def leg_cov(cx, hbm_peak):
    """K1 covariance assembly, BASELINE config 5 shape (N = 32 768, d = 10): symmetric K(X, X) and a rectangular block."""
    torch, h, L, p = cx.torch, cx.h, cx._lib._lib, cx._lib._ptr
    n, d = 32768, 10
    X = torch.rand(n, d + 1, dtype=torch.float64, device=cx.dev)
    X[:, -1] = (torch.arange(n, device=cx.dev) >= n * 7 // 8).double()
    th = torch.ones(2 * d + 3, dtype=torch.float64, device=cx.dev)
    K = torch.empty(n, n, dtype=torch.float64, device=cx.dev)
    X2 = X.clone()
    h.set_async(True)
    out = []
    for name, x2, n2 in (("symmetric K(X,X)", None, n), ("rectangular K(X,X2)", X2, n)):
        run = lambda: L.mfgp_cov(h._h, p(X), n, None if x2 is None else p(x2), n2, d, p(th), p(K), n)
        for _ in range(2):
            assert run() == 0
        torch.cuda.synchronize()
        e0, e1 = cx.events()
        e0.record(cx.stream)
        for _ in range(5):
            assert run() == 0
        e1.record(cx.stream)
        torch.cuda.synchronize()
        t = e0.elapsed_time(e1) * 1e-3 / 5
        byts = 8.0 * n * n2 + 8.0 * (n + n2) * (d + 1)  # SURVEY 8(d): algorithmic bytes of cov(N, N2, d)
        # spot-check the result that was timed: exact symmetry / zero rows cannot be checked cheaply here, so compare
        # 4096 sampled entries against the closed form evaluated by torch in fp64
        idx = torch.randint(0, n, (4096, 2), device=cx.dev)
        xi, xj = X[idx[:, 0]], (X if x2 is None else x2)[idx[:, 1]]
        r2 = ((xi[:, :d] - xj[:, :d]) ** 2).sum(1)
        hi, hj = xi[:, d], xj[:, d]
        ref = torch.exp(-0.5 * r2) * (1.0 + hi * hj)  # theta = 1: s_i = s_j = 1, delta term on HF x HF pairs
        got = K[idx[:, 0], idx[:, 1]]
        assert float((got - ref).abs().max()) < 1e-12, "cov spot check failed"
        out.append({"kernel": f"cov_stream_kernel {name}", "bound": "hbm", "achieved": byts / t / 1e9, "peak": hbm_peak,
                    "unit": "GB/s", "frac": byts / t / 1e9 / hbm_peak, "N": n, "N2": n2, "d": d, "ms": t * 1e3, "alg_bytes": byts})
    assert h.sync() == 0
    del K, X, X2
    return out


def leg_svgp_step(cx, peak):
    """K7: one training step (ELBO + gradient + Adam on the device) of the Goku single-bin SVGP (BASELINE config 3 shape on
    the Goku arrays: L = P = 64 latents, M = 300, B = 1164), device loop with CUDA-graph replay."""
    from multi_fidelity_gpflow_b200.data import PowerSpecs
    from multi_fidelity_gpflow_b200.kernels import SquaredExponential
    from multi_fidelity_gpflow_b200.singlebin_svgp import SingleBinSVGP

    ps = PowerSpecs().read_from_npz(os.path.join(ROOT, "tests", "golden", "goku.npz"))
    X, Y = ps.training_arrays()
    d, P, M = X.shape[1] - 1, Y.shape[1], 300
    cx.h.set_stream(None)
    cx.h.set_async(False)
    mdl = SingleBinSVGP(X, Y, SquaredExponential(lengthscales=np.ones(d)), SquaredExponential(lengthscales=np.ones(d)), P,
                        ps.extras["Z_kmeans300"], handle=cx.h)
    mdl.optimize_on_device((X, Y), max_iters=3, initial_lr=0.005)
    def call(steps):
        cx.torch.cuda.synchronize()
        t0 = time.perf_counter()
        mdl.optimize_on_device((X, Y), max_iters=steps, initial_lr=0.005)
        assert np.all(np.isfinite(mdl.loss_history)) and mdl.loss_history[-1] < mdl.loss_history[0]
        return time.perf_counter() - t0

    # Every CALL moves the unconstrained parameters and both Adam moments host -> device -> host (3 x 46 MB of q_sqrt for
    # 64 latents, pageable memory), runs its first step eagerly and captures the graph; the replayed step is what training
    # runs thousands of times.  Two call lengths separate the two: step = (t(n2) - t(n1)) / (n2 - n1).
    # Wall-clock calls on a shared host: a descheduled thread adds tens of milliseconds to single calls (seen as 9-95 ms
    # outliers on some boxes), always upwards -- so each length is the MINIMUM of three calls.
    n1, n2 = 20, 120
    t1 = min(call(n1) for _ in range(3))
    t2 = min(call(n2) for _ in range(3))
    dt = (t2 - t1) / (n2 - n1)
    per_call = t1 - n1 * dt
    B = X.shape[0]
    flops = 3.0 * P * (M**3 / 3 + 3.0 * M * M * B)  # SURVEY 8(d): svgp_elbo forward L (M^3/3 + 3 M^2 B), x3 with backward
    cx.h.set_stream(cx.stream.cuda_stream)
    return {"kernel": "SVGP step (K7: batched cov/potrf/trtri + DMMA GEMMs + epilogues, CUDA-graph replay)", "bound": "tensor",
            "achieved": flops / dt / 1e12, "peak": peak / 1e12, "unit": "TFLOP/s", "frac": flops / dt / peak, "L": P, "M": M,
            "B": B, "ms": dt * 1e3, "alg_flops": flops, "timing": f"steady-state replayed step, (t({n2} steps) - t({n1} steps)) / {n2 - n1}, each t the minimum of 3 calls",
            "per_call_ms": per_call * 1e3, "ms_amortised_over_20_steps": t1 / n1 * 1e3}


def leg_goku_per_bin(cx, peak):
    """BASELINE config 2 on the Goku arrays (C2g): one linear MF GPR per k-bin, 64 bins x N = 1164, d = 10, NLML + gradient
    through the batched blocked path (N > 64: K1 -> batched potrf / trtri -> DMMA GEMMs -> K5), host buffers."""
    from multi_fidelity_gpflow_b200.data import PowerSpecs

    ps = PowerSpecs().read_from_npz(os.path.join(ROOT, "tests", "golden", "goku.npz"))
    X, Y = ps.training_arrays()
    N, P = Y.shape
    d = X.shape[1] - 1
    rng = np.random.default_rng(7)
    th = np.exp(0.2 * rng.standard_normal((P, 2 * d + 3)))
    nz = np.full(P, 1e-3)
    h = cx.h
    h.set_stream(None)
    h.set_async(False)
    nl, gr = h.gpr_batched_nlml_grad(X, Y, th, nz)  # warm-up
    ts = []
    for _ in range(9):  # host wall clock per call; the median is robust against a descheduled host thread (see leg_svgp_step)
        t0 = time.perf_counter()
        nl, gr = h.gpr_batched_nlml_grad(X, Y, th, nz)
        ts.append(time.perf_counter() - t0)
    dt = float(np.median(ts))
    # verify bin 0 against the single-problem path (same building blocks, different batching)
    v0, g0 = h.gpr_nlml_grad(X, np.ascontiguousarray(Y[:, :1]), th[0], 1e-3)
    assert abs(v0 - nl[0]) < 1e-10 * abs(v0) and np.max(np.abs(g0 - gr[0])) < 1e-8 * np.max(np.abs(g0))
    flops = P * (float(N) ** 3 + 4.0 * N * N)
    h.set_stream(cx.stream.cuda_stream)
    return {"kernel": "batched exact GPR, 64 bins x N=1164 (K1 + batched potrf/trtri + DMMA GEMMs + K5)", "bound": "tensor",
            "achieved": flops / dt / 1e12, "peak": peak / 1e12, "unit": "TFLOP/s", "frac": flops / dt / peak, "bins": P, "N": N,
            "ms": dt * 1e3, "ms_min": min(ts) * 1e3, "ms_max": max(ts) * 1e3, "timing": "median of 9 C-ABI calls with host buffers",
            "evals_per_s": 1.0 / dt, "alg_flops": flops}


def leg_exact_gp(cx, peak):
    """BASELINE config 5: 32 768-point two-fidelity exact GP, NLML and NLML + gradient.  world 1: the single-GPU path.
    world > 1: 2-D block-cyclic distributed Cholesky (panel broadcasts over NVLink), asserted against rank 0's single-GPU
    value computed in the same run."""
    from multi_fidelity_gpflow_b200.data import synthetic_two_fidelity
    from multi_fidelity_gpflow_b200.dist_chol import distributed_gpr_nlml, process_grid

    torch, h = cx.torch, cx.h
    N = cx.args.exact_n
    X, Y, theta, noise = synthetic_two_fidelity(N)
    h.set_stream(None)
    h.set_async(False)
    out = {"N": N, "d": 10}

    def timed(fn, reps):
        best, val = 1e30, None
        for _ in range(reps):
            cx.barrier()
            t0 = time.perf_counter()
            val = fn()
            torch.cuda.synchronize()
            best = min(best, cx.max_over_ranks(time.perf_counter() - t0))
        return best, val

    single = single_g = None
    if cx.rank == 0:  # the single-GPU answer: the measurement at world 1, the in-run reference at world > 1
        # warm-up at full size, WITH the gradient: the stream-ordered pool grows to the 26 GB working set (K, W, G) once; the
        # value-only call needs K alone
        h.gpr_nlml_grad(X, Y, theta, noise)
        t0 = time.perf_counter()
        single = h.gpr_nlml(X, Y, theta, noise)
        t1 = time.perf_counter()
        sv, single_g = h.gpr_nlml_grad(X, Y, theta, noise)
        t2 = time.perf_counter()
        assert abs(sv - single) < 1e-11 * abs(single)
        out["single_gpu"] = {"nlml_ms": (t1 - t0) * 1e3, "nlml_grad_ms": (t2 - t1) * 1e3,
                             "potrf_flops_tflops": N**3 / 3 / (t1 - t0) / 1e12,
                             "alg_tflops_nlml_grad": (N**3 + 4.0 * N * N) / (t2 - t1) / 1e12,
                             "frac_of_fp64_peak_nlml_grad": (N**3 + 4.0 * N * N) / (t2 - t1) / peak,
                             "note": "host wall time of the C-ABI call with host buffers (H2D of X, Y inside)"}
        torch.cuda.empty_cache()
    if cx.world > 1:
        from multi_fidelity_gpflow_b200.dist_chol import GpuOps

        nb = cx.args.dist_nb
        ops = GpuOps(h)
        ops.stats = {}
        h._dist_ops = ops
        t_v, v = timed(lambda: distributed_gpr_nlml(h, X, Y, theta, noise, nbd=nb), 3)
        t_g, (v2, g2) = timed(lambda: distributed_gpr_nlml(h, X, Y, theta, noise, nbd=nb, want_grad=True), 2)
        ok = True
        if cx.rank == 0:
            ev, eg = abs(v - single) / abs(single), float(np.max(np.abs(g2 - single_g)) / np.max(np.abs(single_g)))
            out["dist_vs_single_gpu"] = {"nlml_rel_err": ev, "grad_rel_err": eg}
            ok = ev < 1e-9 and eg < 1e-7 and abs(v2 - v) <= 1e-12 * abs(v)
        P, Q = process_grid(cx.world)
        out["critical_path_messages"] = ops.stats.get("critical_messages")
        if getattr(ops, "p2p_error", None):
            out["peer_memory_unavailable"] = ops.p2p_error[:200]
        out.update({"grid": [P, Q], "block": nb, "dist_potrf_n32768_ms": t_v * 1e3,
                    "dist_potrf_n32768_tflops": N**3 / 3 / t_v / 1e12,
                    "dist_potrf_n32768_frac_of_N_x_peak": N**3 / 3 / t_v / (cx.world * peak),
                    "dist_nlml_grad_ms": t_g * 1e3, "dist_nlml_grad_alg_tflops": (N**3 + 4.0 * N * N) / t_g / 1e12,
                    "dist_nlml_grad_frac_of_N_x_peak": (N**3 + 4.0 * N * N) / t_g / (cx.world * peak),
                    "timing": "host wall clock around the whole call (assembly + factorisation + solves [+ gradient]) "
                              "bracketed by barrier + synchronize, max over ranks, best of 3 / 2"})
        assert ok, f"distributed exact GP disagrees with the single-GPU path: {out.get('dist_vs_single_gpu')}"
        h._dist_ops = None  # drop the cached multi-GB block columns
        torch.cuda.empty_cache()
    h.set_stream(cx.stream.cuda_stream)
    return out


def leg_dp_svgp(cx):
    """BASELINE config 4 (Goku z=0 latent inference: L = 15, M = 300, W mixing), one data-parallel training step: rows of
    the batch shard across ranks, one in-place all-reduce of the flat device gradient (~0.69 M doubles)."""
    from multi_fidelity_gpflow_b200.data import PowerSpecs
    from multi_fidelity_gpflow_b200.kernels import SquaredExponential
    from multi_fidelity_gpflow_b200.linear_svgp import LatentMFCoregionalizationSVGP

    torch, dist, h = cx.torch, cx.dist, cx.h
    ps = PowerSpecs().read_from_npz(os.path.join(ROOT, "tests", "golden", "goku.npz"))
    X, Y = ps.training_arrays()
    d, P = X.shape[1] - 1, Y.shape[1]
    h.set_stream(None)
    h.set_async(False)
    created = False
    if not dist.is_initialized():  # world 1: a one-rank NCCL group so the same code path (incl. the collective call) runs
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", str(29800 + os.getpid() % 100))
        dist.init_process_group("nccl", rank=0, world_size=1, device_id=cx.dev)
        created = True
    import copy

    base = LatentMFCoregionalizationSVGP(X, Y, SquaredExponential(lengthscales=np.ones(d)), SquaredExponential(lengthscales=np.ones(d)),
                                         num_latents=15, num_inducing=300, num_outputs=P, handle=h)  # num_data = 1164
    mk = lambda: copy.deepcopy(base)
    out = {"L": 15, "M": 300, "P": P,
           "grad_doubles": int(15 * (2 * d + 3) + 300 * (d + 1) + P * 15 + 300 * 15 + 15 * 300 * 300 + 1)}
    steps = 42  # 2 eager + 40 replays of the captured step
    solo = dist.new_group([0]) if cx.world > 1 else None
    for B in (X.shape[0], 256):
        data = (X[:B], Y[:B])
        mk().optimize_data_parallel(data, max_iters=2, initial_lr=0.005)  # warm-up (NCCL channels, pool)
        m = mk()
        t = {}
        m.optimize_data_parallel(data, max_iters=steps, initial_lr=0.005, timing=t)
        out[f"dp_svgp_ms_per_step_B{B}"] = cx.max_over_ranks(t["ms_per_step"])
        out[f"dp_svgp_graph_setup_ms_B{B}"] = t.get("setup_ms")
        assert np.all(np.isfinite(m.loss_history))
        if cx.world > 1 and cx.rank == 0:  # same trajectory as one rank (sub-group of rank 0), checked in the run
            r = mk()
            r.optimize_data_parallel(data, max_iters=steps, initial_lr=0.005, group=solo)
            err = float(np.max(np.abs(np.array(m.loss_history) / np.array(r.loss_history) - 1.0)))
            out[f"dp_svgp_loss_rel_err_vs_one_rank_B{B}"] = err
            assert err < 1e-9, f"data-parallel SVGP trajectory differs from one rank: {err}"
    if created:
        dist.destroy_process_group()
    h.set_stream(cx.stream.cuda_stream)
    return out


# ---------------------------------------------------------------------------------------------
def run_mine(args):
    cx = Ctx(args)
    torch, h, dev, stream, rank, world = cx.torch, cx.h, cx.dev, cx.stream, cx.rank, cx.world

    # CPU baseline first (rank 0, N=1 only), in a separate process so no fork happens after CUDA init
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "0",
                              "--sample-evals", str(4 * args.sample_evals), "--cpu-potrf"], capture_output=True, text=True, cwd=ROOT)
        for ln in out.stdout.splitlines():
            if ln.startswith("{"):
                cpu = json.loads(ln)["cpu_baseline"]

    sampler = ClockSampler(cx.local)
    sampler.start()  # before the warm-up: nvidia-smi needs ~0.5 s to deliver its first sample

    R = args.restarts
    Xh, Yh = load_hbs()
    thh, nzh = make_thetas(R, 1000 + rank)
    nprob = R * NBINS
    X = torch.from_numpy(Xh).to(dev)
    Y = torch.from_numpy(np.ascontiguousarray(Yh)).to(dev)
    th = torch.from_numpy(thh).to(dev)
    nz = torch.from_numpy(nzh).to(dev)
    nlml = torch.empty(nprob, dtype=torch.float64, device=dev)
    grad = torch.empty(nprob, 2 * DIM + 4, dtype=torch.float64, device=dev)
    peak = max(h.fp64_peak(1, 20000), h.fp64_peak(0, 20000))  # measured FP64 pipe peak (DMMA / DFMA microbenchmarks)
    hbm_peak, hbm_src = 6547.8, "fallback 6547.8 GB/s (MEASURED_PEAKS.json absent)"
    try:
        hbm_peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
        hbm_src = "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        pass

    h.set_async(True)

    def step():
        h.gpr_batched_nlml_grad(X, Y, th, nz, nlml=nlml, grad=grad)

    for _ in range(args.warmup):
        step()
    cx.barrier()
    e0, e1 = cx.events()
    sampler.mark("t0")
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    cx.barrier()
    sampler.mark("t1")
    sec = e0.elapsed_time(e1) * 1e-3
    clocks = sampler.stop()
    assert h.sync() == 0
    assert bool(torch.isfinite(nlml).all()) and bool(torch.isfinite(grad).all())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, nlml, grad)
    sec = cx.max_over_ranks(sec)
    value = world * R * args.steps / sec
    kernel_sec = sec / args.steps  # one K6 launch per step
    achieved = ALG_FLOPS_PER_BIN * nprob / kernel_sec

    # e2e: same metric through the public binding with HOST (pinned) buffers, sync on return
    h.set_async(False)
    pin = lambda a: torch.from_numpy(a).pin_memory().numpy()
    Xp, Yp, thp, nzp = pin(Xh), pin(np.ascontiguousarray(Yh)), pin(thh), pin(nzh)
    nlml_h = torch.empty(nprob, dtype=torch.float64).pin_memory().numpy()
    grad_h = torch.empty(nprob, 2 * DIM + 4, dtype=torch.float64).pin_memory().numpy()
    for _ in range(max(1, min(args.warmup, 3))):
        h.gpr_batched_nlml_grad(Xp, Yp, thp, nzp, nlml=nlml_h, grad=grad_h)
    cx.barrier()
    e2e_steps = max(3, args.steps // 2)
    e0.record(stream)
    for _ in range(e2e_steps):
        h.gpr_batched_nlml_grad(Xp, Yp, thp, nzp, nlml=nlml_h, grad=grad_h)
    e1.record(stream)
    cx.barrier()
    e2e_sec = cx.max_over_ranks(e0.elapsed_time(e1) * 1e-3)
    np.testing.assert_allclose(nlml_h, nlml.cpu().numpy(), rtol=1e-12)
    # verify what was timed on a DIFFERENT device code path: a sample of the step's problems re-evaluated with the large-N
    # building blocks (K1 tile kernel -> blocked potrf -> trtri) and three lines of host algebra
    for b in np.arange(0, nprob, max(1, nprob // 8))[:8]:
        K = np.zeros((NPTS, NPTS + 1))
        K[:, :NPTS] = h.cov(Xh, None, thh[b])
        K[np.arange(NPTS), np.arange(NPTS)] += nzh[b]
        Lf, Wf = h.potrf(K, want_inverse=True)
        a = Wf[:, :NPTS] @ Yh[:, b % NBINS]
        v = 0.5 * float(a @ a) + float(np.sum(np.log(np.diag(Lf)))) + 0.5 * NPTS * math.log(2.0 * math.pi)
        assert abs(v - nlml_h[b]) < 1e-9 * abs(v), (b, v, nlml_h[b])
    h2d = Xp.nbytes + Yp.nbytes + thp.nbytes + nzp.nbytes
    d2h = nlml_h.nbytes + grad_h.nbytes + 4
    del th, nz, nlml, grad, thp, nzp, nlml_h, grad_h
    torch.cuda.empty_cache()

    extra, roof_extra, multi = {}, [], {}
    if not args.no_extra:
        if world == 1:
            pr = leg_potrf(cx, peak)
            roof_extra.append(pr)
            extra = {"potrf_n16384_tflops": pr["achieved"], "potrf_n16384_frac_of_fp64_peak": pr["frac"],
                     "potrf_n16384_residual_rel": pr["residual_rel"], "fp64_peak_tflops_measured": peak / 1e12}
            roof_extra.extend(leg_cov(cx, hbm_peak))
            roof_extra.append(leg_svgp_step(cx, peak))
            roof_extra.append(leg_goku_per_bin(cx, peak))
        multi["exact_gp_n32768"] = leg_exact_gp(cx, peak)
        multi["dp_svgp_goku_latent"] = leg_dp_svgp(cx)
        if world > 1:
            eg = multi["exact_gp_n32768"]
            extra.update({k: eg[k] for k in ("dist_potrf_n32768_tflops", "dist_potrf_n32768_frac_of_N_x_peak", "dist_nlml_grad_ms")})
        extra["dp_svgp_ms_per_step"] = multi["dp_svgp_goku_latent"]["dp_svgp_ms_per_step_B1164"]
        extra["dp_svgp_ms_per_step_B256"] = multi["dp_svgp_goku_latent"]["dp_svgp_ms_per_step_B256"]

    if rank == 0:
        traffic, traffic_src = None, None
        tr = os.path.join(ROOT, "profiles", "r02_traffic_gpr_small.json")
        if os.path.exists(tr):
            try:
                tj = json.load(open(tr))
                # per-launch DRAM bytes of the ncu capture, scaled to this run's problems per launch (the kernel streams
                # theta / noise in and nlml / grad out once per problem; the K^L scratch stays in L2)
                traffic = tj["dram_bytes_per_problem"] * nprob
                traffic_src = f"profiles/r02_traffic_gpr_small.json ({tj.get('source')}, git {tj.get('git_head')})"
            except Exception:
                pass
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": sec / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": DATA, "config": config(R, extra),
            "roofline": {"bound": "tensor", "achieved": achieved / 1e12, "peak": peak / 1e12, "unit": "TFLOP/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "gpr_small_v4_kernel<7,5>",  # the only K6 kernel in libmfgp.so (csrc/gpr_small_v4.cu)
                         "peak_source": "measured live: FP64 pipe microbenchmark (DMMA m8n8k4 / DFMA), "
                                        "MEASURED_PEAKS.json has no FP64 entry",
                         "alg_flops_per_bin": ALG_FLOPS_PER_BIN, "alg_io_bytes": nprob * (13 + 1 + 1 + 14) * 8,
                         "hbm_peak_gbs": hbm_peak, "hbm_peak_source": hbm_src},
            "cpu_baseline": cpu,
            "e2e": {"value": world * R * e2e_steps / e2e_sec, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": args.steps, "clocks": clocks,
        }
        if roof_extra:
            line["roofline_extra"] = roof_extra
        if multi:
            line["multi_gpu"] = multi
        print(json.dumps(line), flush=True)
    if world > 1:
        cx.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="mine", choices=["mine", "reference"])
    ap.add_argument("--restarts", type=int, default=98304, help="hyper-parameter sets per step (x49 bins); 98304 = ~0.12 s per step")
    ap.add_argument("--sample-evals", type=int, default=256, help="CPU arm: 49-bin evals per step")
    ap.add_argument("--exact-n", type=int, default=32768, help="size of the BASELINE config-5 exact GP leg")
    ap.add_argument("--dist-nb", type=int, default=1024, help="block size of the distributed Cholesky")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--cpu-potrf", action="store_true", help="reference arm: add the LAPACK dpotrf line")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's nlml / grad to DIR/*.npy")
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs applies to the GPU arm")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_mine(args)


if __name__ == "__main__":
    main()
