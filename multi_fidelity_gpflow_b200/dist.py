"""One-process-per-GPU partitioning of the hot path (torch.distributed; NCCL on GPUs, gloo in the
CPU tests).  How each sub-path shards (SURVEY 8(e)):

* independent bins / restarts  -> contiguous slices per rank, NO data-path collective
  (`shard_range`, `gather_bins` only to assemble the result vector);
* SVGP minibatch ELBO          -> rows of (X, Y) shard across ranks; every rank evaluates its rows
  with the global scale and kl_mult / world, then ONE all-reduce(sum) of the flat
  [loss, kl, gradients] vector.  `dp_svgp_adam` is the training loop: parameters, Adam moments and the
  flat gradient stay in device memory, the kernels write the gradient pieces straight into the buffer
  NCCL reduces in place, and the host never synchronises inside the loop.  `dp_svgp_value_and_grad` is
  the one-evaluation form for host-driven optimisers (L-BFGS).
"""
from __future__ import annotations

import numpy as np


def shard_range(n: int, rank: int, world: int):
    """Contiguous, balanced [lo, hi) of n items for `rank` (first n % world ranks get one extra)."""
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def _dist():
    import torch.distributed as dist

    return dist


def gather_bins(local: np.ndarray, n_total: int, group=None) -> np.ndarray:
    """All-gather per-rank slices (along axis 0) produced with shard_range back into the full array."""
    import torch

    dist = _dist()
    world = dist.get_world_size(group)
    dev = "cuda" if dist.get_backend(group) == "nccl" else "cpu"
    counts = [shard_range(n_total, r, world) for r in range(world)]
    width = int(np.prod(local.shape[1:])) if local.ndim > 1 else 1
    mx = max(hi - lo for lo, hi in counts)
    buf = torch.zeros(mx * width, dtype=torch.float64, device=dev)
    buf[: local.size] = torch.from_numpy(np.ascontiguousarray(local, dtype=np.float64).ravel()).to(dev)
    outs = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(outs, buf, group=group)
    parts = [o.cpu().numpy()[: (hi - lo) * width].reshape((hi - lo,) + local.shape[1:]) for o, (lo, hi) in zip(outs, counts)]
    return np.concatenate(parts, axis=0)


def dp_svgp_value_and_grad(local_fn, X, Y, num_data, kl_mult=1.0, group=None):
    """Data-parallel SVGP objective.

    local_fn(X_rows, Y_rows, scale, kl_mult) -> dict(elbo, kl, g_* ...) evaluated on this rank's rows
    (mfgp_svgp_elbo_grad through Handle.svgp_elbo_grad).  Returns the same dict for the GLOBAL batch:
    identical (to rounding) on every rank after one all-reduce.
    """
    import torch

    dist = _dist()
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    B = X.shape[0]
    lo, hi = shard_range(B, rank, world)
    scale = float(num_data) / B if num_data is not None else 1.0
    r = local_fn(X[lo:hi], Y[lo:hi], scale, kl_mult / world)
    keys = [k for k in sorted(r) if k.startswith("g_") and r[k] is not None]
    # elbo_r = scale*VE_r - KL  ->  sum_r (elbo_r + KL) - KL
    flat = np.concatenate([[r["elbo"] + r["kl"]]] + [np.ravel(np.asarray(r[k], dtype=np.float64)) for k in keys])
    dev = "cuda" if dist.get_backend(group) == "nccl" else "cpu"
    t = torch.from_numpy(flat).to(dev)
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    flat = t.cpu().numpy()
    out = {"kl": r["kl"], "elbo": float(flat[0]) - r["kl"]}
    o = 1
    for k in keys:
        n = int(np.size(r[k]))
        out[k] = flat[o:o + n].reshape(np.shape(r[k])) if np.ndim(r[k]) else float(flat[o])
        o += n
    for k in r:
        if k.startswith("g_") and r[k] is None:
            out[k] = None
    return out


# ------------------------------------------------------------------------------------------------
# Data-parallel SVGP training loop on device memory (SURVEY 8(e) row 2)
# ------------------------------------------------------------------------------------------------
class SvgpDeviceOps:
    """The three per-step calls of the data-parallel loop through the C-ABI (include/mfgp.h) on torch CUDA tensors.
    The CPU schedule test (tests/test_host_logic.py) substitutes a double with the same three methods."""

    def __init__(self, handle):
        import torch

        from . import _lib

        self.torch, self._lib, self.h, self.L = torch, _lib, handle, _lib._lib
        self.device = torch.device("cuda", torch.cuda.current_device())

    def begin(self):
        self.h.set_stream(self.torch.cuda.current_stream().cuda_stream)  # NCCL's stream: the three calls and the all-reduce are ordered
        self.h.set_async(True)

    def end(self):
        self.torch.cuda.current_stream().synchronize()
        self.h.set_async(False)
        info = self.h.sync()
        self.h.set_stream(None)
        if info:
            raise self._lib.NotPositiveDefiniteError(f"data-parallel SVGP: Cholesky of Kuu failed (pivot {info})")

    def _chk(self, rc, what):
        if rc != 0:
            raise self._lib.MFGPError(f"{what}: rc={rc}: {self.L.mfgp_last_error(self.h._h).decode()}")

    def make_cfg(self, L, M, P, B, d, hetero, scale, kl_mult, lik_lower, masked, lik_per_output, jitter=1e-6):
        return self._lib.SvgpCfg(L, M, P, B, d, int(hetero), float(scale), float(kl_mult), float(jitter), float(lik_lower),
                                 int(masked), int(lik_per_output))

    def constrain(self, cfg, has_W, u, c):
        import ctypes as C

        p = self._lib._ptr
        self._chk(self.L.mfgp_svgp_constrain(self.h._h, C.byref(cfg), int(has_W), p(u), p(c)), "mfgp_svgp_constrain")

    def elbo_grad_flat(self, cfg, X, Y, has_W, c, nranks, eg):
        import ctypes as C

        p = self._lib._ptr
        self._chk(self.L.mfgp_svgp_elbo_grad_flat(self.h._h, C.byref(cfg), p(X), p(Y), int(has_W), p(c), int(nranks), p(eg)),
                  "mfgp_svgp_elbo_grad_flat")

    def gather(self, X, Y, seed, pos0, step, B, lo, Xb, Yb):
        self.h.minibatch_gather(X, Y, seed, pos0, B, lo=lo, count=Xb.shape[0], step=step, Xb=Xb, Yb=Yb)

    def adam_update(self, cfg, has_W, u, m, v, mask, c, eg, lr_t, step, b1, b2, eps, loss_hist, kl_hist, scratch):
        import ctypes as C

        p = self._lib._ptr
        self._chk(self.L.mfgp_svgp_adam_update(self.h._h, C.byref(cfg), int(has_W), p(u), p(m), p(v), p(mask), p(c), p(eg), p(lr_t),
                                               p(step), float(b1), float(b2), float(eps), p(loss_hist), p(kl_hist), p(scratch)),
                  "mfgp_svgp_adam_update")


def dp_svgp_adam(handle_or_ops, X, Y, shape, u, mask, lr_t, beta1, beta2, eps=1e-7, num_data=None, kl_mult=1.0,
                 group=None, timing=None, use_graph=None, minibatch=None):
    """len(lr_t) data-parallel Adam steps.  Every rank passes the same GLOBAL (mini)batch X [B, d+1], Y, the same flat
    unconstrained parameter vector `u` (layout of mfgp_svgp_adam), trainable mask and per-step factors `lr_t`
    (optimizers.adam_step_factors); rank r evaluates rows shard_range(B, r, world).
    minibatch=(B, seed, pos0): X, Y are the whole data set instead, held by every rank, and step t's global batch is the B
    rows at positions pos0 + t B ... of the shuffled stream (include/mfgp.h: minibatch stream); rank r gathers its rows
    shard_range(B, r, world) of it at the start of each step, reading the device step counter (ops.gather), and the ELBO
    scale is num_data / B.

    shape: dict(L, M, P, d, has_W, hetero, masked, lik_per_output, lik_lower).
    Returns (u_final, loss_hist, kl_hist) as NumPy arrays, identical on every rank (same reduced gradient, same update).
    timing (optional dict): receives 'ms_per_step' measured with device events around the steady-state steps (the replayed
    steps when a graph is used, else the whole loop; max over ranks is the caller's job) and 'setup_ms', the wall time of the
    two eager steps + capture + instantiation that a graph costs once per call.
    use_graph (default: on CUDA when there are more than 3 steps): the step -- ~60 kernel launches plus the NCCL all-reduce --
    is launch-latency bound for the reference's model sizes, so after two eager steps ONE step is captured as a CUDA graph
    (the step counter and the per-step factors live on the device, so the same graph serves every step) and replayed."""
    import torch

    dist = _dist()
    ops = handle_or_ops if hasattr(handle_or_ops, "elbo_grad_flat") else SvgpDeviceOps(handle_or_ops)
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    dev = ops.device
    X = np.ascontiguousarray(X, dtype=np.float64)
    Y = np.ascontiguousarray(Y, dtype=np.float64)
    B, d = X.shape[0], X.shape[1] - 1
    if minibatch is not None:
        B, seed, pos0 = minibatch
    if B < world:
        raise ValueError(f"batch of {B} rows cannot be sharded over {world} ranks")
    lo, hi = shard_range(B, rank, world)
    scale = float(num_data) / B if num_data is not None else 1.0
    cfg = ops.make_cfg(shape["L"], shape["M"], shape["P"], hi - lo, d, shape.get("hetero", False), scale, kl_mult,
                       shape.get("lik_lower", 1e-6), shape.get("masked", False), shape.get("lik_per_output", False))
    has_W = bool(shape["has_W"])
    n, nsteps = int(np.size(u)), int(len(lr_t))
    f64 = dict(dtype=torch.float64, device=dev)
    if minibatch is None:
        Xd, Yd = torch.from_numpy(X[lo:hi].copy()).to(dev), torch.from_numpy(Y[lo:hi].copy()).to(dev)
    else:  # the whole data set stays on the device; Xd, Yd receive this rank's rows of each step's batch
        Xall, Yall = torch.from_numpy(X).to(dev), torch.from_numpy(Y).to(dev)
        Xd, Yd = torch.empty((hi - lo, d + 1), **f64), torch.empty((hi - lo, Y.shape[1]), **f64)
    ud = torch.from_numpy(np.ascontiguousarray(u, dtype=np.float64).ravel().copy()).to(dev)
    md, vd, c = torch.zeros(n, **f64), torch.zeros(n, **f64), torch.empty(n, **f64)
    eg = torch.zeros(n + 2, **f64)
    mk = None if mask is None else torch.from_numpy(np.ascontiguousarray(mask, dtype=np.uint8)).to(dev)
    lrd = torch.from_numpy(np.ascontiguousarray(lr_t, dtype=np.float64)).to(dev)
    step = torch.zeros(1, dtype=torch.int32, device=dev)
    loss_h, kl_h, scratch = torch.zeros(nsteps, **f64), torch.zeros(nsteps, **f64), torch.zeros(2, **f64)
    if hasattr(ops, "begin"):
        ops.begin()
    graph = lib_h = None
    try:
        use_events = timing is not None and dev.type == "cuda"
        timed_steps = nsteps
        if use_events:
            import time as _time

            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            dist.barrier(group=group)
            t_setup = _time.perf_counter()
            e0.record()

        def one_step():
            if minibatch is not None:
                ops.gather(Xall, Yall, seed, pos0, step, B, lo, Xd, Yd)
            ops.constrain(cfg, has_W, ud, c)
            ops.elbo_grad_flat(cfg, Xd, Yd, has_W, c, world, eg)
            if world > 1:
                dist.all_reduce(eg, op=dist.ReduceOp.SUM, group=group)  # in place on the buffer the kernels wrote
            ops.adam_update(cfg, has_W, ud, md, vd, mk, c, eg, lrd, step, beta1, beta2, eps, loss_h, kl_h, scratch)

        if use_graph is None:
            use_graph = dev.type == "cuda" and nsteps > 3
        done = 0
        if use_graph:
            lib_h = getattr(ops, "h", None)
            if lib_h is not None:
                lib_h.workspace(lib_h.WS_MEASURE)
            for _ in range(2):  # eager: first-call attribute opt-ins, pool growth, NCCL channel set-up
                one_step()
            if lib_h is not None:
                # the captured step takes its temporaries from one arena allocated here, outside the capture: no allocation
                # nodes in the graph, hence no graph-owned memory left behind (include/mfgp.h: mfgp_workspace)
                lib_h.workspace(lib_h.WS_FIXED)
            graph = torch.cuda.CUDAGraph()
            cur = torch.cuda.current_stream()
            side = torch.cuda.Stream()
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                if hasattr(ops, "h"):
                    ops.h.set_stream(side.cuda_stream)
                with torch.cuda.graph(graph, stream=side, capture_error_mode="relaxed"):
                    one_step()  # recorded, not executed
            cur.wait_stream(side)
            if hasattr(ops, "h"):
                ops.h.set_stream(cur.cuda_stream)
            if use_events:  # steady state = the replayed steps
                torch.cuda.current_stream().synchronize()
                timing["setup_ms"] = (_time.perf_counter() - t_setup) * 1e3
                dist.barrier(group=group)
                e0.record()
                timed_steps = nsteps - 2
            for _ in range(2, nsteps):
                graph.replay()
            done = nsteps
        for _ in range(done, nsteps):
            one_step()
        if use_events:
            e1.record()
    finally:  # the handle leaves async mode / the caller's stream even when a step raises
        if hasattr(ops, "end"):
            ops.end()
        if graph is not None:
            torch.cuda.current_stream().synchronize()
            del graph
        if lib_h is not None:
            lib_h.workspace(lib_h.WS_POOL)
            lib_h.graph_mem_trim()  # nothing to return unless a step outgrew the measured arena
    if use_events:
        timing["ms_per_step"] = e0.elapsed_time(e1) / max(timed_steps, 1)
        timing["graph"] = bool(use_graph)
    return ud.cpu().numpy(), loss_h.cpu().numpy(), kl_h.cpu().numpy()
