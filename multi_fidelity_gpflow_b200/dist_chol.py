"""Distributed exact-GP NLML for ONE large problem across the GPUs of a box (SURVEY 8(e), row 3; BASELINE config 5).

Layout: 2-D block-cyclic.  The N x N covariance is cut into nb x nb blocks; block (i, j), i >= j, lives on the rank
at grid position (i mod P, j mod Q) of a P x Q process grid (8 GPUs: 2 x 4).  Every rank assembles its own blocks from
the replicated inputs with the fused covariance kernel (no communication), then the right-looking Cholesky runs

    step k   diag owner        : L_kk, W_kk = L_kk^-1            (mfgp_potrf_inv)        -> broadcast W_kk
             column k mod Q    : L_ik = A_ik W_kk^T  (local rows) (mfgp_gemm, DMMA)       -> P panel broadcasts (NVLink)
             everyone          : A_ij -= L_ik L_jk^T for the local blocks i >= j > k      (mfgp_gemm, DMMA)
             everyone          : a_k = W_kk y_k ; y[k+1:] -= L[k+1:, k] a_k               (replicated, O(N nb))

with LOOK-AHEAD on three CUDA streams: the CRITICAL stream factors the diagonal block, broadcasts its inverse, solves
and broadcasts only the single block (k+1, k) and completes the next diagonal block, so potrf(k+1) starts ~0.3 ms after
potrf(k) ends; the PANEL stream solves and broadcasts the bulk of panel k and updates block column k+1; the MAIN stream
applies panel k to the rest of the trailing matrix.  NLML = 1/2 |a|^2 + sum log L_ii + N/2 log 2 pi  (GPflow GPR.log_marginal_likelihood,
reference call sites mfgpflow/linear.py:206,227).  P = 1 gives the 1-D block-cyclic column layout of round 1.

All device arithmetic goes through libmfgp.so (`GpuOps`); torch supplies buffers, streams and NCCL.  The block
operations are behind a four-method interface so that the schedule (ownership, broadcasts, look-ahead ordering) is
also exercised on CPU by a world-size-2/4 gloo test with a NumPy double (tests/test_dist_chol_cpu.py) -- that double
lives in tests/, the product path has no CPU fallback."""
from __future__ import annotations

import math

import numpy as np


def process_grid(world: int) -> tuple[int, int]:
    """P x Q with P <= Q, both as close to sqrt(world) as the factorisation allows (8 -> 2 x 4, 4 -> 2 x 2, 2 -> 1 x 2)."""
    p = int(math.isqrt(world))
    while world % p:
        p -= 1
    return p, world // p


class GpuOps:
    """Block operations on torch CUDA tensors through the C-ABI (include/mfgp.h)."""

    def __init__(self, handle):
        import torch

        from . import _lib

        self.torch, self._lib, self.h = torch, _lib, handle
        self.L = _lib._lib
        self.device = torch.device("cuda", torch.cuda.current_device())

    def begin(self):
        self.h.set_async(True)  # library calls only enqueue; finish() collects the status

    def _chk(self, rc, what):
        if rc != 0:
            raise self._lib.MFGPError(f"{what}: rc={rc}: {self.L.mfgp_last_error(self.h._h).decode()}")

    @staticmethod
    def _vptr(t):
        """Address of a row-major VIEW (unit column stride; the row stride is passed as the leading dimension)."""
        import ctypes

        if t.dim() == 2 and t.stride(1) != 1:
            raise ValueError("matrix views must have unit column stride")
        return ctypes.c_void_p(t.data_ptr())

    # -- streams ---------------------------------------------------------------------------------------
    def new_stream(self, high_priority=False):
        # the panel stream is high priority: its small GEMMs / potrf must not queue behind the trailing update's CTAs
        return self.torch.cuda.Stream(priority=-1 if high_priority else 0)

    def use(self, stream):
        """Context manager: torch's current stream AND the library's stream."""
        ops = self

        class _Ctx:
            def __enter__(self_inner):
                self_inner.ctx = ops.torch.cuda.stream(stream)
                self_inner.ctx.__enter__()
                ops.h.set_stream(stream.cuda_stream)

            def __exit__(self_inner, *exc):
                return self_inner.ctx.__exit__(*exc)

        return _Ctx()

    timeline = None  # set to a dict to get a device timeline of the schedule: {label: ms since the first recorded event}

    def record(self, stream, label=None):
        timed = self.timeline is not None and label is not None
        ev = self.torch.cuda.Event(enable_timing=timed)
        ev.record(stream)
        if timed:
            self.timeline.setdefault("_events", []).append((label, ev))
        return ev

    def timeline_ms(self):
        """After finish(): {label: milliseconds after the first labelled event} for one call (diagnostics only)."""
        evs = (self.timeline or {}).pop("_events", [])
        if not evs:
            return {}
        t0 = evs[0][1]
        return {lab: t0.elapsed_time(e) for lab, e in evs}

    def wait(self, stream, event):
        if event is not None:
            stream.wait_event(event)

    def finish(self):
        self.torch.cuda.synchronize()
        self.h.set_async(False)
        info = self.h.sync()
        self.h.set_stream(None)
        if info:
            raise self._lib.NotPositiveDefiniteError(f"distributed potrf: pivot {info} of a diagonal block not positive")

    # -- NVLink peer memory for the critical-path messages --------------------------------------------------
    def peer_buffers(self, count, nb, group):
        """`count` symmetric nb x nb blocks (torch symmetric memory: every rank's allocation is mapped into every peer
        over NVLink).  Returns (local [count, nb, nb], handle, [peer views]) or None when peer memory is unavailable."""
        try:
            import torch.distributed as dist
            import torch.distributed._symmetric_memory as symm

            pg = group if group is not None else dist.group.WORLD
            local = symm.empty((count, nb, nb), dtype=self.torch.float64, device=self.device)
            hdl = symm.rendezvous(local, pg)
            world = dist.get_world_size(pg)
            peers = [hdl.get_buffer(r, (count, nb, nb), self.torch.float64) for r in range(world)]
            return local, hdl, peers
        except Exception as e:  # no P2P / unsupported build: the NCCL broadcasts remain (reported, not silent)
            self.p2p_error = repr(e)
            return None

    def peer_publish(self, hdl, peers, local_block, k, me, channel):
        """Owner side: store block k into every peer's copy with direct NVLink writes (ONE kernel of the library for up to
        8 destinations, mfgp_peer_store), then raise every peer's signal."""
        others = [r for r in range(len(peers)) if r != me]
        for o in range(0, len(others), 8):
            grp = others[o:o + 8]
            self.h.peer_store(local_block, [peers[r][k].data_ptr() for r in grp], local_block.numel())
        for r in others:
            hdl.put_signal(r, channel, 30000)

    def peer_wait(self, hdl, src, channel):
        hdl.wait_signal(src, channel, 30000)

    # -- block arithmetic -------------------------------------------------------------------------------
    def cov(self, Xa, Xb, theta, out):
        ptr = self._vptr
        self._chk(self.L.mfgp_cov(self.h._h, ptr(Xa), Xa.shape[0], ptr(Xb), Xb.shape[0], Xa.shape[1] - 1, ptr(theta), ptr(out),
                                  out.stride(0)), "cov")

    def cov_grad(self, X, theta, G, scale, out):
        """out[2d+4] <- scale * sum_ij G_ij dK_ij/dtheta (lower triangle of G, off-diagonal twice), last entry trace(G)."""
        ptr = self._vptr
        self._chk(self.L.mfgp_cov_grad(self.h._h, ptr(X), X.shape[0], X.shape[1] - 1, ptr(theta), ptr(G), G.stride(0),
                                       float(scale), ptr(out)), "cov_grad")

    def potrf_inv(self, A, W):
        ptr = self._vptr
        self._chk(self.L.mfgp_potrf_inv(self.h._h, ptr(A), A.shape[0], A.stride(0), ptr(W), W.stride(0)), "potrf_inv")

    def tall_skinny_update(self, m, k, alpha, A, X, Y):
        """Y[m, :nc] += alpha * A[m, k] X[k, :nc]  (nc = X.shape[1] <= 2): one HBM-bound pass over A (mfgp_tall_skinny_update)."""
        ptr = self._vptr
        self._chk(self.L.mfgp_tall_skinny_update(self.h._h, m, k, X.shape[1], float(alpha), ptr(A), A.stride(0), ptr(X), X.stride(0),
                                                 ptr(Y), Y.stride(0)), "tall_skinny_update")

    def gemm(self, ta, tb, m, n, k, alpha, A, B, beta, C):
        ptr = self._vptr
        self._chk(self.L.mfgp_gemm(self.h._h, b"T" if ta else b"N", b"T" if tb else b"N", m, n, k, float(alpha), ptr(A),
                                   A.stride(0), ptr(B), B.stride(0), float(beta), ptr(C), C.stride(0)), "gemm")


def distributed_gpr_nlml(handle_or_ops, X, Y, theta, noise, nbd=1024, group=None, grid=None, lookahead=True, profile=None,
                         want_grad=False):
    """Every rank passes the same host X [N, d+1], Y [N, 1], theta [2d+3], noise.  Returns the NLML (same on all ranks);
    with want_grad=True returns (nlml, grad[2d+4]) with grad = d nlml / d [theta, noise] (constrained space), the analogue
    of tape.gradient at linear.py:207.

    Gradient (SURVEY 8(e) row 3), designed for 180 GB of HBM per GPU rather than for minimal memory: every panel is
    already broadcast to every rank by the factorisation, so each rank simply KEEPS the factor (N^2/2 doubles) and the
    diagonal-block inverses.  Then nothing else needs communication: rank r builds the block ROWS k = r (mod world) of
    W = L^-1 by block back-substitution (row k = e_k^T L^-1 is independent of the other rows), accumulates its share
    sum_k W_k^T W_k of K^-1, contracts it with dK/dtheta recomputed on the fly (K5), and ONE all-reduce of 2d+4 numbers
    finishes  d nlml/d theta = -1/2 tr((alpha alpha^T - K^-1) dK/dtheta).  Flops per rank: 2/3 N^3 / world.

    `handle_or_ops`: a `_lib.Handle` (product path) or an object with GpuOps' interface (CPU schedule tests).
    `profile`: optional dict; when given every phase is bracketed by a device synchronize and its wall time is
    accumulated there (serialises the two streams -- for diagnosis only)."""
    import time

    import torch
    import torch.distributed as dist

    class _Phase:
        def __init__(self, name):
            self.name = name

        def __enter__(self):
            if profile is not None:
                torch.cuda.synchronize()
                self.t0 = time.perf_counter()

        def __exit__(self, *exc):
            if profile is not None:
                torch.cuda.synchronize()
                profile[self.name] = profile.get(self.name, 0.0) + time.perf_counter() - self.t0

    if hasattr(handle_or_ops, "potrf_inv"):
        ops = handle_or_ops
    else:  # a library handle: keep the GpuOps (and with it the cached streams / workspaces) on the handle
        ops = getattr(handle_or_ops, "_dist_ops", None)
        if ops is None:
            ops = GpuOps(handle_or_ops)
            handle_or_ops._dist_ops = ops
    if hasattr(ops, "begin"):
        ops.begin()
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    P, Q = grid if grid is not None else process_grid(world)
    if P * Q != world:
        raise ValueError(f"process grid {P}x{Q} does not match world size {world}")
    p, q = rank // Q, rank % Q
    dev = ops.device
    X = np.ascontiguousarray(X, dtype=np.float64)
    Y = np.ascontiguousarray(Y, dtype=np.float64)
    N0, d = X.shape[0], X.shape[1] - 1
    if Y.ndim != 2 or Y.shape[1] != 1:
        raise ValueError("single-output problem expected (SURVEY config C5)")
    nb = int(nbd)
    if nb % 2:
        raise ValueError("block size must be even (16-byte aligned rows)")
    nblk = (N0 + nb - 1) // nb
    N = nblk * nb
    npad = N - N0
    # padding rows: fidelity 2.0 -> zero covariance (reference linear.py:82), noise on the diagonal, y = 0;
    # they add npad * log(noise)/2 to sum log L_ii, removed at the end
    if npad:
        Xp = np.zeros((N, d + 1))
        Xp[:N0] = X
        Xp[N0:, d] = 2.0
        Yp = np.zeros((N, 1))
        Yp[:N0] = Y
        X, Y = Xp, Yp
    Xd = torch.from_numpy(X).to(dev)
    thd = torch.from_numpy(np.ascontiguousarray(theta, dtype=np.float64)).to(dev)
    y = torch.zeros(N, 2, dtype=torch.float64, device=dev)  # column 1 pads the leading dimension to an even number
    y[:, 0] = torch.from_numpy(Y[:, 0].copy()).to(dev)

    R = [i for i in range(nblk) if i % P == p]   # local block rows
    Cb = [j for j in range(nblk) if j % Q == q]  # local block columns

    def first_local_row(j):  # index into R of the first local block row >= j
        return max(0, -(-(j - p) // P))

    # Streams and buffers are created once per (N, nb, grid) and kept on the ops object -- like the library handle's own
    # workspaces -- so that repeated evaluations (an optimiser loop) allocate nothing: cudaMalloc/cudaFree of the
    # multi-GB block columns would otherwise serialise the device and dominate the call.
    cache = getattr(ops, "_dist_chol_ws", None)
    key = (N, nb, P, Q, d, str(dev))
    if cache is None or cache.get("key") != key:
        cache = {"key": key, "s_main": ops.new_stream(), "s_pan": ops.new_stream(True), "s_crit": ops.new_stream(True), "cols": {}}
        for j in Cb:
            nr = len(R) - first_local_row(j)
            if nr > 0:
                cache["cols"][j] = torch.empty(nr * nb, nb, dtype=torch.float64, device=dev)
        cache["pans"] = [torch.empty(max(nblk - 1, 1) * nb, nb, dtype=torch.float64, device=dev) for _ in range(2)]
        cache["Wks"] = [torch.empty(nb, nb, dtype=torch.float64, device=dev) for _ in range(2)]
        cache["blks"] = [torch.empty(nb, nb, dtype=torch.float64, device=dev) for _ in range(2)]
        cache["piece"] = torch.empty(((nblk + P - 1) // P) * nb, nb, dtype=torch.float64, device=dev)
        cache["Rloc"] = torch.empty(max(len(R), 1) * nb, nb, dtype=torch.float64, device=dev)
        cache["Xr"] = torch.empty(max(len(R), 1) * nb, d + 1, dtype=torch.float64, device=dev)
        # Critical-path messages (inv(L_kk) and the early block (k+1, k)): one symmetric slot PER STEP (2 x nblk x nb^2 doubles
        # -- 0.5 GB at N = 32 768, nothing next to 180 GB of HBM), so a slot is never reused inside a factorisation and the
        # owner can store it into every peer without asking whether the previous tenant has been consumed.
        cache["p2p"] = None
        if world > 1 and hasattr(ops, "peer_buffers"):
            pw = ops.peer_buffers(nblk, nb, group)
            pb = ops.peer_buffers(nblk, nb, group) if pw is not None else None
            if pw is not None and pb is not None:
                cache["p2p"] = {"W": pw, "B": pb}
        try:
            ops._dist_chol_ws = cache
        except AttributeError:
            pass
    if want_grad and "Lcols" not in cache:
        cache["Lcols"] = [torch.empty(max(nblk - k - 1, 1) * nb, nb, dtype=torch.float64, device=dev) for k in range(nblk)]
        cache["Wd"] = [torch.empty(nb, nb, dtype=torch.float64, device=dev) for _ in range(nblk)]
        cache["Kinv"] = torch.empty(N, N, dtype=torch.float64, device=dev)
        cache["Xrow"] = torch.empty(nb, N, dtype=torch.float64, device=dev)
        cache["tmpb"] = torch.empty(nb, nb, dtype=torch.float64, device=dev)
    if lookahead:
        # One communicator: NCCL executes its collectives in issue order (W_k, blk_k, panel k, W_k+1, ...), which is also
        # the dependency order.  A second communicator for the small broadcasts was measured 10x SLOWER on 4 GPUs (two NCCL
        # kernels of different communicators spin against each other).
        s_main, s_pan, s_crit = cache["s_main"], cache["s_pan"], cache["s_crit"]
    else:  # reference schedule: the same steps, one stream
        s_main = s_pan = s_crit = cache["s_main"]

    # ---- assembly (no communication) -------------------------------------------------------------------
    cols = cache["cols"]
    with ops.use(s_main), _Phase("assembly"):
        Xr = cache["Xr"]
        if R:
            Xr[:len(R) * nb].view(len(R), nb, d + 1).copy_(Xd.view(nblk, nb, d + 1)[p::P])
        for j in Cb:
            f = first_local_row(j)
            nr = len(R) - f
            if nr <= 0:
                continue
            A = cols[j]
            ops.cov(Xr[f * nb:len(R) * nb], Xd[j * nb:(j + 1) * nb], thd, A)
            if R[f] == j:
                A[:nb].diagonal().add_(noise)
    ev_main = ops.record(s_main, "assembled") if hasattr(ops, "timeline") else ops.record(s_main)

    logdet = torch.zeros(1, dtype=torch.float64, device=dev)
    quad = torch.zeros(1, dtype=torch.float64, device=dev)
    pans, Wks, blks, piece, Rloc = cache["pans"], cache["Wks"], cache["blks"], cache["piece"], cache["Rloc"]
    p2p = cache.get("p2p") if lookahead else None
    if isinstance(getattr(ops, "stats", None), dict):
        ops.stats["critical_messages"] = "nvlink peer stores + signals" if p2p is not None else "nccl broadcast"
    W_of = (lambda k: p2p["W"][0][k]) if p2p is not None else (lambda k: Wks[k % 2])
    blk_of = (lambda k: p2p["B"][0][k]) if p2p is not None else (lambda k: blks[k % 2])
    ak = torch.zeros(nb, 2, dtype=torch.float64, device=dev)
    a_all = torch.zeros(N, 2, dtype=torch.float64, device=dev) if want_grad else None
    ev_W, ev_blk, ev_pan, ev_la, ev_done = {}, {}, {}, {}, {-1: ev_main}

    def rank_of(i, j):
        return (i % P) * Q + (j % Q)

    def local_off(j, i):
        """Row offset of block row i inside cols[j] (i is local, i >= j)."""
        return ((i - p) // P - first_local_row(j)) * nb

    def gather_local_rows(k, pan, out):
        """out <- panel-k rows of the local block rows > k, contiguous (strided block slice of the global-order panel)."""
        fk = first_local_row(k + 1)
        n = len(R) - fk
        if n > 0:
            s0 = R[fk] - (k + 1)
            out[:n * nb].view(n, nb, nb).copy_(pan[:(nblk - k - 1) * nb].view(nblk - k - 1, nb, nb)[s0::P])
        return out

    def apply_panel(k, j, pan, rows, skip_diag):
        """cols[j] -= L[i, k] L[j, k]^T for the local block rows i >= j (i > j when skip_diag); rows = gather_local_rows(k)."""
        if j not in cols:
            return
        f = first_local_row(j + 1 if skip_diag else j)
        m = (len(R) - f) * nb
        if m <= 0:
            return
        fk, fj = first_local_row(k + 1), first_local_row(j)
        ops.gemm(False, True, m, nb, nb, -1.0, rows[(f - fk) * nb:], pan[(j - k - 1) * nb:(j - k) * nb], 1.0, cols[j][(f - fj) * nb:])

    # Who applies panel k to block column j (so that no block is ever updated from two streams at once):
    #   diagonal block (j, j):  main for k <= j-3, crit for k = j-2 (from pan_k) and k = j-1 (from the early block blk_k)
    #   rows below it:          main for k <= j-2, pan (look-ahead) for k = j-1
    def crit_step(k):
        """Critical path of step k: factor the diagonal block, broadcast its inverse, solve + broadcast the ONE block
        (k+1, k) and finish the next diagonal block, so that potrf(k+1) never waits for the bulk of panel k."""
        buf = k % 2
        Wk, blk = W_of(k), blk_of(k)
        # Block (k, k) has received its main-stream updates once main has finished step k-3 (panels k-2 and k-1 are applied to
        # it by THIS stream).  With one message slot per step (peer-memory path) that is all potrf(k) has to wait for, so it
        # overlaps main's step k-2; the two-buffer NCCL path must also wait until main's step k-2 has released W/blk[k % 2].
        # (Device timeline, 8 GPUs, N = 32 768: waiting for done[k-2] here throttled every second potrf by 4-5 ms while main
        # was still busy with a trailing update the diagonal block does not depend on.)
        ops.wait(s_crit, ev_done.get(k - 3 if p2p is not None else k - 2))
        with _Phase("diag_potrf_inv"):
            if rank == rank_of(k, k):
                A = cols[k]
                ops.potrf_inv(A[:nb], Wk)
                logdet.add_(torch.log(A[:nb].diagonal()).sum())
        with _Phase("bcast_W"):
            if p2p is not None:  # direct NVLink stores + signal: never queues behind the panel broadcasts
                if rank == rank_of(k, k):
                    ops.peer_publish(p2p["W"][1], p2p["W"][2], Wk, k, rank, 0)
                else:
                    ops.peer_wait(p2p["W"][1], rank_of(k, k), 0)
            else:
                dist.broadcast(Wk, src=rank_of(k, k), group=group)
        ev_W[k] = ops.record(s_crit, f"W{k}") if hasattr(ops, "timeline") else ops.record(s_crit)
        if k + 1 >= nblk:
            return
        ops.wait(s_crit, ev_done.get(k - 2))  # column k below the diagonal and block (k+1, k+1) carry main's step k-2
        with _Phase("early_block"):
            src = rank_of(k + 1, k)
            if rank == src:
                ops.wait(s_crit, ev_la.get(k - 1))  # block (k+1, k) carries panel k-1 (look-ahead of the previous step)
                o = local_off(k, k + 1)
                ops.gemm(False, True, nb, nb, nb, 1.0, cols[k][o:o + nb], Wk, 0.0, blk)
                cols[k][o:o + nb].copy_(blk)
            if p2p is not None:
                if rank == src:
                    ops.peer_publish(p2p["B"][1], p2p["B"][2], blk, k, rank, 1)
                else:
                    ops.peer_wait(p2p["B"][1], src, 1)
            else:
                dist.broadcast(blk, src=src, group=group)
            ev_blk[k] = ops.record(s_crit, f"blk{k}") if hasattr(ops, "timeline") else ops.record(s_crit)
            if rank == rank_of(k + 1, k + 1):
                D = cols[k + 1][:nb]
                if k >= 1:
                    ops.wait(s_crit, ev_pan.get(k - 1))
                    L1 = pans[(k - 1) % 2][nb:2 * nb]  # L[k+1, k-1]
                    ops.gemm(False, True, nb, nb, nb, -1.0, L1, L1, 1.0, D)
                ops.gemm(False, True, nb, nb, nb, -1.0, blk, blk, 1.0, D)

    def pan_step(k):
        """Bulk of step k: rest of the panel solve, the P panel broadcasts, look-ahead update of column k+1."""
        nbelow = nblk - k - 1
        if nbelow == 0:
            return
        buf = k % 2
        pan, Wk = pans[buf], W_of(k)
        kq = k % Q
        ops.wait(s_pan, ev_done.get(k - 2))  # rows of column k carry panels <= k-2; pans[buf] is no longer read by main
        ops.wait(s_pan, ev_blk.get(k))       # W_k and the solved block (k+1, k) are in place
        with _Phase("panel_solve"):
            if q == kq and k in cols:
                A = cols[k]
                off = (first_local_row(k + 2) - first_local_row(k)) * nb  # skip the diagonal block and block k+1
                m = A.shape[0] - off
                if m > 0:
                    tmp = piece[:m]
                    ops.gemm(False, True, m, nb, nb, 1.0, A[off:], Wk, 0.0, tmp)
                    A[off:].copy_(tmp)
        for pp in range(P):  # one broadcast per process row of column kq: rows i > k, i = pp (mod P)
            i0 = k + 1 + ((pp - (k + 1)) % P)
            if i0 >= nblk:
                continue
            cnt = (nblk - 1 - i0) // P + 1
            src = pp * Q + kq
            if rank == src:
                o = local_off(k, i0)
                buf_t = cols[k][o:o + cnt * nb]
            else:
                buf_t = piece[:cnt * nb]
            with _Phase("bcast_panel"):
                dist.broadcast(buf_t, src=src, group=group)
                pan[:nbelow * nb].view(nbelow, nb, nb)[i0 - (k + 1)::P].copy_(buf_t.view(cnt, nb, nb))
        ev_pan[k] = ops.record(s_pan, f"pan{k}") if hasattr(ops, "timeline") else ops.record(s_pan)
        ops.wait(s_pan, ev_done.get(k - 1))  # main has finished applying panel k-1 to the same rows of column k+1
        with _Phase("lookahead_update"):
            if k + 1 in cols:
                rows = gather_local_rows(k, pan, piece)  # `piece` is idle between the broadcasts of two steps
                apply_panel(k, k + 1, pan, rows, skip_diag=True)
        ev_la[k] = ops.record(s_pan, f"la{k}") if hasattr(ops, "timeline") else ops.record(s_pan)

    def main_step(k):
        """Forward substitution piece (replicated) and the trailing update of the block columns > k+1."""
        nbelow = nblk - k - 1
        buf = k % 2
        pan, Wk = pans[buf], W_of(k)
        ops.wait(s_main, ev_W.get(k))
        ops.wait(s_main, ev_pan.get(k))
        with _Phase("forward_subst"):  # a_k = W_kk y_k ; y[k+1:] -= L[k+1:, k] a_k
            if hasattr(ops, "tall_skinny_update") and nb <= 3072:
                ak.zero_()
                ops.tall_skinny_update(nb, nb, 1.0, Wk, y[k * nb:(k + 1) * nb], ak)
            else:
                ops.gemm(False, False, nb, 2, nb, 1.0, Wk, y[k * nb:(k + 1) * nb], 0.0, ak)
            quad.add_((ak[:, 0] * ak[:, 0]).sum())
            if want_grad:  # keep the factor: panel k, inv(L_kk) and a_k (every rank has them anyway)
                a_all[k * nb:(k + 1) * nb].copy_(ak)
                cache["Wd"][k].copy_(Wk)
                if nbelow:
                    cache["Lcols"][k][:nbelow * nb].copy_(pan[:nbelow * nb])
            if nbelow:
                if hasattr(ops, "tall_skinny_update") and nb <= 3072:
                    ops.tall_skinny_update(nbelow * nb, nb, -1.0, pan, ak, y[(k + 1) * nb:])
                else:
                    ops.gemm(False, False, nbelow * nb, 2, nb, -1.0, pan, ak, 1.0, y[(k + 1) * nb:])
        with _Phase("trailing_update"):
            if nbelow > 1:
                rows = gather_local_rows(k, pan, Rloc)
                for j in Cb:
                    if j >= k + 2:
                        apply_panel(k, j, pan, rows, skip_diag=(j == k + 2))
        ev_done[k] = ops.record(s_main, f"done{k}") if hasattr(ops, "timeline") else ops.record(s_main)

    t_issue0 = time.perf_counter()
    with ops.use(s_crit):
        ops.wait(s_crit, ev_main)
        if p2p is not None:  # every rank has finished READING the previous call's slots before anybody overwrites them
            p2p["W"][1].barrier(2, 30000)
        crit_step(0)
    for k in range(nblk):
        with ops.use(s_pan):
            pan_step(k)
        if k + 1 < nblk:
            with ops.use(s_crit):
                crit_step(k + 1)
        with ops.use(s_main):
            main_step(k)
    with ops.use(s_main):
        ops.wait(s_main, ev_W.get(nblk - 1))
        dist.all_reduce(logdet, group=group)
    gout = None
    if want_grad:
        with ops.use(s_main), _Phase("gradient"):
            Lcols, Wd, Kinv, Xrow, tmpb = cache["Lcols"], cache["Wd"], cache["Kinv"], cache["Xrow"], cache["tmpb"]
            # alpha = L^-T a by block back-substitution (replicated: O(N^2))
            alpha = torch.zeros(N, 2, dtype=torch.float64, device=dev)
            tvec = torch.empty(nb, 2, dtype=torch.float64, device=dev)
            for k in range(nblk - 1, -1, -1):
                nbelow = nblk - k - 1
                tvec.copy_(a_all[k * nb:(k + 1) * nb])
                if nbelow:
                    ops.gemm(True, False, nb, 2, nbelow * nb, -1.0, Lcols[k], alpha[(k + 1) * nb:], 1.0, tvec)
                ops.gemm(True, False, nb, 2, nb, 1.0, Wd[k], tvec, 0.0, alpha[k * nb:(k + 1) * nb])
            # this rank's share of K^-1 = sum_k W_k^T W_k over its block rows k of W = L^-1
            Kinv.zero_()
            for k in range(rank, nblk, world):
                Xrow[:, k * nb:(k + 1) * nb].copy_(Wd[k])
                for j in range(k - 1, -1, -1):  # W_kj = -(sum_{i=j+1..k} W_ki L_ij) inv(L_jj)
                    ops.gemm(False, False, nb, nb, (k - j) * nb, 1.0, Xrow[:, (j + 1) * nb:], Lcols[j], 0.0, tmpb)
                    ops.gemm(False, False, nb, nb, nb, -1.0, tmpb, Wd[j], 0.0, Xrow[:, j * nb:])
                for c in range(k + 1):  # lower block columns of W_k^T W_k
                    ops.gemm(True, False, (k + 1 - c) * nb, nb, nb, 1.0, Xrow[:, c * nb:], Xrow[:, c * nb:], 1.0,
                             Kinv[c * nb:, c * nb:])
            if rank == 0:  # G = alpha alpha^T - K^-1: the rank-1 term once
                ops.gemm(False, True, N, N, 2, -1.0, alpha, alpha, 1.0, Kinv)
            gout = torch.zeros(2 * d + 4, dtype=torch.float64, device=dev)
            ops.cov_grad(Xd, thd, Kinv, 0.5, gout)  # +1/2 sum (K^-1 - alpha alpha^T) dK = -1/2 sum G dK
            dist.all_reduce(gout, group=group)
    t_issue1 = time.perf_counter()
    ops.finish()
    stats = getattr(ops, "stats", None)
    if isinstance(stats, dict):  # host time to ISSUE the factorisation vs. time until the device has finished it
        stats["host_issue_s"] = t_issue1 - t_issue0
        stats["device_done_s"] = time.perf_counter() - t_issue0
    ld = float(logdet.item()) - (0.5 * npad * math.log(noise) if npad else 0.0)
    nlml = 0.5 * float(quad.item()) + ld + 0.5 * N0 * math.log(2.0 * math.pi)
    if not want_grad:
        return nlml
    grad = gout.cpu().numpy().copy()
    grad[2 * d + 3] -= 0.5 * npad / noise  # the padding rows' log(noise)/2 terms
    return nlml, grad
