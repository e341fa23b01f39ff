"""Input gradients of the cached SVGP posterior (mfgp_svgp_posterior_predict_grad) against prediction alone and against
central differences.  Prints one JSON document.

  a  HBS single-bin (L = 49) and latent (L = 10, W [49, 10]) models, M = 50, Ns = 1 and 10, host buffers: wall time of
     posterior().predict_f_grad against posterior().predict_f alone and against the 2d + 1 = 11 predict_f calls of
     central differences
  b  HBS single-bin at Ns = 262 144, device buffers: kernel time of one fused grad launch against the predict launch
     (CUDA events, alternating in the same run); (latent, point) pairs/s and the share of the live DMMA peak on
     4M(M+1) + 6M + 4Md flop per pair: the four triangular products V = Wm K_s, U = Lq^T V, Lq U and beta = Wm^T r, the
     three reductions of predict, and the two contractions beta . g_j and alpha . g_j per coordinate (assembly of K_s
     and g_j, exp and the mix not counted)
  c  Goku single-bin (L = 64) and latent (L = 15, W [64, 15]), M = 300, d = 10, Ns = 36 and 4096, host buffers: blocked
     route, predict_grad against predict
Every leg checks a sample of its timed outputs against the autograd oracle (tests/_svgp_grad_oracle.py; 1e-7 relative, atol
1e-7 max|ref|) and mean / var bitwise against predict.  Wall times are medians of 200 calls after a warm-up.
Usage: python scripts/svgp_posterior_grad_bench.py [--out profiles/r06_svgp_posterior_grad.json]"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from multi_fidelity_gpflow_b200 import _lib  # noqa: E402
from multi_fidelity_gpflow_b200.linear_svgp import LatentMFCoregionalizationSVGP  # noqa: E402
from multi_fidelity_gpflow_b200.singlebin_svgp import SingleBinSVGP  # noqa: E402
from oracle import mfgp_oracle as onp  # noqa: E402
from scripts.svgp_posterior_bench import gpu_info, perturbed, se, wall  # noqa: E402
from tests._svgp_grad_oracle import svgp_predict_grad_x  # noqa: E402


def close(got, ref):
    np.testing.assert_allclose(got, ref, rtol=1e-7, atol=1e-7 * np.abs(ref).max())


def check_oracle(Xs, Z, th, W, q_mu, q_sqrt, dm, dv):
    """dm / dv [Ns, P, d] (the C ABI's layout) or [Ns, P, d+1] (predict_f_grad's)."""
    _, _, rdm, rdv = svgp_predict_grad_x(Xs, Z, th, q_mu, np.tril(q_sqrt), W)
    k = dm.shape[-1]
    close(dm, rdm[..., :k])
    close(dv, rdv[..., :k])


def leg_a(h):
    ds = onp.load_dataset("hbs")
    X, Y, Xt = ds["X"], ds["Y"], ds["X_test"]
    d = X.shape[1] - 1
    rng = np.random.default_rng(0)
    out = {}
    for name, mdl in (("singlebin_L49", SingleBinSVGP(X, Y, se(5), se(5), 49, ds["Z_kmeans50"], handle=h)),
                      ("latent_L10", LatentMFCoregionalizationSVGP(X, Y, se(5), se(5), 10, num_inducing=50, handle=h))):
        M, L = mdl.q_mu.shape
        mdl.q_mu.assign(0.3 * rng.standard_normal((M, L)))
        mdl.q_sqrt.assign(mdl.q_sqrt.numpy() + 0.02 * np.tril(rng.standard_normal((L, M, M))))
        post = mdl.posterior()
        res = {}
        for ns in (1, 10):
            Xs = np.ascontiguousarray(Xt[:ns])
            mean, var, dm, dv = post.predict_f_grad(Xs)
            pm, pv = post.predict_f(Xs)
            assert np.array_equal(mean, pm) and np.array_equal(var, pv)
            check_oracle(Xs, mdl.Z.numpy(), mdl._thetas(d), mdl._W(), mdl.q_mu.numpy(), mdl.q_sqrt.numpy(), dm, dv)

            def central():
                for j in range(d):
                    for s in (1e-5, -1e-5):
                        xp = Xs.copy()
                        xp[:, j] += s
                        post.predict_f(xp)
                post.predict_f(Xs)

            grad = wall(lambda: post.predict_f_grad(Xs))
            pred = wall(lambda: post.predict_f(Xs))
            fd = wall(central)
            res[f"Ns{ns}"] = {"predict_f_grad_s": grad, "predict_f_s": pred, "central_differences_2d_plus_1_predict_f_s": fd,
                              "grad_over_predict": grad[0] / pred[0], "central_differences_over_grad": fd[0] / grad[0]}
        out[name] = res
        post.post.close()
    return out


def leg_b(h, peak):
    import torch

    ds = onp.load_dataset("hbs")
    Z = ds["Z_kmeans50"]
    L, M, d, Ns = 49, Z.shape[0], 5, 262144
    rng = np.random.default_rng(1)
    th, W, q_mu, q_sqrt = perturbed(rng, Z, L, d, L, False)
    post = h.svgp_posterior(Z, th, W, q_mu, q_sqrt)
    Xs = np.hstack([rng.random((Ns, d)), rng.integers(0, 2, (Ns, 1)).astype(float)])
    dXs = torch.from_numpy(Xs).cuda()
    empty = lambda *s: torch.empty(s, dtype=torch.float64, device="cuda")
    gm, gv, gdm, gdv = empty(Ns, L), empty(Ns, L), empty(Ns, L, d), empty(Ns, L, d)
    pm, pv = empty(Ns, L), empty(Ns, L)
    stream = torch.cuda.current_stream()
    h.set_stream(stream.cuda_stream)
    h.set_async(True)
    grad_fn = lambda: post.predict_grad(dXs, gm, gv, gdm, gdv)
    pred_fn = lambda: post.predict(dXs, pm, pv)

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
            grad_fn()
            pred_fn()
        torch.cuda.synchronize()
        grad, pred = [], []
        for _ in range(5):  # alternating: both see the same clocks and neighbours
            grad.append(timed(grad_fn, 10))
            pred.append(timed(pred_fn, 10))
        assert h.sync() == 0
    finally:
        h.set_async(False)
        h.set_stream(None)
    t, tp = float(np.median(grad)), float(np.median(pred))
    assert torch.equal(gm, pm) and torch.equal(gv, pv)
    idx = np.concatenate([np.arange(16), Ns - 1 - np.arange(16)])
    check_oracle(Xs[idx], Z, th, None, q_mu, q_sqrt, gdm.cpu().numpy()[idx], gdv.cpu().numpy()[idx])
    pairs = L * Ns
    flop = pairs * (4 * M * (M + 1) + 6 * M + 4 * M * d)
    post.close()
    return {"L": L, "M": M, "d": d, "Ns": Ns, "grad_kernel_s": t, "grad_kernel_s_runs": grad, "predict_kernel_s": tp,
            "predict_kernel_s_runs": pred, "grad_over_predict": t / tp, "pairs_per_s": pairs / t, "flop": flop,
            "flop_per_s": flop / t, "fp64_peak_flop_per_s": peak, "share_of_fp64_peak": flop / peak / t}


def leg_c(h):
    ds = onp.load_dataset("goku")
    Z, Xt = ds["Z_kmeans300"], ds["X_test"]
    d = Z.shape[1] - 1
    rng = np.random.default_rng(2)
    out = {}
    for name, L, mixing in (("singlebin_L64", 64, False), ("latent_L15", 15, True)):
        th, W, q_mu, q_sqrt = perturbed(rng, Z, L, d, 64, mixing)
        post = h.svgp_posterior(Z, th, W, q_mu, q_sqrt)
        res = {}
        for ns in (36, 4096):
            Xs = Xt if ns == 36 else np.hstack([rng.random((ns, d)), rng.integers(0, 2, (ns, 1)).astype(float)])
            mean, var, dm, dv = post.predict_grad(Xs)
            pm, pv = post.predict(Xs)
            assert np.array_equal(mean, pm) and np.array_equal(var, pv)
            check_oracle(Xs[:8], Z, th, W, q_mu, q_sqrt, dm[:8], dv[:8])
            grad = wall(lambda: post.predict_grad(Xs))
            pred = wall(lambda: post.predict(Xs))
            res[f"Ns{ns}"] = {"predict_grad_s": grad, "predict_s": pred, "grad_over_predict": grad[0] / pred[0]}
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
