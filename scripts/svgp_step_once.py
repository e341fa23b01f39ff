"""Goku single-bin SVGP device-loop step time (K7) -- for tile-config / fusion A/B runs.  Prints ms per step."""
import os, sys, time
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from multi_fidelity_gpflow_b200 import _lib
from multi_fidelity_gpflow_b200.data import PowerSpecs
from multi_fidelity_gpflow_b200.kernels import SquaredExponential
from multi_fidelity_gpflow_b200.singlebin_svgp import SingleBinSVGP
from multi_fidelity_gpflow_b200.linear_svgp import LatentMFCoregionalizationSVGP
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ps = PowerSpecs().read_from_npz(os.path.join(ROOT, "tests", "golden", "goku.npz"))
X, Y = ps.training_arrays()
d, P = X.shape[1] - 1, Y.shape[1]
se = lambda: SquaredExponential(lengthscales=np.ones(d))
which = sys.argv[1] if len(sys.argv) > 1 else "single"
mdl = SingleBinSVGP(X, Y, se(), se(), P, ps.extras["Z_kmeans300"]) if which == "single" else \
    LatentMFCoregionalizationSVGP(X, Y, se(), se(), num_latents=15, num_inducing=300, num_outputs=P)
mdl.optimize_on_device((X, Y), max_iters=3, initial_lr=0.005)
def timed(steps):
    if which != "single":
        mdl.loss_history, mdl.kl_history = [], []
    torch.cuda.synchronize(); t0 = time.perf_counter()
    mdl.optimize_on_device((X, Y), max_iters=steps, initial_lr=0.005)
    return time.perf_counter() - t0
steps = 20
long_steps = int(sys.argv[2]) if len(sys.argv) > 2 else 0
t20 = timed(steps)
print(f"{which}: {t20 / steps * 1e3:.3f} ms per step  loss {mdl.loss_history[-1]:.6f}")
if long_steps > steps:
    # the per-call cost (parameters + Adam moments host<->device, the eager first step, graph capture) is the same for
    # both lengths: the difference isolates the replayed step
    tl = timed(long_steps)
    print(f"{which}: steady state {(tl - t20) / (long_steps - steps) * 1e3:.3f} ms per step; per-call cost {(t20 - steps * (tl - t20) / (long_steps - steps)) * 1e3:.1f} ms")
