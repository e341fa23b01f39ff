"""ctypes binding of libmfgp.so (C-ABI declared in include/mfgp.h).

There is NO CPU fallback: importing this module without the built library raises, and
creating a handle without a CUDA device raises.  Buffers may be NumPy arrays (host
pointers; the library stages them through its stream) or CUDA tensors / any object with
``data_ptr()`` or ``__cuda_array_interface__`` (device pointers, zero-copy).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmfgp.so")


class MFGPError(RuntimeError):
    pass


class NotPositiveDefiniteError(np.linalg.LinAlgError):
    """Mirror of TF's InvalidArgumentError 'Cholesky decomposition was not successful'."""


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m multi_fidelity_gpflow_b200.build` "
            "(nvcc, sm_100a). This package has no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    vp, i, l, d = C.c_void_p, C.c_int, C.c_long, C.c_double
    i64, u64 = C.c_longlong, C.c_ulonglong
    sig = {
        "mfgp_version": ([], i),
        "mfgp_create": ([i, C.POINTER(vp)], i),
        "mfgp_destroy": ([vp], i),
        "mfgp_set_stream": ([vp, vp], i),
        "mfgp_reset_stream": ([vp], i),
        "mfgp_set_async": ([vp, i], i),
        "mfgp_sync": ([vp, C.POINTER(i)], i),
        "mfgp_last_error": ([vp], C.c_char_p),
        "mfgp_sm_count": ([vp], i),
        "mfgp_cov": ([vp, vp, i, vp, i, i, vp, vp, l], i),
        "mfgp_cov_diag": ([vp, vp, i, i, vp, vp], i),
        "mfgp_cov_grad": ([vp, vp, i, i, vp, vp, l, d, vp], i),
        "mfgp_gpr_nlml": ([vp, vp, vp, i, i, i, vp, d, vp], i),
        "mfgp_gpr_nlml_grad": ([vp, vp, vp, i, i, i, vp, d, vp, vp], i),
        "mfgp_gpr_predict": ([vp, vp, vp, i, i, i, vp, i, vp, d, vp, vp], i),
        "mfgp_gpr_batched_nlml_grad": ([vp, vp, i, i, vp, l, i, i, vp, vp, vp, vp, vp], i),
        "mfgp_gpr_batched_adam": ([vp, vp, i, i, vp, l, i, i, vp, vp, vp, vp, vp, d, d, d, i, i, vp, vp, vp], i),
        "mfgp_gpr_batched_lbfgs": ([vp, vp, i, i, vp, l, i, i, vp, vp, i, i, vp, vp, vp, vp, vp, vp], i),
        "mfgp_gpr_posterior_create": ([vp, vp, i, i, vp, l, i, i, i, vp, vp, vp, C.POINTER(vp)], i),
        "mfgp_gpr_posterior_predict": ([vp, vp, vp, i, vp, vp], i),
        "mfgp_gpr_posterior_predict_grad": ([vp, vp, vp, i, vp, vp, vp, vp], i),
        "mfgp_gpr_posterior_predict_cov": ([vp, vp, vp, i, vp, vp], i),
        "mfgp_gpr_posterior_sample": ([vp, vp, vp, i, i, d, vp, vp, vp], i),
        "mfgp_gpr_posterior_destroy": ([vp], i),
        "mfgp_graph_nparams": ([i, i], i),
        "mfgp_graph_cov": ([vp, vp, i, i, i, vp, vp, l], i),
        "mfgp_graph_cov_diag": ([vp, vp, i, i, i, vp, vp], i),
        "mfgp_graph_gpr_nlml_grad": ([vp, vp, vp, i, i, i, i, vp, d, vp, vp], i),
        "mfgp_svgp_elbo_grad": ([vp, vp, vp, vp, vp, vp, vp, vp, vp, d, vp, vp, vp, vp, vp, vp, vp, vp], i),
        "mfgp_svgp_elbo_grad_v": ([vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp], i),
        "mfgp_svgp_predict": ([vp, vp, vp, i, vp, vp, vp, vp, vp, vp, vp], i),
        "mfgp_svgp_posterior_create": ([vp, vp, vp, vp, vp, vp, vp, vp, C.POINTER(vp)], i),
        "mfgp_svgp_posterior_predict": ([vp, vp, vp, i, vp, vp], i),
        "mfgp_svgp_posterior_predict_grad": ([vp, vp, vp, i, vp, vp, vp, vp], i),
        "mfgp_svgp_posterior_predict_cov": ([vp, vp, vp, i, vp, vp], i),
        "mfgp_svgp_posterior_sample": ([vp, vp, vp, i, i, d, vp, vp, vp], i),
        "mfgp_svgp_posterior_destroy": ([vp], i),
        "mfgp_svgp_adam": ([vp, vp, vp, vp, i, vp, vp, vp, vp, vp, d, d, d, i, vp, vp], i),
        "mfgp_svgp_adam_minibatch": ([vp, vp, vp, vp, i, u64, i64, i, vp, vp, vp, vp, vp, d, d, d, i, vp, vp], i),
        "mfgp_minibatch_gather": ([vp, vp, i, vp, i, i, u64, i64, vp, i, i, i, vp, vp], i),
        "mfgp_svgp_natgrad": ([vp, vp, d, vp, vp, vp, vp, vp], i),
        "mfgp_svgp_natgrad_adam": ([vp, vp, vp, vp, i, u64, i64, i, vp, vp, vp, vp, vp, vp, d, d, d, i, vp, vp, vp], i),
        "mfgp_svgp_flat_size": ([vp, i], l),
        "mfgp_svgp_constrain": ([vp, vp, i, vp, vp], i),
        "mfgp_svgp_elbo_grad_flat": ([vp, vp, vp, vp, i, vp, i, vp], i),
        "mfgp_svgp_adam_update": ([vp, vp, i, vp, vp, vp, vp, vp, vp, vp, vp, d, d, d, vp, vp, vp], i),
        "mfgp_gemm": ([vp, C.c_char, C.c_char, i, i, i, d, vp, l, vp, l, d, vp, l], i),
        "mfgp_potrf": ([vp, vp, i, l], i),
        "mfgp_potrf_inv": ([vp, vp, i, l, vp, l], i),
        "mfgp_tall_skinny_update": ([vp, i, i, i, d, vp, l, vp, l, vp, l], i),
        "mfgp_peer_store": ([vp, vp, l, i, C.POINTER(vp)], i),
        "mfgp_graph_mem_trim": ([vp], i),
        "mfgp_workspace": ([vp, i, C.POINTER(l)], i),
        "mfgp_fp64_peak": ([vp, i, i, C.POINTER(d)], i),
    }
    for name, (args, res) in sig.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = res
    return lib


_lib = _load()
EXPORTED_SYMBOLS = [
    "mfgp_version", "mfgp_create", "mfgp_destroy", "mfgp_set_stream", "mfgp_reset_stream", "mfgp_set_async", "mfgp_sync",
    "mfgp_last_error", "mfgp_sm_count", "mfgp_cov", "mfgp_cov_diag", "mfgp_cov_grad", "mfgp_gpr_nlml", "mfgp_gpr_nlml_grad",
    "mfgp_gpr_predict", "mfgp_gpr_batched_nlml_grad", "mfgp_gpr_batched_adam", "mfgp_gpr_batched_lbfgs",
    "mfgp_gpr_posterior_create", "mfgp_gpr_posterior_predict", "mfgp_gpr_posterior_predict_grad",
    "mfgp_gpr_posterior_predict_cov", "mfgp_gpr_posterior_sample", "mfgp_gpr_posterior_destroy",
    "mfgp_graph_nparams", "mfgp_graph_cov", "mfgp_graph_cov_diag", "mfgp_graph_gpr_nlml_grad", "mfgp_svgp_elbo_grad", "mfgp_svgp_elbo_grad_v", "mfgp_svgp_predict",
    "mfgp_svgp_posterior_create", "mfgp_svgp_posterior_predict", "mfgp_svgp_posterior_predict_grad",
    "mfgp_svgp_posterior_predict_cov", "mfgp_svgp_posterior_sample", "mfgp_svgp_posterior_destroy", "mfgp_svgp_adam", "mfgp_svgp_adam_minibatch", "mfgp_minibatch_gather",
    "mfgp_svgp_natgrad", "mfgp_svgp_natgrad_adam",
    "mfgp_svgp_flat_size", "mfgp_svgp_constrain", "mfgp_svgp_elbo_grad_flat", "mfgp_svgp_adam_update", "mfgp_gemm",
    "mfgp_potrf", "mfgp_potrf_inv", "mfgp_tall_skinny_update", "mfgp_peer_store", "mfgp_graph_mem_trim", "mfgp_workspace", "mfgp_fp64_peak",
]


class SvgpCfg(C.Structure):
    _fields_ = [
        ("L", C.c_int), ("M", C.c_int), ("P", C.c_int), ("B", C.c_int), ("d", C.c_int), ("hetero", C.c_int),
        ("scale", C.c_double), ("kl_mult", C.c_double), ("jitter", C.c_double), ("lik_lower", C.c_double),
        ("masked", C.c_int), ("lik_per_output", C.c_int),
    ]


class LbfgsOpts(C.Structure):
    _fields_ = [("m", C.c_int), ("maxiter", C.c_int), ("maxfun", C.c_int), ("maxls", C.c_int), ("ftol", C.c_double),
                ("gtol", C.c_double)]


# status codes of mfgp_gpr_batched_lbfgs (include/mfgp.h: MFGP_LBFGS_*)
LBFGS_STATUS = {1: "pgtol", 2: "ftol", 3: "maxiter", 4: "maxfun", 5: "abnormal", 6: "not_pd"}
LBFGS_NOT_PD = 6


# ---- DLPack consumer (dlpack.h, DLManagedTensor ABI v0) -------------------------------------------------------
# TF tensors (tf.experimental.dlpack.to_dlpack), CuPy / JAX arrays and anything else with __dlpack__ cross the C-ABI
# zero-copy: the capsule's DLManagedTensor is read with ctypes, checked (float64, C-contiguous, CPU / CUDA memory) and its
# data address passed to the library, which decides host vs device by itself (cudaPointerGetAttributes).
class _DLDevice(C.Structure):
    _fields_ = [("device_type", C.c_int), ("device_id", C.c_int)]


class _DLDataType(C.Structure):
    _fields_ = [("code", C.c_uint8), ("bits", C.c_uint8), ("lanes", C.c_uint16)]


class _DLTensor(C.Structure):
    _fields_ = [("data", C.c_void_p), ("device", _DLDevice), ("ndim", C.c_int), ("dtype", _DLDataType),
                ("shape", C.POINTER(C.c_int64)), ("strides", C.POINTER(C.c_int64)), ("byte_offset", C.c_uint64)]


class _DLManagedTensor(C.Structure):
    _fields_ = [("dl_tensor", _DLTensor), ("manager_ctx", C.c_void_p), ("deleter", C.c_void_p)]


_KDL_FLOAT = 2
_DL_DEVICES = {1: "cpu", 2: "cuda", 3: "cuda_host", 13: "cuda_managed"}
_capsule_get = C.pythonapi.PyCapsule_GetPointer
_capsule_get.restype, _capsule_get.argtypes = C.c_void_p, [C.py_object, C.c_char_p]
_capsule_valid = C.pythonapi.PyCapsule_IsValid
_capsule_valid.restype, _capsule_valid.argtypes = C.c_int, [C.py_object, C.c_char_p]


def _is_capsule(x):
    return type(x).__name__ == "PyCapsule"


def from_dlpack_capsule(capsule, dtype_code=_KDL_FLOAT, bits=64):
    """(address, shape, device kind) of an UNCONSUMED "dltensor" capsule.  The capsule stays owned by the caller (it is
    not renamed to "used_dltensor"): its deleter runs when the capsule is garbage-collected, after the library call."""
    if not _capsule_valid(capsule, b"dltensor"):
        raise TypeError("expected an unconsumed DLPack capsule named 'dltensor'")
    t = C.cast(_capsule_get(capsule, b"dltensor"), C.POINTER(_DLManagedTensor)).contents.dl_tensor
    if (t.dtype.code, t.dtype.bits, t.dtype.lanes) != (dtype_code, bits, 1):
        raise TypeError(f"DLPack tensor must be float{bits} (got code {t.dtype.code}, {t.dtype.bits} bits, {t.dtype.lanes} lanes)")
    if t.device.device_type not in _DL_DEVICES:
        raise TypeError(f"DLPack device type {t.device.device_type} is neither CPU nor CUDA memory")
    shape = tuple(int(t.shape[i]) for i in range(t.ndim))
    if bool(t.strides):  # NULL = compact row-major
        expect = 1
        for i in range(t.ndim - 1, -1, -1):
            if shape[i] != 1 and int(t.strides[i]) != expect:
                raise ValueError("DLPack tensor must be C-contiguous")
            expect *= shape[i]
    return (t.data or 0) + int(t.byte_offset), shape, _DL_DEVICES[t.device.device_type]


def _ptr(x):
    """Raw address of a float64/int32 C-contiguous buffer: host ndarray, torch / CuPy device tensor, a DLPack capsule, or
    any object exporting __dlpack__ (TF eager tensors, JAX arrays)."""
    if x is None:
        return None
    if isinstance(x, np.ndarray):
        if not x.flags["C_CONTIGUOUS"]:
            raise ValueError("array must be C-contiguous")
        return C.c_void_p(x.ctypes.data)
    if hasattr(x, "data_ptr"):
        if hasattr(x, "is_contiguous") and not x.is_contiguous():
            raise ValueError("tensor must be contiguous")
        return C.c_void_p(x.data_ptr())
    if hasattr(x, "__cuda_array_interface__"):
        return C.c_void_p(x.__cuda_array_interface__["data"][0])
    if _is_capsule(x) or hasattr(x, "__dlpack__"):
        cap = x if _is_capsule(x) else x.__dlpack__()
        addr, _, _ = from_dlpack_capsule(cap)
        p = C.c_void_p(addr)
        p._dlpack_owner = cap  # keeps the exporter's memory alive for as long as the pointer object lives (the call)
        return p
    raise TypeError(f"unsupported buffer type {type(x)}")


def _seed(seed):
    """A minibatch stream seed: an integer in [0, 2^64)."""
    seed = int(seed)
    if not 0 <= seed < 1 << 64:
        raise ValueError(f"seed must be an integer in [0, 2**64), got {seed}")
    return seed


def _any_nonzero(a):
    """Whether a host array or device tensor holds a nonzero entry."""
    return bool((a != 0).any())


def as_f64(x):
    """Host arrays -> contiguous float64 ndarray; device tensors and DLPack exporters pass through (must be float64)."""
    if hasattr(x, "data_ptr") or hasattr(x, "__cuda_array_interface__"):
        return x
    if not isinstance(x, np.ndarray) and hasattr(x, "__dlpack__") and hasattr(x, "shape"):
        return x
    return np.ascontiguousarray(x, dtype=np.float64)


class Handle:
    """One per GPU per thread (include/mfgp.h threading contract)."""

    def __init__(self, device: int = 0):
        h = C.c_void_p()
        rc = _lib.mfgp_create(device, C.byref(h))
        if rc != 0:
            raise MFGPError(f"mfgp_create(device={device}) failed with {rc}: no usable CUDA device (no CPU fallback)")
        self._h = h
        self.device = device

    def __deepcopy__(self, memo):
        return self  # a handle is a device resource (stream, workspaces): copies of a model share it

    def __copy__(self):
        return self

    def close(self):
        if getattr(self, "_h", None):
            _lib.mfgp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- helpers -----------------------------------------------------------------------------
    def _check(self, rc, what):
        if rc == 0:
            return
        msg = _lib.mfgp_last_error(self._h).decode()
        if rc > 0:
            raise NotPositiveDefiniteError(f"{what}: {msg}")
        if rc == -1:
            raise ValueError(f"{what}: {msg}")
        raise MFGPError(f"{what}: rc={rc}: {msg}")

    def set_stream(self, cuda_stream_ptr):
        """cuda_stream_ptr: integer cudaStream_t (0 = legacy default stream); None = handle's own stream."""
        if cuda_stream_ptr is None:
            self._check(_lib.mfgp_reset_stream(self._h), "reset_stream")
        else:
            self._check(_lib.mfgp_set_stream(self._h, C.c_void_p(cuda_stream_ptr)), "set_stream")

    def set_async(self, flag: bool):
        self._check(_lib.mfgp_set_async(self._h, int(flag)), "set_async")

    def sync(self) -> int:
        info = C.c_int(0)
        self._check(_lib.mfgp_sync(self._h, C.byref(info)), "sync")
        return info.value

    @property
    def sm_count(self):
        return _lib.mfgp_sm_count(self._h)

    # -- K1 ------------------------------------------------------------------------------------
    def cov(self, X, X2, theta, out=None):
        X = as_f64(X)
        N, d = X.shape[0], X.shape[1] - 1
        if X2 is not None:
            X2 = as_f64(X2)
            N2 = X2.shape[0]
        else:
            N2 = N
        theta = as_f64(theta)
        K = np.empty((N, N2)) if out is None else out
        self._check(_lib.mfgp_cov(self._h, _ptr(X), N, _ptr(X2), N2, d, _ptr(theta), _ptr(K), K.shape[1] if len(K.shape) == 2 else N2), "mfgp_cov")
        return K

    def cov_diag(self, X, theta, out=None):
        X = as_f64(X)
        N, d = X.shape[0], X.shape[1] - 1
        theta = as_f64(theta)
        o = np.empty(N) if out is None else out
        self._check(_lib.mfgp_cov_diag(self._h, _ptr(X), N, d, _ptr(theta), _ptr(o)), "mfgp_cov_diag")
        return o

    # -- exact GPR -----------------------------------------------------------------------------
    def gpr_nlml(self, X, Y, theta, noise):
        X, Y, theta = as_f64(X), as_f64(Y), as_f64(theta)
        N, d, P = X.shape[0], X.shape[1] - 1, Y.shape[1]
        out = np.empty(1)
        self._check(_lib.mfgp_gpr_nlml(self._h, _ptr(X), _ptr(Y), N, d, P, _ptr(theta), float(noise), _ptr(out)), "mfgp_gpr_nlml")
        return float(out[0])

    def gpr_nlml_grad(self, X, Y, theta, noise):
        X, Y, theta = as_f64(X), as_f64(Y), as_f64(theta)
        N, d, P = X.shape[0], X.shape[1] - 1, Y.shape[1]
        out, g = np.empty(1), np.empty(2 * d + 4)
        self._check(
            _lib.mfgp_gpr_nlml_grad(self._h, _ptr(X), _ptr(Y), N, d, P, _ptr(theta), float(noise), _ptr(out), _ptr(g)),
            "mfgp_gpr_nlml_grad",
        )
        return float(out[0]), g

    def gpr_predict(self, X, Y, Xs, theta, noise):
        X, Y, Xs, theta = as_f64(X), as_f64(Y), as_f64(Xs), as_f64(theta)
        N, d, P, Ns = X.shape[0], X.shape[1] - 1, Y.shape[1], Xs.shape[0]
        mean, var = np.empty((Ns, P)), np.empty(Ns)
        self._check(
            _lib.mfgp_gpr_predict(self._h, _ptr(X), _ptr(Y), N, d, P, _ptr(Xs), Ns, _ptr(theta), float(noise), _ptr(mean), _ptr(var)),
            "mfgp_gpr_predict",
        )
        return mean, var

    def gpr_batched_nlml_grad(self, X, Y, thetas, noises, nlml=None, grad=None, info=None, want_grad=True):
        """Host arrays or device tensors.  Y is [N, ycols]; B = thetas.shape[0] problems, problem b uses
        column b % ycols (B > ycols = several hyper-parameter sets per bin).  A non-positive Cholesky pivot raises
        NotPositiveDefiniteError unless a per-problem `info` array (int32 [B]) is passed: then info[b] holds the 1-based
        failing pivot of problem b (0 = ok), its nlml / grad are NaN, and the call returns normally."""
        X, Y, thetas, noises = as_f64(X), as_f64(Y), as_f64(thetas), as_f64(noises)
        N, d = X.shape[0], X.shape[1] - 1
        ycols = ldy = Y.shape[1]
        B = thetas.shape[0]
        if nlml is None:
            nlml = np.empty(B)
        if grad is None and want_grad:
            grad = np.empty((B, 2 * d + 4))
        rc = _lib.mfgp_gpr_batched_nlml_grad(
            self._h, _ptr(X), N, d, _ptr(Y), ldy, ycols, B, _ptr(thetas), _ptr(noises), _ptr(nlml), _ptr(grad), _ptr(info)
        )
        if not (rc > 0 and info is not None):  # with a per-problem info[] a failed Cholesky is that problem's status, not an error
            self._check(rc, "mfgp_gpr_batched_nlml_grad")
        return nlml, grad

    def gpr_posterior(self, X, Y, thetas, noises, P=1, info=None):
        """Factor B = thetas.shape[0] exact GPs once (include/mfgp.h: mfgp_gpr_posterior_create) and return a
        GprPosterior whose predict() reuses the factors.  Y is [N, ycols]; problem b uses columns
        Y[:, c : c + P] with c = (b * P) % ycols.  A non-positive Cholesky pivot raises NotPositiveDefiniteError unless a
        per-problem `info` array (int32 [B]) is passed: then info[b] holds problem b's pivot (0 = ok) and it predicts NaN."""
        X, Y, thetas, noises = as_f64(X), as_f64(Y), as_f64(thetas), as_f64(noises)
        N, d = X.shape[0], X.shape[1] - 1
        ycols = ldy = Y.shape[1]
        B = thetas.shape[0]
        out = C.c_void_p()
        rc = _lib.mfgp_gpr_posterior_create(self._h, _ptr(X), N, d, _ptr(Y), ldy, ycols, int(P), B, _ptr(thetas),
                                            _ptr(noises), _ptr(info), C.byref(out))
        if not (rc > 0 and info is not None):
            self._check(rc, "mfgp_gpr_posterior_create")
        return GprPosterior(self, out, B, N, d, int(P))

    def svgp_adam(self, X, Y, L, M, P, has_W, u, m, v, mask, lr_t, beta1, beta2, eps=1e-7, scale=1.0, kl_mult=1.0,
                  hetero=False, jitter=1e-6, lik_lower=1e-6, masked=False, lik_per_output=False):
        """len(lr_t) full-batch Adam steps on the device; u, m, v (flat layout of include/mfgp.h) are updated in place.
        Returns (loss_hist, kl_hist)."""
        X, Y, lr_t = as_f64(X), as_f64(Y), as_f64(lr_t)
        B, d = X.shape[0], X.shape[1] - 1
        cfg = SvgpCfg(L, M, P, B, d, int(hetero), float(scale), float(kl_mult), float(jitter), float(lik_lower), int(masked),
                      int(lik_per_output))
        n = int(lr_t.shape[0])
        loss, kl = np.empty(n), np.empty(n)
        mk = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        rc = _lib.mfgp_svgp_adam(self._h, C.byref(cfg), _ptr(X), _ptr(Y), int(bool(has_W)), _ptr(u), _ptr(m), _ptr(v),
                                 None if mk is None else C.c_void_p(mk.ctypes.data), _ptr(lr_t), float(beta1), float(beta2),
                                 float(eps), n, _ptr(loss), _ptr(kl))
        self._check(rc, "mfgp_svgp_adam")
        return loss, kl

    def svgp_adam_minibatch(self, X, Y, L, M, P, has_W, u, m, v, mask, lr_t, beta1, beta2, eps=1e-7, batch_size=None, seed=0,
                            pos0=0, scale=1.0, kl_mult=1.0, hetero=False, jitter=1e-6, lik_lower=1e-6, masked=False,
                            lik_per_output=False):
        """len(lr_t) Adam steps on minibatches of `batch_size` rows of the shuffled stream over the N rows of X, Y (include/
        mfgp.h: minibatch stream), starting at stream position pos0; otherwise as svgp_adam.  scale is the caller's
        (num_data / batch_size).  Returns (loss_hist, kl_hist), each step's minibatch estimate."""
        X, Y, lr_t = as_f64(X), as_f64(Y), as_f64(lr_t)
        N, d = X.shape[0], X.shape[1] - 1
        cfg = SvgpCfg(L, M, P, int(batch_size), d, int(hetero), float(scale), float(kl_mult), float(jitter), float(lik_lower),
                      int(masked), int(lik_per_output))
        n = int(lr_t.shape[0])
        loss, kl = np.empty(n), np.empty(n)
        mk = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        rc = _lib.mfgp_svgp_adam_minibatch(self._h, C.byref(cfg), _ptr(X), _ptr(Y), N, _seed(seed), int(pos0), int(bool(has_W)),
                                           _ptr(u), _ptr(m), _ptr(v), None if mk is None else C.c_void_p(mk.ctypes.data),
                                           _ptr(lr_t), float(beta1), float(beta2), float(eps), n, _ptr(loss), _ptr(kl))
        self._check(rc, "mfgp_svgp_adam_minibatch")
        return loss, kl

    def svgp_natgrad_adam(self, X, Y, L, M, P, has_W, u, m, v, mask, lr_t, gamma_t, beta1, beta2, eps=1e-7, batch_size=None,
                          seed=0, pos0=0, scale=1.0, kl_mult=1.0, hetero=False, jitter=1e-6, lik_lower=1e-6, masked=False,
                          lik_per_output=False, info=None):
        """len(lr_t) steps of GPflow's natural-gradient recipe on the device (include/mfgp.h: mfgp_svgp_natgrad_adam): a
        natural-gradient step with gamma_t[t] on q_mu and q_sqrt, then Adam on every other entry.  batch_size None: every
        evaluation uses all rows of X, Y; otherwise the two evaluations of step t read stream positions pos0 + 2 t B ...
        and pos0 + (2 t + 1) B ....  u, m, v are updated in place as in svgp_adam.  A latent whose natural-gradient step
        fails raises NotPositiveDefiniteError unless a per-latent `info` array (int32 [L]) is passed: then info[l] holds
        its first failure's pivot (0 = ok) and the call returns normally.  Returns (loss_hist, kl_hist)."""
        X, Y, lr_t, gamma_t = as_f64(X), as_f64(Y), as_f64(lr_t), as_f64(gamma_t)
        n = int(lr_t.shape[0])
        if tuple(gamma_t.shape) != (n,):
            raise ValueError(f"gamma_t must hold one step size per step ({n}), got shape {tuple(gamma_t.shape)}")
        N, d = X.shape[0], X.shape[1] - 1
        B = N if batch_size is None else int(batch_size)
        cfg = SvgpCfg(L, M, P, B, d, int(hetero), float(scale), float(kl_mult), float(jitter), float(lik_lower), int(masked),
                      int(lik_per_output))
        loss, kl = np.empty(n), np.empty(n)
        mk = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        inf = np.zeros(L, dtype=np.int32) if info is None else info
        rc = _lib.mfgp_svgp_natgrad_adam(self._h, C.byref(cfg), _ptr(X), _ptr(Y), 0 if batch_size is None else N, _seed(seed),
                                         int(pos0), int(bool(has_W)), _ptr(u), _ptr(m), _ptr(v),
                                         None if mk is None else C.c_void_p(mk.ctypes.data), _ptr(lr_t), _ptr(gamma_t),
                                         float(beta1), float(beta2), float(eps), n, _ptr(loss), _ptr(kl), _ptr(inf))
        if not (rc > 0 and info is not None and _any_nonzero(info)):  # natgrad failures are the latents' status with info
            self._check(rc, "mfgp_svgp_natgrad_adam")
        return loss, kl

    def svgp_natgrad(self, q_mu, q_sqrt, g_q_mu, g_q_sqrt, gamma, info=None):
        """One natural-gradient step (include/mfgp.h: mfgp_svgp_natgrad) for all L = q_mu.shape[1] latents: q_mu [M, L] and
        q_sqrt [L, M, M] are updated in place (C-contiguous float64 arrays or device tensors); only the lower triangles of
        q_sqrt and g_q_sqrt are read.  A latent whose step fails raises NotPositiveDefiniteError unless a per-latent
        `info` array (int32 [L]) is passed: then info[l] holds its pivot (0 = ok), that latent keeps its values bit for
        bit and the call returns normally.  Returns info."""
        for a in (q_mu, q_sqrt):
            if isinstance(a, np.ndarray) and not (a.dtype == np.float64 and a.flags.c_contiguous):
                raise ValueError("q_mu and q_sqrt must be C-contiguous float64: they are updated in place")
        g_q_mu, g_q_sqrt = as_f64(g_q_mu), as_f64(g_q_sqrt)
        M, L = q_mu.shape
        if tuple(q_sqrt.shape) != (L, M, M) or tuple(g_q_mu.shape) != (M, L) or tuple(g_q_sqrt.shape) != (L, M, M):
            raise ValueError(f"need q_mu, g_q_mu [M, L] and q_sqrt, g_q_sqrt [L, M, M] with M={M}, L={L}")
        cfg = SvgpCfg(L, M, L, 0, 1, 0, 1.0, 1.0, 0.0, 0.0, 0, 0)
        rc = _lib.mfgp_svgp_natgrad(self._h, C.byref(cfg), float(gamma), _ptr(q_mu), _ptr(q_sqrt), _ptr(g_q_mu), _ptr(g_q_sqrt),
                                    _ptr(info))
        if not (rc > 0 and info is not None):
            self._check(rc, "mfgp_svgp_natgrad")
        return info

    def minibatch_gather(self, X, Y, seed, pos0, batch_size, lo=0, count=None, step=None, Xb=None, Yb=None):
        """Rows of stream positions pos0 + step * batch_size + lo + j, j < count (default batch_size - lo), of the shuffled
        stream over the N rows of X (and Y, or None): (Xb [count, xcols], Yb [count, ycols] or None).  step: an int32
        device tensor holding the step (the data-parallel loop's counter), a host int, or None for 0.  Host arrays or
        device tensors."""
        X = as_f64(X)
        Y = None if Y is None else as_f64(Y)
        N, xcols = X.shape[0], X.shape[1]
        ycols = 0 if Y is None else Y.shape[1]
        count = int(batch_size) - int(lo) if count is None else int(count)
        Xb = np.empty((count, xcols)) if Xb is None else Xb
        if Y is not None and Yb is None:
            Yb = np.empty((count, ycols))
        if step is not None and not hasattr(step, "data_ptr"):
            step = np.array([int(step)], dtype=np.int32)
        rc = _lib.mfgp_minibatch_gather(self._h, _ptr(X), xcols, _ptr(Y), ycols, N, _seed(seed), int(pos0), _ptr(step),
                                        int(batch_size), int(lo), count, _ptr(Xb), _ptr(Yb) if Y is not None else None)
        self._check(rc, "mfgp_minibatch_gather")
        return Xb, Yb

    def gpr_batched_adam(self, X, Y, u, m, v, noises, lr_t, beta1, beta2, eps=1e-7, fix_rho=False, loss_hist=None,
                         theta_out=None, info=None):
        """nsteps = len(lr_t) Adam steps on the device for B = u.shape[0] per-bin GPs; u, m, v [B, 2d+3] are updated in
        place (host arrays or device tensors).  Returns (loss_hist, theta_out)."""
        X, Y, noises, lr_t = as_f64(X), as_f64(Y), as_f64(noises), as_f64(lr_t)
        N, d = X.shape[0], X.shape[1] - 1
        ycols = ldy = Y.shape[1]
        B, nsteps = u.shape[0], int(lr_t.shape[0])
        for a in (u, m, v):
            if isinstance(a, np.ndarray) and not (a.dtype == np.float64 and a.flags.c_contiguous):
                raise ValueError("u, m, v must be C-contiguous float64 (they are updated in place)")
        rc = _lib.mfgp_gpr_batched_adam(self._h, _ptr(X), N, d, _ptr(Y), ldy, ycols, B, _ptr(u), _ptr(m), _ptr(v), _ptr(noises),
                                        _ptr(lr_t), float(beta1), float(beta2), float(eps), int(bool(fix_rho)), nsteps,
                                        _ptr(loss_hist), _ptr(theta_out), _ptr(info))
        if not (rc > 0 and info is not None):  # per-problem status in info[]: the other problems' steps stand
            self._check(rc, "mfgp_gpr_batched_adam")
        return loss_hist, theta_out

    def gpr_batched_lbfgs(self, X, Y, u, noises, fix_rho=False, train_noise=False, m=10, maxiter=15000, maxfun=15000,
                          maxls=20, ftol=2.220446049250313e-09, gtol=1e-5, f=None, nit=None, nfev=None, status=None,
                          info=None):
        """SciPy's L-BFGS-B for B = u.shape[0] per-bin GPs on the device (include/mfgp.h: mfgp_gpr_batched_lbfgs); the
        defaults are scipy.optimize.minimize's.  u [B, 2d+3] (theta = softplus(u)) is updated in place, and so is
        noises [B] when train_noise (noise = 1e-6 + softplus(v)).  Returns (f, nit, nfev, status) [B]; status holds
        MFGP_LBFGS_* codes (LBFGS_STATUS names them).  A start point that is not positive definite raises
        NotPositiveDefiniteError unless a per-problem `info` array (int32 [B]) is passed: then that problem's status is
        not_pd, info[b] its pivot, and the others run on.  Host arrays or device tensors."""
        X, Y = as_f64(X), as_f64(Y)
        if not train_noise:
            noises = as_f64(noises)
        N, d = X.shape[0], X.shape[1] - 1
        ycols = ldy = Y.shape[1]
        B = u.shape[0]
        for a in (u, noises) if train_noise else (u,):
            if isinstance(a, np.ndarray) and not (a.dtype == np.float64 and a.flags.c_contiguous):
                raise ValueError("u (and noises when train_noise) must be C-contiguous float64: they are updated in place")
        f = np.empty(B) if f is None else f
        nit = np.empty(B, dtype=np.int32) if nit is None else nit
        nfev = np.empty(B, dtype=np.int32) if nfev is None else nfev
        status = np.empty(B, dtype=np.int32) if status is None else status
        opts = LbfgsOpts(int(m), int(maxiter), int(maxfun), int(maxls), float(ftol), float(gtol))
        rc = _lib.mfgp_gpr_batched_lbfgs(self._h, _ptr(X), N, d, _ptr(Y), ldy, ycols, B, _ptr(u), _ptr(noises),
                                         int(bool(fix_rho)), int(bool(train_noise)), C.byref(opts), _ptr(f), _ptr(nit),
                                         _ptr(nfev), _ptr(status), _ptr(info))
        if not (rc > 0 and info is not None):  # with info a failed start point is that problem's status
            self._check(rc, "mfgp_gpr_batched_lbfgs")
        return f, nit, nfev, status

    # -- graph-structured multi-fidelity kernel (reference mfgpflow/graph.py) -------------------------------
    def graph_cov(self, X, num_lf, gtheta):
        X, gtheta = as_f64(X), as_f64(gtheta)
        N, d = X.shape[0], X.shape[1] - 1
        K = np.empty((N, N))
        self._check(_lib.mfgp_graph_cov(self._h, _ptr(X), N, d, int(num_lf), _ptr(gtheta), _ptr(K), N), "mfgp_graph_cov")
        return K

    def graph_cov_diag(self, X, num_lf, gtheta):
        X, gtheta = as_f64(X), as_f64(gtheta)
        N, d = X.shape[0], X.shape[1] - 1
        out = np.empty(N)
        self._check(_lib.mfgp_graph_cov_diag(self._h, _ptr(X), N, d, int(num_lf), _ptr(gtheta), _ptr(out)), "mfgp_graph_cov_diag")
        return out

    def graph_gpr_nlml_grad(self, X, Y, num_lf, gtheta, noise, want_grad=True):
        X, Y, gtheta = as_f64(X), as_f64(Y), as_f64(gtheta)
        N, d, P = X.shape[0], X.shape[1] - 1, Y.shape[1]
        n = _lib.mfgp_graph_nparams(int(num_lf), d)
        if gtheta.shape != (n,):
            raise ValueError(f"gtheta must have {n} entries for num_LF={num_lf}, d={d}")
        out, g = np.empty(1), (np.empty(n + 1) if want_grad else None)
        self._check(_lib.mfgp_graph_gpr_nlml_grad(self._h, _ptr(X), _ptr(Y), N, d, P, int(num_lf), _ptr(gtheta), float(noise),
                                                  _ptr(out), _ptr(g)), "mfgp_graph_gpr_nlml_grad")
        return float(out[0]), g

    # -- SVGP ----------------------------------------------------------------------------------
    def svgp_elbo_grad(self, X, Y, Z, thetas, W, q_mu, q_sqrt, lik_var, scale=1.0, kl_mult=1.0, hetero=False,
                       jitter=1e-6, want_grad=True, masked=False):
        """lik_var: scalar (Gaussian / HeteroscedasticGaussian) or a [P] vector (MaskedGaussian: one variance per output);
        g_lik_var comes back as a float or a [P] array accordingly.  masked=True skips the NaN entries of Y."""
        X, Y, Z, thetas, q_mu, q_sqrt = map(as_f64, (X, Y, Z, thetas, q_mu, q_sqrt))
        W = None if W is None else as_f64(W)
        B, d = X.shape[0], X.shape[1] - 1
        M, L = q_mu.shape
        P = L if W is None else W.shape[0]
        per_out = np.ndim(lik_var) > 0 and np.size(lik_var) > 1
        lv = np.ascontiguousarray(np.ravel(lik_var), dtype=np.float64)
        if lv.size != (P if per_out else 1):
            raise ValueError(f"lik_var must be a scalar or have one entry per output ({P}); got {lv.size}")
        cfg = SvgpCfg(L, M, P, B, d, int(hetero), float(scale), float(kl_mult), float(jitter), 0.0, int(masked), int(per_out))
        elbo, kl, glik = np.empty(1), np.empty(1), np.zeros(lv.size)
        if want_grad:
            gZ, gth, gqm, gqs = np.zeros((M, d + 1)), np.zeros((L, 2 * d + 3)), np.zeros((M, L)), np.zeros((L, M, M))
            gW = None if W is None else np.zeros((P, L))
        else:
            gZ = gth = gqm = gqs = gW = None
        rc = _lib.mfgp_svgp_elbo_grad_v(
            self._h, C.byref(cfg), _ptr(X), _ptr(Y), _ptr(Z), _ptr(thetas), _ptr(W), _ptr(q_mu), _ptr(q_sqrt),
            _ptr(lv), _ptr(elbo), _ptr(kl), _ptr(gZ), _ptr(gth), _ptr(gW), _ptr(gqm), _ptr(gqs),
            _ptr(glik) if want_grad else None,
        )
        self._check(rc, "mfgp_svgp_elbo_grad")
        return dict(elbo=float(elbo[0]), kl=float(kl[0]), g_Z=gZ, g_thetas=gth, g_W=gW, g_q_mu=gqm, g_q_sqrt=gqs,
                    g_lik_var=glik.copy() if per_out else float(glik[0]))

    def svgp_predict(self, Xs, Z, thetas, W, q_mu, q_sqrt, jitter=1e-6):
        Xs, Z, thetas, q_mu, q_sqrt = map(as_f64, (Xs, Z, thetas, q_mu, q_sqrt))
        W = None if W is None else as_f64(W)
        Ns, d = Xs.shape[0], Xs.shape[1] - 1
        M, L = q_mu.shape
        P = L if W is None else W.shape[0]
        cfg = SvgpCfg(L, M, P, Ns, d, 0, 1.0, 1.0, float(jitter), 0.0, 0, 0)
        mean, var = np.empty((Ns, P)), np.empty((Ns, P))
        rc = _lib.mfgp_svgp_predict(self._h, C.byref(cfg), _ptr(Xs), Ns, _ptr(Z), _ptr(thetas), _ptr(W), _ptr(q_mu),
                                    _ptr(q_sqrt), _ptr(mean), _ptr(var))
        self._check(rc, "mfgp_svgp_predict")
        return mean, var

    def svgp_posterior(self, Z, thetas, W, q_mu, q_sqrt, jitter=1e-6, info=None):
        """Factor the inducing covariances of the L = q_mu.shape[1] latents once (include/mfgp.h:
        mfgp_svgp_posterior_create) and return an SvgpPosterior whose predict() gives what svgp_predict gives for the same
        arguments.  W [P, L] or None (P = L).  A non-positive Cholesky pivot raises NotPositiveDefiniteError unless a
        per-latent `info` array (int32 [L]) is passed: then info[l] holds latent l's pivot (0 = ok) and it predicts NaN."""
        Z, thetas, q_mu, q_sqrt = map(as_f64, (Z, thetas, q_mu, q_sqrt))
        W = None if W is None else as_f64(W)
        M, L = q_mu.shape
        d = Z.shape[1] - 1
        P = L if W is None else W.shape[0]
        cfg = SvgpCfg(L, M, P, 0, d, 0, 1.0, 1.0, float(jitter), 0.0, 0, 0)
        out = C.c_void_p()
        rc = _lib.mfgp_svgp_posterior_create(self._h, C.byref(cfg), _ptr(Z), _ptr(thetas), _ptr(W), _ptr(q_mu), _ptr(q_sqrt),
                                             _ptr(info), C.byref(out))
        if not (rc > 0 and info is not None):
            self._check(rc, "mfgp_svgp_posterior_create")
        return SvgpPosterior(self, out, L, M, P, d)

    # -- building blocks -------------------------------------------------------------------------
    def cov_grad(self, X, theta, G, scale=1.0):
        """scale * sum_ij G_ij dK_ij/dtheta (lower triangle of the symmetric G, off-diagonal twice) and, last, scale * trace(G)."""
        X, theta, G = as_f64(X), as_f64(theta), as_f64(G)
        N, d = X.shape[0], X.shape[1] - 1
        out = np.empty(2 * d + 4)
        self._check(_lib.mfgp_cov_grad(self._h, _ptr(X), N, d, _ptr(theta), _ptr(G), G.shape[1], float(scale), _ptr(out)), "mfgp_cov_grad")
        return out

    def gemm(self, ta, tb, A, B, alpha=1.0, beta=0.0, C_in=None):
        A, B = as_f64(A), as_f64(B)
        m = A.shape[1] if ta else A.shape[0]
        k = A.shape[0] if ta else A.shape[1]
        n = B.shape[0] if tb else B.shape[1]
        Cm = np.zeros((m, n)) if C_in is None else np.ascontiguousarray(C_in, dtype=np.float64).copy()
        rc = _lib.mfgp_gemm(self._h, b"T" if ta else b"N", b"T" if tb else b"N", m, n, k, float(alpha), _ptr(A),
                            A.shape[1], _ptr(B), B.shape[1], float(beta), _ptr(Cm), n)
        self._check(rc, "mfgp_gemm")
        return Cm

    def potrf(self, A, want_inverse=False):
        """A: [N, lda>=N even] lower-valid.  Returns L (in a copy) and optionally inv(L)."""
        A = np.ascontiguousarray(A, dtype=np.float64).copy()
        N, lda = A.shape
        if want_inverse:
            Wm = np.empty((N, lda))
            self._check(_lib.mfgp_potrf_inv(self._h, _ptr(A), N, lda, _ptr(Wm), lda), "mfgp_potrf_inv")
            return A, Wm
        self._check(_lib.mfgp_potrf(self._h, _ptr(A), N, lda), "mfgp_potrf")
        return A

    def potrf_device(self, A_dev, N, lda):
        self._check(_lib.mfgp_potrf(self._h, _ptr(A_dev), N, lda), "mfgp_potrf")

    def peer_store(self, src, dst_ptrs, count):
        """One kernel: `count` doubles from `src` into every raw device address in `dst_ptrs` (peer GPUs' mapped buffers or local)."""
        arr = (C.c_void_p * len(dst_ptrs))(*[C.c_void_p(int(p)) for p in dst_ptrs])
        self._check(_lib.mfgp_peer_store(self._h, _ptr(src), int(count), len(dst_ptrs), arr), "mfgp_peer_store")

    WS_POOL, WS_MEASURE, WS_FIXED = 0, 1, 2

    def workspace(self, mode: int) -> int:
        """Source of the following calls' temporaries (include/mfgp.h: mfgp_workspace); returns the measured bytes."""
        out = C.c_long(0)
        self._check(_lib.mfgp_workspace(self._h, int(mode), C.byref(out)), "mfgp_workspace")
        return int(out.value)

    def graph_mem_trim(self):
        """Return the memory that destroyed CUDA graphs still reserve on this device to the driver (see include/mfgp.h)."""
        self._check(_lib.mfgp_graph_mem_trim(self._h), "mfgp_graph_mem_trim")

    def fp64_peak(self, kind: int, iters: int = 20000) -> float:
        out = C.c_double(0.0)
        self._check(_lib.mfgp_fp64_peak(self._h, kind, iters, C.byref(out)), "mfgp_fp64_peak")
        return out.value


class _Posterior:
    """A device-resident posterior owned by this object: freed by close() or when the object is collected."""

    _destroy = None  # the C-ABI destroy function of the subclass's posterior type

    def __init__(self, handle, ptr):
        self.handle, self._p = handle, ptr

    def _xs(self, Xs):
        """Xs as float64 [Ns, d+1], after checking that the posterior is open."""
        if not self._p:
            raise ValueError(f"{type(self).__name__} is closed")
        Xs = as_f64(Xs)
        if Xs.shape[1] != self.d + 1:
            raise ValueError(f"Xs must have {self.d + 1} columns")
        return Xs

    def close(self):
        if getattr(self, "_p", None):
            type(self)._destroy(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class GprPosterior(_Posterior):
    """Device-resident factors of B exact GPs (W = L^-1, a = W Y) made by Handle.gpr_posterior: a snapshot of the
    hyper-parameters and data at creation.  predict() returns mean [B, Ns, P] and var [B, Ns]."""

    _destroy = _lib.mfgp_gpr_posterior_destroy

    def __init__(self, handle, ptr, B, N, d, P):
        super().__init__(handle, ptr)
        self.B, self.N, self.d, self.P = B, N, d, P

    def predict(self, Xs, mean=None, var=None):
        """Host arrays or device tensors; mean / var (optional outputs) may be device tensors (zero-copy)."""
        Xs = self._xs(Xs)
        Ns = Xs.shape[0]
        mean = np.empty((self.B, Ns, self.P)) if mean is None else mean
        var = np.empty((self.B, Ns)) if var is None else var
        self.handle._check(_lib.mfgp_gpr_posterior_predict(self.handle._h, self._p, _ptr(Xs), Ns, _ptr(mean), _ptr(var)),
                           "mfgp_gpr_posterior_predict")
        return mean, var

    def predict_grad(self, Xs, mean=None, var=None, dmean=None, dvar=None):
        """predict() plus the gradients with respect to the d continuous coordinates of each test point:
        (mean [B, Ns, P], var [B, Ns], dmean [B, Ns, P, d], dvar [B, Ns, d]).  Host arrays or device tensors."""
        Xs = self._xs(Xs)
        Ns = Xs.shape[0]
        mean = np.empty((self.B, Ns, self.P)) if mean is None else mean
        var = np.empty((self.B, Ns)) if var is None else var
        dmean = np.empty((self.B, Ns, self.P, self.d)) if dmean is None else dmean
        dvar = np.empty((self.B, Ns, self.d)) if dvar is None else dvar
        self.handle._check(_lib.mfgp_gpr_posterior_predict_grad(self.handle._h, self._p, _ptr(Xs), Ns, _ptr(mean), _ptr(var),
                                                                _ptr(dmean), _ptr(dvar)), "mfgp_gpr_posterior_predict_grad")
        return mean, var, dmean, dvar

    def predict_cov(self, Xs, mean=None, cov=None):
        """Mean [B, Ns, P] and the joint covariance [B, Ns, Ns] over the test points (the same for every column of a
        problem).  mean is predict()'s mean and diag(cov) predict()'s var, bit for bit.  Host arrays or device tensors."""
        Xs = self._xs(Xs)
        Ns = Xs.shape[0]
        mean = np.empty((self.B, Ns, self.P)) if mean is None else mean
        cov = np.empty((self.B, Ns, Ns)) if cov is None else cov
        self.handle._check(_lib.mfgp_gpr_posterior_predict_cov(self.handle._h, self._p, _ptr(Xs), Ns, _ptr(mean), _ptr(cov)),
                           "mfgp_gpr_posterior_predict_cov")
        return mean, cov

    def sample(self, Xs, z, jitter=1e-6, samples=None, info=None):
        """Joint draws [B, Ns, S, P]: samples[b] = mean[b] + L_b z[b] over the test-point axis, L_b L_b^T = cov[b] +
        jitter I, for standard normals z [B, Ns, S, P].  A problem whose factor fails raises NotPositiveDefiniteError
        unless a per-problem `info` array (int32 [B]) is passed: then info[b] holds its 1-based pivot (0 = ok) and its
        samples are NaN.  Host arrays or device tensors."""
        Xs = self._xs(Xs)
        Ns = Xs.shape[0]
        z = as_f64(z)
        if tuple(z.shape[:2]) != (self.B, Ns) or len(z.shape) != 4 or z.shape[3] != self.P:
            raise ValueError(f"z must be [B={self.B}, Ns={Ns}, S, P={self.P}]")
        S = int(z.shape[2])
        samples = np.empty((self.B, Ns, S, self.P)) if samples is None else samples
        rc = _lib.mfgp_gpr_posterior_sample(self.handle._h, self._p, _ptr(Xs), Ns, S, float(jitter), _ptr(z), _ptr(samples),
                                            _ptr(info))
        if not (rc > 0 and info is not None):
            self.handle._check(rc, "mfgp_gpr_posterior_sample")
        return samples

    def draw_f(self, Xs, num_samples=None, full_cov=True, full_output_cov=False, seed=None, info=None):
        """GPflow's predict_f_samples over every problem: [B, Ns, S, P] (S = 1 when num_samples is None), from
        z = np.random.default_rng(seed).standard_normal((B, Ns, S, P)).  full_cov=True: sample() with GPflow's default
        jitter 1e-6; full_cov=False: mean + sqrt(var) z from predict(), without jitter."""
        if full_output_cov:
            raise NotImplementedError("full_output_cov: the outputs of an exact GP are independent given its kernel")
        Xs = self._xs(Xs)
        S = 1 if num_samples is None else int(num_samples)
        z = np.random.default_rng(seed).standard_normal((self.B, Xs.shape[0], S, self.P))
        if full_cov:
            return self.sample(Xs, z, jitter=1e-6, info=info)
        mean, var = self.predict(Xs)
        return mean[:, :, None, :] + np.sqrt(var)[:, :, None, None] * z


class SvgpPosterior(_Posterior):
    """Device-resident factors of an SVGP (Wm = Lm^-1, tril(q_sqrt), q_mu, W) made by Handle.svgp_posterior: a snapshot of
    the parameters at creation.  predict() returns mean [Ns, P] and var [Ns, P], as Handle.svgp_predict."""

    _destroy = _lib.mfgp_svgp_posterior_destroy

    def __init__(self, handle, ptr, L, M, P, d):
        super().__init__(handle, ptr)
        self.L, self.M, self.P, self.d = L, M, P, d

    def predict(self, Xs, mean=None, var=None):
        """Host arrays or device tensors; mean / var (optional outputs) may be device tensors (zero-copy)."""
        Xs = self._xs(Xs)
        Ns = Xs.shape[0]
        mean = np.empty((Ns, self.P)) if mean is None else mean
        var = np.empty((Ns, self.P)) if var is None else var
        self.handle._check(_lib.mfgp_svgp_posterior_predict(self.handle._h, self._p, _ptr(Xs), Ns, _ptr(mean), _ptr(var)),
                           "mfgp_svgp_posterior_predict")
        return mean, var

    def predict_grad(self, Xs, mean=None, var=None, dmean=None, dvar=None):
        """predict() plus the gradients with respect to the d continuous coordinates of each test point:
        (mean [Ns, P], var [Ns, P], dmean [Ns, P, d], dvar [Ns, P, d]).  Host arrays or device tensors."""
        Xs = self._xs(Xs)
        Ns = Xs.shape[0]
        mean = np.empty((Ns, self.P)) if mean is None else mean
        var = np.empty((Ns, self.P)) if var is None else var
        dmean = np.empty((Ns, self.P, self.d)) if dmean is None else dmean
        dvar = np.empty((Ns, self.P, self.d)) if dvar is None else dvar
        self.handle._check(_lib.mfgp_svgp_posterior_predict_grad(self.handle._h, self._p, _ptr(Xs), Ns, _ptr(mean),
                                                                 _ptr(var), _ptr(dmean), _ptr(dvar)),
                           "mfgp_svgp_posterior_predict_grad")
        return mean, var, dmean, dvar

    def predict_cov(self, Xs, mean=None, cov=None):
        """Mean [Ns, P] and each output's joint covariance cov [P, Ns, Ns] over the test points (GPflow
        SVGP.predict_f(full_cov=True)).  mean is predict()'s mean and diag(cov[p]) predict()'s var[:, p], bit for bit.
        Host arrays or device tensors."""
        Xs = self._xs(Xs)
        Ns = Xs.shape[0]
        mean = np.empty((Ns, self.P)) if mean is None else mean
        cov = np.empty((self.P, Ns, Ns)) if cov is None else cov
        self.handle._check(_lib.mfgp_svgp_posterior_predict_cov(self.handle._h, self._p, _ptr(Xs), Ns, _ptr(mean), _ptr(cov)),
                           "mfgp_svgp_posterior_predict_cov")
        return mean, cov

    def sample(self, Xs, z, jitter=1e-6, samples=None, info=None):
        """Draws [P, Ns, S], each output on its own: samples[p] = mean[:, p] + L_p z[p] over the test-point axis,
        L_p L_p^T = cov[p] + jitter I, for standard normals z [P, Ns, S].  An output whose factor fails raises
        NotPositiveDefiniteError unless a per-output `info` array (int32 [P]) is passed: then info[p] holds its 1-based
        pivot (0 = ok) and its samples are NaN.  Host arrays or device tensors."""
        Xs = self._xs(Xs)
        Ns = Xs.shape[0]
        z = as_f64(z)
        if len(z.shape) != 3 or tuple(z.shape[:2]) != (self.P, Ns):
            raise ValueError(f"z must be [P={self.P}, Ns={Ns}, S]")
        S = int(z.shape[2])
        samples = np.empty((self.P, Ns, S)) if samples is None else samples
        rc = _lib.mfgp_svgp_posterior_sample(self.handle._h, self._p, _ptr(Xs), Ns, S, float(jitter), _ptr(z), _ptr(samples),
                                             _ptr(info))
        if not (rc > 0 and info is not None):
            self.handle._check(rc, "mfgp_svgp_posterior_sample")
        return samples

    def draw_f(self, Xs, num_samples=None, full_cov=True, full_output_cov=False, seed=None, info=None):
        """GPflow's predict_f_samples with full_output_cov=False: [P, Ns, S] (S = 1 when num_samples is None), from
        z = np.random.default_rng(seed).standard_normal((P, Ns, S)).  full_cov=True: sample() with GPflow's default
        jitter 1e-6; full_cov=False: mean + sqrt(var) z from predict(), without jitter."""
        if full_output_cov:
            raise NotImplementedError("full_output_cov: draws correlated across the outputs through W are not supported")
        Xs = self._xs(Xs)
        S = 1 if num_samples is None else int(num_samples)
        z = np.random.default_rng(seed).standard_normal((self.P, Xs.shape[0], S))
        if full_cov:
            return self.sample(Xs, z, jitter=1e-6, info=info)
        mean, var = self.predict(Xs)
        return mean.T[:, :, None] + np.sqrt(var).T[:, :, None] * z


_default = {}


def default_handle(device: int = 0) -> Handle:
    if device not in _default:
        _default[device] = Handle(device)
    return _default[device]
