// api.cu -- extern "C" entry points of libmfgp.so (see include/mfgp.h for the contract).
#include <cuda_runtime.h>

#include <cmath>
#include <vector>

#include "chol.cuh"
#include "common.cuh"
#include "cov.cuh"
#include "gemm.cuh"
#include "gpr.cuh"
#include "gpr_small.cuh"
#include "mathx.cuh"
#include "svgp.cuh"

#define CHECK_H(h) \
    if (!(h)) return MFGP_ERR_ARG

extern "C" {

int mfgp_version(void) { return 100; }

int mfgp_create(int device, mfgp_handle** out) {
    if (!out) return MFGP_ERR_ARG;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return MFGP_ERR_CUDA;  // no CPU fallback
    if (device < 0 || device >= ndev) return MFGP_ERR_ARG;
    mfgp_handle* h = new mfgp_handle();
    h->device = device;
    if (cudaSetDevice(device) != cudaSuccess) { delete h; return MFGP_ERR_CUDA; }
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    h->sm_count = prop.multiProcessorCount;
    cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking);
    {
        // the panel chain of potrf runs on the aux stream next to the trailing update's thousands of CTAs: highest priority,
        // so that its few CTAs are scheduled first
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        cudaStreamCreateWithPriority(&h->aux_stream, cudaStreamNonBlocking, hi);
    }
    cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking);
    for (auto& e : h->ev) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    h->stream = h->own_stream;
    cudaMalloc(&h->d_info, sizeof(int));
    cudaMemset(h->d_info, 0, sizeof(int));
    cudaMallocHost(&h->h_info, sizeof(int));
    *h->h_info = 0;
    // keep freed temporaries in the pool: no trim at synchronisation points
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        unsigned long long thr = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    if (cudaGetLastError() != cudaSuccess) { delete h; return MFGP_ERR_CUDA; }
    *out = h;
    return 0;
}

int mfgp_destroy(mfgp_handle* h) {
    CHECK_H(h);
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    if (h->ws.arena) cudaFree(h->ws.arena);  // a workspace arena left behind by a caller that never went back to MFGP_WS_POOL
    for (auto& e : h->ev) cudaEventDestroy(e);
    cudaStreamDestroy(h->own_stream);
    cudaStreamDestroy(h->aux_stream);
    cudaStreamDestroy(h->copy_stream);
    cudaFree(h->d_info);
    cudaFreeHost(h->h_info);
    delete h;
    return 0;
}

int mfgp_set_stream(mfgp_handle* h, void* s) {
    CHECK_H(h);
    h->stream = static_cast<cudaStream_t>(s);
    return 0;
}
int mfgp_reset_stream(mfgp_handle* h) {
    CHECK_H(h);
    h->stream = h->own_stream;
    return 0;
}
int mfgp_set_async(mfgp_handle* h, int async) {
    CHECK_H(h);
    h->async = async;
    return 0;
}
int mfgp_sync(mfgp_handle* h, int* info_out) {
    CHECK_H(h);
    cudaSetDevice(h->device);
    CUDA_TRY(h, cudaMemcpyAsync(h->h_info, h->d_info, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    const int info = *h->h_info;
    if (info) CUDA_TRY(h, cudaMemsetAsync(h->d_info, 0, sizeof(int), h->stream));
    if (info_out) *info_out = info;
    return 0;
}
const char* mfgp_last_error(mfgp_handle* h) { return h ? h->err : "null handle"; }
int mfgp_sm_count(mfgp_handle* h) { return h ? h->sm_count : 0; }

// ---------------------------------------------------------------------------------------------
int mfgp_cov(mfgp_handle* h, const double* X, int N, const double* X2, int N2, int d, const double* theta, double* K,
             long ldk) {
    CHECK_H(h);
    if (!X || !theta || !K || N < 0 || d < 1 || d > MFGP_MAX_D) return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_cov: bad argument");
    cudaSetDevice(h->device);
    const bool sym = (X2 == nullptr);
    if (sym) N2 = N;
    if (ldk < N2) return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_cov: ldk < N2");
    if (N == 0 || N2 == 0) return 0;
    Scope sc(h);
    CovArgs c{};
    c.Xa = sc.in(X, (size_t)N * (d + 1));
    c.Na = N;
    c.Xb = sym ? c.Xa : sc.in(X2, (size_t)N2 * (d + 1));
    c.Nb = N2;
    c.d = d;
    c.theta = sc.in(theta, 2 * d + 3);
    c.theta_stride = 0;
    c.K = sc.out(K, (size_t)N * ldk);
    c.ldk = ldk;
    c.symmetric = sym;
    c.mirror = sym;
    c.batch = 1;
    if (!sc.ok) return sc.finish();
    if (launch_cov(h->stream, c)) return mfgp_fail(h, MFGP_ERR_CUDA, "cov launch failed");
    return sc.finish();
}

int mfgp_cov_diag(mfgp_handle* h, const double* X, int N, int d, const double* theta, double* out) {
    CHECK_H(h);
    if (!X || !theta || !out || N < 0 || d < 1 || d > MFGP_MAX_D) return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_cov_diag: bad argument");
    cudaSetDevice(h->device);
    if (N == 0) return 0;
    Scope sc(h);
    const double* dX = sc.in(X, (size_t)N * (d + 1));
    const double* dth = sc.in(theta, 2 * d + 3);
    double* dout = sc.out(out, N);
    if (!sc.ok) return sc.finish();
    if (launch_cov_diag(h->stream, dX, N, d, dth, 0, dout, 0, 1)) return mfgp_fail(h, MFGP_ERR_CUDA, "cov_diag launch failed");
    return sc.finish();
}

// ---------------------------------------------------------------------------------------------
// Small shared-kernel GPR (N <= 64: the reference's own HBS multi-bin model, tests/test_ho2021_multibin.py): the P-column
// objective is the SUM over columns of the one-column objectives at the same hyper-parameters -- and so is its gradient,
// -1/2 tr((sum_p alpha_p alpha_p^T - P K^-1) dK) -- so one launch of the batched K6 kernel (problem p = column p) followed
// by a fixed-order reduction replaces the ~30 launches of the blocked path (213 us -> ~60 us per evaluation).
namespace {
__global__ void small_shared_fill_kernel(const double* __restrict__ theta, const double* __restrict__ noise, int np, int P,
                                         double* __restrict__ th, double* __restrict__ nz) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < P * np) th[i] = theta[i % np];
    if (i < P) nz[i] = noise[0];
}
__global__ void small_shared_reduce_kernel(const double* __restrict__ nl, const double* __restrict__ g, int P, int ng,
                                           double* __restrict__ nlml, double* __restrict__ grad) {
    const int q = threadIdx.x;  // one thread per output, columns summed in index order (deterministic)
    if (q == 0) {
        double s = 0.0;
        for (int p = 0; p < P; ++p) s += nl[p];
        *nlml = s;
    } else if (grad && q <= ng) {
        double s = 0.0;
        for (int p = 0; p < P; ++p) s += g[(long)p * ng + (q - 1)];
        grad[q - 1] = s;
    }
}
}  // namespace

static int gpr_common(mfgp_handle* h, const double* X, const double* Y, int N, int d, int P, const double* theta,
                      double noise, double* nlml, double* grad) {
    CHECK_H(h);
    if (!X || !Y || !theta || !nlml || N < 1 || P < 1 || d < 1 || d > MFGP_MAX_D)
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_gpr_nlml: bad argument");
    cudaSetDevice(h->device);
    Scope sc(h);
    const double* dX = sc.in(X, (size_t)N * (d + 1));
    const double* dY = sc.in(Y, (size_t)N * P);
    const double* dth = sc.in(theta, 2 * d + 3);
    const double* dnz = sc.in(&noise, 1);
    double* dn = sc.out(nlml, 1);
    double* dg = grad ? sc.out(grad, 2 * d + 4) : nullptr;
    if (!sc.ok) return sc.finish();
    if (N <= MFGP_SMALL_MAX_N && d <= MFGP_SMALL_MAX_D && P <= 8192) {
        const int np = 2 * d + 3;
        double* th = sc.alloc<double>((size_t)P * np);
        double* nz = sc.alloc<double>(P);
        double* nl = sc.alloc<double>(P);
        double* gg = grad ? sc.alloc<double>((size_t)P * (np + 1)) : nullptr;
        if (!sc.ok) return sc.finish();
        small_shared_fill_kernel<<<(P * np + 255) / 256, 256, 0, h->stream>>>(dth, dnz, np, P, th, nz);
        SmallArgs a{};
        a.X = dX; a.N = N; a.d = d; a.Y = dY; a.ldy = P; a.ycols = P; a.B = P;
        a.theta = th; a.noise = nz; a.nlml = nl; a.grad = gg; a.info = nullptr; a.d_info = h->d_info;
        if (launch_gpr_small(h->stream, a)) return mfgp_fail(h, MFGP_ERR_CUDA, "gpr_small launch failed");
        small_shared_reduce_kernel<<<1, 64, 0, h->stream>>>(nl, gg, P, np + 1, dn, dg);
        return sc.finish();
    }
    int rc = gpr_nlml_grad_device(h, sc, dX, dY, P, 0, 0, 0, N, d, P, 1, dth, dnz, dn, dg, nullptr);
    if (rc) return rc;
    return sc.finish();
}

int mfgp_gpr_nlml(mfgp_handle* h, const double* X, const double* Y, int N, int d, int P, const double* theta,
                  double noise, double* nlml) {
    return gpr_common(h, X, Y, N, d, P, theta, noise, nlml, nullptr);
}
int mfgp_gpr_nlml_grad(mfgp_handle* h, const double* X, const double* Y, int N, int d, int P, const double* theta,
                       double noise, double* nlml, double* grad) {
    if (!grad) return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_gpr_nlml_grad: grad is NULL");
    return gpr_common(h, X, Y, N, d, P, theta, noise, nlml, grad);
}

int mfgp_gpr_predict(mfgp_handle* h, const double* X, const double* Y, int N, int d, int P, const double* Xs, int Ns,
                     const double* theta, double noise, double* mean, double* var) {
    CHECK_H(h);
    if (!X || !Y || !Xs || !theta || !mean || !var || N < 1 || P < 1 || Ns < 1 || d < 1 || d > MFGP_MAX_D)
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_gpr_predict: bad argument");
    cudaSetDevice(h->device);
    Scope sc(h);
    const double* dX = sc.in(X, (size_t)N * (d + 1));
    const double* dY = sc.in(Y, (size_t)N * P);
    const double* dXs = sc.in(Xs, (size_t)Ns * (d + 1));
    const double* dth = sc.in(theta, 2 * d + 3);
    const double* dnz = sc.in(&noise, 1);
    double* dm = sc.out(mean, (size_t)Ns * P);
    double* dv = sc.out(var, Ns);
    if (!sc.ok) return sc.finish();
    int rc = gpr_predict_device(h, sc, dX, dY, N, d, P, dXs, Ns, dth, dnz, dm, dv);
    if (rc) return rc;
    return sc.finish();
}

// Large batches with HOST theta / results: the call is pipelined in chunks -- hyper-parameters of chunk c+1 travel to the
// device (H2D engine, aux stream) and results of chunk c-1 travel back (D2H engine, copy stream) while chunk c is being
// evaluated, so the end-to-end rate through the C-ABI approaches the device rate instead of (H2D + kernel + D2H) in series.
static int batched_small_pipelined(mfgp_handle* h, const double* X, int N, int d, const double* Y, long ldy, int ycols, int B,
                                   const double* theta, const double* noise, double* nlml, double* grad, int* info) {
    const int np = 2 * d + 3;
    Scope sc(h);
    cudaStream_t s = h->stream, sin = h->aux_stream, sout = h->copy_stream;
    const double* dX = sc.in(X, (size_t)N * (d + 1));
    const double* dY = sc.in(Y, (size_t)N * ldy);
    double* dth = sc.alloc<double>((size_t)B * np);
    double* dnz = sc.alloc<double>(B);
    double* dn = sc.alloc<double>(B);
    double* dg = grad ? sc.alloc<double>((size_t)B * (np + 1)) : nullptr;
    int* di = info ? sc.alloc<int>(B, true) : nullptr;
    if (!sc.ok) return sc.finish();
    const long wave = (long)h->sm_count * 12;  // one resident wave of warps
    long chunk = ((B / 8 + wave - 1) / wave) * wave;
    if (chunk < 4 * wave) chunk = 4 * wave;
    const int nch = (int)((B + chunk - 1) / chunk);
    std::vector<cudaEvent_t> ev(2 * nch + 2);
    for (auto& e : ev) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    cudaEventRecord(ev[2 * nch], s);  // buffers exist (stream-ordered allocation) and X, Y are staged
    cudaStreamWaitEvent(sin, ev[2 * nch], 0);
    cudaStreamWaitEvent(sout, ev[2 * nch], 0);
    for (int c = 0; c < nch; ++c) {
        const long b0 = (long)c * chunk, nb = (B - b0) < chunk ? (B - b0) : chunk;
        cudaMemcpyAsync(dth + b0 * np, theta + b0 * np, (size_t)nb * np * 8, cudaMemcpyHostToDevice, sin);
        cudaMemcpyAsync(dnz + b0, noise + b0, (size_t)nb * 8, cudaMemcpyHostToDevice, sin);
        cudaEventRecord(ev[c], sin);
    }
    int rc = 0;
    for (int c = 0; c < nch && rc == 0; ++c) {
        const long b0 = (long)c * chunk, nb = (B - b0) < chunk ? (B - b0) : chunk;
        cudaStreamWaitEvent(s, ev[c], 0);
        SmallArgs a{};
        a.X = dX; a.N = N; a.d = d; a.Y = dY; a.ldy = ldy; a.ycols = ycols; a.B = (int)nb; a.prob0 = (int)(b0 % ycols);
        a.theta = dth + b0 * np; a.noise = dnz + b0; a.nlml = dn + b0; a.grad = dg ? dg + b0 * (np + 1) : nullptr;
        a.info = di ? di + b0 : nullptr; a.d_info = h->d_info;
        if (launch_gpr_small(s, a)) rc = mfgp_fail(h, MFGP_ERR_CUDA, "gpr_small launch failed");
        cudaEventRecord(ev[nch + c], s);
        cudaStreamWaitEvent(sout, ev[nch + c], 0);
        cudaMemcpyAsync(nlml + b0, dn + b0, (size_t)nb * 8, cudaMemcpyDeviceToHost, sout);
        if (dg) cudaMemcpyAsync(grad + b0 * (np + 1), dg + b0 * (np + 1), (size_t)nb * (np + 1) * 8, cudaMemcpyDeviceToHost, sout);
        if (di) cudaMemcpyAsync(info + b0, di + b0, (size_t)nb * sizeof(int), cudaMemcpyDeviceToHost, sout);
    }
    cudaEventRecord(ev[2 * nch + 1], sout);
    cudaStreamWaitEvent(s, ev[2 * nch + 1], 0);  // the handle's stream owns the result (and the frees) again
    sc.host_out = true;                          // host outputs were written: finish() must synchronise
    const int fin = sc.finish();
    for (auto& e : ev) cudaEventDestroy(e);
    return rc ? rc : fin;
}

int mfgp_gpr_batched_nlml_grad(mfgp_handle* h, const double* X, int N, int d, const double* Y, long ldy, int ycols,
                               int B, const double* theta, const double* noise, double* nlml, double* grad, int* info) {
    CHECK_H(h);
    if (!X || !Y || !theta || !noise || !nlml || N < 1 || B < 0 || d < 1 || d > MFGP_MAX_D || ycols < 1 || ldy < ycols)
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_gpr_batched_nlml_grad: bad argument");
    cudaSetDevice(h->device);
    if (B == 0) return 0;
    {
        const bool host_io = !mfgp_is_device_ptr(theta) && !mfgp_is_device_ptr(noise) && !mfgp_is_device_ptr(nlml) &&
                             (!grad || !mfgp_is_device_ptr(grad)) && (!info || !mfgp_is_device_ptr(info));
        if (host_io && N <= MFGP_SMALL_MAX_N && d <= MFGP_SMALL_MAX_D && B >= 16L * h->sm_count * 12)
            return batched_small_pipelined(h, X, N, d, Y, ldy, ycols, B, theta, noise, nlml, grad, info);
    }
    Scope sc(h);
    const double* dX = sc.in(X, (size_t)N * (d + 1));
    const double* dY = sc.in(Y, (size_t)N * ldy);
    const double* dth = sc.in(theta, (size_t)B * (2 * d + 3));
    const double* dnz = sc.in(noise, B);
    double* dn = sc.out(nlml, B);
    double* dg = grad ? sc.out(grad, (size_t)B * (2 * d + 4)) : nullptr;
    int* di = info ? sc.out(info, B, true) : nullptr;
    if (!sc.ok) return sc.finish();
    if (N <= MFGP_SMALL_MAX_N && d <= MFGP_SMALL_MAX_D) {
        SmallArgs a{};
        a.X = dX; a.N = N; a.d = d; a.Y = dY; a.ldy = ldy; a.ycols = ycols; a.B = B;
        a.theta = dth; a.noise = dnz; a.nlml = dn; a.grad = dg; a.info = di; a.d_info = h->d_info;
        if (launch_gpr_small(h->stream, a))
            return mfgp_fail(h, MFGP_ERR_CUDA, "gpr_small launch failed");
    } else {
        // blocked path, chunked so that 3 N^2 workspaces per problem fit comfortably
        const long chunk =
            chunk_by_free_memory((size_t)3 * N * round_up(N, 2) * 8 + (size_t)chol_dinv_count(N, 1) * 8, 1, 16384);
        for (long b0 = 0; b0 < B; b0 += chunk) {
            const int nb = (int)((B - b0) < chunk ? (B - b0) : chunk);
            Scope inner(h);
            int rc = gpr_nlml_grad_device(h, inner, dX, dY, ldy, 1, (int)b0, ycols, N, d, 1, nb, dth + b0 * (2 * d + 3),
                                          dnz + b0, dn + b0, dg ? dg + b0 * (2 * d + 4) : nullptr, di ? di + b0 : nullptr, B);
            if (rc) return rc;
            if (!inner.ok) return inner.finish();
        }
    }
    return sc.finish();
}

// ---------------------------------------------------------------------------------------------
// Cached posteriors (include/mfgp.h).  One cudaMalloc block holds the device copies of the inputs and the factors; it
// belongs to the device, not to the handle that created it.
}  // extern "C"

struct PosteriorMem {
    int device;
    void* mem;
};
struct mfgp_gpr_posterior {
    PosteriorMem m;
    GprPosteriorData q;
};
struct mfgp_svgp_posterior {
    PosteriorMem m;
    SvgpPosteriorData q;
};

namespace {
// Offsets of consecutive arrays of doubles in one block, each 256-byte aligned: add() every array, allocate tot bytes,
// then at() gives each array's address.
struct Carve {
    size_t tot = 0;
    size_t add(size_t count) {
        const size_t o = tot;
        tot += (count * sizeof(double) + 255) & ~(size_t)255;
        return o;
    }
    static double* at(void* mem, size_t off) { return reinterpret_cast<double*>(static_cast<char*>(mem) + off); }
};

// The end of a create call: the block is freed when the call fails (rc < 0, or a failed factorisation without an info
// array to report it in); otherwise *out becomes a new posterior that owns it.
template <class Post, class Data>
int publish_posterior(mfgp_handle* h, int rc, const int* info, void* mem, const Data& q, Post** out) {
    if (rc < 0 || (rc > 0 && !info)) {
        cudaFree(mem);
        return rc;
    }
    *out = new Post{{h->device, mem}, q};
    return rc;
}

// The checks every predict call of a posterior starts with.  Returns 1 when there is work, else what the call returns
// (0 for Ns == 0, or the error code).  Makes the handle's device current.
template <class Post>
int posterior_predict_prologue(mfgp_handle* h, const Post* post, const double* Xs, int Ns, const double* mean,
                               const double* var, const char* name) {
    CHECK_H(h);
    if (!post || !Xs || !mean || !var || Ns < 0) return mfgp_fail(h, MFGP_ERR_ARG, "%s: bad argument", name);
    if (post->m.device != h->device)
        return mfgp_fail(h, MFGP_ERR_ARG, "%s: the posterior lives on device %d, the handle on %d", name, post->m.device,
                         h->device);
    if (Ns == 0) return 0;
    cudaSetDevice(h->device);
    return 1;
}

int free_posterior_mem(const PosteriorMem& m) {
    int prev = 0;
    cudaGetDevice(&prev);
    cudaSetDevice(m.device);
    const cudaError_t e = cudaFree(m.mem);
    cudaSetDevice(prev);
    return e == cudaSuccess ? 0 : MFGP_ERR_CUDA;
}

// Problems whose factorisation failed: NaN on the diagonal of W and in a (real columns), so both predict routes give NaN.
__global__ void posterior_poison_kernel(const int* __restrict__ info, int B, int N, long ld, int P, int Pp, double* __restrict__ W,
                                        double* __restrict__ a) {
    const double qnan = __longlong_as_double(0x7ff8000000000000ll);
    for (long b = blockIdx.x; b < B; b += gridDim.x) {
        if (!info[b]) continue;
        for (int i = threadIdx.x; i < N; i += blockDim.x) W[b * N * ld + (long)i * ld + i] = qnan;
        for (long i = threadIdx.x; i < (long)N * Pp; i += blockDim.x)
            if (i % Pp < P) a[b * N * Pp + i] = qnan;
    }
}
}  // namespace

extern "C" {

int mfgp_gpr_posterior_create(mfgp_handle* h, const double* X, int N, int d, const double* Y, long ldy, int ycols, int P,
                              int B, const double* theta, const double* noise, int* info, mfgp_gpr_posterior** out) {
    CHECK_H(h);
    if (out) *out = nullptr;
    if (!out || !X || !Y || !theta || !noise || N < 1 || d < 1 || d > MFGP_MAX_D || P < 1 || B < 1 || ycols < P ||
        ycols % P != 0 || ldy < ycols)
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_gpr_posterior_create: bad argument (ycols must be a multiple of P)");
    cudaSetDevice(h->device);
    const int np = 2 * d + 3, Pp = (int)round_up(P, 2);
    const long ld = round_up(N, 2);
    Carve c;
    const size_t oX = c.add((size_t)N * (d + 1)), oT = c.add((size_t)B * np), oN = c.add(B), oW = c.add((size_t)B * N * ld),
                 oA = c.add((size_t)B * N * Pp);
    void* mem = nullptr;
    CUDA_TRY(h, cudaMalloc(&mem, c.tot));
    double *dX = Carve::at(mem, oX), *dT = Carve::at(mem, oT), *dN = Carve::at(mem, oN), *dW = Carve::at(mem, oW),
           *dA = Carve::at(mem, oA);
    const int rc = [&]() -> int {
        Scope sc(h);
        cudaStream_t s = h->stream;
        CUDA_TRY(h, cudaMemcpyAsync(dX, X, (size_t)N * (d + 1) * sizeof(double), cudaMemcpyDefault, s));
        CUDA_TRY(h, cudaMemcpyAsync(dT, theta, (size_t)B * np * sizeof(double), cudaMemcpyDefault, s));
        CUDA_TRY(h, cudaMemcpyAsync(dN, noise, (size_t)B * sizeof(double), cudaMemcpyDefault, s));
        const double* dY = sc.in(Y, (size_t)N * ldy);
        int* di = info ? sc.out(info, B, true) : sc.alloc<int>(B, true);
        if (!sc.ok) return sc.finish();
        // the blocked batched route of mfgp_gpr_batched_nlml_grad, chunked so that its workspaces fit comfortably
        const size_t per = ((size_t)3 * N * ld + (size_t)chol_dinv_count(N, 1) + (size_t)2 * N * Pp + N) * sizeof(double);
        const long chunk = chunk_by_free_memory(per, 1, 16384);
        for (long b0 = 0; b0 < B; b0 += chunk) {
            const int nb = (int)((B - b0) < chunk ? (B - b0) : chunk);
            Scope inner(h);
            GprFactor f;
            MFGP_TRY(gpr_factor(h, inner, dX, dY, ldy, P, (int)b0, ycols, N, d, P, nb, dT + b0 * np, dN + b0, di + b0, f, true,
                               B));
            if (!inner.ok) return inner.finish();
            CUDA_TRY(h, cudaMemcpyAsync(dW + b0 * N * ld, f.W, (size_t)nb * N * ld * sizeof(double), cudaMemcpyDeviceToDevice, s));
            CUDA_TRY(h, cudaMemcpyAsync(dA + b0 * N * Pp, f.a, (size_t)nb * N * Pp * sizeof(double), cudaMemcpyDeviceToDevice, s));
        }
        posterior_poison_kernel<<<(unsigned)(B < 4096 ? B : 4096), 128, 0, s>>>(di, B, N, ld, P, Pp, dW, dA);
        sc.host_out = true;  // always synchronise: the factorisation status decides what the call returns
        return sc.finish();
    }();
    return publish_posterior(h, rc, info, mem, GprPosteriorData{N, d, P, Pp, B, ld, dX, dT, dN, dW, dA}, out);
}

}  // extern "C"

namespace {
// mfgp_gpr_posterior_predict and _predict_grad: one body, the gradients when dmean != NULL.
int posterior_predict(mfgp_handle* h, const mfgp_gpr_posterior* post, const double* Xs, int Ns, double* mean, double* var,
                      double* dmean, double* dvar, const char* name) {
    if (const int rc = posterior_predict_prologue(h, post, Xs, Ns, mean, var, name); rc <= 0) return rc;
    const GprPosteriorData& q = post->q;
    Scope sc(h);
    const double* dXs = sc.in(Xs, (size_t)Ns * (q.d + 1));
    double* dm = sc.out(mean, (size_t)q.B * Ns * q.P);
    double* dv = sc.out(var, (size_t)q.B * Ns);
    double* ddm = dmean ? sc.out(dmean, (size_t)q.B * Ns * q.P * q.d) : nullptr;
    double* ddv = dmean ? sc.out(dvar, (size_t)q.B * Ns * q.d) : nullptr;
    if (!sc.ok) return sc.finish();
    if (gpr_posterior_fused_ok(q.N, q.d, q.P)) {
        if (gpr_posterior_predict_fused(h->stream, q, dXs, Ns, dm, dv, ddm, ddv))
            return mfgp_fail(h, MFGP_ERR_CUDA, "%s: fused kernel launch failed", name);
    } else {
        MFGP_TRY(gpr_posterior_predict_blocked(h, q, dXs, Ns, dm, dv, ddm, ddv));
    }
    return sc.finish();
}
}  // namespace

extern "C" {

int mfgp_gpr_posterior_predict(mfgp_handle* h, const mfgp_gpr_posterior* post, const double* Xs, int Ns, double* mean,
                               double* var) {
    return posterior_predict(h, post, Xs, Ns, mean, var, nullptr, nullptr, "mfgp_gpr_posterior_predict");
}

int mfgp_gpr_posterior_predict_grad(mfgp_handle* h, const mfgp_gpr_posterior* post, const double* Xs, int Ns, double* mean,
                                    double* var, double* dmean, double* dvar) {
    if (!dmean || !dvar) {
        CHECK_H(h);
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_gpr_posterior_predict_grad: bad argument (dmean and dvar are required)");
    }
    return posterior_predict(h, post, Xs, Ns, mean, var, dmean, dvar, "mfgp_gpr_posterior_predict_grad");
}

}  // extern "C"

namespace {
// mfgp_gpr_posterior_predict_cov and _sample: one body, the samples when `sample`.
int posterior_joint(mfgp_handle* h, const mfgp_gpr_posterior* post, const double* Xs, int Ns, double* mean, double* cov,
                    bool sample, int S, double jitter, const double* z, double* samples, int* info, const char* name) {
    CHECK_H(h);
    if (!post || !Xs || Ns < 0 ||
        (sample ? (!z || !samples || S < 0 || !std::isfinite(jitter) || jitter < 0.0) : (!mean || !cov)))
        return mfgp_fail(h, MFGP_ERR_ARG, "%s: bad argument", name);
    if (post->m.device != h->device)
        return mfgp_fail(h, MFGP_ERR_ARG, "%s: the posterior lives on device %d, the handle on %d", name, post->m.device,
                         h->device);
    const GprPosteriorData& q = post->q;
    const long SP = sample ? (long)S * q.P : 0;
    if (sample) {
        const size_t bytes = (size_t)q.B * Ns * SP * sizeof(double);
        const char *zc = reinterpret_cast<const char*>(z), *sc = reinterpret_cast<const char*>(samples);
        if (zc < sc + bytes && sc < zc + bytes && bytes) return mfgp_fail(h, MFGP_ERR_ARG, "%s: z and samples overlap", name);
    }
    if (Ns == 0 || (sample && S == 0)) return 0;
    cudaSetDevice(h->device);
    Scope sc(h);
    const double* dXs = sc.in(Xs, (size_t)Ns * (q.d + 1));
    double* dm = sample ? sc.alloc<double>((size_t)q.B * Ns * q.P) : sc.out(mean, (size_t)q.B * Ns * q.P);
    GprJointOut j{};
    j.SP = SP;
    j.jitter = jitter;
    if (sample) {
        j.z = sc.in(z, (size_t)q.B * Ns * SP);
        j.samples = sc.out(samples, (size_t)q.B * Ns * SP);
        j.info = info ? sc.out(info, q.B, true) : sc.alloc<int>(q.B, true);
    } else {
        j.cov = sc.out(cov, (size_t)q.B * Ns * Ns);
    }
    if (!sc.ok) return sc.finish();
    if (gpr_posterior_joint_fused_ok(q.N, q.d, q.P, Ns)) {
        if (gpr_posterior_joint_fused(h->stream, q, dXs, Ns, dm, j, h->d_info))
            return mfgp_fail(h, MFGP_ERR_CUDA, "%s: fused kernel launch failed", name);
    } else {
        double* dv = sc.alloc<double>((size_t)q.B * Ns);
        if (!sc.ok) return sc.finish();
        // mean and diag(cov) are _predict's bits: when _predict runs the fused kernel (N <= 64 with Ns > 64), so do they
        j.mean_var_given = gpr_posterior_fused_ok(q.N, q.d, q.P);
        if (j.mean_var_given && gpr_posterior_predict_fused(h->stream, q, dXs, Ns, dm, dv))
            return mfgp_fail(h, MFGP_ERR_CUDA, "%s: fused kernel launch failed", name);
        MFGP_TRY(gpr_posterior_predict_blocked(h, q, dXs, Ns, dm, dv, nullptr, nullptr, &j));
    }
    return sc.finish();
}
}  // namespace

extern "C" {

int mfgp_gpr_posterior_predict_cov(mfgp_handle* h, const mfgp_gpr_posterior* post, const double* Xs, int Ns, double* mean,
                                   double* cov) {
    return posterior_joint(h, post, Xs, Ns, mean, cov, false, 0, 0.0, nullptr, nullptr, nullptr,
                           "mfgp_gpr_posterior_predict_cov");
}

int mfgp_gpr_posterior_sample(mfgp_handle* h, const mfgp_gpr_posterior* post, const double* Xs, int Ns, int S,
                              double jitter, const double* z, double* samples, int* info) {
    return posterior_joint(h, post, Xs, Ns, nullptr, nullptr, true, S, jitter, z, samples, info,
                           "mfgp_gpr_posterior_sample");
}

int mfgp_gpr_posterior_destroy(mfgp_gpr_posterior* post) {
    if (!post) return 0;
    const int rc = free_posterior_mem(post->m);
    delete post;
    return rc;
}

// ---------------------------------------------------------------------------------------------
// Cached SVGP posterior (include/mfgp.h): the memory model of mfgp_gpr_posterior, the factors of svgp_factor.
int mfgp_svgp_posterior_create(mfgp_handle* h, const mfgp_svgp_cfg* cfg, const double* Z, const double* theta,
                               const double* W, const double* q_mu, const double* q_sqrt, int* info,
                               mfgp_svgp_posterior** out) {
    CHECK_H(h);
    if (out) *out = nullptr;
    if (!out || !cfg || !Z || !theta || !q_mu || !q_sqrt)
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_svgp_posterior_create: NULL argument");
    const int L = cfg->L, M = cfg->M, P = cfg->P, d = cfg->d;
    if (L < 1 || M < 1 || P < 1 || d < 1 || d > MFGP_MAX_D || (!W && L != P))
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_svgp_posterior_create: bad configuration");
    cudaSetDevice(h->device);
    const int np = 2 * d + 3;
    const long ld = round_up(M, 2);
    Carve c;
    const size_t oZ = c.add((size_t)M * (d + 1)), oT = c.add((size_t)L * np), oW = c.add(W ? (size_t)P * L : 0),
                 oWm = c.add((size_t)L * M * ld), oLq = c.add((size_t)L * M * ld), oQ = c.add((size_t)M * L);
    void* mem = nullptr;
    CUDA_TRY(h, cudaMalloc(&mem, c.tot));
    double *dZ = Carve::at(mem, oZ), *dT = Carve::at(mem, oT), *dW = W ? Carve::at(mem, oW) : nullptr,
           *dWm = Carve::at(mem, oWm), *dLq = Carve::at(mem, oLq), *dQ = Carve::at(mem, oQ);
    const int rc = [&]() -> int {
        Scope sc(h);
        cudaStream_t s = h->stream;
        CUDA_TRY(h, cudaMemcpyAsync(dZ, Z, (size_t)M * (d + 1) * sizeof(double), cudaMemcpyDefault, s));
        CUDA_TRY(h, cudaMemcpyAsync(dT, theta, (size_t)L * np * sizeof(double), cudaMemcpyDefault, s));
        if (W) CUDA_TRY(h, cudaMemcpyAsync(dW, W, (size_t)P * L * sizeof(double), cudaMemcpyDefault, s));
        CUDA_TRY(h, cudaMemcpyAsync(dQ, q_mu, (size_t)M * L * sizeof(double), cudaMemcpyDefault, s));
        const double* dqs = sc.in(q_sqrt, (size_t)L * M * M);
        int* di = info ? sc.out(info, L, true) : sc.alloc<int>(L, true);
        if (!sc.ok) return sc.finish();
        Fwd f{};
        f.Wm = dWm;
        f.Lq = dLq;
        f.ldM = ld;
        f.sMM = (long)M * ld;
        MFGP_TRY(svgp_factor(h, sc, L, M, d, cfg->jitter, dZ, dT, dqs, di, f));
        // a failed latent: NaN on the diagonal of Wm (P = 0: q_mu is left as it is); it reaches every output of the latent
        posterior_poison_kernel<<<(unsigned)(L < 4096 ? L : 4096), 128, 0, s>>>(di, L, M, ld, 0, 1, dWm, nullptr);
        sc.host_out = true;  // always synchronise: the factorisation status decides what the call returns
        return sc.finish();
    }();
    return publish_posterior(h, rc, info, mem, SvgpPosteriorData{L, M, P, d, ld, dZ, dT, dW, dWm, dLq, dQ}, out);
}

}  // extern "C"

namespace {
// mfgp_svgp_posterior_predict and _predict_grad: one body, the gradients when dmean != NULL.  With W the fused route
// writes the latents to [L][Ns] (and [L][Ns][d]) scratch and the mix kernels form the outputs.
int svgp_posterior_predict(mfgp_handle* h, const mfgp_svgp_posterior* post, const double* Xs, int Ns, double* mean,
                           double* var, double* dmean, double* dvar, const char* name) {
    if (const int rc = posterior_predict_prologue(h, post, Xs, Ns, mean, var, name); rc <= 0) return rc;
    const SvgpPosteriorData& q = post->q;
    Scope sc(h);
    const double* dXs = sc.in(Xs, (size_t)Ns * (q.d + 1));
    double* dm = sc.out(mean, (size_t)Ns * q.P);
    double* dv = sc.out(var, (size_t)Ns * q.P);
    double* ddm = dmean ? sc.out(dmean, (size_t)Ns * q.P * q.d) : nullptr;
    double* ddv = dmean ? sc.out(dvar, (size_t)Ns * q.P * q.d) : nullptr;
    if (!sc.ok) return sc.finish();
    if (svgp_posterior_fused_ok(q.L, q.M, q.d)) {
        if (!q.W) {
            if (svgp_posterior_predict_fused(h->stream, q, dXs, Ns, dm, dv, 1, q.P, ddm, ddv))
                return mfgp_fail(h, MFGP_ERR_CUDA, "%s: fused kernel launch failed", name);
        } else {
            const size_t lat = (size_t)q.L * Ns;
            double* g = sc.alloc<double>(2 * lat);  // latent marginals [L][Ns], mean then var
            double* gd = dmean ? sc.alloc<double>(2 * lat * q.d) : nullptr;  // latent gradients [L][Ns][d], mean then var
            if (!sc.ok) return sc.finish();
            if (svgp_posterior_predict_fused(h->stream, q, dXs, Ns, g, g + lat, Ns, 1, gd, dmean ? gd + lat * q.d : nullptr) ||
                launch_svgp_mix(h->stream, g, g + lat, q.L, Ns, q.P, q.W, dm, dv) ||
                (dmean && launch_svgp_grad_mix(h->stream, gd, gd + lat * q.d, q.L, Ns, q.P, q.d, q.W, ddm, ddv)))
                return mfgp_fail(h, MFGP_ERR_CUDA, "%s: fused kernel launch failed", name);
        }
    } else {
        MFGP_TRY(svgp_posterior_predict_blocked(h, q, dXs, Ns, dm, dv, ddm, ddv));
    }
    return sc.finish();
}
}  // namespace

extern "C" {

int mfgp_svgp_posterior_predict(mfgp_handle* h, const mfgp_svgp_posterior* post, const double* Xs, int Ns, double* mean,
                                double* var) {
    return svgp_posterior_predict(h, post, Xs, Ns, mean, var, nullptr, nullptr, "mfgp_svgp_posterior_predict");
}

int mfgp_svgp_posterior_predict_grad(mfgp_handle* h, const mfgp_svgp_posterior* post, const double* Xs, int Ns,
                                     double* mean, double* var, double* dmean, double* dvar) {
    if (!dmean || !dvar) {
        CHECK_H(h);
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_svgp_posterior_predict_grad: bad argument (dmean and dvar are required)");
    }
    return svgp_posterior_predict(h, post, Xs, Ns, mean, var, dmean, dvar, "mfgp_svgp_posterior_predict_grad");
}

int mfgp_svgp_posterior_destroy(mfgp_svgp_posterior* post) {
    if (!post) return 0;
    const int rc = free_posterior_mem(post->m);
    delete post;
    return rc;
}

// ---------------------------------------------------------------------------------------------
int mfgp_cov_grad(mfgp_handle* h, const double* X, int N, int d, const double* theta, const double* G, long ldg, double scale,
                  double* out) {
    CHECK_H(h);
    if (!X || !theta || !G || !out || N < 1 || d < 1 || d > MFGP_MAX_D || ldg < N)
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_cov_grad: bad argument");
    cudaSetDevice(h->device);
    Scope sc(h);
    const double* dX = sc.in(X, (size_t)N * (d + 1));
    const double* dth = sc.in(theta, 2 * d + 3);
    const double* dG = sc.in(G, (size_t)N * ldg);
    double* dout = sc.out(out, 2 * d + 4);
    if (!sc.ok) return sc.finish();
    CovGradArgs cg{};
    cg.Xa = dX; cg.Na = N; cg.Xb = dX; cg.Nb = N; cg.d = d;
    cg.theta = dth; cg.theta_stride = 2 * d + 3;
    cg.G = dG; cg.ldg = ldg; cg.strideG = 0;
    cg.sym_lower = 1;
    cg.out = dout; cg.out_stride = 2 * d + 4;
    cg.out_scale = scale;
    cg.accumulate = 0;
    cg.rowgrad = nullptr;
    cg.batch = 1;
    cg.partial = sc.alloc<double>((size_t)cov_grad_partial_count(cg));
    if (!sc.ok) return sc.finish();
    if (launch_cov_grad(h->stream, cg)) return mfgp_fail(h, MFGP_ERR_CUDA, "cov_grad launch failed");
    return sc.finish();
}

// ---------------------------------------------------------------------------------------------
// Device-resident Adam loop for the batched per-bin GPs (SURVEY 8(f) rank 1; reference loop mfgpflow/linear.py:190-221).
namespace {
__global__ void adam_softplus_kernel(const double* __restrict__ u, double* __restrict__ theta, long n) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) theta[i] = softplus_fwd(u[i]);
}
// One thread per (problem, parameter): chain rule, moment update, step, and theta for the NEXT evaluation.
__global__ void adam_update_kernel(double* __restrict__ u, double* __restrict__ m, double* __restrict__ v,
                                   double* __restrict__ theta, const double* __restrict__ grad, const double* __restrict__ nlml,
                                   const double* __restrict__ lr_t, int step, double b1, double b2, double eps, int fix_rho,
                                   int np, int B, double* __restrict__ loss_hist, const int* __restrict__ step_info,
                                   int* __restrict__ first_info) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long)B * np) return;
    const int b = (int)(i / np), q = (int)(i % np);
    if (q == 0) {
        if (loss_hist) loss_hist[(long)step * B + b] = nlml[b];
        if (first_info && step_info[b] && !first_info[b]) first_info[b] = step_info[b];
    }
    if (fix_rho && q == 0) return;
    const double th = theta[i];
    const double g = grad[(long)b * (np + 1) + q] * (1.0 - exp(-th));  // d theta / d u = sigmoid(u) = 1 - exp(-theta)
    double mi = m[i], vi = v[i];
    mi += (g - mi) * (1.0 - b1);
    vi += (g * g - vi) * (1.0 - b2);
    const double un = u[i] - lr_t[step] * mi / (sqrt(vi) + eps);
    m[i] = mi;
    v[i] = vi;
    u[i] = un;
    theta[i] = softplus_fwd(un);
}
}  // namespace

int mfgp_gpr_batched_adam(mfgp_handle* h, const double* X, int N, int d, const double* Y, long ldy, int ycols, int B,
                          double* u, double* m, double* v, const double* noise, const double* lr_t, double beta1,
                          double beta2, double eps, int fix_rho, int nsteps, double* loss_hist, double* theta_out, int* info) {
    CHECK_H(h);
    if (!X || !Y || !u || !m || !v || !noise || !lr_t || N < 1 || B < 0 || d < 1 || ycols < 1 || ldy < ycols || nsteps < 0)
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_gpr_batched_adam: bad argument");
    if (N > MFGP_SMALL_MAX_N || d > MFGP_SMALL_MAX_D)
        return mfgp_fail(h, MFGP_ERR_UNSUPPORTED, "mfgp_gpr_batched_adam: N <= 64 and d <= 16 only");
    cudaSetDevice(h->device);
    if (B == 0 || nsteps == 0) return 0;
    const int np = 2 * d + 3;
    const size_t n = (size_t)B * np;
    Scope sc(h);
    const double* dX = sc.in(X, (size_t)N * (d + 1));
    const double* dY = sc.in(Y, (size_t)N * ldy);
    const double* dnz = sc.in(noise, B);
    const double* dlr = sc.in(lr_t, nsteps);
    double* du = sc.inout(u, n);
    double* dm = sc.inout(m, n);
    double* dv = sc.inout(v, n);
    double* dl = loss_hist ? sc.out(loss_hist, (size_t)nsteps * B) : nullptr;
    double* dto = theta_out ? sc.out(theta_out, n) : nullptr;
    int* di = info ? sc.out(info, B, true) : nullptr;
    double* dth = sc.alloc<double>(n);
    double* dn = sc.alloc<double>(B);
    double* dg = sc.alloc<double>((size_t)B * (np + 1));
    int* dsi = sc.alloc<int>(B);
    if (!sc.ok) return sc.finish();
    const int tb = 256;
    const unsigned gb = (unsigned)((n + tb - 1) / tb);
    adam_softplus_kernel<<<gb, tb, 0, h->stream>>>(du, dth, (long)n);
    SmallArgs a{};
    a.X = dX; a.N = N; a.d = d; a.Y = dY; a.ldy = ldy; a.ycols = ycols; a.B = B;
    a.theta = dth; a.noise = dnz; a.nlml = dn; a.grad = dg; a.info = dsi; a.d_info = h->d_info;
    for (int s = 0; s < nsteps; ++s) {
        if (launch_gpr_small(h->stream, a)) return mfgp_fail(h, MFGP_ERR_CUDA, "gpr_small launch failed");
        adam_update_kernel<<<gb, tb, 0, h->stream>>>(du, dm, dv, dth, dg, dn, dlr, s, beta1, beta2, eps, fix_rho, np, B, dl, dsi, di);
    }
    if (dto) CUDA_TRY(h, cudaMemcpyAsync(dto, dth, n * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    return sc.finish();
}

// ---------------------------------------------------------------------------------------------
int mfgp_gemm(mfgp_handle* h, char transa, char transb, int m, int n, int k, double alpha, const double* A, long lda,
              const double* B, long ldb, double beta, double* C, long ldc) {
    CHECK_H(h);
    cudaSetDevice(h->device);
    const bool ta = (transa == 'T' || transa == 't'), tb = (transb == 'T' || transb == 't');
    const long arows = ta ? k : m, brows = tb ? n : k;
    if (!A || !B || !C || m < 0 || n < 0 || k < 0) return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_gemm: bad argument");
    if ((lda & 1) || (ldb & 1)) return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_gemm: lda/ldb must be even");
    Scope sc(h);
    GemmArgs g;
    g.transA = ta; g.transB = tb; g.M = m; g.N = n; g.K = k; g.alpha = alpha; g.beta = beta;
    g.A = sc.in(A, (size_t)arows * lda); g.lda = lda;
    g.B = sc.in(B, (size_t)brows * ldb); g.ldb = ldb;
    double* dC;
    if (mfgp_is_device_ptr(C)) dC = C;
    else {
        dC = sc.alloc<double>((size_t)m * ldc);
        if (dC && beta != 0.0) cudaMemcpyAsync(dC, C, (size_t)m * ldc * 8, cudaMemcpyHostToDevice, h->stream);
        sc.outs.push_back({C, dC, (size_t)m * ldc * 8});
        sc.host_out = true;
    }
    g.C = dC; g.ldc = ldc;
    if (!sc.ok) return sc.finish();
    if (launch_gemm(h->stream, g)) return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_gemm: launch failed (alignment?)");
    return sc.finish();
}

static int potrf_common(mfgp_handle* h, double* A, int N, long lda, double* Winv, long ldw) {
    CHECK_H(h);
    if (!A || N < 1 || lda < N || (lda & 1)) return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_potrf: bad argument (lda must be even)");
    if (Winv && (ldw < N || (ldw & 1))) return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_potrf_inv: bad ldw");
    cudaSetDevice(h->device);
    Scope sc(h);
    double* dA;
    if (mfgp_is_device_ptr(A)) dA = A;
    else {
        dA = sc.alloc<double>((size_t)N * lda);
        if (dA) cudaMemcpyAsync(dA, A, (size_t)N * lda * 8, cudaMemcpyHostToDevice, h->stream);
        sc.outs.push_back({A, dA, (size_t)N * lda * 8});
        sc.host_out = true;
    }
    CholArgs ch{};
    ch.A = dA; ch.N = N; ch.lda = lda; ch.strideA = 0; ch.batch = 1;
    ch.dinv = sc.alloc<double>((size_t)chol_dinv_count(N, 1));
    ch.logd = sc.alloc<double>(N);
    ch.d_info = h->d_info; ch.aux = h->aux_stream; ch.ev = h->ev;
    if (!sc.ok) return sc.finish();
    if (launch_potrf(h->stream, ch)) return mfgp_fail(h, MFGP_ERR_CUDA, "potrf launch failed");
    if (Winv) {
        double* dW = sc.out(Winv, (size_t)N * ldw);
        double* scratch = sc.alloc<double>((size_t)N * ldw);
        if (!sc.ok) return sc.finish();
        if (launch_trtri(h->stream, ch, dW, ldw, 0, scratch)) return mfgp_fail(h, MFGP_ERR_CUDA, "trtri launch failed");
    }
    return sc.finish();
}
int mfgp_potrf(mfgp_handle* h, double* A, int N, long lda) { return potrf_common(h, A, N, lda, nullptr, 0); }
int mfgp_potrf_inv(mfgp_handle* h, double* A, int N, long lda, double* Winv, long ldw) {
    if (!Winv) return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_potrf_inv: Winv is NULL");
    return potrf_common(h, A, N, lda, Winv, ldw);
}

// ---- tall-skinny update ---------------------------------------------------------------------------------
// Y[M, 0:nc] += alpha * A[M, K] X[K, 0:nc] for nc <= 2 right-hand sides: the forward-substitution step of the distributed
// Cholesky (y[k+1:] -= L[k+1:, k] a_k, M up to N rows, K = block size).  HBM bound (every row of A is read once); the 64-wide
// GEMM tiles would compute 32x more columns than exist.  One warp per row, 128-bit loads, X staged in shared memory.
__global__ void __launch_bounds__(256) tall_skinny_kernel(int M, int K, int nc, double alpha, const double* __restrict__ A, long lda,
                                                          const double* __restrict__ X, long ldx, double* __restrict__ Y, long ldy) {
    extern __shared__ double xs[];  // [K][2]
    for (int i = threadIdx.x; i < K; i += blockDim.x) {
        xs[2 * i] = X[(long)i * ldx];
        xs[2 * i + 1] = nc > 1 ? X[(long)i * ldx + 1] : 0.0;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warps = (blockDim.x >> 5) * gridDim.x;
    for (int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < M; r += warps) {
        const double* row = A + (long)r * lda;
        double s0 = 0.0, s1 = 0.0;
        for (int k = 2 * lane; k + 1 < K; k += 64) {
            const double2 a = *reinterpret_cast<const double2*>(row + k);
            s0 = fma(a.x, xs[2 * k], s0);
            s1 = fma(a.x, xs[2 * k + 1], s1);
            s0 = fma(a.y, xs[2 * k + 2], s0);
            s1 = fma(a.y, xs[2 * k + 3], s1);
        }
        if ((K & 1) && lane == 0) {
            s0 = fma(row[K - 1], xs[2 * (K - 1)], s0);
            s1 = fma(row[K - 1], xs[2 * (K - 1) + 1], s1);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s0 += __shfl_xor_sync(0xffffffffu, s0, o);
            s1 += __shfl_xor_sync(0xffffffffu, s1, o);
        }
        if (lane == 0) {
            Y[(long)r * ldy] = fma(alpha, s0, Y[(long)r * ldy]);
            if (nc > 1) Y[(long)r * ldy + 1] = fma(alpha, s1, Y[(long)r * ldy + 1]);
        }
    }
}

int mfgp_tall_skinny_update(mfgp_handle* h, int M, int K, int nc, double alpha, const double* A, long lda, const double* X,
                            long ldx, double* Y, long ldy) {
    CHECK_H(h);
    if (!A || !X || !Y || M < 0 || K < 1 || K > 3072 || nc < 1 || nc > 2 || lda < K || (lda & 1) || (reinterpret_cast<size_t>(A) & 15) ||
        ldx < nc || ldy < nc)
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_tall_skinny_update: bad argument (1 <= nc <= 2, K <= 3072 [X is staged in 48 KB of shared memory], even lda, 16-byte aligned A)");
    if (!mfgp_is_device_ptr(A) || !mfgp_is_device_ptr(X) || !mfgp_is_device_ptr(Y))
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_tall_skinny_update: device pointers only");
    if (M == 0) return 0;
    cudaSetDevice(h->device);
    long blocks = (M + 7) / 8;
    const long cap = (long)h->sm_count * 8;
    if (blocks > cap) blocks = cap;
    tall_skinny_kernel<<<(unsigned)blocks, 256, (size_t)K * 16, h->stream>>>(M, K, nc, alpha, A, lda, X, ldx, Y, ldy);
    CUDA_TRY(h, cudaGetLastError());
    return 0;
}

// ---- one-to-many store over peer memory ----------------------------------------------------------------
// The critical-path messages of the distributed Cholesky (inv(L_kk) and the early block (k+1, k), nb x nb doubles) go to
// every other GPU of the box.  With the peers' buffers mapped into this process (symmetric memory over NVLink / NVSwitch)
// that is ONE kernel: each 16-byte piece of the source is read once and stored to every destination, so the transfers to
// the peers run concurrently on all NVLink lanes and never queue behind the bulk panel broadcasts of the NCCL stream.
struct PeerDsts {
    double* p[MFGP_PEER_MAX];
};
__global__ void __launch_bounds__(256) peer_store_kernel(const double2* __restrict__ src, long n2, int ndst, PeerDsts d) {
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += (long)gridDim.x * blockDim.x) {
        const double2 v = src[i];
#pragma unroll
        for (int k = 0; k < MFGP_PEER_MAX; ++k)
            if (k < ndst) reinterpret_cast<double2*>(d.p[k])[i] = v;
    }
}

int mfgp_workspace(mfgp_handle* h, int mode, long* bytes) {
    CHECK_H(h);
    if (mode != MFGP_WS_POOL && mode != MFGP_WS_MEASURE && mode != MFGP_WS_FIXED)
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_workspace: mode must be MFGP_WS_POOL, _MEASURE or _FIXED");
    cudaSetDevice(h->device);
    mfgp_ws_state& w = h->ws;
    const long measured = w.mode == MFGP_WS_MEASURE ? (long)w.need : 0;
    if (bytes) *bytes = measured;
    if (w.arena) {  // leaving FIXED (or re-entering it): the arena goes back to the pool in stream order
        CUDA_TRY(h, cudaFreeAsync(w.arena, h->stream));
        w.arena = nullptr;
        w.cap = w.off = 0;
    }
    if (mode == MFGP_WS_FIXED) {
        if (w.mode != MFGP_WS_MEASURE) return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_workspace: MFGP_WS_FIXED follows MFGP_WS_MEASURE");
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        cudaStreamIsCapturing(h->stream, &cs);
        if (cs != cudaStreamCaptureStatusNone)
            return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_workspace: allocate the arena outside the stream capture");
        const size_t cap = measured > 0 ? (size_t)measured : 256;
        void* p = nullptr;
        CUDA_TRY(h, cudaMallocAsync(&p, cap, h->stream));
        w.arena = static_cast<char*>(p);
        w.cap = cap;
    }
    w.mode = mode;
    w.base_depth = w.depth;
    w.cur = w.need = w.off = w.spilled = 0;
    return 0;
}

int mfgp_graph_mem_trim(mfgp_handle* h) {
    CHECK_H(h);
    cudaSetDevice(h->device);
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    CUDA_TRY(h, cudaDeviceGraphMemTrim(h->device));
    return 0;
}

int mfgp_peer_store(mfgp_handle* h, const double* src, long count, int ndst, double* const* dsts) {
    CHECK_H(h);
    if (!src || !dsts || count < 0 || (count & 1) || ndst < 0 || ndst > MFGP_PEER_MAX || (reinterpret_cast<size_t>(src) & 15))
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_peer_store: bad argument (even count, 16-byte aligned, <= %d destinations)", MFGP_PEER_MAX);
    if (ndst == 0 || count == 0) return 0;
    cudaSetDevice(h->device);
    PeerDsts d{};
    for (int k = 0; k < ndst; ++k) {
        if (!dsts[k] || (reinterpret_cast<size_t>(dsts[k]) & 15)) return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_peer_store: destination %d unaligned", k);
        d.p[k] = dsts[k];
    }
    const long n2 = count / 2;
    long blocks = (n2 + 255) / 256;
    const long cap = (long)h->sm_count * 8;
    if (blocks > cap) blocks = cap;
    peer_store_kernel<<<(unsigned)blocks, 256, 0, h->stream>>>(reinterpret_cast<const double2*>(src), n2, ndst, d);
    CUDA_TRY(h, cudaGetLastError());
    return 0;
}

// ---- FP64 pipe microbenchmarks ---------------------------------------------------------------
__global__ void __launch_bounds__(256) dfma_peak_kernel(double* out, int iters) {
    double a[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = 1.0 + 1e-9 * (threadIdx.x + i);
    const double x = 1.0000001, y = 1e-9;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 16; ++i) a[i] = fma(a[i], x, y);
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += a[i];
    if (s == 123.456) out[0] = s;
}
__global__ void __launch_bounds__(256) dmma_peak_kernel(double* out, int iters) {
    double c[16][2];
#pragma unroll
    for (int i = 0; i < 16; ++i) c[i][0] = c[i][1] = 0.0;
    const double a = 1.0 + 1e-9 * threadIdx.x, b = 1e-9;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 16; ++i) dmma(c[i][0], c[i][1], a, b);
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += c[i][0] + c[i][1];
    if (s == 123.456) out[0] = s;
}

// kind 2: both instruction streams in one loop, sized for equal pipe time (8 DMMA x 16 cycles = 64 DFMA x 2 cycles per
// sub-partition): if DMMA and DFMA share one FP64 datapath the loop takes the SUM of the two times (same FLOP/s as either
// alone), if they are separate units it takes the MAX (twice the FLOP/s).  The answer decides what "FP64 pipe busy" can
// mean for a kernel that mixes both, like K6.
__global__ void __launch_bounds__(256) dmix_peak_kernel(double* out, int iters) {
    double c[8][2], a[16];
#pragma unroll
    for (int i = 0; i < 8; ++i) c[i][0] = c[i][1] = 0.0;
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = 1.0 + 1e-9 * (threadIdx.x + i);
    const double am = 1.0 + 1e-9 * threadIdx.x, bm = 1e-9, x = 1.0000001, y = 1e-9;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
#pragma unroll
            for (int i = 0; i < 2; ++i) dmma(c[2 * r + i][0], c[2 * r + i][1], am, bm);
#pragma unroll
            for (int i = 0; i < 16; ++i) a[i] = fma(a[i], x, y);
        }
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += c[i][0] + c[i][1];
#pragma unroll
    for (int i = 0; i < 16; ++i) s += a[i];
    if (s == 123.456) out[0] = s;
}

int mfgp_fp64_peak(mfgp_handle* h, int kind, int iters, double* flops) {
    CHECK_H(h);
    if (!flops || iters < 1) return MFGP_ERR_ARG;
    cudaSetDevice(h->device);
    double* d = nullptr;
    CUDA_TRY(h, cudaMalloc(&d, 8));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    const int blocks = h->sm_count * 4;  // 4 CTAs x 8 warps per SM
    float best = 1e30f;
    for (int rep = 0; rep < 4; ++rep) {
        cudaEventRecord(e0, h->stream);
        if (kind == 0) dfma_peak_kernel<<<blocks, 256, 0, h->stream>>>(d, iters);
        else if (kind == 1) dmma_peak_kernel<<<blocks, 256, 0, h->stream>>>(d, iters);
        else dmix_peak_kernel<<<blocks, 256, 0, h->stream>>>(d, iters);
        cudaEventRecord(e1, h->stream);
        cudaEventSynchronize(e1);
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        if (rep > 0 && ms < best) best = ms;
    }
    const double per_thread = kind == 0 ? 16.0 * 2.0 : kind == 1 ? 16.0 * (2.0 * 8 * 8 * 4) / 32.0
                                                     : 8.0 * (2.0 * 8 * 8 * 4) / 32.0 + 64.0 * 2.0;
    *flops = per_thread * iters * 256.0 * blocks / (best * 1e-3);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d);
    CUDA_TRY(h, cudaGetLastError());
    return 0;
}

}  // extern "C"
