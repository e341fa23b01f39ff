// minibatch.cu -- the shuffled-epoch row stream of the minibatch SVGP loops and the kernel that gathers one batch of it.
//
// The rule (include/mfgp.h: "Minibatch stream"; tests/_minibatch_twin.py is its NumPy twin) is integer-only and stateless,
// so the gather kernel evaluates it inside a captured CUDA graph from the device step counter, and every rank of a
// data-parallel run draws its slice of the same global batch without communicating.
#include "svgp.cuh"

namespace {

constexpr int MB_ROUNDS = 8;

__device__ __forceinline__ unsigned long long splitmix64(unsigned long long z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

__device__ __forceinline__ unsigned mix32(unsigned x) {
    x ^= x >> 16;
    x *= 0x7FEB352Du;
    x ^= x >> 15;
    x *= 0x846CA68Bu;
    x ^= x >> 16;
    return x;
}

// Row of stream position p: epoch e = p / N, offset i = p mod N, row = pi_{seed,e}(i).  pi is an 8-round balanced
// Feistel network on 2k-bit values (4^k >= N), cycle-walked until the value is below N.
__device__ __forceinline__ long long stream_row(long long p, long long N, int k, unsigned long long seed) {
    const unsigned long long e = (unsigned long long)(p / N);
    const unsigned long long se = splitmix64(splitmix64(seed) ^ e);
    unsigned key[MB_ROUNDS];
#pragma unroll
    for (int r = 0; r < MB_ROUNDS; ++r) key[r] = (unsigned)splitmix64(se ^ (unsigned long long)r);
    const unsigned mask = (1u << k) - 1u;
    unsigned long long x = (unsigned long long)(p % N);
    do {
        unsigned l = (unsigned)(x >> k), r = (unsigned)x & mask;
#pragma unroll
        for (int j = 0; j < MB_ROUNDS; ++j) {
            const unsigned t = l ^ (mix32(r ^ key[j]) & mask);
            l = r;
            r = t;
        }
        x = ((unsigned long long)l << k) | r;
    } while (x >= (unsigned long long)N);
    return (long long)x;
}

// One warp per batch row j < count: the row of position pos0 + (*step) B + lo + j, its X and Y columns copied by the lanes
// (NaN entries of a masked Y travel as they are).
__global__ void minibatch_gather_kernel(const double* __restrict__ X, int xcols, const double* __restrict__ Y, int ycols,
                                        long long N, int k, unsigned long long seed, long long pos0,
                                        const int* __restrict__ step, long long B, long long lo, int count,
                                        double* __restrict__ Xb, double* __restrict__ Yb) {
    const int lane = threadIdx.x & 31;
    const long long base = pos0 + (step ? (long long)*step : 0ll) * B + lo;
    const long nwarps = ((long)gridDim.x * blockDim.x) >> 5;
    for (long j = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < count; j += nwarps) {
        const long long row = stream_row(base + j, N, k, seed);
        for (int c = lane; c < xcols; c += 32) Xb[j * xcols + c] = X[row * xcols + c];
        if (Y)
            for (int c = lane; c < ycols; c += 32) Yb[j * ycols + c] = Y[row * ycols + c];
    }
}

}  // namespace

int launch_minibatch_gather(cudaStream_t s, const MinibatchStream& ms, const int* step, int B, int lo, int count, double* Xb,
                            double* Yb) {
    if (count <= 0) return 0;
    int k = 0;
    while ((1ll << (2 * k)) < (long long)ms.N) ++k;
    const long blocks = ((long)count + 7) / 8;
    minibatch_gather_kernel<<<(unsigned)(blocks < 4096 ? blocks : 4096), 256, 0, s>>>(
        ms.X, ms.xcols, ms.Y, ms.ycols, ms.N, k, ms.seed, ms.pos0, step, B, lo, count, Xb, Yb);
    return cudaGetLastError() == cudaSuccess ? 0 : MFGP_ERR_CUDA;
}

extern "C" int mfgp_minibatch_gather(mfgp_handle* h, const double* X, int xcols, const double* Y, int ycols, int N,
                                     unsigned long long seed, long long pos0, const int* step, int B, int lo, int count,
                                     double* Xb, double* Yb) {
    if (!h) return MFGP_ERR_ARG;
    if (!X || !Xb || xcols < 1 || ycols < 0 || (!Y != !Yb) || (Y && ycols < 1) || N < 1 || B < 1 || B > N || pos0 < 0 ||
        lo < 0 || count < 0 || (long)lo + count > B)
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_minibatch_gather: bad arguments (need 1 <= B <= N, pos0 >= 0, "
                                          "0 <= lo, lo + count <= B, Y and Yb both given or both NULL)");
    if (count == 0) return 0;
    cudaSetDevice(h->device);
    Scope sc(h);
    const MinibatchStream ms{sc.in(X, (size_t)N * xcols), xcols, Y ? sc.in(Y, (size_t)N * ycols) : nullptr, Y ? ycols : 0,
                             N, seed, pos0};
    const int* dstep = step ? sc.in(step, 1) : nullptr;
    double* dXb = sc.out(Xb, (size_t)count * xcols);
    double* dYb = Y ? sc.out(Yb, (size_t)count * ycols) : nullptr;
    if (!sc.ok) return sc.finish();
    if (launch_minibatch_gather(h->stream, ms, dstep, B, lo, count, dXb, dYb))
        return mfgp_fail(h, MFGP_ERR_CUDA, "mfgp_minibatch_gather: launch failed");
    return sc.finish();
}
