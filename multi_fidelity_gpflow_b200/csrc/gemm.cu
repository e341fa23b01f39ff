// gemm.cu -- batched fp64 GEMM for sm_100a on the FP64 tensor path, operand tiles fed by TMA.
//
// tcgen05.mma has no f64 kind, so the FP64 tensor path on Blackwell is the warp-level
// mma.sync.m8n8k4.f64 (SASS: DMMA.8x8x4).  This kernel feeds it from a 4-stage shared-memory ring that the TMA unit
// fills (cp.async.bulk.tensor, SASS UTMALDG) and mbarriers hand over: one elected thread arms the stage's barrier with
// the byte count and issues the tile copies, the eight MMA warps wait on the barrier's phase.  No thread computes an
// address or a bounds predicate for the operand stream: the tensor maps carry shapes and strides (incl. the strided
// batch dimensions), out-of-range rows / k are zero-filled by the hardware, and the 128-byte swizzle of the tensor
// map produces the bank-conflict-free layout the 8-byte fragment loads need:
//   * K-major operand (contiguous along k): one box [rows][16 k] per stage; a row is 128 bytes and its 16-byte chunk c
//     lands at chunk c ^ (row & 7); an MMA row-fragment uses rows {2g + b} of a 16-row group, so the four rows of a
//     half-warp land in four different bank octets.
//   * M-major operand (contiguous along m/n): rows / 16 boxes [16 k][16 m] per stage (2 KB each); inside a box k-row k is
//     128 bytes and chunk c of it lands at c ^ (k & 7); an MMA fragment takes the rows {0-3, 8-11} or {4-7, 12-15} of a
//     box (frag_row below), which makes the 16 lanes of a half-warp hit 16 distinct 8-byte bank pairs.
//   Both layouts and the epilogue mapping are modelled on the CPU in tests/test_gemm_layout_model.py.
// Warp tile 64x32 (128x128 CTA, 8 warps) or 32x32 (64x64 CTA, 4 warps): 12 (8) LDS.64 per
// 32 (16) DMMA.  Triangular operands are expressed as per-tile k ranges (GemmKRange).
#include "gemm.cuh"
#include "common.cuh"

#include <cuda.h>  // CUtensorMap (types only: the encoder is fetched through cudaGetDriverEntryPoint, libcuda is not linked)

#include <cstdint>

#include "mathx.cuh"

namespace {

constexpr int BK = 16;
constexpr int STAGES = 4;

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, int src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(dst), "l"(src), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}
__device__ __forceinline__ double lds64(uint32_t addr) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];\n" : "=d"(v) : "r"(addr));
    return v;
}

// ---- TMA / mbarrier primitives -------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(bar), "r"(parity)
        : "memory");
}
// 4-D tiled copy: coordinates (contiguous dimension, row dimension, batch, outer batch)
__device__ __forceinline__ void tma_load(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n" ::"r"(dst),
                 "l"(tm), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}

// One stage of one operand, issued by the lanes of warp 0.  K-major: a single box [ROWS][BK] (lane 0).  M-major: ROWS / 16
// boxes [BK][16], one per lane, so that the eight boxes of a 128-row operand are issued side by side, not one after another.
template <bool KMAJOR, int ROWS>
__device__ __forceinline__ void tma_operand(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int row0, int k0, int b1, int b2, int lane) {
    if (KMAJOR) {
        if (lane == 0) tma_load(dst, tm, bar, k0, row0, b1, b2);
    } else {
        if (lane < ROWS / 16) tma_load(dst + lane * 2048, tm, bar, row0 + 16 * lane, k0, b1, b2);
    }
}

// tile-local row of MMA row g (0..7) of fragment f inside a warp tile starting at w0 (a multiple of 32)
template <bool KMAJOR>
__device__ __forceinline__ int frag_row(int w0, int f, int g) {
    return KMAJOR ? w0 + (f >> 1) * 16 + 2 * g + (f & 1)
                  : w0 + (f >> 1) * 16 + 8 * ((g >> 1) & 1) + 4 * (f & 1) + 2 * (g >> 2) + (g & 1);
}
// shared address (bytes, relative to the 1024-byte aligned tile base) of element (row, k): the TMA 128-byte swizzle
template <bool KMAJOR, int ROWS>
__device__ __forceinline__ uint32_t frag_addr(int row, int k) {
    return KMAJOR ? (uint32_t)(row * 128 + (((k >> 1) ^ (row & 7)) << 4) + ((k & 1) << 3))
                  : (uint32_t)((row >> 4) * 2048 + k * 128 + ((((row & 15) >> 1) ^ (k & 7)) << 4) + ((row & 1) << 3));
}

struct KernelArgs {
    int M, N, K;
    double alpha, beta;
    const double* A;
    long lda, strideA;
    const double* B;
    long ldb, strideB;
    double* C;
    long ldc, strideC;
    int krange, lower_only, vec_ok;
    int batch;
    long strideA2, strideB2, strideC2;
    int bA1, bA2, bB1, bB2;  // 1: the operand has that batch dimension in its tensor map (0: broadcast, coordinate 0)
};

template <int BM, int BN, int WM, int WN, bool TA, bool TB>
__global__ void __launch_bounds__((BM / WM) * (BN / WN) * 32, (BM * BN == 128 * 128 ? 1 : 2))
    dgemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, KernelArgs p) {
    constexpr int NWN = BN / WN;
    constexpr int NT = (BM / WM) * NWN * 32;
    constexpr int MT = WM / 8, NTL = WN / 8;
    constexpr bool A_KM = !TA, B_KM = TB;
    constexpr int A_BYTES = BM * BK * 8, B_BYTES = BN * BK * 8, STAGE_BYTES = A_BYTES + B_BYTES;
    extern __shared__ __align__(128) unsigned char smem_dyn[];
    __shared__ __align__(8) unsigned long long full_bar[STAGES];

    const int i0 = blockIdx.y * BM, j0 = blockIdx.x * BN;
    if (p.lower_only && j0 >= i0 + BM) return;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const int wm0 = (warp / NWN) * WM, wn0 = (warp % NWN) * WN;
    const int b1 = blockIdx.z % p.batch, b2 = blockIdx.z / p.batch;
    double* __restrict__ C = p.C + (long)b1 * p.strideC + (long)b2 * p.strideC2;

    int klo = 0, khi = p.K;
    switch (p.krange & 3) {
        case KR_LO_I: klo = i0; break;
        case KR_LO_J: klo = j0; break;
        case KR_LO_MAXIJ: klo = i0 > j0 ? i0 : j0; break;
        default: break;
    }
    switch (p.krange & 12) {
        case KR_HI_I: khi = min(khi, i0 + BM); break;
        case KR_HI_J: khi = min(khi, j0 + BN); break;
        case KR_HI_MINIJ: khi = min(khi, min(i0 + BM, j0 + BN)); break;
        default: break;
    }
    // k ranges start and end on multiples of the tile sizes (or at K, beyond which the tensor map zero-fills), so whole
    // BK-wide boxes are loaded and no partial-k predicate is needed
    const int nk = (khi > klo && p.alpha != 0.0) ? (khi - klo + BK - 1) / BK : 0;
    // the 128-byte swizzle is a function of the shared-memory ADDRESS: tile bases must be 1024-byte aligned
    const uint32_t sraw = (uint32_t)__cvta_generic_to_shared(smem_dyn);
    const uint32_t sbase = (sraw + 1023u) & ~1023u;
    unsigned char* smem_raw = smem_dyn + (sbase - sraw);
    const uint32_t bar0 = (uint32_t)__cvta_generic_to_shared(full_bar);

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) mbar_init(bar0 + 8 * s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncthreads();

    // Warp 0 feeds the ring: lane 0 arms the stage's barrier with the byte count (the phase cannot complete before that
    // arrival, whatever the order in which the copies land), then the lanes issue the boxes.
    auto load_stage = [&](int stage, int k0) {
        const uint32_t sa = sbase + stage * STAGE_BYTES, sb = sa + A_BYTES, bar = bar0 + 8 * stage;
        if (lane == 0) mbar_expect_tx(bar, STAGE_BYTES);
        __syncwarp();
        tma_operand<A_KM, BM>(sa, &tmA, bar, i0, k0, p.bA1 ? b1 : 0, p.bA2 ? b2 : 0, lane);
        tma_operand<B_KM, BN>(sb, &tmB, bar, j0, k0, p.bB1 ? b1 : 0, p.bB2 ? b2 : 0, lane);
    };

    double acc[MT][NTL][2];
    int arow[MT], bcol[NTL];
#pragma unroll
    for (int m = 0; m < MT; ++m) arow[m] = frag_row<A_KM>(wm0, m, g);
#pragma unroll
    for (int n = 0; n < NTL; ++n) bcol[n] = frag_row<B_KM>(wn0, n, g);

    if (warp == 0) {
#pragma unroll
        for (int s = 0; s < STAGES - 1; ++s)
            if (s < nk) load_stage(s, klo + s * BK);
    }

#pragma unroll
    for (int m = 0; m < MT; ++m)
#pragma unroll
        for (int n = 0; n < NTL; ++n) acc[m][n][0] = acc[m][n][1] = 0.0;

    for (int it = 0; it < nk; ++it) {
        // stage (it - 1) % STAGES was read in the previous iteration: once every warp is past this barrier it may be refilled
        __syncthreads();
        const int nxt = it + STAGES - 1;
        if (warp == 0 && nxt < nk) load_stage(nxt % STAGES, klo + nxt * BK);
        mbar_wait(bar0 + 8 * (it % STAGES), (it / STAGES) & 1);  // the TMA bytes of stage `it` have landed
        const uint32_t sa = sbase + (it % STAGES) * STAGE_BYTES, sb = sa + A_BYTES;
#pragma unroll
        for (int kk = 0; kk < BK / 4; ++kk) {
            double af[MT], bf[NTL];
            const int k = kk * 4 + t;
#pragma unroll
            for (int m = 0; m < MT; ++m) af[m] = lds64(sa + frag_addr<A_KM, BM>(arow[m], k));
#pragma unroll
            for (int n = 0; n < NTL; ++n) bf[n] = lds64(sb + frag_addr<B_KM, BN>(bcol[n], k));
#pragma unroll
            for (int m = 0; m < MT; ++m)
#pragma unroll
                for (int n = 0; n < NTL; ++n) dmma(acc[m][n][0], acc[m][n][1], af[m], bf[n]);
        }
    }

    // ---- epilogue through shared memory -----------------------------------------------------------
    // The accumulator fragments own 16-byte pieces scattered over 8 rows; reading/writing C straight from
    // them half-uses every 128-byte line and starves on outstanding-miss slots (measured: the beta*C read
    // ran at 1.6 TB/s).  Instead the C tile is moved with full-line cp.async / 128-bit stores and the
    // fragments touch only shared memory.  The pipeline buffers are free at this point.
    constexpr int CP = (BM * (BN + 2) * 8 <= STAGES * STAGE_BYTES) ? BN + 2 : BN;  // padded pitch (doubles)
    double* ct = reinterpret_cast<double*>(smem_raw);
    const double alpha = p.alpha, beta = p.beta;
    const bool full = p.vec_ok && (i0 + BM <= p.M) && (j0 + BN <= p.N);
    __syncthreads();  // every warp is done reading the last stage
    if (beta != 0.0) {
        if (full) {
#pragma unroll 4
            for (int idx = tid; idx < BM * BN / 2; idx += NT) {
                const int r = idx / (BN / 2), c = idx % (BN / 2);
                cp_async16(sbase + (r * CP + 2 * c) * 8, C + (long)(i0 + r) * p.ldc + j0 + 2 * c, 16);
            }
            cp_async_commit();
            cp_async_wait<0>();
        } else {
            for (int idx = tid; idx < BM * BN; idx += NT) {
                const int r = idx / BN, c = idx % BN;
                ct[r * CP + c] = (i0 + r < p.M && j0 + c < p.N) ? C[(long)(i0 + r) * p.ldc + j0 + c] : 0.0;
            }
        }
        __syncthreads();
    }
    auto merge2 = [&](int r, int c, double v0, double v1) {  // tile-local row r, columns c, c+1 (c even)
        double2* q = reinterpret_cast<double2*>(ct + r * CP + c);
        double2 o = make_double2(alpha * v0, alpha * v1);
        if (beta != 0.0) {
            const double2 old = *q;
            o.x = fma(beta, old.x, o.x);
            o.y = fma(beta, old.y, o.y);
        }
        *q = o;
    };
#pragma unroll
    for (int m = 0; m < MT; ++m) {
        const int r = arow[m];
        if (B_KM) {
            // fragment pair (2q, 2q+1) holds columns 16q + 4t + {0,1,2,3}
#pragma unroll
            for (int q = 0; q < NTL / 2; ++q) {
                const int c = wn0 + q * 16 + 4 * t;
                merge2(r, c, acc[m][2 * q][0], acc[m][2 * q + 1][0]);
                merge2(r, c + 2, acc[m][2 * q][1], acc[m][2 * q + 1][1]);
            }
        } else {
#pragma unroll
            for (int n = 0; n < NTL; ++n) merge2(r, frag_row<false>(wn0, n, 2 * t), acc[m][n][0], acc[m][n][1]);
        }
    }
    __syncthreads();
    if (full) {
#pragma unroll 4
        for (int idx = tid; idx < BM * BN / 2; idx += NT) {
            const int r = idx / (BN / 2), c = idx % (BN / 2);
            *reinterpret_cast<double2*>(C + (long)(i0 + r) * p.ldc + j0 + 2 * c) =
                *reinterpret_cast<const double2*>(ct + r * CP + 2 * c);
        }
    } else {
        for (int idx = tid; idx < BM * BN; idx += NT) {
            const int r = idx / BN, c = idx % BN;
            if (i0 + r < p.M && j0 + c < p.N) C[(long)(i0 + r) * p.ldc + j0 + c] = ct[r * CP + c];
        }
    }
}

// ---- tensor maps -------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPointByVersion("cuTensorMapEncodeTiled", &p, 12000, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            p = nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

// Operand `base` with op-rows of extent `rows` (M or N) and contraction extent K.  kmajor: element (r, k) at base[r * ld + k];
// else at base[k * ld + r].  Dimensions 2, 3: the two strided batch levels (extent 1 when the operand is broadcast).
bool make_operand_map(CUtensorMap* tm, const double* base, bool kmajor, int rows, int K, long ld, int tile_rows, int nb1, long s1,
                      int nb2, long s2) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return false;
    if (K < 1) K = 1;  // K == 0 (C = beta C): no box is ever requested, the map only has to be well formed
    const cuuint64_t inner = kmajor ? (cuuint64_t)K : (cuuint64_t)rows, outer = kmajor ? (cuuint64_t)rows : (cuuint64_t)K;
    const cuuint64_t dims[4] = {inner, outer, (cuuint64_t)(s1 ? nb1 : 1), (cuuint64_t)(s2 ? nb2 : 1)};
    // strides of dimensions 1..3 in bytes (multiples of 16: ld and the batch strides are even)
    const cuuint64_t one_matrix = (cuuint64_t)ld * 8 * outer;
    const cuuint64_t strides[3] = {(cuuint64_t)ld * 8, s1 ? (cuuint64_t)s1 * 8 : one_matrix, s2 ? (cuuint64_t)s2 * 8 : one_matrix};
    const cuuint32_t box[4] = {16, (cuuint32_t)(kmajor ? tile_rows : BK), 1, 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 4, const_cast<double*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int BM, int BN, int WM, int WN, bool TA, bool TB>
int launch_cfg(cudaStream_t s, const GemmArgs& a, const KernelArgs& ka) {
    constexpr int NT = (BM / WM) * (BN / WN) * 32;
    constexpr int SMEM = STAGES * (BM + BN) * BK * 8 + 1024;  // + alignment slack for the 1024-byte swizzle atoms
    static SmemOptIn optin;
    if (!optin.ensure(dgemm_kernel<BM, BN, WM, WN, TA, TB>, SMEM)) return -2;
    CUtensorMap tmA, tmB;
    if (!make_operand_map(&tmA, a.A, !TA, a.M, a.K, a.lda, BM, a.batch, a.strideA, a.batch2, a.strideA2) ||
        !make_operand_map(&tmB, a.B, TB, a.N, a.K, a.ldb, BN, a.batch, a.strideB, a.batch2, a.strideB2))
        return -3;
    dim3 grid((a.N + BN - 1) / BN, (a.M + BM - 1) / BM, a.batch * a.batch2);
    dgemm_kernel<BM, BN, WM, WN, TA, TB><<<grid, NT, SMEM, s>>>(tmA, tmB, ka);
    return cudaGetLastError() == cudaSuccess ? 0 : -2;
}

template <bool TA, bool TB>
int launch_t(cudaStream_t s, const GemmArgs& a, const KernelArgs& ka, int cfg) {
    if (cfg == 1) return launch_cfg<64, 64, 32, 32, TA, TB>(s, a, ka);
    if (cfg == 2) return launch_cfg<128, 64, 64, 32, TA, TB>(s, a, ka);
    return launch_cfg<128, 128, 64, 32, TA, TB>(s, a, ka);
}

}  // namespace

int launch_gemm(cudaStream_t s, const GemmArgs& a) {
    if (a.M <= 0 || a.N <= 0 || a.batch <= 0 || a.batch2 <= 0) return 0;
    auto al16 = [](const void* p) { return (reinterpret_cast<size_t>(p) & 15) == 0; };
    if (!al16(a.A) || !al16(a.B) || (a.lda & 1) || (a.ldb & 1) || (a.strideA & 1) || (a.strideB & 1) || (a.strideA2 & 1) || (a.strideB2 & 1)) return -1;
    KernelArgs ka;
    ka.M = a.M; ka.N = a.N; ka.K = a.K;
    ka.alpha = a.alpha; ka.beta = a.beta;
    ka.A = a.A; ka.lda = a.lda; ka.strideA = a.strideA;
    ka.B = a.B; ka.ldb = a.ldb; ka.strideB = a.strideB;
    ka.C = a.C; ka.ldc = a.ldc; ka.strideC = a.strideC;
    ka.krange = a.krange; ka.lower_only = a.lower_only;
    ka.batch = a.batch; ka.strideA2 = a.strideA2; ka.strideB2 = a.strideB2; ka.strideC2 = a.strideC2;
    ka.bA1 = a.strideA != 0; ka.bA2 = a.strideA2 != 0; ka.bB1 = a.strideB != 0; ka.bB2 = a.strideB2 != 0;
    ka.vec_ok = al16(a.C) && !(a.ldc & 1) && !(a.strideC & 1) && !(a.strideC2 & 1);
    // tile config: 0 = 128x128 (1 CTA/SM; the only one safe for the in-place panel solve), 1 = 64x64,
    // 2 = 128x64 (2 CTAs/SM: one CTA's prologue/epilogue hides behind the other's main loop) -- the default.
    int cfg;
    if (a.small_tiles >= 0) cfg = a.small_tiles;
    else {
        // 64x64 tiles when the grid would be small, or when 128-row tiles would pad M by > 12 % more than 64-row tiles do:
        // M = 300 (the SVGP inducing-point count) is 384 in 128-row tiles but 320 in 64-row tiles -- measured on the Goku
        // single-bin SVGP step: 7.93 -> 7.03 ms (profiles/r02_svgp_tile_config.log)
        const long ctas = (long)((a.M + 127) / 128) * ((a.N + 63) / 64) * a.batch * a.batch2;
        const double pad128 = (double)((a.M + 127) / 128 * 128) / a.M, pad64 = (double)((a.M + 63) / 64 * 64) / a.M;
        cfg = (ctas < 2 * 148 || pad128 > 1.12 * pad64) ? 1 : 2;
    }
    if (!a.transA && !a.transB) return launch_t<false, false>(s, a, ka, cfg);
    if (!a.transA && a.transB) return launch_t<false, true>(s, a, ka, cfg);
    if (a.transA && !a.transB) return launch_t<true, false>(s, a, ka, cfg);
    return launch_t<true, true>(s, a, ka, cfg);
}
