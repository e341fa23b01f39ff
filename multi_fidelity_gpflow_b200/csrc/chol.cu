// chol.cu -- K2: blocked right-looking fp64 Cholesky (lower, row-major); K4: triangular inverse.
//
// potrf (NB = 128):  for each diagonal block
//     diag kernel   one CTA factors the 128x128 block with the trailing matrix held in
//                   REGISTERS (2-D cyclic ownership, one published column + one barrier per
//                   step) and inverts the factor in shared memory            [latency bound]
//     panel         A21 <- A21 * inv(L11)^T      (DMMA GEMM, in place)
//     trailing      A22 <- A22 - A21 A21^T       (DMMA GEMM, lower tiles only) [FP64 pipe bound]
// trtri: inv(L) by log2(N/128) levels of batched merges
//     [W11 0; W21 W22],  W21 = -W22 (L21 W11)    two DMMA GEMMs per level, every level a full grid.
// These replace tf.linalg.cholesky / triangular_solve behind GPflow's GPR / SVGP objectives
// (reference call sites linear.py:206, singlebin_svgp.py:83, linear_svgp.py:184).
#include "chol.cuh"
#include "common.cuh"

#include "gemm.cuh"
#include "mathx.cuh"

namespace {

constexpr int NB = CHOL_NB;

struct DiagArgs {
    double* A;  // top-left of the diagonal block (batch 0)
    long lda, strideA;
    int nb;       // rows in this block (<= 128)
    int k0;       // global index of the first row (for info)
    double* dinv;  // [128*128] for this block (batch 0)
    long stride_dinv;
    double* logd;  // + k0 (batch 0)
    long stride_logd;
    int* d_info;
    int* info_vec;
};

// ---- DMMA tile helpers (same swizzled 8x8-tile layout as gpr_small_v4.cu) ---------------------------
__device__ __forceinline__ int tslot(int i, int j) { return i * (i + 1) / 2 + j; }  // i >= j
__device__ __forceinline__ int tile_off(int r, int c) { return r * 8 + ((((c >> 1) ^ (r & 2))) << 1) + (c & 1); }

constexpr int DT = NB / 8;                  // 16 tile rows
constexpr int DTRI = DT * (DT + 1) / 2;     // 136 lower tiles
// Warps of the diagonal-block kernel.  The kernel is latency bound (ncu, round 1: one warp per scheduler issues an
// instruction every 6 cycles; 23 % of them are address arithmetic), so more warps per scheduler shorten it directly:
// measured (profiles/r02_potrf_diag_warps.log) with 4 / 8 / 16 warps: potrf_inv of a 1024 block 924 / 802 / 792 us, potrf
// N = 8192 19.2 / 20.3 / 20.3 TFLOP/s, N = 16 384 29.1 / 29.5 / 29.5 (cuSOLVER 29.5).
constexpr int DIAG_WARPS = 8;
constexpr int DIAG_THREADS = 32 * DIAG_WARPS;

// One CTA factors a 128x128 diagonal block on the FP64 tensor path and inverts the factor:
//   left-looking over 8-wide block columns; tile rows are dealt round-robin to the DIAG_WARPS warps;
//   the 8x8 diagonal tile is factored redundantly in registers by one warp (no shuffles);
//   W = L^-1 is then built column by column (columns are independent -> no block barriers).
__global__ void __launch_bounds__(DIAG_THREADS, 1) potrf_diag_kernel(DiagArgs p) {
    extern __shared__ __align__(16) double sm[];
    double* Lt = sm;                 // [DTRI][64] L tiles (diagonal slots: L_kk, lower)
    double* Wt = Lt + DTRI * 64;     // [DTRI][64] W = L^-1 tiles
    double* lg = Wt + DTRI * 64;     // [DT] log-products of pivots per diagonal tile
    __shared__ int bad;
    const int nb = p.nb;
    const int ntb = (nb + 7) / 8;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const int cst = tile_off(g, 2 * t);
    const int km0 = tile_off(g, t), km1 = tile_off(g, t + 4);
    const int mm0 = tile_off(t, g), mm1 = tile_off(t + 4, g);
    const long bz = blockIdx.x;
    double* __restrict__ A = p.A + bz * p.strideA;
    if (tid == 0) bad = 0;

    // ---- load the lower triangle into tiles; pad with identity up to a multiple of 8 ---------------
    // 128-bit loads, 8 in flight per thread (a load->store chain per element exposed one L2/DRAM round trip
    // per iteration: 77k of the kernel's 237k cycles in the first profile).
    for (int idx = tid; idx < ntb * (ntb + 1) / 2 * 64; idx += DIAG_THREADS) Lt[idx] = 0.0;
    __syncthreads();
    {
        const bool vec = ((reinterpret_cast<size_t>(A) & 15) == 0) && ((p.lda & 1) == 0);
        constexpr int UN = 8;
        for (int base = 0; base < nb * (NB / 2); base += DIAG_THREADS * UN) {
            double2 v[UN];
#pragma unroll
            for (int u = 0; u < UN; ++u) {
                const int idx = base + u * DIAG_THREADS + tid;
                const int r = idx >> 6, c = (idx & 63) * 2;
                v[u] = make_double2(0.0, 0.0);
                if (r < nb && c <= r) {
                    const double* src = A + (long)r * p.lda + c;
                    if (vec) v[u] = *reinterpret_cast<const double2*>(src);
                    else {
                        v[u].x = src[0];
                        if (c + 1 <= r) v[u].y = src[1];
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < UN; ++u) {
                const int idx = base + u * DIAG_THREADS + tid;
                const int r = idx >> 6, c = (idx & 63) * 2;
                if (r < nb && c <= r) {
                    if (c + 1 > r) v[u].y = 0.0;  // strictly-upper element of a diagonal tile
                    *reinterpret_cast<double2*>(Lt + tslot(r >> 3, c >> 3) * 64 + tile_off(r & 7, c & 7)) = v[u];
                }
            }
        }
    }
    for (int r = nb + tid; r < ntb * 8; r += DIAG_THREADS) Lt[tslot(r >> 3, r >> 3) * 64 + tile_off(r & 7, r & 7)] = 1.0;
    __syncthreads();

    // Left-looking with a one-column look-ahead: while warp 0 factors the 8x8 diagonal tile of column kb
    // (a ~2k-cycle dependent chain), warps 1-3 already apply the terms k < kb to column kb+1; only the last
    // term (k = kb) of each column sits on the critical path.
    auto update_tiles = [&](int col, int kfrom, int kto, int w, int nw) {
        // tile (i, col) -= sum_{k=kfrom}^{kto-1} L_ik L_col,k^T for rows i = col + w, col + w + nw, ... (4 chains per pass)
        for (int ibase = col + w; ibase < ntb; ibase += 4 * nw) {
            double acc[4][2];
            int row[4];
#pragma unroll
            for (int s4 = 0; s4 < 4; ++s4) {
                row[s4] = ibase + s4 * nw;
                if (row[s4] < ntb) {
                    const double2 v = *reinterpret_cast<const double2*>(Lt + tslot(row[s4], col) * 64 + cst);
                    acc[s4][0] = v.x;
                    acc[s4][1] = v.y;
                }
            }
#pragma unroll 1
            for (int k = kfrom; k < kto; ++k) {
                const double* tb = Lt + tslot(col, k) * 64;
                const double b0 = tb[km0], b1 = tb[km1];
#pragma unroll
                for (int s4 = 0; s4 < 4; ++s4)
                    if (row[s4] < ntb) {
                        const double* ta = Lt + tslot(row[s4], k) * 64;
                        dmma(acc[s4][0], acc[s4][1], -ta[km0], b0);
                        dmma(acc[s4][0], acc[s4][1], -ta[km1], b1);
                    }
            }
#pragma unroll
            for (int s4 = 0; s4 < 4; ++s4)
                if (row[s4] < ntb)
                    *reinterpret_cast<double2*>(Lt + tslot(row[s4], col) * 64 + cst) = make_double2(acc[s4][0], acc[s4][1]);
        }
    };
#pragma unroll 1
    for (int kb = 0; kb < ntb; ++kb) {
        // ---- finish column kb: only the term k = kb-1 is still missing (earlier terms were applied one step ahead)
        if (kb > 0) update_tiles(kb, kb - 1, kb, warp, DIAG_WARPS);
        __syncthreads();
        // ---- warp 0: diagonal tile (redundant register Cholesky + inverse); warps 1-3: look-ahead on column kb+1
        if (warp != 0) {
            if (kb + 1 < ntb && kb > 0) update_tiles(kb + 1, 0, kb, warp - 1, DIAG_WARPS - 1);
        } else {
            double* td = Lt + tslot(kb, kb) * 64;
            double* tw = Wt + tslot(kb, kb) * 64;
            double a[8][8], rinv[8];
#pragma unroll
            for (int r = 0; r < 8; ++r)
#pragma unroll
                for (int c = 0; c <= r; ++c) a[r][c] = td[tile_off(r, c)];
            double prod = 1.0;
            int mybad = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                double piv = a[j][j];
                if (!(piv > 0.0)) {
                    if (!mybad) mybad = p.k0 + 8 * kb + j + 1;
                    piv = nan("");
                }
                prod *= piv;
                const double ri = rsqrt(piv);
                rinv[j] = ri;
                a[j][j] = piv * ri;  // L_jj = sqrt(piv)
#pragma unroll
                for (int i = j + 1; i < 8; ++i) a[i][j] *= ri;
#pragma unroll
                for (int k = j + 1; k < 8; ++k)
#pragma unroll
                    for (int i = k; i < 8; ++i) a[i][k] = fma(-a[i][j], a[k][j], a[i][k]);
            }
            const int c = lane & 7;
            double w[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                double s = (i == c) ? 1.0 : 0.0;
#pragma unroll
                for (int k = 0; k < i; ++k) s = fma(-a[i][k], w[k], s);
                w[i] = s * rinv[i];
            }
            __syncwarp();
            // all lanes hold the same L_kk: same-address stores collapse to one write each
#pragma unroll
            for (int r = 0; r < 8; ++r)
#pragma unroll
                for (int cc = 0; cc < 8; ++cc) td[tile_off(r, cc)] = (cc <= r) ? a[r][cc] : 0.0;
            if (lane < 8) {
#pragma unroll
                for (int i = 0; i < 8; ++i) tw[tile_off(i, c)] = w[i];
            }
            if (lane == 0) {
                lg[kb] = log(prod);
                if (mybad && bad == 0) bad = mybad;
            }
        }
        __syncthreads();
        // ---- panel: L_ik = A_ik inv(L_kk)^T for rows i = kb + 1 + warp + DIAG_WARPS s ---------------------
        {
            const double* tw = Wt + tslot(kb, kb) * 64;
            const double wb0 = tw[km0], wb1 = tw[km1];
#pragma unroll
            for (int s = 0; s < (DT + DIAG_WARPS - 1) / DIAG_WARPS; ++s) {
                const int i = kb + 1 + warp + DIAG_WARPS * s;
                if (i < ntb) {
                    double* ta = Lt + tslot(i, kb) * 64;
                    const double a0 = ta[km0], a1 = ta[km1];
                    double c0 = 0.0, c1 = 0.0;
                    dmma(c0, c1, a0, wb0);
                    dmma(c0, c1, a1, wb1);
                    __syncwarp();
                    *reinterpret_cast<double2*>(ta + cst) = make_double2(c0, c1);
                }
            }
        }
        __syncthreads();
    }

    // ---- write L back (lower, strict upper of the block zeroed) and log L_ii ------------------------------
    for (int idx = tid; idx < nb * NB; idx += DIAG_THREADS) {
        const int r = idx >> 7, c = idx & (NB - 1);
        if (c < nb) A[(long)r * p.lda + c] = (c <= r) ? Lt[tslot(r >> 3, c >> 3) * 64 + tile_off(r & 7, c & 7)] : 0.0;
    }
    if (tid < nb) p.logd[bz * p.stride_logd + tid] = 0.0;  // per-row logs are folded into the first row of each tile
    __syncthreads();
    if (tid < ntb) p.logd[bz * p.stride_logd + 8 * tid] = 0.5 * lg[tid];

    // ---- W = L^-1: column block j owned by warp j % DIAG_WARPS (columns are independent) ------------------
#pragma unroll 1
    for (int j = warp; j < ntb; j += DIAG_WARPS) {
#pragma unroll 1
        for (int i = j + 1; i < ntb; ++i) {
            double c0 = 0.0, c1 = 0.0, d0 = 0.0, d1 = 0.0;  // two interleaved accumulator chains
            int k = j;
#pragma unroll 1
            for (; k + 1 < i; k += 2) {
                const double* ta = Lt + tslot(i, k) * 64;
                const double* tb = Wt + tslot(k, j) * 64;
                const double* ta2 = Lt + tslot(i, k + 1) * 64;
                const double* tb2 = Wt + tslot(k + 1, j) * 64;
                dmma(c0, c1, ta[km0], tb[mm0]);
                dmma(d0, d1, ta2[km0], tb2[mm0]);
                dmma(c0, c1, ta[km1], tb[mm1]);
                dmma(d0, d1, ta2[km1], tb2[mm1]);
            }
            if (k < i) {
                const double* ta = Lt + tslot(i, k) * 64;
                const double* tb = Wt + tslot(k, j) * 64;
                dmma(c0, c1, ta[km0], tb[mm0]);
                dmma(c0, c1, ta[km1], tb[mm1]);
            }
            c0 += d0;
            c1 += d1;
            double* tij = Wt + tslot(i, j) * 64;
            *reinterpret_cast<double2*>(tij + cst) = make_double2(c0, c1);  // T = sum_k L_ik W_kj
            __syncwarp();
            const double* tw = Wt + tslot(i, i) * 64;
            double w0 = 0.0, w1 = 0.0;
            dmma(w0, w1, -tw[km0], tij[mm0]);
            dmma(w0, w1, -tw[km1], tij[mm1]);
            __syncwarp();
            *reinterpret_cast<double2*>(tij + cst) = make_double2(w0, w1);
            __syncwarp();
        }
    }
    __syncthreads();
    double* __restrict__ D = p.dinv + bz * p.stride_dinv;
    for (int idx = tid; idx < NB * NB; idx += DIAG_THREADS) {
        const int r = idx >> 7, c = idx & (NB - 1);
        D[idx] = (r < nb && c <= r) ? Wt[tslot(r >> 3, c >> 3) * 64 + tile_off(r & 7, c & 7)] : 0.0;
    }
    if (tid == 0 && bad) {
        atomicCAS(p.d_info, 0, bad);
        if (p.info_vec) atomicCAS(p.info_vec + bz, 0, bad);
    }
}

constexpr size_t DIAG_SMEM = (size_t)(2 * DTRI * 64 + DT + 2) * 8;

// W diagonal blocks <- dinv; everything else of W <- 0 (done by memset before)
__global__ void place_diag_kernel(const double* __restrict__ dinv, long stride_dinv, int nblk, double* __restrict__ W,
                                  long ldw, long strideW, int N) {
    const int kb = blockIdx.x, bz = blockIdx.y;
    const double* D = dinv + bz * stride_dinv + (long)kb * NB * NB;
    double* Wb = W + bz * strideW + (long)kb * NB * ldw + kb * NB;
    const int nb = min(NB, N - kb * NB);
    for (int idx = threadIdx.x; idx < NB * NB; idx += blockDim.x) {
        const int i = idx >> 7, j = idx & (NB - 1);
        if (i < nb && j < nb) Wb[(long)i * ldw + j] = D[idx];
    }
}

}  // namespace

int launch_potrf(cudaStream_t s, const CholArgs& a) {
    if (a.N <= 0 || a.batch <= 0) return 0;
    static SmemOptIn optin;
    if (!optin.ensure(potrf_diag_kernel, DIAG_SMEM)) return -2;
    const int N = a.N;
    const int nblk = chol_nblk(N);
    const long stride_dinv = (long)nblk * NB * NB;
    // outer block: the trailing update is a rank-OB GEMM (OB / 128 panels of 128 columns); wider = fewer read-modify-write
    // passes over the trailing matrix and longer DMMA main loops per tile, at the price of more skinny inner updates on
    // the panel stream.  Measured on B200 (scripts/potrf_once.py): see DESIGN.md section 5.
    // measured with the TMA-fed GEMM (profiles/r02_potrf_outer_block.log): N = 8192: 128 -> 18.0, 256 -> 19.2, 384 -> 18.6 TFLOP/s;
    // N = 16 384: 256 -> 27.7, 384 -> 28.6, 512 -> 29.0, 768 -> 28.9; N = 32 768: 512 -> 32.6, 768 -> 33.2, 1024 -> 33.4
    const int OB = N <= 12288 ? 2 * NB : (N <= 24576 ? 4 * NB : 8 * NB);
    // Look-ahead: the latency-bound chain  diag -> panel -> inner update -> diag -> panel  runs on the aux stream and
    // overlaps the FP64-bound trailing update of the previous outer step; the main stream hands over the next
    // OB columns early.
    const bool la = a.aux != nullptr && a.ev != nullptr && N > 2 * OB;
    cudaStream_t sp = la ? a.aux : s;
    if (la) {
        cudaEventRecord(a.ev[0], s);
        cudaStreamWaitEvent(sp, a.ev[0], 0);
    }
    auto diag = [&](int k0, int nb) {
        DiagArgs d;
        d.A = a.A + (long)k0 * a.lda + k0;
        d.lda = a.lda;
        d.strideA = a.strideA;
        d.nb = nb;
        d.k0 = k0;
        d.dinv = a.dinv + (long)(k0 / NB) * NB * NB;
        d.stride_dinv = stride_dinv;
        d.logd = a.logd + k0;
        d.stride_logd = N;
        d.d_info = a.d_info;
        d.info_vec = a.info_vec;
        potrf_diag_kernel<<<a.batch, DIAG_THREADS, DIAG_SMEM, sp>>>(d);
    };
    // rows [r0, N) of block column [k0, k0+nb)  <-  (same) * inv(L_kk)^T     (in place, one 128-wide column tile)
    auto panel = [&](int k0, int nb, int r0) -> int {
        if (N - r0 <= 0) return 0;
        double* P = a.A + (long)r0 * a.lda + k0;
        GemmArgs g;
        g.transA = false; g.transB = true;
        g.M = N - r0; g.N = nb; g.K = nb;
        g.A = P; g.lda = a.lda; g.strideA = a.strideA;
        g.B = a.dinv + (long)(k0 / NB) * NB * NB; g.ldb = NB; g.strideB = stride_dinv;
        g.C = P; g.ldc = a.lda; g.strideC = a.strideA;
        g.batch = a.batch;
        g.small_tiles = 0;
        return launch_gemm(sp, g);
    };
    // C[rows r0.., cols c0..c0+nc) -= P[rows r0.., k0..k0+kw) * P[rows c0..c0+nc, k0..k0+kw)^T
    auto update = [&](cudaStream_t st, int r0, int c0, int nc, int k0, int kw, int lower) -> int {
        if (N - r0 <= 0 || nc <= 0) return 0;
        GemmArgs t;
        t.transA = false; t.transB = true;
        t.M = N - r0; t.N = nc; t.K = kw;
        t.alpha = -1.0; t.beta = 1.0;
        t.A = a.A + (long)r0 * a.lda + k0; t.lda = a.lda; t.strideA = a.strideA;
        t.B = a.A + (long)c0 * a.lda + k0; t.ldb = a.lda; t.strideB = a.strideA;
        t.C = a.A + (long)r0 * a.lda + c0; t.ldc = a.lda; t.strideC = a.strideA;
        t.batch = a.batch;
        t.lower_only = lower;
        return launch_gemm(st, t);
    };
    int step = 0;
    for (int K0 = 0; K0 < N; K0 += OB, ++step) {
        const int w = N - K0 < OB ? N - K0 : OB;
        cudaEvent_t ev_col = la ? a.ev[2 * (step & 1)] : nullptr, ev_panel = la ? a.ev[2 * (step & 1) + 1] : nullptr;
        if (la && step > 0) cudaStreamWaitEvent(sp, ev_col, 0);  // columns [K0, K0+w) fully updated
        // factor the outer block column panel by panel (left-looking inside the block: panel j first receives the
        // rank-(j*128) update from the panels already finished in this block)
        for (int j0 = 0; j0 < w; j0 += NB) {
            const int nbj = w - j0 < NB ? w - j0 : NB;
            if (j0 > 0 && update(sp, K0 + j0, K0 + j0, nbj, K0, j0, 0)) return -2;
            diag(K0 + j0, nbj);
            if (panel(K0 + j0, nbj, K0 + j0 + nbj)) return -2;
        }
        const int rem = N - K0 - w;
        if (rem <= 0) break;
        if (la) {
            cudaEventRecord(ev_panel, sp);
            cudaStreamWaitEvent(s, ev_panel, 0);
        }
        // trailing <- trailing - P P^T with P = A[K0+w:, K0:K0+w]  (rank-w update, lower tiles)
        const int ncol = la ? (rem < OB ? rem : OB) : 0;
        if (la) {
            if (update(s, K0 + w, K0 + w, ncol, K0, w, 1)) return -2;  // next outer block column first (lower tiles)
            cudaEventRecord(a.ev[2 * ((step + 1) & 1)], s);
        }
        if (rem - ncol > 0 && update(s, K0 + w + ncol, K0 + w + ncol, rem - ncol, K0, w, 1)) return -2;
    }
    if (la) {  // the main stream owns the result again
        cudaEventRecord(a.ev[0], sp);
        cudaStreamWaitEvent(s, a.ev[0], 0);
    }
    return cudaGetLastError() == cudaSuccess ? 0 : -2;
}

int launch_trtri(cudaStream_t s, const CholArgs& a, double* W, long ldw, long strideW, double* scratch) {
    if (a.N <= 0 || a.batch <= 0) return 0;
    const int N = a.N;
    const int nblk = chol_nblk(N);
    const long stride_dinv = (long)nblk * NB * NB;
    for (int b = 0; b < a.batch; ++b)
        cudaMemsetAsync(W + b * strideW, 0, sizeof(double) * (size_t)N * ldw, s);
    place_diag_kernel<<<dim3(nblk, a.batch), 256, 0, s>>>(a.dinv, stride_dinv, nblk, W, ldw, strideW, N);
    for (long sz = NB; sz < N; sz *= 2) {
        // pairs c: first half [c*2sz, c*2sz+sz), second half [c*2sz+sz, min(c*2sz+2sz, N))
        const int nfull = (int)(N / (2 * sz));                 // pairs whose second half is full
        const int rem2 = (int)(N - nfull * 2 * sz - sz);       // rows in the ragged last second half
        for (int pass = 0; pass < 2; ++pass) {
            int npairs, s2;
            long c0;
            if (pass == 0) { npairs = nfull; s2 = (int)sz; c0 = 0; }
            else { npairs = rem2 > 0 ? 1 : 0; s2 = rem2; c0 = nfull; }
            if (npairs == 0) continue;
            const long o1 = c0 * 2 * sz;  // first-half offset of the first pair in this pass
            const long pstepL = 2 * sz * a.lda + 2 * sz, pstepW = 2 * sz * ldw + 2 * sz;
            // T = L21 * W11      (s2 x sz) = (s2 x sz) (sz x sz lower)
            GemmArgs g;
            g.transA = false; g.transB = false;
            g.M = s2; g.N = (int)sz; g.K = (int)sz;
            g.A = a.A + (o1 + sz) * a.lda + o1; g.lda = a.lda; g.strideA = pstepL; g.strideA2 = a.strideA;
            g.B = W + o1 * ldw + o1; g.ldb = ldw; g.strideB = pstepW; g.strideB2 = strideW;
            g.C = scratch + (o1 + sz) * ldw + o1; g.ldc = ldw; g.strideC = pstepW; g.strideC2 = strideW;
            g.batch = npairs; g.batch2 = a.batch;
            g.krange = KR_LO_J;
            if (launch_gemm(s, g)) return -2;
            // W21 = -W22 * T     (s2 x sz) = (s2 x s2 lower) (s2 x sz)
            GemmArgs h;
            h.transA = false; h.transB = false;
            h.M = s2; h.N = (int)sz; h.K = s2;
            h.alpha = -1.0;
            h.A = W + (o1 + sz) * ldw + (o1 + sz); h.lda = ldw; h.strideA = pstepW; h.strideA2 = strideW;
            h.B = g.C; h.ldb = ldw; h.strideB = pstepW; h.strideB2 = strideW;
            h.C = W + (o1 + sz) * ldw + o1; h.ldc = ldw; h.strideC = pstepW; h.strideC2 = strideW;
            h.batch = npairs; h.batch2 = a.batch;
            h.krange = KR_HI_I;
            if (launch_gemm(s, h)) return -2;
        }
    }
    return cudaGetLastError() == cudaSuccess ? 0 : -2;
}
