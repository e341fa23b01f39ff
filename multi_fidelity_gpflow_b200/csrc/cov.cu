// cov.cu -- K1: fused multi-fidelity covariance assembly; K5: gradient contraction with
// on-the-fly recomputation of dK/dtheta.
//
// Replaces LinearMultiFidelityKernel.K / K_diag (reference mfgpflow/linear.py:55-136): no
// gather / meshgrid / scatter -- every output element selects its block from the two
// fidelity flags:   K_ij = s_i s_j k_L(x_i, x_j) + h_i h_j k_delta(x_i, x_j)
//   s = 1 (fid 0) | rho (fid 1) | 0 (anything else, linear.py:82), h = [fid == 1].
// The squared distance uses the expanded form GPflow's SquaredExponential uses
// (|a|^2 + |b|^2 - 2 a.b on length-scaled inputs), folded into the exp argument.
//
// Tiling: one CTA = 64 x 64 outputs, 256 threads, 4x4 register block per thread.  X tiles
// are staged in shared memory already divided by the length-scales, k-major so that the
// inner loop is 2+2 128-bit LDS per 16 DFMA.  A warp covers 4 thread-rows x 8 thread-cols,
// so both the direct store (row segments) and the mirrored store of the symmetric case
// (column segments) are written as full 128-byte lines with 128-bit STG.
#include "cov.cuh"
#include "common.cuh"

#include "mathx.cuh"

#include <cstdio>

namespace {

struct TileSmem {
    double* aL;  // [d][64] scaled coords of the row points (kernel_L length-scales)
    double* bL;  // [d][64] ... of the column points
    double* aD;  // kernel_delta length-scales
    double* bD;
    double* haL;  // [64] -0.5 |a|^2
    double* hbL;
    double* haD;
    double* hbD;
    double* fa;  // [64] s_a
    double* sb;  // [64] s_b
    double* ga;  // [64] h_a * var_D
    double* hb;  // [64] h_b
    double* th;  // [2d+3] theta, then [2d] inverse length-scales (L then D)
    int* flags;  // [2] any HF row / any HF col
    double* etab;  // [64] 2^(j/64) for fexp_tab
};

__device__ inline TileSmem carve(double* base, int d) {
    TileSmem t;
    const int T = COV_TILE;
    t.aL = base;
    t.bL = t.aL + d * T;
    t.aD = t.bL + d * T;
    t.bD = t.aD + d * T;
    t.haL = t.bD + d * T;
    t.hbL = t.haL + T;
    t.haD = t.hbL + T;
    t.hbD = t.haD + T;
    t.fa = t.hbD + T;
    t.sb = t.fa + T;
    t.ga = t.sb + T;
    t.hb = t.ga + T;
    t.th = t.hb + T;
    t.flags = reinterpret_cast<int*>(t.th + 4 * MFGP_MAX_D + 4);
    t.etab = t.th + 4 * MFGP_MAX_D + 4 + 2;
    return t;
}

__host__ __device__ inline size_t tile_smem_bytes(int d) { return (size_t)(4 * d * COV_TILE + 8 * COV_TILE + 4 * MFGP_MAX_D + 4) * 8 + 16 + 64 * 8; }

// Loads theta and both 64-point tiles.  Must be called by all 256 threads.
__device__ inline void load_tiles(const TileSmem& t, const double* __restrict__ Xa, int Na, int i0,
                                  const double* __restrict__ Xb, int Nb, int j0, int d,
                                  const double* __restrict__ theta) {
    const int tid = threadIdx.x;
    const int T = COV_TILE;
    if (tid < 2 * d + 3) t.th[tid] = theta[tid];
    if (tid < 2) t.flags[tid] = 0;
    fexp_table_fill(t.etab, tid, blockDim.x);
    __syncthreads();
    if (tid < 2 * d) {
        // inverse length-scales: th[2d+3 + k] = 1/lsL[k], th[3d+3 + k] = 1/lsD[k]
        int k = tid < d ? tid : tid - d;
        double ls = tid < d ? t.th[1 + k] : t.th[2 + d + k];
        t.th[2 * d + 3 + tid] = 1.0 / ls;
    }
    __syncthreads();
    if (tid < 2 * T) {
        const int which = tid >> 6;  // 0: row points, 1: col points
        const int r = tid & (T - 1);
        const double* X = which ? Xb : Xa;
        const int Np = which ? Nb : Na;
        const int p = (which ? j0 : i0) + r;
        const double rho = t.th[0], vD = t.th[2 + 2 * d];
        double s = 0.0, h = 0.0;
        bool live = false;
        if (p < Np) {
            double fid = X[(long)p * (d + 1) + d];
            if (fid == 0.0) {
                s = 1.0;
                live = true;
            } else if (fid == 1.0) {
                s = rho;
                h = 1.0;
                live = true;
            }
        }
        double nL = 0.0, nD = 0.0;
        double* cL = which ? t.bL : t.aL;
        double* cD = which ? t.bD : t.aD;
        for (int k = 0; k < d; ++k) {
            double x = live ? X[(long)p * (d + 1) + k] : 0.0;
            double xl = x * t.th[2 * d + 3 + k];
            double xd = x * t.th[3 * d + 3 + k];
            cL[k * T + r] = xl;
            cD[k * T + r] = xd;
            nL = fma(xl, xl, nL);
            nD = fma(xd, xd, nD);
        }
        if (which) {
            t.hbL[r] = -0.5 * nL;
            t.hbD[r] = -0.5 * nD;
            t.sb[r] = s;
            t.hb[r] = h;
        } else {
            t.haL[r] = -0.5 * nL;
            t.haD[r] = -0.5 * nD;
            t.fa[r] = s;
            t.ga[r] = h * vD;
        }
        if (h != 0.0) t.flags[which] = 1;  // benign race: all writers store 1
    }
    __syncthreads();
}

// acc[a][b] = sum_k A[k][r0+a] * B[k][col(b)],  col(b) = {2tx, 2tx+1, 32+2tx, 33+2tx}
__device__ inline void tile_dots(const double* __restrict__ A, const double* __restrict__ B, int d, int r0, int tx,
                                 double acc[4][4]) {
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;
#pragma unroll 2
    for (int k = 0; k < d; ++k) {
        const double2 a01 = *reinterpret_cast<const double2*>(A + k * COV_TILE + r0);
        const double2 a23 = *reinterpret_cast<const double2*>(A + k * COV_TILE + r0 + 2);
        const double2 b01 = *reinterpret_cast<const double2*>(B + k * COV_TILE + 2 * tx);
        const double2 b23 = *reinterpret_cast<const double2*>(B + k * COV_TILE + 32 + 2 * tx);
        const double av[4] = {a01.x, a01.y, a23.x, a23.y};
        const double bv[4] = {b01.x, b01.y, b23.x, b23.y};
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) acc[a][b] = fma(av[a], bv[b], acc[a][b]);
    }
}

// Streaming-kernel variant: ACCUMULATES onto acc (the caller seeds it with the exponent's additive terms, which saves a
// zero-fill and an add per element) and unrolls fully when the dimension is a compile-time constant (D > 0), so the
// panel rows are immediate offsets of one base register instead of a loop with address arithmetic.
template <int D>
__device__ __forceinline__ void tile_dots_acc(const double* __restrict__ A, const double* __restrict__ B, int d, int r0, int tx,
                                              double acc[4][4]) {
    const double* pa = A + r0;
    const double* pb = B + 2 * tx;
    auto step = [&](int k) {
        const double2 a01 = *reinterpret_cast<const double2*>(pa + k * COV_TILE);
        const double2 a23 = *reinterpret_cast<const double2*>(pa + k * COV_TILE + 2);
        const double2 b01 = *reinterpret_cast<const double2*>(pb + k * COV_TILE);
        const double2 b23 = *reinterpret_cast<const double2*>(pb + k * COV_TILE + 32);
        const double av[4] = {a01.x, a01.y, a23.x, a23.y};
        const double bv[4] = {b01.x, b01.y, b23.x, b23.y};
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) acc[a][b] = fma(av[a], bv[b], acc[a][b]);
    };
    if constexpr (D > 0) {
#pragma unroll
        for (int k = 0; k < D; ++k) step(k);
    } else {
#pragma unroll 2
        for (int k = 0; k < d; ++k) step(k);
    }
}

__device__ inline int col_of(int tx, int b) { return (b < 2 ? 0 : 32) + 2 * tx + (b & 1); }

__device__ inline void tile_index(long t, int TJ, int symmetric, int& I, int& J) {
    if (symmetric) {
        long i = (long)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
        while ((i + 1) * (i + 2) / 2 <= t) ++i;
        while (i * (i + 1) / 2 > t) --i;
        I = (int)i;
        J = (int)(t - i * (i + 1) / 2);
    } else {
        I = (int)(t / TJ);
        J = (int)(t % TJ);
    }
}

__global__ void __launch_bounds__(256, 2) cov_kernel(CovArgs p, int TJ, int vec_ok) {
    extern __shared__ __align__(16) double smem[];
    const TileSmem t = carve(smem, p.d);
    int I, J;
    tile_index(blockIdx.x, TJ, p.symmetric, I, J);
    const int b = blockIdx.z;
    const int i0 = I * COV_TILE, j0 = J * COV_TILE;
    load_tiles(t, p.Xa, p.Na, i0, p.Xb, p.Nb, j0, p.d, p.theta + (long)b * p.theta_stride);

    const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
    const int tx = (w & 1) * 8 + (lane & 7);
    const int ty = (w >> 1) * 4 + (lane >> 3);
    const int r0 = ty * 4;

    double acc[4][4], val[4][4];
    const double vL = t.th[1 + p.d];
    tile_dots(t.aL, t.bL, p.d, r0, tx, acc);
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int cc = col_of(tx, c);
            // (s_a s_b) and (h_a + h_b) are commutative: K(X,X) comes out exactly symmetric
            val[a][c] = (t.fa[r0 + a] * t.sb[cc]) * vL * fexp_tab(acc[a][c] + (t.haL[r0 + a] + t.hbL[cc]), t.etab);
        }
    if (t.flags[0] && t.flags[1]) {  // tile touches the HF x HF block: add the discrepancy GP
        tile_dots(t.aD, t.bD, p.d, r0, tx, acc);
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int cc = col_of(tx, c);
                const double g = t.ga[r0 + a] * t.hb[cc];
                if (g != 0.0) val[a][c] += g * fexp_tab(acc[a][c] + (t.haD[r0 + a] + t.hbD[cc]), t.etab);
            }
    }
    if (p.symmetric && I == J) {
        const double dg = p.diag_add_vec ? p.diag_add_vec[b] : p.diag_add;
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int c = 0; c < 4; ++c)
                if (r0 + a == col_of(tx, c)) val[a][c] += dg;
    }

    double* __restrict__ K = p.K + (long)b * p.strideK;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const int i = i0 + r0 + a;
        if (i >= p.Na) continue;
#pragma unroll
        for (int hblk = 0; hblk < 2; ++hblk) {
            const int j = j0 + hblk * 32 + 2 * tx;
            double* dst = K + (long)i * p.ldk + j;
            if (vec_ok && j + 1 < p.Nb) {
                *reinterpret_cast<double2*>(dst) = make_double2(val[a][2 * hblk], val[a][2 * hblk + 1]);
            } else {
                if (j < p.Nb) dst[0] = val[a][2 * hblk];
                if (j + 1 < p.Nb) dst[1] = val[a][2 * hblk + 1];
            }
        }
    }
    if (p.symmetric && p.mirror && I != J) {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int j = j0 + col_of(tx, c);
            if (j >= p.Nb) continue;
            const int i = i0 + r0;
            double* dst = K + (long)j * p.ldk + i;
            if (vec_ok && i + 3 < p.Na) {
                *reinterpret_cast<double2*>(dst) = make_double2(val[0][c], val[1][c]);
                *reinterpret_cast<double2*>(dst + 2) = make_double2(val[2][c], val[3][c]);
            } else {
#pragma unroll
                for (int a = 0; a < 4; ++a)
                    if (i + a < p.Na) dst[a] = val[a][c];
            }
        }
    }
}

__global__ void cov_diag_kernel(const double* __restrict__ X, int N, int d, const double* __restrict__ theta,
                                long theta_stride, double* __restrict__ out, long out_stride) {
    const int b = blockIdx.y;
    const double* th = theta + (long)b * theta_stride;
    const double rho = th[0], vL = th[1 + d], vD = th[2 + 2 * d];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
        const double fid = X[(long)i * (d + 1) + d];
        double v = 0.0;
        if (fid == 0.0) v = vL;
        else if (fid == 1.0) v = __dadd_rn(__dmul_rn(vL, __dmul_rn(rho, rho)), vD);  // K_diag_L * rho^2 + K_diag_delta (linear.py:127)
        out[(long)b * out_stride + i] = v;
    }
}

// ---------------------------------------------------------------------------------------------
// K5: out[q] = sum_ij G_ij dK_ij/dtheta_q with dK recomputed in registers (never stored).
// ---------------------------------------------------------------------------------------------
__device__ inline double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

template <bool ROWGRAD>
__global__ void __launch_bounds__(256, 2) cov_grad_kernel(CovGradArgs p, int TJ, long ntiles) {
    extern __shared__ __align__(16) double smem[];
    const int d = p.d;
    const TileSmem t = carve(smem, d);
    double* red = smem + tile_smem_bytes(d) / 8;  // [8 warps][2d+4]
    int I, J;
    tile_index(blockIdx.x, TJ, p.sym_lower, I, J);
    const int b = blockIdx.z;
    const int i0 = I * COV_TILE, j0 = J * COV_TILE;
    load_tiles(t, p.Xa, p.Na, i0, p.Xb, p.Nb, j0, d, p.theta + (long)b * p.theta_stride);

    const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
    const int tx = (w & 1) * 8 + (lane & 7);
    const int ty = (w >> 1) * 4 + (lane >> 3);
    const int r0 = ty * 4;
    const int nq = 2 * d + 4;
    const bool hh = t.flags[0] && t.flags[1];

    // weights G (with symmetric-lower multiplicity) for this thread's 4x4 block
    const double* __restrict__ G = p.G + (long)b * p.strideG;
    double TL[4][4], TD[4][4], acc[4][4];
    double s_diag = 0.0;
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int i = i0 + r0 + a, j = j0 + col_of(tx, c);
            double g = 0.0;
            if (i < p.Na && j < p.Nb) {
                if (p.sym_lower) {
                    if (j < i) g = 2.0 * G[(long)i * p.ldg + j];
                    else if (j == i) {
                        g = G[(long)i * p.ldg + j];
                        s_diag += g;
                    }
                } else {
                    g = G[(long)i * p.ldg + j];
                }
            }
            TL[a][c] = g;
            TD[a][c] = g;
        }
    tile_dots(t.aL, t.bL, d, r0, tx, acc);
    const double vL = t.th[1 + d];
    double s_vL = 0.0, s_rho = 0.0, s_vD = 0.0;
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int cc = col_of(tx, c);
            const double kl = (t.fa[r0 + a] * t.sb[cc]) * vL * fexp_tab(acc[a][c] + (t.haL[r0 + a] + t.hbL[cc]), t.etab);
            const double v = TL[a][c] * kl;  // G_ij * K^L_ij
            TL[a][c] = v;
            s_vL += v;
            // dK^L/drho = K^L (h_i + h_j) / rho ;  ga > 0 <=> h_a == 1
            s_rho += v * ((t.ga[r0 + a] != 0.0 ? 1.0 : 0.0) + t.hb[cc]);
        }
    if (hh) {
        tile_dots(t.aD, t.bD, d, r0, tx, acc);
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int cc = col_of(tx, c);
                const double g = t.ga[r0 + a] * t.hb[cc];
                const double v = (g != 0.0) ? TD[a][c] * g * fexp_tab(acc[a][c] + (t.haD[r0 + a] + t.hbD[cc]), t.etab) : 0.0;
                TD[a][c] = v;
                s_vD += v;
            }
    }
    double* myred = red + w * nq;
    {
        const double r_rho = warp_sum(s_rho), r_vL = warp_sum(s_vL), r_vD = warp_sum(s_vD), r_dg = warp_sum(s_diag);
        if (lane == 0) {
            myred[0] = r_rho;
            myred[1 + d] = r_vL;
            myred[2 + 2 * d] = hh ? r_vD : 0.0;
            myred[3 + 2 * d] = r_dg;
        }
    }
    double* __restrict__ rg = ROWGRAD ? p.rowgrad + (long)b * p.rowgrad_stride : nullptr;
    for (int k = 0; k < d; ++k) {
        double sL = 0.0, sD = 0.0;
        double zr[4] = {0.0, 0.0, 0.0, 0.0};
        const double ilL = t.th[2 * d + 3 + k], ilD = t.th[3 * d + 3 + k];
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            const double xa = t.aL[k * COV_TILE + r0 + a];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const double df = t.bL[k * COV_TILE + col_of(tx, c)] - xa;
                const double tv = TL[a][c] * df;
                sL = fma(tv, df, sL);
                if (ROWGRAD) zr[a] = fma(tv, ilL, zr[a]);
            }
        }
        if (hh) {
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                const double xa = t.aD[k * COV_TILE + r0 + a];
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const double df = t.bD[k * COV_TILE + col_of(tx, c)] - xa;
                    const double tv = TD[a][c] * df;
                    sD = fma(tv, df, sD);
                    if (ROWGRAD) zr[a] = fma(tv, ilD, zr[a]);
                }
            }
        }
        sL = warp_sum(sL);
        sD = warp_sum(sD);
        if (lane == 0) {
            myred[1 + k] = sL;
            myred[2 + d + k] = sD;
        }
        if (ROWGRAD) {
            // dk/dx_i,k = K * (x_j - x_i)_k / ls_k^2 = K * df_scaled / ls_k ; reduce over the 8 lanes sharing a row
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                double z = zr[a];
                z += __shfl_xor_sync(0xffffffffu, z, 1);
                z += __shfl_xor_sync(0xffffffffu, z, 2);
                z += __shfl_xor_sync(0xffffffffu, z, 4);
                const int i = i0 + r0 + a;
                if ((lane & 7) == 0 && i < p.Na && z != 0.0) atomicAdd(rg + (long)i * (d + 1) + k, p.rowgrad_scale * z);
            }
        }
    }
    __syncthreads();
    if (tid < nq) {
        double s = 0.0;
#pragma unroll
        for (int ww = 0; ww < 8; ++ww) s += red[ww * nq + tid];
        p.partial[((long)b * ntiles + blockIdx.x) * nq + tid] = s;
    }
}

__global__ void cov_grad_reduce_kernel(const double* __restrict__ partial, long ntiles, int d,
                                       const double* __restrict__ theta, long theta_stride, double* __restrict__ out,
                                       long out_stride, double scale, int accumulate) {
    const int b = blockIdx.x;
    const int nq = 2 * d + 4;
    const double* th = theta + (long)b * theta_stride;
    __shared__ double sh[8];
    for (int q = 0; q < nq; ++q) {
        double s = 0.0;
        for (long t = threadIdx.x; t < ntiles; t += blockDim.x) s += partial[((long)b * ntiles + t) * nq + q];
        s = warp_sum(s);
        if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
        __syncthreads();
        if (threadIdx.x == 0) {
            double tot = 0.0;
            for (int ww = 0; ww < (int)(blockDim.x >> 5); ++ww) tot += sh[ww];
            double f = 1.0;
            if (q == 0) f = 1.0 / th[0];                            // rho
            else if (q <= d) f = 1.0 / th[q];                       // ls_L[k]: raw sum is in scaled coords -> / ls
            else if (q == d + 1) f = 1.0 / th[d + 1];               // var_L
            else if (q <= 2 * d + 1) f = 1.0 / th[q];               // ls_D[k]
            else if (q == 2 * d + 2) f = 1.0 / th[2 * d + 2];       // var_D
            double v = scale * f * tot;
            double* o = out + (long)b * out_stride + q;
            *o = accumulate ? (*o + v) : v;
        }
        __syncthreads();
    }
}


// ---------------------------------------------------------------------------------------------
// K1 streaming variant (large problems).  Profile of the one-tile-per-CTA kernel above at N = 16 384 (profiles/
// r01_ncu_cov_*): each CTA spends ~1/3 of its life in a serial prologue (theta -> 1/ls -> scale 128 points, three
// barriers, two dependent global round trips) that 2 resident CTAs cannot hide, so neither the FP64 pipe (48 %) nor
// HBM (24-42 %) is busy.  Here the per-point work is done ONCE by cov_prescale_kernel into a k-major workspace
//     P[k][Npad]:  k < d: x/ls_L | k < 2d: x/ls_delta | 2d: -|x/ls_L|^2/2 + log(var_L)/2 | 2d+1: -|x/ls_d|^2/2 + log(var_d)/2
//                  | 2d+2: s in {0,1,rho} | 2d+3: h in {0,1}
// and persistent CTAs walk a contiguous range of tiles, double-buffering the two 64-point panels of the NEXT tile
// with cp.async while the current tile is evaluated and stored.
// ---------------------------------------------------------------------------------------------
__global__ void cov_prescale_kernel(const double* __restrict__ X, int N, int Npad, int d, const double* __restrict__ theta,
                                    long theta_stride, double* __restrict__ P, unsigned char* __restrict__ tflags) {
    const int b = blockIdx.y;
    const double* th = theta + (long)b * theta_stride;
    const int S = 2 * d + 4;
    double* Pb = P + (long)b * S * Npad;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;  // blockDim.x == COV_TILE: one block per tile
    double s = 0.0, h = 0.0;
    bool live = false;
    if (p < N) {
        const double fid = X[(long)p * (d + 1) + d];
        if (fid == 0.0) {
            s = 1.0;
            live = true;
        } else if (fid == 1.0) {
            s = th[0];
            h = 1.0;
            live = true;
        }
    }
    double nL = 0.0, nD = 0.0;
    for (int k = 0; k < d; ++k) {
        const double x = live ? X[(long)p * (d + 1) + k] : 0.0;
        const double xl = x / th[1 + k], xd = x / th[2 + d + k];
        Pb[(long)k * Npad + p] = xl;
        Pb[(long)(d + k) * Npad + p] = xd;
        nL = fma(xl, xl, nL);
        nD = fma(xd, xd, nD);
    }
    Pb[(long)(2 * d) * Npad + p] = fma(-0.5, nL, 0.5 * log(th[1 + d]));
    Pb[(long)(2 * d + 1) * Npad + p] = fma(-0.5, nD, 0.5 * log(th[2 + 2 * d]));
    Pb[(long)(2 * d + 2) * Npad + p] = s;
    Pb[(long)(2 * d + 3) * Npad + p] = h;
    // per-tile flags: bit 0 = some HF point, bit 1 = some row scale != 1 (HF with rho != 1, dead or padding rows)
    const int any_h = __syncthreads_or(h != 0.0), any_s = __syncthreads_or(s != 1.0);
    if (threadIdx.x == 0) tflags[(long)b * gridDim.x + blockIdx.x] = (unsigned char)((any_h ? 1 : 0) | (any_s ? 2 : 0));
}

__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
    const unsigned sa = (unsigned)__cvta_generic_to_shared(dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(src));
}

struct CovStreamArgs {
    const double* Pa;  // [batch][S][Napad]
    const double* Pb;  // [batch][S][Nbpad]
    const unsigned char* fa;  // [batch][TI]
    const unsigned char* fb;  // [batch][TJ]
    int Na, Nb, Napad, Nbpad, d, TI, TJ;
    long ntiles;  // per batch
    long total;   // batch * ntiles
    long per_cta;
    double* K;
    long ldk, strideK;
    int symmetric, mirror, vec_ok;
    double diag_add;
    const double* diag_add_vec;
};

// D: input dimension when it is one of the specialised values (5, 10), else 0 = run-time d.  SYM: lower triangle of K(X, X)
// with optional mirroring (2 CTAs per SM: the mirror staging buffer); otherwise rectangular, 3 CTAs per SM.
template <int D, bool SYM>
__global__ void __launch_bounds__(256, SYM ? 2 : 3) cov_stream_kernel(CovStreamArgs p) {
    extern __shared__ __align__(16) double smem[];
    __shared__ __align__(16) double etab[512];  // static: the table's shared address is an immediate in every lookup
    const int d = D > 0 ? D : p.d, S = 2 * d + 4, T = COV_TILE;
    const int panel = S * T;             // doubles per 64-point panel
    double* stage0 = smem;               // stage s: [a panel | b panel]
    constexpr int MROW = 18;             // staging row stride (16 values + 2 pad: 16-byte aligned rows, fewer bank conflicts)
    double* mstage = stage0 + 4 * panel; // SYM only: [8 warps][32][MROW] transposed blocks of the mirrored tile
    const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
    const int tx = (w & 1) * 8 + (lane & 7);
    const int ty = (w >> 1) * 4 + (lane >> 3);
    const int r0 = ty * 4;
    fexp512_table_fill(etab, tid, blockDim.x);

    const long w0 = (long)blockIdx.x * p.per_cta;
    long w1 = w0 + p.per_cta;
    if (w1 > p.total) w1 = p.total;
    if (w0 >= w1) return;

    // walk the tiles of this CTA in linear order (row-major; lower triangle when symmetric) without re-decoding
    auto advance = [&](int& b, int& I, int& J) {
        ++J;
        if (SYM ? (J > I) : (J == p.TJ)) {
            J = 0;
            if (++I == p.TI) {
                I = 0;
                ++b;
            }
        }
    };
    // cp.async work split: thread -> (panel row k0 + 8m, 16-byte chunk o); constant across tiles
    const int ck0 = tid >> 5, co = (tid & 31) * 2;
    auto issue = [&](int stage, int b, int I, int J) {
        double* sa = stage0 + (size_t)stage * 2 * panel + ck0 * T + co;
        double* sb = sa + panel;
        const double* ga = p.Pa + (long)b * S * p.Napad + (long)I * T + (long)ck0 * p.Napad + co;
        const double* gb = p.Pb + (long)b * S * p.Nbpad + (long)J * T + (long)ck0 * p.Nbpad + co;
        for (int k = ck0; k < S; k += 8) {
            cp_async16(sa, ga);
            cp_async16(sb, gb);
            sa += 8 * T;
            sb += 8 * T;
            ga += 8 * (long)p.Napad;
            gb += 8 * (long)p.Nbpad;
        }
        asm volatile("cp.async.commit_group;\n" ::);
    };

    int b, I, J;
    {
        b = (int)(w0 / p.ntiles);
        tile_index(w0 - (long)b * p.ntiles, p.TJ, SYM, I, J);
    }
    issue(0, b, I, J);
    int nfla = p.fa[(long)b * p.TI + I], nflb = p.fb[(long)b * p.TJ + J];
    int stage = 0;
    for (long wi = w0; wi < w1; ++wi) {
        asm volatile("cp.async.wait_group 0;\n" ::);
        __syncthreads();  // current stage landed for everyone; the other stage is no longer being read
        const int fla = nfla, flb = nflb;
        int nb = b, nI = I, nJ = J;
        if (wi + 1 < w1) {
            advance(nb, nI, nJ);
            issue(stage ^ 1, nb, nI, nJ);
            nfla = p.fa[(long)nb * p.TI + nI];  // consumed one tile later: the load latency is off the critical path
            nflb = p.fb[(long)nb * p.TJ + nJ];
        }
        const double* A = stage0 + (size_t)stage * 2 * panel;
        const double* B = A + panel;

        double acc[4][4], val[4][4];
        {
            const double* hA = A + 2 * d * T;
            const double* hB = B + 2 * d * T;
            const double2 ha01 = *reinterpret_cast<const double2*>(hA + r0), ha23 = *reinterpret_cast<const double2*>(hA + r0 + 2);
            const double2 hb01 = *reinterpret_cast<const double2*>(hB + 2 * tx), hb23 = *reinterpret_cast<const double2*>(hB + 32 + 2 * tx);
            const double ha[4] = {ha01.x, ha01.y, ha23.x, ha23.y}, hb[4] = {hb01.x, hb01.y, hb23.x, hb23.y};
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[a][c] = ha[a] + hb[c];  // commutative: K(X, X) stays exactly symmetric
            tile_dots_acc<D>(A, B, d, r0, tx, acc);
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int c = 0; c < 4; ++c) val[a][c] = fexp512(acc[a][c], etab);
        }
        if ((fla | flb) & 2) {  // some row scale differs from 1: (s_a s_b) is commutative -> K(X,X) exactly symmetric
            const double* sA = A + (2 * d + 2) * T;
            const double* sB = B + (2 * d + 2) * T;
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int c = 0; c < 4; ++c) val[a][c] *= sA[r0 + a] * sB[col_of(tx, c)];
        }
        if ((fla & 1) && (flb & 1)) {  // tile touches the HF x HF block: add the discrepancy GP
            const double* hA = A + (2 * d + 1) * T;
            const double* hB = B + (2 * d + 1) * T;
            const double* gA = A + (2 * d + 3) * T;
            const double* gB = B + (2 * d + 3) * T;
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[a][c] = hA[r0 + a] + hB[col_of(tx, c)];
            tile_dots_acc<D>(A + d * T, B + d * T, d, r0, tx, acc);
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    if (gA[r0 + a] * gB[col_of(tx, c)] != 0.0) val[a][c] += fexp512(acc[a][c], etab);
        }
        const int i0 = I * T, j0 = J * T;
        if (SYM && I == J) {
            const double dg = p.diag_add_vec ? p.diag_add_vec[b] : p.diag_add;
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    if (r0 + a == col_of(tx, c)) val[a][c] += dg;
        }
        double* __restrict__ K = p.K + (long)b * p.strideK;
        if (p.vec_ok && i0 + T <= p.Na && j0 + T <= p.Nb) {  // interior tile: unguarded 128-bit stores
            double* dst = K + (long)(i0 + r0) * p.ldk + j0 + 2 * tx;
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                *reinterpret_cast<double2*>(dst) = make_double2(val[a][0], val[a][1]);
                *reinterpret_cast<double2*>(dst + 32) = make_double2(val[a][2], val[a][3]);
                dst += p.ldk;
            }
            if (SYM && p.mirror && I != J) {
                // Mirrored tile: a direct STG of the transposed 4x4 blocks touches 8 half-filled lines per instruction and
                // backs up the LSU.  Instead each warp transposes its 16 x 32 block through a private staging buffer and
                // every lane hands ONE full 128-byte row to the bulk-copy engine (cp.async.bulk, asynchronous, no registers).
                double* M = mstage + w * (32 * MROW);
                asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");  // previous tile's rows have left the buffer
                __syncwarp();
                const int lx = lane & 7, ly = lane >> 3;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    double* q = M + ((c >> 1) * 16 + 2 * lx + (c & 1)) * MROW + 4 * ly;
                    *reinterpret_cast<double2*>(q) = make_double2(val[0][c], val[1][c]);
                    *reinterpret_cast<double2*>(q + 2) = make_double2(val[2][c], val[3][c]);
                }
                asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
                __syncwarp();
                {
                    const int col = (lane >> 4) * 32 + (w & 1) * 16 + (lane & 15);
                    double* dst = K + (long)(j0 + col) * p.ldk + i0 + 16 * (w >> 1);
                    const unsigned src = (unsigned)__cvta_generic_to_shared(M + lane * MROW);
                    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], 128;\n" ::"l"(dst), "r"(src) : "memory");
                    asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
                }
            }
        } else {
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                const int i = i0 + r0 + a;
                if (i >= p.Na) continue;
#pragma unroll
                for (int hblk = 0; hblk < 2; ++hblk) {
                    const int j = j0 + hblk * 32 + 2 * tx;
                    double* dst = K + (long)i * p.ldk + j;
                    if (p.vec_ok && j + 1 < p.Nb) {
                        *reinterpret_cast<double2*>(dst) = make_double2(val[a][2 * hblk], val[a][2 * hblk + 1]);
                    } else {
                        if (j < p.Nb) dst[0] = val[a][2 * hblk];
                        if (j + 1 < p.Nb) dst[1] = val[a][2 * hblk + 1];
                    }
                }
            }
            if (SYM && p.mirror && I != J) {
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const int j = j0 + col_of(tx, c);
                    if (j >= p.Nb) continue;
                    const int i = i0 + r0;
                    double* dst = K + (long)j * p.ldk + i;
                    if (p.vec_ok && i + 3 < p.Na) {
                        *reinterpret_cast<double2*>(dst) = make_double2(val[0][c], val[1][c]);
                        *reinterpret_cast<double2*>(dst + 2) = make_double2(val[2][c], val[3][c]);
                    } else {
#pragma unroll
                        for (int a = 0; a < 4; ++a)
                            if (i + a < p.Na) dst[a] = val[a][c];
                    }
                }
            }
        }
        b = nb;
        I = nI;
        J = nJ;
        stage ^= 1;
    }
    if (SYM) asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory");  // shared memory must outlive the bulk copies that read it
}

// ---------------------------------------------------------------------------------------------
// Rectangular streaming variant on the FP64 tensor path.  The profile of the DFMA version (profiles/r02_ncu_cov_rect.md)
// shows a kernel bound by instruction issue and the FP64 datapath together (50 warp instructions per 32 outputs, 21 of
// them FP64), not by HBM.  DMMA does not shorten the datapath time (one m8n8k4 = 8 DFMA warp instructions of work) but it
// needs 1/8 of the issue slots and half the shared-memory loads, and the exponent's additive terms ride along as two
// extra k columns:   x_ij = sum_k a_ik b_jk + hA_i * 1 + 1 * hB_j   ->  K' = d + 2  (d = 10: exactly three k4 steps).
// Warp w owns rows 16 (w >> 1) .. +16 and columns 32 (w & 1) .. +32 of the 64 x 64 tile = 2 x 4 m8n8 accumulator tiles;
// lane (g, t) ends up with rows 8 mi + g, columns 8 ni + 2t, 2t + 1: every STG.128 writes 8 rows x 64 contiguous bytes.
// Panel rows are padded to 68 doubles in shared memory so that the 8-byte fragment loads (address t * 68 + g) of a
// half-warp fall into 16 different bank pairs.
// ---------------------------------------------------------------------------------------------
constexpr int COV_PS = 68;  // shared-memory pitch of a panel row (doubles)

// acc[mi][ni][2] += sum over the d coordinate rows starting at row `c0` + the two augmented columns built from row `hrow`
template <int D>
__device__ __forceinline__ void tile_dmma(const double* __restrict__ Ar, const double* __restrict__ Bc, int d, int c0, int hrow,
                                          int t, double acc[2][4][2]) {
    // Ar = A panel + first row of this warp + g; Bc = B panel + first column of this warp + g
    auto step = [&](int ks, bool regular) {
        const int k = 4 * ks + t;
        double a[2], b[4];
        if (regular) {
            const double* pa = Ar + (c0 + k) * COV_PS;
            const double* pb = Bc + (c0 + k) * COV_PS;
            a[0] = pa[0]; a[1] = pa[8];
            b[0] = pb[0]; b[1] = pb[8]; b[2] = pb[16]; b[3] = pb[24];
        } else {
            // k < d: coordinate; k == d: (hA_i, 1); k == d + 1: (1, hB_j); beyond: zero padding
            const int row = (k < d ? c0 + k : hrow) * COV_PS;
            const bool la = k <= d, lb = k < d || k == d + 1;
            const double ca = k == d + 1 ? 1.0 : 0.0, cb = k == d ? 1.0 : 0.0;
            a[0] = la ? Ar[row] : ca; a[1] = la ? Ar[row + 8] : ca;
            b[0] = lb ? Bc[row] : cb; b[1] = lb ? Bc[row + 8] : cb; b[2] = lb ? Bc[row + 16] : cb; b[3] = lb ? Bc[row + 24] : cb;
        }
#pragma unroll
        for (int mi = 0; mi < 2; ++mi)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni) dmma(acc[mi][ni][0], acc[mi][ni][1], a[mi], b[ni]);
    };
    if constexpr (D > 0) {
        constexpr int KS = (D + 2 + 3) / 4;
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) step(ks, 4 * ks + 3 < D);
    } else {
        const int KS = (d + 2 + 3) / 4;
        for (int ks = 0; ks < KS; ++ks) step(ks, false);
    }
}

// 3 CTAs per SM at 80 registers; 2 CTAs at 126 registers measured 3 % (N = 32 768) to 8 % (N = 16 384) slower.
template <int D>
__global__ void __launch_bounds__(256, 3) cov_stream_rect_kernel(CovStreamArgs p) {
    extern __shared__ __align__(16) double smem[];
    __shared__ __align__(16) double etab[512];  // static: the table's shared address is an immediate in every lookup
    const int d = D > 0 ? D : p.d, S = 2 * d + 4, T = COV_TILE;
    constexpr int PS = COV_PS;
    const int panel = S * PS;            // doubles per 64-point panel
    double* stage0 = smem;               // stage s: [a panel | b panel]
    const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const int wr = (w >> 1) * 16, wc = (w & 1) * 32;  // first row / column of this warp inside the tile
    fexp512_table_fill(etab, tid, blockDim.x);

    const long w0 = (long)blockIdx.x * p.per_cta;
    long w1 = w0 + p.per_cta;
    if (w1 > p.total) w1 = p.total;
    if (w0 >= w1) return;

    auto advance = [&](int& b, int& I, int& J) {
        if (++J == p.TJ) {
            J = 0;
            if (++I == p.TI) {
                I = 0;
                ++b;
            }
        }
    };
    // cp.async work split: thread -> (panel row k0 + 8m, 16-byte chunk o); constant across tiles
    const int ck0 = tid >> 5, co = (tid & 31) * 2;
    auto issue = [&](int stage, int b, int I, int J) {
        double* sa = stage0 + (size_t)stage * 2 * panel + ck0 * PS + co;
        double* sb = sa + panel;
        const double* ga = p.Pa + (long)b * S * p.Napad + (long)I * T + (long)ck0 * p.Napad + co;
        const double* gb = p.Pb + (long)b * S * p.Nbpad + (long)J * T + (long)ck0 * p.Nbpad + co;
        for (int k = ck0; k < S; k += 8) {
            cp_async16(sa, ga);
            cp_async16(sb, gb);
            sa += 8 * PS;
            sb += 8 * PS;
            ga += 8 * (long)p.Napad;
            gb += 8 * (long)p.Nbpad;
        }
        asm volatile("cp.async.commit_group;\n" ::);
    };

    int b, I, J;
    {
        b = (int)(w0 / p.ntiles);
        tile_index(w0 - (long)b * p.ntiles, p.TJ, 0, I, J);
    }
    issue(0, b, I, J);
    int nfla = p.fa[(long)b * p.TI + I], nflb = p.fb[(long)b * p.TJ + J];
    int stage = 0;
    for (long wi = w0; wi < w1; ++wi) {
        asm volatile("cp.async.wait_group 0;\n" ::);
        __syncthreads();  // current stage landed for everyone; the other stage is no longer being read
        const int fla = nfla, flb = nflb;
        int nb = b, nI = I, nJ = J;
        if (wi + 1 < w1) {
            advance(nb, nI, nJ);
            issue(stage ^ 1, nb, nI, nJ);
            nfla = p.fa[(long)nb * p.TI + nI];  // consumed one tile later: the load latency is off the critical path
            nflb = p.fb[(long)nb * p.TJ + nJ];
        }
        const double* A = stage0 + (size_t)stage * 2 * panel;
        const double* B = A + panel;
        const double* Ar = A + wr + g;
        const double* Bc = B + wc + g;

        double acc[2][4][2], val[2][4][2];
#pragma unroll
        for (int mi = 0; mi < 2; ++mi)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
        tile_dmma<D>(Ar, Bc, d, 0, 2 * d, t, acc);
#pragma unroll
        for (int mi = 0; mi < 2; ++mi)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                for (int e = 0; e < 2; ++e) val[mi][ni][e] = fexp512(acc[mi][ni][e], etab);
        // element (mi, ni, e) of this lane: row wr + 8 mi + g, column wc + 8 ni + 2 t + e
        if ((fla | flb) & 2) {  // some row scale differs from 1
            const double* sA = A + (2 * d + 2) * PS + wr + g;
            const double* sB = B + (2 * d + 2) * PS + wc + 2 * t;
#pragma unroll
            for (int mi = 0; mi < 2; ++mi)
#pragma unroll
                for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                    for (int e = 0; e < 2; ++e) val[mi][ni][e] *= sA[8 * mi] * sB[8 * ni + e];
        }
        if ((fla & 1) && (flb & 1)) {  // tile touches the HF x HF block: add the discrepancy GP
#pragma unroll
            for (int mi = 0; mi < 2; ++mi)
#pragma unroll
                for (int ni = 0; ni < 4; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
            tile_dmma<D>(Ar, Bc, d, d, 2 * d + 1, t, acc);
            const double* gA = A + (2 * d + 3) * PS + wr + g;
            const double* gB = B + (2 * d + 3) * PS + wc + 2 * t;
#pragma unroll
            for (int mi = 0; mi < 2; ++mi)
#pragma unroll
                for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                    for (int e = 0; e < 2; ++e)
                        if (gA[8 * mi] * gB[8 * ni + e] != 0.0) val[mi][ni][e] += fexp512(acc[mi][ni][e], etab);
        }
        const int i0 = I * T + wr + g, j0 = J * T + wc + 2 * t;
        double* __restrict__ K = p.K + (long)b * p.strideK;
        if (p.vec_ok && I * T + T <= p.Na && J * T + T <= p.Nb) {  // interior tile: unguarded 128-bit stores
#pragma unroll
            for (int mi = 0; mi < 2; ++mi) {
                double* dst = K + (long)(i0 + 8 * mi) * p.ldk + j0;
#pragma unroll
                for (int ni = 0; ni < 4; ++ni)
                    *reinterpret_cast<double2*>(dst + 8 * ni) = make_double2(val[mi][ni][0], val[mi][ni][1]);
            }
        } else {
#pragma unroll
            for (int mi = 0; mi < 2; ++mi) {
                const int i = i0 + 8 * mi;
                if (i >= p.Na) continue;
#pragma unroll
                for (int ni = 0; ni < 4; ++ni) {
                    const int j = j0 + 8 * ni;
                    double* dst = K + (long)i * p.ldk + j;
                    if (p.vec_ok && j + 1 < p.Nb) {
                        *reinterpret_cast<double2*>(dst) = make_double2(val[mi][ni][0], val[mi][ni][1]);
                    } else {
                        if (j < p.Nb) dst[0] = val[mi][ni][0];
                        if (j + 1 < p.Nb) dst[1] = val[mi][ni][1];
                    }
                }
            }
        }
        b = nb;
        I = nI;
        J = nJ;
        stage ^= 1;
    }
}

}  // namespace

static bool aligned16(const void* p) { return (reinterpret_cast<size_t>(p) & 15) == 0; }

static int launch_cov_stream(cudaStream_t s, const CovArgs& a, int TI, int TJ, long ntiles, int vec_ok) {
    const int S = 2 * a.d + 4, T = COV_TILE;
    const int Napad = TI * T, Nbpad = TJ * T;
    const bool same = a.symmetric || (a.Xa == a.Xb && a.Na == a.Nb);
    const size_t pa = (size_t)a.batch * S * Napad, pb = same ? 0 : (size_t)a.batch * S * Nbpad;
    const size_t fbytes = (((size_t)a.batch * (TI + (same ? 0 : TJ))) + 15) & ~(size_t)15;
    double* ws = nullptr;
    if (mfgp_ws_malloc(reinterpret_cast<void**>(&ws), (pa + pb) * sizeof(double) + fbytes, s) != cudaSuccess) return -2;
    unsigned char* fl = reinterpret_cast<unsigned char*>(ws + pa + pb);
    cov_prescale_kernel<<<dim3(TI, a.batch), T, 0, s>>>(a.Xa, a.Na, Napad, a.d, a.theta, a.theta_stride, ws, fl);
    if (!same)
        cov_prescale_kernel<<<dim3(TJ, a.batch), T, 0, s>>>(a.Xb, a.Nb, Nbpad, a.d, a.theta, a.theta_stride, ws + pa,
                                                            fl + (size_t)a.batch * TI);
    CovStreamArgs q{};
    q.Pa = ws;
    q.Pb = same ? ws : ws + pa;
    q.fa = fl;
    q.fb = same ? fl : fl + (size_t)a.batch * TI;
    q.Na = a.Na; q.Nb = a.Nb; q.Napad = Napad; q.Nbpad = same ? Napad : Nbpad; q.d = a.d; q.TI = TI; q.TJ = same ? TI : TJ;
    if (!a.symmetric) q.TJ = TJ;
    q.ntiles = ntiles;
    q.total = ntiles * a.batch;
    q.K = a.K; q.ldk = a.ldk; q.strideK = a.strideK;
    q.symmetric = a.symmetric; q.mirror = a.mirror; q.vec_ok = vec_ok;
    q.diag_add = a.diag_add; q.diag_add_vec = a.diag_add_vec;
    const int sms = mfgp_current_dev_info().sms;
    const bool sym = a.symmetric != 0;
    // The tensor-path variant pays off when d + 2 fills whole k4 steps: measured at N = 32 768 (profiles/r02_cov_stream_variants.log)
    // d = 10: 2.49 ms against 2.58 ms for the DFMA kernel; d = 5 (K' = 7 padded to 8): 2.19 against 2.08; run-time d = 7: 2.67 / 2.47.
    const bool dm = !sym && a.d == 10;
    const size_t smem = (size_t)(4 * S * (dm ? COV_PS : T) + (sym ? 8 * 32 * 18 : 0)) * sizeof(double);
    const int slots = sym ? 2 : 3;  // resident CTAs per SM (launch bounds of the two variants)

    // contiguous chunks of tiles per CTA; measured at N = 32 768: 8 chunks per resident CTA slot / <= 64 tiles 3930 GB/s,
    // 32 / <= 16 tiles 4057 GB/s (shorter tail, better balance between the two dies)
    constexpr int cps = 32, per_max = 16;
    long per = (q.total + (long)sms * slots * cps - 1) / ((long)sms * slots * cps);
    if (per < 1) per = 1;
    if (per > per_max) per = per_max;
    q.per_cta = per;
    const long grid = (q.total + per - 1) / per;
    bool ok = true;
    auto go = [&](auto kernel, SmemOptIn& optin) {
        ok = optin.ensure(kernel, smem);
        if (ok) kernel<<<(unsigned)grid, 256, smem, s>>>(q);
    };
    // the reference's data sets have d = 5 (HBS2021) and d = 10 (Goku): those dimensions are compiled in
    static SmemOptIn o5s, o5r, o10s, o10r, o0s, o0r;
    if (a.d == 5) sym ? go(cov_stream_kernel<5, true>, o5s) : go(cov_stream_kernel<5, false>, o5r);
    else if (a.d == 10) sym ? go(cov_stream_kernel<10, true>, o10s) : go(cov_stream_rect_kernel<10>, o10r);
    else sym ? go(cov_stream_kernel<0, true>, o0s) : go(cov_stream_kernel<0, false>, o0r);
    ok = ok && cudaGetLastError() == cudaSuccess;
    mfgp_ws_free(ws, s);
    return ok ? 0 : -2;
}

int launch_cov(cudaStream_t s, const CovArgs& a) {
    if (a.d < 1 || a.d > MFGP_MAX_D) return -1;
    if (a.Na <= 0 || a.Nb <= 0 || a.batch <= 0) return 0;
    const int TI = (a.Na + COV_TILE - 1) / COV_TILE, TJ = (a.Nb + COV_TILE - 1) / COV_TILE;
    const long ntiles = a.symmetric ? (long)TI * (TI + 1) / 2 : (long)TI * TJ;
    const int vec_ok = aligned16(a.K) && (a.ldk % 2 == 0) && (a.strideK % 2 == 0);
    constexpr long stream_min = 1024;
    if (ntiles * (a.route_batch > 0 ? a.route_batch : a.batch) >= stream_min) return launch_cov_stream(s, a, TI, TJ, ntiles, vec_ok);
    const size_t smem = tile_smem_bytes(a.d);
    static SmemOptIn optin;
    if (!optin.ensure(cov_kernel, tile_smem_bytes(MFGP_MAX_D))) return -2;
    dim3 grid((unsigned)ntiles, 1, a.batch);
    cov_kernel<<<grid, 256, smem, s>>>(a, TJ, vec_ok);
    return cudaGetLastError() == cudaSuccess ? 0 : -2;
}

int launch_cov_diag(cudaStream_t s, const double* X, int N, int d, const double* theta, long theta_stride,
                    double* out, long out_stride, int batch) {
    if (N <= 0 || batch <= 0) return 0;
    dim3 grid((N + 255) / 256, batch);
    cov_diag_kernel<<<grid, 256, 0, s>>>(X, N, d, theta, theta_stride, out, out_stride);
    return cudaGetLastError() == cudaSuccess ? 0 : -2;
}

static long grad_ntiles(const CovGradArgs& a) {
    const int TI = (a.Na + COV_TILE - 1) / COV_TILE, TJ = (a.Nb + COV_TILE - 1) / COV_TILE;
    return a.sym_lower ? (long)TI * (TI + 1) / 2 : (long)TI * TJ;
}

long cov_grad_partial_count(const CovGradArgs& a) { return (long)a.batch * grad_ntiles(a) * (2 * a.d + 4); }

int launch_cov_grad(cudaStream_t s, const CovGradArgs& a) {
    if (a.d < 1 || a.d > MFGP_MAX_D) return -1;
    if (a.Na <= 0 || a.Nb <= 0 || a.batch <= 0) return 0;
    const int TJ = (a.Nb + COV_TILE - 1) / COV_TILE;
    const long ntiles = grad_ntiles(a);
    const size_t smem = tile_smem_bytes(a.d) + (size_t)8 * (2 * a.d + 4) * 8;
    static SmemOptIn optin_rg, optin_norg;
    const size_t mx = tile_smem_bytes(MFGP_MAX_D) + 8 * (2 * MFGP_MAX_D + 4) * 8;
    if (!(a.rowgrad ? optin_rg.ensure(cov_grad_kernel<true>, mx) : optin_norg.ensure(cov_grad_kernel<false>, mx))) return -2;
    dim3 grid((unsigned)ntiles, 1, a.batch);
    if (a.rowgrad) cov_grad_kernel<true><<<grid, 256, smem, s>>>(a, TJ, ntiles);
    else cov_grad_kernel<false><<<grid, 256, smem, s>>>(a, TJ, ntiles);
    cov_grad_reduce_kernel<<<a.batch, 256, 0, s>>>(a.partial, ntiles, a.d, a.theta, a.theta_stride, a.out,
                                                   a.out_stride, a.out_scale, a.accumulate);
    return cudaGetLastError() == cudaSuccess ? 0 : -2;
}
