// gpr_small_v4.cu -- K6 v4: batched small-matrix NLML + analytic gradient, one warp per problem,
// PERSISTENT grid, compact instruction stream, 12 problems in flight per SM.
//
// What changed against v2/v3 (deleted; see git history), and why (profiles/r01_ncu_gpr_small_final.csv):
//   * v3's fully unrolled body is ~300 KB of SASS; with 8 warps at 8 different program counters the dominant
//     stall was `no_instruction` (2.0 cycles per issued instruction) and the 234 registers capped the SM at 8 warps.
//     Here the covariance assembly / dK recompute (the exp-heavy part) and the 8x8 diagonal-tile factorisation are
//     single-copy runtime loops; only the DMMA tile products are unrolled (a few KB).  The kernel fits the 32 KB
//     L1.5 instruction cache, needs no __syncthreads re-alignment, and runs at <= 168 registers = 12 warps per SM.
//   * K^-1 = W^T W is formed IN PLACE row block by row block (LAPACK lauum order), so its accumulators are one block
//     row (14 doubles) instead of the whole triangle (56 doubles).
//   * a = W y and alpha = W^T a are DFMA dot products + 4-lane shuffles instead of one-column DMMA products
//     (a one-column DMMA wastes 7/8 of the FP64 pipe time it occupies).
//   * tiles are packed by COLUMN: tile(i, j) = column base(j) + (i - j), so the left-looking update addresses
//     tile(kb + u, k) as pointer + constant.
//   * the discrepancy kernel (HF x HF pairs only) is evaluated pair-wise from the raw inputs; no per-warp copy of
//     delta-scaled coordinates; the row scale s_i and -|x_i|^2/2 + log(var_L)/2 are one interleaved array.
//
// Algorithm (per problem; N <= 64 padded to NT tiles of 8):
//   1  K = fused MF covariance (+ noise; identity on padding rows) -> lower tiles in shared memory
//   2  left-looking tile Cholesky; diagonal slot keeps inv(L_kk); panel = A_ik inv(L_kk)^T (DMMA)
//   3  W = L^-1 row block by row block: W_ij = -W_ii sum_k L_ik W_kj (DMMA)
//   4  a = W y, alpha = W^T a;  nlml = |a|^2/2 + sum log L_ii + N/2 log 2 pi
//   5  K^-1 in place, G = alpha alpha^T - K^-1 (weighted by multiplicity)
//   6  gradient: sum G o dK/dtheta with K^L recomputed tile by tile
// Replaces, per bin, GPR.log_marginal_likelihood + tape.gradient (reference mfgpflow/linear.py:206-207).
#include <cmath>
#include <cstdint>

#include "common.cuh"
#include "gpr_small.cuh"
#include "mathx.cuh"

namespace {

// One CTA per SM; its warp count (= problems in flight per SM) is chosen at launch: as many as shared memory allows,
// at most 12 (168 registers per thread).  One 12-warp CTA measured 8 % faster than 3 x 4 or 2 x 6 warps.
constexpr int MAX_WPC = 12;
// The 8x8 diagonal tiles are factored per lane: a cooperative, shuffle-based factorisation measured 766 k against 790 k evals/s.
// Tiles assembled per loop iteration (2 * n independent exp chains per lane).  Measured: 2 -> 791 k, 4 -> 783 k, 7 -> 760 k
// evals/s: more chains only add register pressure at the 168-register cap.
constexpr int TILES_PER_ITER = 2;
constexpr double LOG2PI = 1.8378770664093454835606594728112;

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// element offset (doubles) inside a 64-double tile: 16-byte chunks of a row XOR-swizzled by (row & 2)
__host__ __device__ __forceinline__ constexpr int tile_off(int r, int c) {
    return r * 8 + ((((c >> 1) ^ (r & 2))) << 1) + (c & 1);
}
template <int NT>
__host__ __device__ __forceinline__ constexpr int cslot(int i, int j) {  // i >= j, packed by column
    return j * NT - j * (j - 1) / 2 + (i - j);
}

template <int NT>
__device__ __forceinline__ int cslot_rt(int i, int j) {
    return j * NT - j * (j - 1) / 2 + (i - j);
}

template <int NT>
struct WarpMem {
    static constexpr int NP = 8 * NT;
    static constexpr int NTRI = NT * (NT + 1) / 2;
    double* tiles;  // [NTRI][64]
    double* xL;     // [d][NP]   inputs / ls_L
    double* hs;     // [NP][2]   { -|xL|^2/2 + log(var_L)/2 , row scale s in {0, 1, rho} }
    double* yv;     // [NP]      y, later alpha
    double* av;     // [NP]      a = W y
    double* inv;    // [2d]      1/ls_L, 1/ls_delta
    double* red;    // [2d+4]
    unsigned char* hidx;  // [NP] indices of the HF rows
    __host__ __device__ static size_t doubles(int d) {
        return (size_t)NTRI * 64 + (size_t)d * NP + 4 * NP + 2 * d + (2 * d + 4) + NP / 8 + 2;
    }
    __device__ WarpMem(double* base, int d) {
        tiles = base;
        xL = tiles + NTRI * 64;
        hs = xL + d * NP;
        yv = hs + 2 * NP;
        av = yv + NP;
        inv = av + NP;
        red = inv + 2 * d;
        hidx = reinterpret_cast<unsigned char*>(red + 2 * d + 4);
    }
};

// K^L C-fragment of tile (i, j): rows 8i+g, columns 8j+2t, 8j+2t+1.  Expanded-square distance folded into the
// exponent; log(var_L) is split over the two row terms.  With DS > 0 the scaled coordinates are returned for reuse.
template <int NT, int DS>
__device__ __forceinline__ void kl_tile(const WarpMem<NT>& m, const double* etab, int d, int i, int j, int g, int t, double& k0,
                                        double& k1, double* xr, double* xc0, double* xc1) {
    constexpr int NP = 8 * NT;
    const int r = 8 * i + g, c = 8 * j + 2 * t;
    double e0 = 0.0, e1 = 0.0;
    if constexpr (DS > 0) {
#pragma unroll
        for (int q = 0; q < DS; ++q) {
            const double a = m.xL[q * NP + r];
            const double2 b = *reinterpret_cast<const double2*>(m.xL + q * NP + c);
            xr[q] = a;
            xc0[q] = b.x;
            xc1[q] = b.y;
            e0 = fma(a, b.x, e0);
            e1 = fma(a, b.y, e1);
        }
    } else {
        for (int q = 0; q < d; ++q) {
            const double a = m.xL[q * NP + r];
            const double2 b = *reinterpret_cast<const double2*>(m.xL + q * NP + c);
            e0 = fma(a, b.x, e0);
            e1 = fma(a, b.y, e1);
        }
    }
    const double2 hr = *reinterpret_cast<const double2*>(m.hs + 2 * r);
    const double2 h0 = *reinterpret_cast<const double2*>(m.hs + 2 * c);
    const double2 h1 = *reinterpret_cast<const double2*>(m.hs + 2 * c + 2);
    k0 = (hr.y * h0.y) * fexp_tab(e0 + (hr.x + h0.x), etab);
    k1 = (hr.y * h1.y) * fexp_tab(e1 + (hr.x + h1.x), etab);
}

template <int NT>
__device__ __forceinline__ void next_tile(int& i, int& j) {  // column-packed order
    if (++i == NT) {
        ++j;
        i = j;
    }
}

template <int NT, int DS>
__global__ void __launch_bounds__(MAX_WPC * 32, 1) gpr_small_v4_kernel(SmallArgs p, int warp_doubles) {
    constexpr int NP = 8 * NT;
    constexpr int NTRI = NT * (NT + 1) / 2;
    extern __shared__ __align__(16) double smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int N = p.N, d = (DS > 0) ? DS : p.d;
    const double* etab = smem;  // 2^(j/64), shared by the CTA
    fexp_table_fill(smem, threadIdx.x, blockDim.x);
    __syncthreads();
    const WarpMem<NT> m(smem + 64 + (size_t)warp * warp_doubles, d);
    const int g = lane >> 2, t = lane & 3;
    const int cst = tile_off(g, 2 * t);                                // C fragment: row g, cols 2t, 2t+1
    const int km0 = tile_off(g, t), km1 = tile_off(g, t + 4);          // K-major fragment: (row g, col t + 4s)
    const int mm0 = tile_off(t, g), mm1 = tile_off(t + 4, g);          // M-major fragment: (row t + 4s, col g)
    const int nq = 2 * d + 4;
    const int wpc = blockDim.x >> 5;
    double* scr = p.scratch + ((size_t)blockIdx.x * wpc + warp) * (NTRI * 64) + 2 * lane;

    for (int prob = blockIdx.x * wpc + warp; prob < p.B; prob += gridDim.x * wpc) {
        // ---- setup --------------------------------------------------------------------------------
        const double* __restrict__ theta = p.theta + (size_t)prob * (2 * d + 3);
        if (lane < 2 * d) m.inv[lane] = 1.0 / theta[lane < d ? 1 + lane : 2 + lane];
        const double rho = theta[0], vL = theta[1 + d], vD = theta[2 + 2 * d];
        const double noise = p.noise[prob];
        const double hlv = 0.5 * log(vL);
        __syncwarp();
        int nH = 0;
        unsigned long long hfmask = 0ull;  // bit r: row r is a high-fidelity point
#pragma unroll
        for (int pass = 0; pass < (NP + 31) / 32; ++pass) {
            const int r = lane + 32 * pass;
            bool live = false, hf = false;
            if (r < N) {
                const double fid = p.X[(size_t)r * (d + 1) + d];
                hf = (fid == 1.0);
                live = hf || (fid == 0.0);
            }
            if (r < NP) {
                double nL = 0.0;
                for (int q = 0; q < d; ++q) {
                    const double x = live ? p.X[(size_t)r * (d + 1) + q] * m.inv[q] : 0.0;
                    m.xL[q * NP + r] = x;
                    nL = fma(x, x, nL);
                }
                *reinterpret_cast<double2*>(m.hs + 2 * r) = make_double2(fma(-0.5, nL, hlv), live ? (hf ? rho : 1.0) : 0.0);
                m.yv[r] = (r < N) ? p.Y[(size_t)r * p.ldy + (prob + p.prob0) % p.ycols] : 0.0;
            }
            const unsigned hm = __ballot_sync(0xffffffffu, hf);
            if (hf) m.hidx[nH + __popc(hm & ((1u << lane) - 1u))] = (unsigned char)r;
            nH += __popc(hm);
            hfmask |= (unsigned long long)hm << (32 * pass);
        }
        __syncwarp();

        // ---- 1: covariance tiles --------------------------------------------------------------------
        {
            constexpr int TPI = TILES_PER_ITER;  // tiles per iteration = 2 * TPI independent exp chains per lane
            int i = 0, j = 0;
#pragma unroll 1
            for (int s = 0; s < NTRI; s += TPI) {
                int ti[TPI], tj[TPI];
                double k0[TPI], k1[TPI];
#pragma unroll
                for (int u = 0; u < TPI; ++u) {
                    const bool live = (s + u < NTRI);
                    ti[u] = live ? i : 0;  // tail of the last iteration: recompute tile 0, discard
                    tj[u] = live ? j : 0;
                    if (live) next_tile<NT>(i, j);
                }
#pragma unroll
                for (int u = 0; u < TPI; ++u) kl_tile<NT, 0>(m, etab, d, ti[u], tj[u], g, t, k0[u], k1[u], nullptr, nullptr, nullptr);
#pragma unroll
                for (int u = 0; u < TPI; ++u) {
                    if (s + u >= NTRI) break;
                    // K^L is needed again by the gradient: park it in the L2-resident scratch (own lane's values)
                    if (p.grad) __stcg(reinterpret_cast<double2*>(scr + (s + u) * 64), make_double2(k0[u], k1[u]));
                    if (ti[u] == tj[u]) {  // diagonal: + noise (real rows) or identity (padding rows keep the factorisation well posed)
                        const double dg = (8 * ti[u] + g < N) ? noise : 1.0;
                        if (g == 2 * t) k0[u] += dg;
                        if (g == 2 * t + 1) k1[u] += dg;
                    }
                    *reinterpret_cast<double2*>(m.tiles + (s + u) * 64 + cst) = make_double2(k0[u], k1[u]);
                }
            }
        }
        __syncwarp();
        // discrepancy GP on HF x HF pairs (lower triangle incl. diagonal), straight from the raw inputs
        const int npairs = nH * (nH + 1) / 2;
        for (int tt = lane; tt < npairs; tt += 32) {
            int pi = (int)((sqrt(8.0 * tt + 1.0) - 1.0) * 0.5);
            while ((pi + 1) * (pi + 2) / 2 <= tt) ++pi;
            while (pi * (pi + 1) / 2 > tt) --pi;
            const int pj = tt - pi * (pi + 1) / 2;
            const int ri = m.hidx[pi], rj = m.hidx[pj];  // ri >= rj
            double ee = 0.0;
            for (int q = 0; q < d; ++q) {
                const double df = (p.X[(size_t)ri * (d + 1) + q] - p.X[(size_t)rj * (d + 1) + q]) * m.inv[d + q];
                ee = fma(df, df, ee);
            }
            const double kd = vD * fexp_tab(-0.5 * ee, etab);
            double* tl = m.tiles + cslot_rt<NT>(ri >> 3, rj >> 3) * 64;
            tl[tile_off(ri & 7, rj & 7)] += kd;
            if ((ri >> 3) == (rj >> 3) && ri != rj) tl[tile_off(rj & 7, ri & 7)] += kd;  // diagonal tiles are kept fully symmetric
        }
        __syncwarp();

        // ---- 2: left-looking tile Cholesky ------------------------------------------------------------
        int bad = 0;
        double lmant = 1.0;  // prod(pivots) = lmant * 2^lexp, renormalised after every diagonal tile
        int lexp = 0;
        {
#pragma unroll 1
            for (int kb = 0; kb < NT; ++kb) {
                const int cnt = NT - kb;
                double acc[NT][2];
#pragma unroll
                for (int u = 0; u < NT; ++u) acc[u][0] = acc[u][1] = 0.0;
                double* pk = m.tiles + kb * 64;  // tile(kb, 0); tile(kb + u, k) = pk + u * 64
#pragma unroll 1
                for (int k = 0; k < kb; ++k) {
                    const double b0 = pk[km0], b1 = pk[km1];
                    dmma(acc[0][0], acc[0][1], b0, b0);
                    dmma(acc[0][0], acc[0][1], b1, b1);
#pragma unroll
                    for (int u = 1; u < NT; ++u) {
                        // cnt is warp-uniform: the break jumps past the tiles below the matrix.  Written as `if (u < cnt)`,
                        // ptxas predicates the block instead, and 72 % of these loads and DMMAs issued for nothing.
                        if (u >= cnt) break;
                        const double a0 = pk[u * 64 + km0], a1 = pk[u * 64 + km1];
                        dmma(acc[u][0], acc[u][1], a0, b0);
                        dmma(acc[u][0], acc[u][1], a1, b1);
                    }
                    pk += (NT - k - 1) * 64;
                }
                // pk == tile(kb, kb).  acc = K - sum
#pragma unroll
                for (int u = 0; u < NT; ++u)
                    if (u < cnt) {
                        const double2 c = *reinterpret_cast<const double2*>(pk + u * 64 + cst);
                        acc[u][0] = c.x - acc[u][0];
                        acc[u][1] = c.y - acc[u][1];
                    }
                __syncwarp();
#pragma unroll
                for (int u = 0; u < NT; ++u)
                    if (u < cnt) *reinterpret_cast<double2*>(pk + u * 64 + cst) = make_double2(acc[u][0], acc[u][1]);
                __syncwarp();
                // K-major fragments of the raw panel tiles (re-using acc as storage), before they are overwritten
#pragma unroll
                for (int u = 1; u < NT; ++u)
                    if (u < cnt) {
                        acc[u][0] = pk[u * 64 + km0];
                        acc[u][1] = pk[u * 64 + km1];
                    }
                // diagonal tile: every lane factors the 8x8 block in registers (no shuffles), lanes 0-7 invert it
                {
                    double a[8][8], rinv[8];
#pragma unroll
                    for (int r = 0; r < 8; ++r)
#pragma unroll
                        for (int c2 = 0; c2 <= r / 2; ++c2) {
                            const double2 v = *reinterpret_cast<const double2*>(pk + r * 8 + ((c2 ^ (r & 2)) << 1));
                            a[r][2 * c2] = v.x;
                            a[r][2 * c2 + 1] = v.y;
                        }
                    double prod = 1.0;
                    int hiv[8], hmin = 0x7fffffff, hmax = 0;  // pivot sign / NaN test on the high words (integer pipe)
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const double piv = a[j][j];
                        hiv[j] = __double2hiint(piv);
                        hmin = min(hmin, hiv[j]);
                        hmax = max(hmax, hiv[j]);
                        prod *= piv;
                        const double ri = frsqrt(piv);
                        rinv[j] = ri;
#pragma unroll
                        for (int i = j + 1; i < 8; ++i) a[i][j] *= ri;
#pragma unroll
                        for (int k = j + 1; k < 8; ++k)
#pragma unroll
                            for (int i = k; i < 8; ++i) a[i][k] = fma(-a[i][j], a[k][j], a[i][k]);
                    }
                    if (hmin <= 0 || hmax >= 0x7ff00000) {  // a pivot <= 0 (or denormal), inf or NaN: report the first one
                        if (!bad) {
#pragma unroll
                            for (int j = 7; j >= 0; --j)
                                if (hiv[j] <= 0 || hiv[j] >= 0x7ff00000) bad = 8 * kb + j + 1;
                        }
                        prod = nan("");
                    }
                    {
                        const int ph = __double2hiint(prod);
                        lexp += ((ph >> 20) & 0x7ff) - 1023;
                        lmant *= __hiloint2double((ph & 0x800fffff) | 0x3ff00000, __double2loint(prod));
                    }
                    const int c = lane & 7;  // column c of inv(L_kk) by forward substitution
                    double w[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        double s = (i == c) ? 1.0 : 0.0;
#pragma unroll
                        for (int k = 0; k < i; ++k) s = fma(-a[i][k], w[k], s);
                        w[i] = s * rinv[i];
                    }
                    __syncwarp();  // every lane has read the raw diagonal tile
                    if (lane < 8) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) pk[tile_off(i, c)] = w[i];
                    }
                }
                __syncwarp();
                // panel: L_ik = A_ik inv(L_kk)^T
                {
                    const double wb0 = pk[km0], wb1 = pk[km1];
#pragma unroll
                    for (int u = 1; u < NT; ++u) {
                        if (u >= cnt) break;
                        double c0 = 0.0, c1 = 0.0;
                        dmma(c0, c1, acc[u][0], wb0);
                        dmma(c0, c1, acc[u][1], wb1);
                        *reinterpret_cast<double2*>(pk + u * 64 + cst) = make_double2(c0, c1);
                    }
                }
                __syncwarp();
            }
        }

        // ---- 3: W = L^-1, row block by row block -------------------------------------------------------
#pragma unroll
        for (int i = 1; i < NT; ++i) {
            double la[NT][2], acc[NT][2];
#pragma unroll
            for (int k = 0; k < i; ++k) {
                la[k][0] = m.tiles[cslot<NT>(i, k) * 64 + km0];
                la[k][1] = m.tiles[cslot<NT>(i, k) * 64 + km1];
            }
#pragma unroll
            for (int j = 0; j < i; ++j) {
                acc[j][0] = acc[j][1] = 0.0;
#pragma unroll
                for (int k = j; k < i; ++k) {
                    dmma(acc[j][0], acc[j][1], la[k][0], m.tiles[cslot<NT>(k, j) * 64 + mm0]);
                    dmma(acc[j][0], acc[j][1], la[k][1], m.tiles[cslot<NT>(k, j) * 64 + mm1]);
                }
            }
#pragma unroll
            for (int j = 0; j < i; ++j)
                *reinterpret_cast<double2*>(m.tiles + cslot<NT>(i, j) * 64 + cst) = make_double2(acc[j][0], acc[j][1]);
            __syncwarp();
            const double w0 = -m.tiles[cslot<NT>(i, i) * 64 + km0], w1 = -m.tiles[cslot<NT>(i, i) * 64 + km1];
#pragma unroll
            for (int j = 0; j < i; ++j) {
                acc[j][0] = acc[j][1] = 0.0;
                dmma(acc[j][0], acc[j][1], w0, m.tiles[cslot<NT>(i, j) * 64 + mm0]);
                dmma(acc[j][0], acc[j][1], w1, m.tiles[cslot<NT>(i, j) * 64 + mm1]);
            }
            __syncwarp();
#pragma unroll
            for (int j = 0; j < i; ++j)
                *reinterpret_cast<double2*>(m.tiles + cslot<NT>(i, j) * 64 + cst) = make_double2(acc[j][0], acc[j][1]);
            __syncwarp();
        }

        // ---- 4: a = W y, alpha = W^T a, value ------------------------------------------------------------
        double quad = 0.0;
        {
            double2 yy[NT];
#pragma unroll
            for (int j = 0; j < NT; ++j) yy[j] = *reinterpret_cast<const double2*>(m.yv + 8 * j + 2 * t);
#pragma unroll
            for (int i = 0; i < NT; ++i) {
                double s = 0.0;
#pragma unroll
                for (int j = 0; j <= i; ++j) {
                    const double2 w = *reinterpret_cast<const double2*>(m.tiles + cslot<NT>(i, j) * 64 + cst);
                    s = fma(w.x, yy[j].x, s);
                    s = fma(w.y, yy[j].y, s);
                }
                s = quad_sum(s);
                if (t == 0) {
                    m.av[8 * i + g] = s;
                    quad = fma(s, s, quad);
                }
            }
            __syncwarp();
#pragma unroll
            for (int j = 0; j < NT; ++j) {
                double s = 0.0;
#pragma unroll
                for (int i = j; i < NT; ++i) {
                    s = fma(m.tiles[cslot<NT>(i, j) * 64 + mm0], m.av[8 * i + t], s);
                    s = fma(m.tiles[cslot<NT>(i, j) * 64 + mm1], m.av[8 * i + t + 4], s);
                }
                s = quad_sum(s);
                if (t == 0) m.yv[8 * j + g] = s;  // alpha overwrites y
            }
            quad = warp_sum(quad);
            if (lane == 0) {
                const double logdet2 = log(lmant) + 0.69314718055994530942 * (double)lexp;  // sum log(pivot) = 2 sum log L_ii
                p.nlml[prob] = 0.5 * quad + 0.5 * logdet2 + 0.5 * N * LOG2PI;
                if (p.info) p.info[prob] = bad;
                if (bad) atomicCAS(p.d_info, 0, bad);
            }
        }
        if (!p.grad) {
            __syncwarp();
            continue;
        }
        __syncwarp();

        // ---- 5: K^-1 = W^T W in place (row blocks ascending), G = w o (alpha alpha^T - K^-1) -----------------
        double s_dg = 0.0;
#pragma unroll
        for (int i = 0; i < NT; ++i) {
            double acc[NT][2];
#pragma unroll
            for (int j = 0; j <= i; ++j) acc[j][0] = acc[j][1] = 0.0;
#pragma unroll
            for (int k = i; k < NT; ++k) {
                const double a0 = m.tiles[cslot<NT>(k, i) * 64 + mm0], a1 = m.tiles[cslot<NT>(k, i) * 64 + mm1];
#pragma unroll
                for (int j = 0; j <= i; ++j) {
                    const double b0 = (j == i) ? a0 : m.tiles[cslot<NT>(k, j) * 64 + mm0];
                    const double b1 = (j == i) ? a1 : m.tiles[cslot<NT>(k, j) * 64 + mm1];
                    dmma(acc[j][0], acc[j][1], a0, b0);
                    dmma(acc[j][0], acc[j][1], a1, b1);
                }
            }
            __syncwarp();  // row block i of W is dead from here on
            const int r = 8 * i + g;
            const double alr = m.yv[r];
#pragma unroll
            for (int j = 0; j <= i; ++j) {
                const int c0 = 8 * j + 2 * t;
                const double2 alc = *reinterpret_cast<const double2*>(m.yv + c0);
                double g0 = fma(alr, alc.x, -acc[j][0]), g1 = fma(alr, alc.y, -acc[j][1]);
                // multiplicity: strictly lower counted twice, diagonal once; upper part of diagonal tiles and padding zero
                double w0 = (c0 < r) ? 2.0 : (c0 == r ? 1.0 : 0.0), w1 = (c0 + 1 < r) ? 2.0 : (c0 + 1 == r ? 1.0 : 0.0);
                if (r >= N) w0 = w1 = 0.0;
                g0 *= w0;
                g1 *= w1;
                if (j == i) {
                    if (c0 == r) s_dg += g0;
                    if (c0 + 1 == r) s_dg += g1;
                }
                *reinterpret_cast<double2*>(m.tiles + cslot<NT>(i, j) * 64 + cst) = make_double2(g0, g1);
            }
        }
        __syncwarp();

        // ---- 6: gradient contraction --------------------------------------------------------------------
        // discrepancy kernel first (needs G at the HF x HF pairs, before T^L overwrites anything)
        for (int q = lane; q < nq; q += 32) m.red[q] = 0.0;
        __syncwarp();
        for (int t0 = 0; t0 < npairs; t0 += 32) {
            const int tt = t0 + lane;
            double td = 0.0;
            int ri = 0, rj = 0;
            if (tt < npairs) {
                int pi = (int)((sqrt(8.0 * tt + 1.0) - 1.0) * 0.5);
                while ((pi + 1) * (pi + 2) / 2 <= tt) ++pi;
                while (pi * (pi + 1) / 2 > tt) --pi;
                const int pj = tt - pi * (pi + 1) / 2;
                ri = m.hidx[pi];
                rj = m.hidx[pj];
                double ee = 0.0;
                for (int q = 0; q < d; ++q) {
                    const double df = (p.X[(size_t)ri * (d + 1) + q] - p.X[(size_t)rj * (d + 1) + q]) * m.inv[d + q];
                    ee = fma(df, df, ee);
                }
                td = m.tiles[cslot_rt<NT>(ri >> 3, rj >> 3) * 64 + tile_off(ri & 7, rj & 7)] * vD * fexp_tab(-0.5 * ee, etab);
            }
            const double sv = warp_sum(td);
            if (lane == 0) m.red[2 + 2 * d] += sv;
            for (int q = 0; q < d; ++q) {
                const double df = (p.X[(size_t)ri * (d + 1) + q] - p.X[(size_t)rj * (d + 1) + q]) * m.inv[d + q];
                const double sq = warp_sum(td * df * df);
                if (lane == 0) m.red[2 + d + q] += sq;
            }
        }
        double s_vL = 0.0, s_rho = 0.0;
        if constexpr (DS > 0) {
            double sL[DS];
#pragma unroll
            for (int q = 0; q < DS; ++q) sL[q] = 0.0;
            int i = 0, j = 0;
            double2 kna = __ldcg(reinterpret_cast<const double2*>(scr));
            double2 knb = __ldcg(reinterpret_cast<const double2*>(scr + (NTRI > 1 ? 64 : 0)));
#pragma unroll 1
            for (int s = 0; s < NTRI; s += 2) {
                const int ia = i, ja = j;
                next_tile<NT>(i, j);
                const bool two = (s + 1 < NTRI);
                const int ib = two ? i : ia, jb = two ? j : ja;
                next_tile<NT>(i, j);
                const double2 ka = kna, kb = knb;
                if (s + 2 < NTRI) kna = __ldcg(reinterpret_cast<const double2*>(scr + (s + 2) * 64));
                if (s + 3 < NTRI) knb = __ldcg(reinterpret_cast<const double2*>(scr + (s + 3) * 64));
                const double2 ga = *reinterpret_cast<const double2*>(m.tiles + s * 64 + cst);
                double2 gb = *reinterpret_cast<const double2*>(m.tiles + (two ? s + 1 : s) * 64 + cst);
                if (!two) gb.x = gb.y = 0.0;
                const double ta0 = ga.x * ka.x, ta1 = ga.y * ka.y, tb0 = gb.x * kb.x, tb1 = gb.y * kb.y;
                s_vL += (ta0 + ta1) + (tb0 + tb1);
                // exponent of rho in s_i s_j = number of HF points in the pair; only tiles that touch an HF row or column
                if ((((hfmask >> (8 * ia)) | (hfmask >> (8 * ja))) & 0xffull) != 0ull) {
                    const double hr = (double)((hfmask >> (8 * ia + g)) & 1ull);
                    const double hc0 = (double)((hfmask >> (8 * ja + 2 * t)) & 1ull), hc1 = (double)((hfmask >> (8 * ja + 2 * t + 1)) & 1ull);
                    s_rho += ta0 * (hr + hc0) + ta1 * (hr + hc1);
                }
                if ((((hfmask >> (8 * ib)) | (hfmask >> (8 * jb))) & 0xffull) != 0ull) {
                    const double hr = (double)((hfmask >> (8 * ib + g)) & 1ull);
                    const double hc0 = (double)((hfmask >> (8 * jb + 2 * t)) & 1ull), hc1 = (double)((hfmask >> (8 * jb + 2 * t + 1)) & 1ull);
                    s_rho += tb0 * (hr + hc0) + tb1 * (hr + hc1);
                }
                const int ra = 8 * ia + g, ca = 8 * ja + 2 * t, rb = 8 * ib + g, cb = 8 * jb + 2 * t;
#pragma unroll
                for (int q = 0; q < DS; ++q) {
                    const double xra = m.xL[q * NP + ra], xrb = m.xL[q * NP + rb];
                    const double2 xa = *reinterpret_cast<const double2*>(m.xL + q * NP + ca);
                    const double2 xb = *reinterpret_cast<const double2*>(m.xL + q * NP + cb);
                    const double da0 = xra - xa.x, da1 = xra - xa.y, db0 = xrb - xb.x, db1 = xrb - xb.y;
                    sL[q] = fma(ta0 * da0, da0, sL[q]);
                    sL[q] = fma(ta1 * da1, da1, sL[q]);
                    sL[q] = fma(tb0 * db0, db0, sL[q]);
                    sL[q] = fma(tb1 * db1, db1, sL[q]);
                }
            }
#pragma unroll
            for (int q = 0; q < DS; ++q) {
                const double v = warp_sum(sL[q]);
                if (lane == 0) m.red[1 + q] = v;
            }
        } else {
            // generic d: T^L = G o K^L overwrites G, then one pass per dimension
            int i = 0, j = 0;
#pragma unroll 1
            for (int s = 0; s < NTRI; ++s) {
                const double2 kk = __ldcg(reinterpret_cast<const double2*>(scr + s * 64));
                const double2 gg = *reinterpret_cast<const double2*>(m.tiles + s * 64 + cst);
                const double t0 = gg.x * kk.x, t1 = gg.y * kk.y;
                const double hr = (double)((hfmask >> (8 * i + g)) & 1ull);
                const double hc0 = (double)((hfmask >> (8 * j + 2 * t)) & 1ull), hc1 = (double)((hfmask >> (8 * j + 2 * t + 1)) & 1ull);
                s_vL += t0 + t1;
                s_rho += t0 * (hr + hc0) + t1 * (hr + hc1);
                *reinterpret_cast<double2*>(m.tiles + s * 64 + cst) = make_double2(t0, t1);
                next_tile<NT>(i, j);
            }
            for (int q = 0; q < d; ++q) {
                double sL = 0.0;
                i = 0;
                j = 0;
#pragma unroll 1
                for (int s = 0; s < NTRI; ++s) {
                    const double2 tt = *reinterpret_cast<const double2*>(m.tiles + s * 64 + cst);
                    const double xr = m.xL[q * NP + 8 * i + g];
                    const double2 xc = *reinterpret_cast<const double2*>(m.xL + q * NP + 8 * j + 2 * t);
                    const double d0 = xr - xc.x, d1 = xr - xc.y;
                    sL = fma(tt.x * d0, d0, sL);
                    sL = fma(tt.y * d1, d1, sL);
                    next_tile<NT>(i, j);
                }
                sL = warp_sum(sL);
                if (lane == 0) m.red[1 + q] = sL;
            }
        }
        {
            const double a0 = warp_sum(s_rho), a1 = warp_sum(s_vL), a2 = warp_sum(s_dg);
            if (lane == 0) {
                m.red[0] = a0;
                m.red[1 + d] = a1;
                m.red[3 + 2 * d] = a2;
            }
        }
        __syncwarp();
        for (int q = lane; q < nq; q += 32) {
            double f = 1.0;
            if (q == 0) f = 1.0 / rho;
            else if (q <= d) f = m.inv[q - 1];
            else if (q == d + 1) f = 1.0 / vL;
            else if (q <= 2 * d + 1) f = m.inv[d + (q - d - 2)];
            else if (q == 2 * d + 2) f = 1.0 / vD;
            p.grad[(size_t)prob * nq + q] = -0.5 * f * m.red[q];  // d(nlml) = -1/2 sum G dK
        }
        __syncwarp();
    }
}

template <int NT, int DS>
int launch_v4(cudaStream_t st, const SmallArgs& a) {
    const int wd = (int)((WarpMem<NT>::doubles(a.d) + 1) & ~(size_t)1);  // every warp's base stays 16-byte aligned
    const mfgp_dev_info di = mfgp_current_dev_info();
    const int smem_cap = di.smem_optin, sms = di.sms;
    if (smem_cap <= 0 || sms <= 0) return -2;
    int wpc = (int)(((size_t)smem_cap - 64 * 8) / ((size_t)wd * 8));
    if (wpc > MAX_WPC) wpc = MAX_WPC;
    if (wpc < 1) return -1;
    const int want_warps = a.B < sms * wpc ? a.B : sms * wpc;  // few problems: spread them over the SMs first
    if ((want_warps + sms - 1) / sms < wpc) wpc = (want_warps + sms - 1) / sms;
    const size_t bytes = (size_t)wd * 8 * wpc + 64 * 8;
    static SmemOptIn optin;
    if (!optin.ensure(gpr_small_v4_kernel<NT, DS>, bytes)) return -2;
    const int want = (a.B + wpc - 1) / wpc;
    const int grid = want < sms ? want : sms;
    SmallArgs b = a;
    b.scratch = nullptr;
    if (a.grad) {  // one K^L slot per resident warp: <= 148 * 12 * 14 KB = 25 MB, stays in the 126 MB L2
        if (mfgp_ws_malloc(reinterpret_cast<void**>(&b.scratch), (size_t)grid * wpc * WarpMem<NT>::NTRI * 64 * sizeof(double), st) != cudaSuccess) return -2;
    }
    gpr_small_v4_kernel<NT, DS><<<grid, wpc * 32, bytes, st>>>(b, wd);
    const bool ok = cudaGetLastError() == cudaSuccess;
    if (b.scratch) mfgp_ws_free(b.scratch, st);
    return ok ? 0 : -2;
}

template <int NT>
int launch_nt(cudaStream_t st, const SmallArgs& a) {
    return a.d == 5 ? launch_v4<NT, 5>(st, a) : launch_v4<NT, 0>(st, a);
}

}  // namespace

int launch_gpr_small_v4(cudaStream_t st, const SmallArgs& a) {
    if (a.N < 1 || a.N > 64 || a.d < 1 || a.d > MFGP_SMALL_MAX_D) return -1;
    if (a.B <= 0) return 0;
    switch ((a.N + 7) / 8) {
        case 1: return launch_nt<1>(st, a);
        case 2: return launch_nt<2>(st, a);
        case 3: return launch_nt<3>(st, a);
        case 4: return launch_nt<4>(st, a);
        case 5: return launch_nt<5>(st, a);
        case 6: return launch_nt<6>(st, a);
        case 7: return launch_nt<7>(st, a);
        default: return launch_nt<8>(st, a);
    }
}
