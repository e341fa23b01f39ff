// gpr_posterior.cu -- fused prediction from a cached exact-GP posterior (include/mfgp.h: mfgp_gpr_posterior_predict) for
// the small problems of the per-bin emulators (N <= 64, d <= 16, P <= 64): one launch serves every problem and test point.
//
// One CTA per (problem, chunk of test points).  The CTA stages the problem's W = L^-1 (lower), a = W Y and the scaled
// training inputs in shared memory once; each warp then takes 8 test points at a time:
//   K_s^T [8 x N]    built directly in the DMMA A-fragment layout: lane (g, t) evaluates k(x_n, xs_g) for n = 4k + t, so
//                    every lane computes N / 4 distinct entries and K_s never needs a shared-memory round trip
//   V^T = K_s^T W^T  mma.sync.m8n8k4.f64 over the lower-triangular tiles of W only (k-steps 0 .. 2i+1 for row tile i)
//   var = k_ss - sum_n V^2   each lane squares its own V entries, then a fixed-order reduction over the 4 lanes of the point
//   mean = V^T a     DMMA for P >= 8 with the k index permuted to the C-fragment columns the lane already holds
//                    (k-step 2i + e <-> n = 8i + 2t + e), so V feeds the next product without a transpose; DFMA below 8
// Every value of a test point is computed by the lanes of its own row from its own inputs: no cross-point reduction and
// no atomics, so a result does not depend on which other points or problems share the call.
#include <cmath>

#include "gpr.cuh"
#include "gpr_small.cuh"
#include "mathx.cuh"

namespace {

constexpr int PW = 4;            // warps per CTA
constexpr int MAX_P = 64;

__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}
__device__ __forceinline__ double quad_sum(double v) {  // sum over the 4 lanes that share g
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    return v;
}

struct FusedArgs {
    GprPosteriorData q;
    const double* Xs;
    int Ns;
    int gpc;  // 8-point groups per CTA
    double* mean;
    double* var;
};

// Shared-memory pitches (doubles).  W rows: WP = NP + 4 (= 4 or 12 mod 16) puts the B-fragment loads W[8i+g][4k+t] of a
// half-warp into 16 different bank pairs; a rows: AP = round_up(P, 8) + 2 (2 mod 8) does the same for a[8i+2t+e][8j+g].
__host__ __device__ constexpr int w_pitch(int NP) { return NP + 4; }
__host__ __device__ inline int a_pitch(int P) { return ((P + 7) & ~7) + 2; }
// per-point record: [x/ls_L (d)] [x/ls_delta (d)] [-|x/ls_L|^2/2 + log(var_L)/2] [same for delta] [s] [h] [k_ss]
// (odd length: the 8 records of a warp start in 8 different bank pairs)
__host__ __device__ inline int rec_len(int d) { return 2 * d + 5; }

size_t fused_smem_bytes(int NT, int d, int P) {
    const int NP = 8 * NT;
    return sizeof(double) * ((size_t)NP * w_pitch(NP) + (size_t)NP * a_pitch(P) + (size_t)(2 * d + 4) * NP +
                             (size_t)PW * 8 * rec_len(d));
}

// Scaled coordinates and flags of one point, as the covariance kernel K1 prepares them (cov_prescale_kernel): dead rows
// (fidelity not exactly 0 or 1) get zero coordinates and s = h = 0, so their covariance with anything is exactly 0.
// hlL / hlD = log(var_L) / 2, log(var_delta) / 2, computed once per CTA.
__device__ __forceinline__ void prescale_point(const double* __restrict__ x, bool exists, int d, const double* __restrict__ th,
                                               double hlL, double hlD, double* __restrict__ out, int stride) {
    double s = 0.0, h = 0.0;
    bool live = false;
    if (exists) {
        const double fid = x[d];
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
        const double v = live ? x[k] : 0.0;
        const double xl = v / th[1 + k], xd = v / th[2 + d + k];
        out[k * stride] = xl;
        out[(d + k) * stride] = xd;
        nL = fma(xl, xl, nL);
        nD = fma(xd, xd, nD);
    }
    out[(2 * d) * stride] = fma(-0.5, nL, hlL);
    out[(2 * d + 1) * stride] = fma(-0.5, nD, hlD);
    out[(2 * d + 2) * stride] = s;
    out[(2 * d + 3) * stride] = h;
}

template <int NT>
__global__ void __launch_bounds__(PW * 32) gpr_posterior_predict_kernel(FusedArgs p) {
    constexpr int NP = 8 * NT, WP = w_pitch(NP);
    extern __shared__ __align__(16) double sm[];
    __shared__ __align__(16) double etab[512];
    const GprPosteriorData& q = p.q;
    const int N = q.N, d = q.d, P = q.P, AP = a_pitch(P), S1 = rec_len(d);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const long b = blockIdx.y;
    const double* __restrict__ th = q.theta + b * (2 * d + 3);
    double* Ws = sm;                                  // [NP][WP]
    double* As = Ws + NP * WP;                        // [NP][AP]
    double* Xt = As + NP * AP;                        // [2d+4][NP]  training points, k-major
    double* Xw = Xt + (2 * d + 4) * NP + warp * 8 * S1;  // [8][S1]  this warp's test points
    fexp512_table_fill(etab, tid, blockDim.x);
    const double hlL = 0.5 * log(th[1 + d]), hlD = 0.5 * log(th[2 + 2 * d]);

    // ---- stage the problem: W (lower triangle; zero above it and in the padding), a, scaled training inputs
    {
        const double* __restrict__ Wg = q.W + b * N * q.ld;
        for (int idx = tid; idx < NP * NP; idx += blockDim.x) {
            const int r = idx / NP, c = idx - r * NP;
            Ws[r * WP + c] = (r < N && c <= r) ? Wg[(long)r * q.ld + c] : 0.0;
        }
        const double* __restrict__ ag = q.a + b * N * q.Pp;
        for (int idx = tid; idx < NP * AP; idx += blockDim.x) {
            const int r = idx / AP, c = idx - r * AP;
            As[idx] = (r < N && c < P) ? ag[(long)r * q.Pp + c] : 0.0;
        }
        for (int n = tid; n < NP; n += blockDim.x) prescale_point(q.X + (long)n * (d + 1), n < N, d, th, hlL, hlD, Xt + n, NP);
    }
    __syncthreads();
    const double rho = th[0], vL = th[1 + d], vD = th[2 + 2 * d];
    const double kss_hf = __dadd_rn(__dmul_rn(vL, __dmul_rn(rho, rho)), vD);  // K_diag at fidelity 1, as cov_diag_kernel

    for (int grp = warp; grp < p.gpc; grp += PW) {
        const long pt0 = ((long)blockIdx.x * p.gpc + grp) * 8;
        if (pt0 >= p.Ns) break;
        // ---- this group's 8 test points (padding points beyond Ns are dead: K_s = 0, never stored)
        if (lane < 8) {
            const long pt = pt0 + lane;
            const bool exists = pt < p.Ns;
            double* rec = Xw + lane * S1;
            prescale_point(p.Xs + (exists ? pt : 0) * (d + 1), exists, d, th, hlL, hlD, rec, 1);
            rec[2 * d + 4] = rec[2 * d + 3] != 0.0 ? kss_hf : (rec[2 * d + 2] != 0.0 ? vL : 0.0);
        }
        __syncwarp();
        const double* xg = Xw + g * S1;
        const double sg = xg[2 * d + 2], hg = xg[2 * d + 3];

        // ---- K_s^T fragment: ks[k] = k(x_n, xs_g), n = 4k + t
        double ks[2 * NT];
        {
            double e[2 * NT];
#pragma unroll
            for (int k = 0; k < 2 * NT; ++k) e[k] = Xt[2 * d * NP + 4 * k + t] + xg[2 * d];
            for (int c = 0; c < d; ++c) {
                const double xc = xg[c];
                const double* xr = Xt + c * NP + t;
#pragma unroll
                for (int k = 0; k < 2 * NT; ++k) e[k] = fma(xr[4 * k], xc, e[k]);
            }
            const double* sr = Xt + (2 * d + 2) * NP + t;
#pragma unroll
            for (int k = 0; k < 2 * NT; ++k) ks[k] = fexp512(e[k], etab) * (sr[4 * k] * sg);
            if (__any_sync(0xffffffffu, hg != 0.0)) {  // some HF test point: discrepancy GP on the HF x HF pairs
#pragma unroll
                for (int k = 0; k < 2 * NT; ++k) e[k] = Xt[(2 * d + 1) * NP + 4 * k + t] + xg[2 * d + 1];
                for (int c = 0; c < d; ++c) {
                    const double xc = xg[d + c];
                    const double* xr = Xt + (d + c) * NP + t;
#pragma unroll
                    for (int k = 0; k < 2 * NT; ++k) e[k] = fma(xr[4 * k], xc, e[k]);
                }
                const double* hr = Xt + (2 * d + 3) * NP + t;
#pragma unroll
                for (int k = 0; k < 2 * NT; ++k)
                    if (hr[4 * k] * hg != 0.0) ks[k] += fexp512(e[k], etab);
            }
        }

        // ---- V^T = K_s^T W^T over the lower-triangular tiles: v[i][e] = V^T[g][8i + 2t + e]
        double v[NT][2];
#pragma unroll
        for (int i = 0; i < NT; ++i) {
            v[i][0] = v[i][1] = 0.0;
            const double* wr = Ws + (8 * i + g) * WP + t;
#pragma unroll
            for (int k = 0; k <= 2 * i + 1; ++k) dmma(v[i][0], v[i][1], ks[k], wr[4 * k]);
        }

        // ---- var = k_ss - sum_n V^2
        double ss = 0.0;
#pragma unroll
        for (int i = 0; i < NT; ++i) ss = fma(v[i][1], v[i][1], fma(v[i][0], v[i][0], ss));
        ss = quad_sum(ss);
        const long ptg = pt0 + g;
        if (t == 0 && ptg < p.Ns) p.var[b * p.Ns + ptg] = xg[2 * d + 4] - ss;

        // ---- mean = V^T a
        double* mrow = p.mean + (b * p.Ns + ptg) * P;
        if (P >= 8) {
            for (int j = 0; j < (P + 7) / 8; ++j) {
                double c0 = 0.0, c1 = 0.0;
                const double* ar = As + (2 * t) * AP + 8 * j + g;
#pragma unroll
                for (int i = 0; i < NT; ++i) {
                    dmma(c0, c1, v[i][0], ar[(8 * i) * AP]);
                    dmma(c0, c1, v[i][1], ar[(8 * i + 1) * AP]);
                }
                const int col = 8 * j + 2 * t;
                if (ptg < p.Ns) {
                    if (col < P) mrow[col] = c0;
                    if (col + 1 < P) mrow[col + 1] = c1;
                }
            }
        } else {
            for (int c = 0; c < P; ++c) {
                const double* ar = As + (2 * t) * AP + c;
                double m = 0.0;
#pragma unroll
                for (int i = 0; i < NT; ++i) m = fma(v[i][1], ar[(8 * i + 1) * AP], fma(v[i][0], ar[(8 * i) * AP], m));
                m = quad_sum(m);
                if (t == 0 && ptg < p.Ns) mrow[c] = m;
            }
        }
        __syncwarp();  // the group's records are read by every lane before lanes 0-7 overwrite them
    }
}

template <int NT>
int launch_fused(cudaStream_t s, const FusedArgs& a, int B, size_t smem) {
    static SmemOptIn optin;
    if (!optin.ensure(gpr_posterior_predict_kernel<NT>, smem)) return -2;
    const long G = (a.Ns + 7) / 8;
    dim3 grid((unsigned)((G + a.gpc - 1) / a.gpc), (unsigned)B);
    gpr_posterior_predict_kernel<NT><<<grid, PW * 32, smem, s>>>(a);
    return cudaGetLastError() == cudaSuccess ? 0 : -2;
}

}  // namespace

bool gpr_posterior_fused_ok(int N, int d, int P) {
    return N >= 1 && N <= MFGP_SMALL_MAX_N && d >= 1 && d <= MFGP_SMALL_MAX_D && P >= 1 && P <= MAX_P;
}

int gpr_posterior_predict_fused(cudaStream_t s, const GprPosteriorData& q, const double* Xs, int Ns, double* mean,
                                double* var) {
    if (!gpr_posterior_fused_ok(q.N, q.d, q.P)) return -1;
    if (Ns <= 0 || q.B <= 0) return 0;
    const int NT = (q.N + 7) / 8;
    const size_t smem = fused_smem_bytes(NT, q.d, q.P);
    // 8-point groups per CTA: enough CTAs for ~8 per SM, and no more than 256 groups so that a CTA's staging of W and a
    // (read once per CTA) stays small against its arithmetic.  The split never changes a result (see the file comment).
    const long G = (Ns + 7) / 8;
    const long target = (long)mfgp_current_dev_info().sms * 8;
    long gpc = (G * q.B + target - 1) / target;
    if (gpc > 256) gpc = 256;
    if (gpc > G) gpc = G;
    if (gpc < 1) gpc = 1;
    constexpr int MAX_GRID_Y = 65535;
    for (int b0 = 0; b0 < q.B; b0 += MAX_GRID_Y) {
        const int nb = q.B - b0 < MAX_GRID_Y ? q.B - b0 : MAX_GRID_Y;
        FusedArgs a{};
        a.q = q;
        a.q.B = nb;
        a.q.theta = q.theta + (long)b0 * (2 * q.d + 3);
        a.q.noise = q.noise + b0;
        a.q.W = q.W + (long)b0 * q.N * q.ld;
        a.q.a = q.a + (long)b0 * q.N * q.Pp;
        a.Xs = Xs; a.Ns = Ns; a.gpc = (int)gpc;
        a.mean = mean + (long)b0 * Ns * q.P;
        a.var = var + (long)b0 * Ns;
        int rc = 0;
        switch (NT) {
            case 1: rc = launch_fused<1>(s, a, nb, smem); break;
            case 2: rc = launch_fused<2>(s, a, nb, smem); break;
            case 3: rc = launch_fused<3>(s, a, nb, smem); break;
            case 4: rc = launch_fused<4>(s, a, nb, smem); break;
            case 5: rc = launch_fused<5>(s, a, nb, smem); break;
            case 6: rc = launch_fused<6>(s, a, nb, smem); break;
            case 7: rc = launch_fused<7>(s, a, nb, smem); break;
            default: rc = launch_fused<8>(s, a, nb, smem); break;
        }
        if (rc) return rc;
    }
    return 0;
}
