// posterior.cu -- fused prediction from the cached posteriors (include/mfgp.h: mfgp_gpr_posterior_predict, _predict_grad,
// mfgp_svgp_posterior_predict) for the small problems of the per-bin emulators (N or M <= 64, d <= 16): one launch serves
// every problem (or latent) and test point.  Also the input-gradient kernel of the exact posterior's blocked route.
//
// The six fused kernels are built from one set of device pieces (the building blocks below) on one decomposition.  One
// CTA per (problem, chunk of test points) stages the problem's factor W = L^-1 (lower triangle) and its scaled training
// inputs in shared memory once; each warp then takes 8 test points at a time:
//   K_s^T [8 x N]    built directly in the DMMA A-fragment layout: lane (g, t) evaluates k(x_n, xs_g) for n = 4k + t, so
//                    every lane computes N / 4 distinct entries and K_s never needs a shared-memory round trip
//   V^T = K_s^T W^T  mma.sync.m8n8k4.f64 over the lower-triangular tiles of W only (k-steps 0 .. 2i+1 for row tile i);
//                    DMMA returns V in the C-fragment order: slot 2i + e of lane (g, t) holds n = 8i + 2t + e
//   var = k_ss - sum_n V^2   each lane squares its own V entries, then a fixed-order reduction over the 4 lanes of the point
//   V^T T            for a table T [N][P] in shared memory (contract_table): DMMA for P >= 8 with the k index permuted to
//                    the C-fragment columns the lane already holds (k-step 2i + e <-> n = 8i + 2t + e), so V feeds the next
//                    product without a transpose; DFMA and a quad sum below 8
//   V^T F            for a second triangular factor F (upper_tri_product): F is staged transposed with its columns in the
//                    C-fragment order (Ft[c][slot] = F[perm_n(slot)][c]), which keeps the B-fragment loads free of bank conflicts, and the
//                    product comes back in the C layout with the same n as V
// Every value of a test point is computed by the lanes of its own row from its own inputs: no cross-point reduction and
// no atomics, so a result does not depend on which other points or problems share the call.
//
// gpr_posterior_predict_kernel (mfgp_gpr_posterior_predict): mean = V^T a.
//
// gpr_posterior_predict_grad_kernel (mfgp_gpr_posterior_predict_grad) adds d mean / dx* and d var / dx*.  K_s is built in
// its two parts kL and kD in predict's A-fragment layout, so V, var and mean are computed the same way predict computes
// them.  Two quad shuffles per tile and part then move kL and kD to the C-fragment order, where beta = W^T V = K^-1 k_s
// (upper_tri_product with F = W) holds the same n: the dvar sum is lane-local.  alpha = W^T a is formed once per CTA in
// shared memory.  Per coordinate j:  gk_n = dk_n/dx*_j = -kL_n (u*_j - u_nj) / ls_Lj - kD_n (w*_j - w_nj) / ls_dj
// (differences, never the expanded form), dvar_j = -2 sum_n beta_n gk_n (lane-local, then the quad), dmean_:j = alpha^T gk
// (contract_table with gk in the place of V).
//
// gpr_posterior_joint_kernel (mfgp_gpr_posterior_predict_cov / _sample, Ns <= 64): predict's K_s, V, var and mean per
// 8-point group (so mean and diag(Sigma) are predict's bits), V^T to shared memory, then Sigma = K_ss - V^T V on the lower
// 8x8 tiles (DMMA over the training index, K_ss from the point records) with var on the diagonal, mirrored.  _sample goes
// on: L L^T = Sigma + jitter I in shared memory, and samples = mean + L z over the CTA's chunk of the S * P columns.
//
// svgp_posterior_predict_kernel (mfgp_svgp_posterior_predict): the inducing points Z in the place of X, one latent per
// blockIdx.y, W = Wm.  U = Lq^T V (upper_tri_product with F = Lq) never leaves the accumulators: sum U^2 is lane-local.
// var = k_ss - sum V^2 + sum U^2, mean = V^T q_mu.
//
// svgp_posterior_joint_kernel (mfgp_svgp_posterior_predict_cov / _sample, Ns <= 64): one CTA per latent; predict's K_s, V
// and U per 8-point group, V^T and U^T to shared memory, then Sigma_l = K_ss - V^T V + U^T U on the lower 8x8 tiles as the
// exact joint kernel forms K_ss - V^T V, mirrored.  The outputs' mix, diagonal and sampling tail run after it (api.cu).
//
// svgp_posterior_predict_grad_kernel (mfgp_svgp_posterior_predict_grad): predict's values, computed as predict computes
// them, plus the input gradients.  d var / dx*_j = -2 beta . gk with beta = Wm^T (V - Lq U): U stays in a fragment row,
// Lq U runs over the tiles m <= n reading predict's Lt staging in the other direction (lower_tri_product), and beta is
// upper_tri_product with F = Wm.  d mean / dx*_j = alpha . gk with alpha = Wm^T q_mu, formed once per CTA.  gk as in the
// exact grad kernel.
#include <cmath>
#include <type_traits>

#include "gpr.cuh"
#include "gpr_small.cuh"
#include "mathx.cuh"
#include "svgp.cuh"

namespace {

constexpr int PW = 4;            // warps per CTA
constexpr int MAX_P = 64;

struct FusedArgs {
    GprPosteriorData q;
    const double* Xs;
    int Ns;
    int gpc;  // 8-point groups per CTA
    double* mean;
    double* var;
    double* dmean;  // grad kernel only: [B][Ns][P][d]
    double* dvar;   //                   [B][Ns][d]
};

struct SvgpFusedArgs {
    SvgpPosteriorData q;
    const double* Xs;
    int Ns;
    int gpc;  // 8-point groups per CTA
    double* mean;
    double* var;
    long ls, ns;  // output of (latent l, point n) at l * ls + n * ns
};
struct SvgpFusedGradArgs : SvgpFusedArgs {
    double* dmean;  // gradients of (latent l, point n) at (l * ls + n * ns) * d + j
    double* dvar;
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
// grad kernel: a second copy of W (transposed), alpha next to a, and the 2d inverse lengthscales
size_t fused_grad_smem_bytes(int NT, int d, int P) {
    const int NP = 8 * NT;
    return fused_smem_bytes(NT, d, P) + sizeof(double) * ((size_t)NP * w_pitch(NP) + (size_t)NP * a_pitch(P) + 2 * d);
}
// SVGP kernel: Wm and Lq^T, q_mu, the inducing points and the test-point records
size_t svgp_fused_smem_bytes(int NT, int d) {
    const int NP = 8 * NT;
    return sizeof(double) * (2 * (size_t)NP * w_pitch(NP) + NP + (size_t)(2 * d + 4) * NP + (size_t)PW * 8 * rec_len(d));
}
// SVGP grad kernel: a third factor copy (Wm transposed), alpha next to q_mu, and the 2d inverse lengthscales
size_t svgp_fused_grad_smem_bytes(int NT, int d) {
    const int NP = 8 * NT;
    return svgp_fused_smem_bytes(NT, d) + sizeof(double) * ((size_t)NP * w_pitch(NP) + NP + 2 * d);
}

// C-fragment order of the training index: slot 4k + t (k-step k, lane t) holds
// n = 8(k/2) + 2t + (k&1), and back.
__host__ __device__ constexpr int perm_n(int slot) { return 8 * (slot >> 3) + 2 * (slot & 3) + ((slot >> 2) & 1); }
__host__ __device__ constexpr int perm_slot(int n) { return 8 * (n >> 3) + 4 * (n & 1) + ((n >> 1) & 3); }
__host__ __device__ constexpr int slot_off(int k) { return 8 * (k >> 1) + (k & 1); }  // n - 2t of slot k

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

// ---- staging of the fused kernels: one problem's (or latent's) hyperparameters, points and factors in shared memory.

// What the point records of one problem need from its theta th: log(var_L) / 2 and log(var_delta) / 2 (prescale_point),
// and k_ss at fidelity 0 (var_L) and 1 (K_diag at fidelity 1, as cov_diag_kernel).
struct RecordParams {
    const double* th;
    double hlL, hlD, vL, kss_hf;
};
__device__ __forceinline__ RecordParams record_params(const double* th, int d) {
    const double rho = th[0], vL = th[1 + d], vD = th[2 + 2 * d];
    return {th, 0.5 * log(vL), 0.5 * log(vD), vL, __dadd_rn(__dmul_rn(vL, __dmul_rn(rho, rho)), vD)};
}

// Record of test point pt of Xs [Ns][d+1] (rec_len(d) doubles): prescale_point, then k_ss.  pt >= Ns gives a dead
// record: K_s = 0, and the kernels never store its results.
__device__ __forceinline__ void point_record(double* rec, const double* Xs, long pt, long Ns, int d,
                                             const RecordParams& rp) {
    const bool exists = pt < Ns;
    prescale_point(Xs + (exists ? pt : 0) * (d + 1), exists, d, rp.th, rp.hlL, rp.hlD, rec, 1);
    rec[2 * d + 4] = rec[2 * d + 3] != 0.0 ? rp.kss_hf : (rec[2 * d + 2] != 0.0 ? rp.vL : 0.0);
}

// The N training (or inducing) points X [N][d+1] scaled into Xt [2d+4][NP], k-major; the NP - N padding columns are dead.
__device__ __forceinline__ void stage_points(double* Xt, const double* X, int N, int NP, int d, const RecordParams& rp,
                                             int tid) {
    for (int n = tid; n < NP; n += blockDim.x)
        prescale_point(X + (long)n * (d + 1), n < N, d, rp.th, rp.hlL, rp.hlD, Xt + n, NP);
}

// Entry (r, c) of the two staged layouts [NP][WP] of an n x n lower-triangular factor F (leading dimension ld), zero
// outside the triangle and in the padding.  lower_entry: F itself (lower_tri_v).  transposed_entry: F^T with its columns
// in the C-fragment order, Ft[c][slot] = F[perm_n(slot)][c] (upper_tri_product, lower_tri_product).  The kernels stage
// all their copies in one pass over (r, c).
__device__ __forceinline__ double lower_entry(const double* F, long ld, int n, int r, int c) {
    return (r < n && c <= r) ? F[(long)r * ld + c] : 0.0;
}
__device__ __forceinline__ double transposed_entry(const double* F, long ld, int n, int r, int c) {
    const int m = perm_n(c);
    return (m < n && r <= m) ? F[(long)m * ld + r] : 0.0;
}

// Table T [n][P] (leading dimension ld) into Ts [NP][AP] (contract_table's layout), zero in the padding.
__device__ __forceinline__ void stage_table(double* Ts, const double* T, long ld, int n, int P, int AP, int NP, int tid) {
    for (int idx = tid; idx < NP * AP; idx += blockDim.x) {
        const int r = idx / AP, c = idx - r * AP;
        Ts[idx] = (r < n && c < P) ? T[(long)r * ld + c] : 0.0;
    }
}

// Il [2d] = -1/ls_L, -1/ls_delta: the factors of gk_fragment.
__device__ __forceinline__ void stage_inv_ls(double* Il, const double* th, int d, int tid) {
    for (int k = tid; k < d; k += blockDim.x) {
        Il[k] = -1.0 / th[1 + k];
        Il[d + k] = -1.0 / th[2 + d + k];
    }
}

// ---- building blocks of the fused kernels.  A fragment row `double f[2 * NT]` holds one value per training index of
//      the lane's point, in the C-fragment order of the file comment (slot 2i + e <-> n = 8i + 2t + e) unless noted.

// K_s^T fragment in the A-fragment order: ks[k] = k(x_n, xs_g), n = 4k + t, from the training points Xt [2d+4][NP]
// (k-major) and the point record xg (point_record, K1's expanded-square form).
template <int NT>
__device__ __forceinline__ void ks_fragment(double (&ks)[2 * NT], const double* Xt, const double* xg, int d, int t,
                                            const double* etab) {
    constexpr int NP = 8 * NT;
    const double sg = xg[2 * d + 2], hg = xg[2 * d + 3];
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

// A fragment row from the A-fragment order (n = 4k + t) to the C-fragment order, within the quad: slot 2i + e of lane t
// takes n = 8i + 2t + e, which lane (2t + e) & 3 holds in slot 2i + t / 2.
template <int NT>
__device__ __forceinline__ void to_c_order(double (&f)[2 * NT], int lane, int t) {
    const int src0 = (lane & ~3) | ((2 * t) & 3), src1 = (lane & ~3) | ((2 * t + 1) & 3);
    const bool hi = t >= 2;
#pragma unroll
    for (int i = 0; i < NT; ++i) {
        const double a0 = __shfl_sync(0xffffffffu, f[2 * i], src0), b0 = __shfl_sync(0xffffffffu, f[2 * i + 1], src0);
        const double a1 = __shfl_sync(0xffffffffu, f[2 * i], src1), b1 = __shfl_sync(0xffffffffu, f[2 * i + 1], src1);
        f[2 * i] = hi ? b0 : a0;
        f[2 * i + 1] = hi ? b1 : a1;
    }
}

// gk = dk_s/dx*_j in the C-fragment order, from kL and kD in that order (to_c_order) and Il (stage_inv_ls):
// gk_n = -kL_n (u*_j - u_nj) / ls_Lj - kD_n (w*_j - w_nj) / ls_dj, differences formed directly.
template <int NT>
__device__ __forceinline__ void gk_fragment(double (&gk)[2 * NT], const double (&kL)[2 * NT], const double (&kD)[2 * NT],
                                            const double* Xt, const double* xg, const double* Il, int d, int j, int t,
                                            bool anyh) {
    constexpr int NP = 8 * NT;
    const double uj = xg[j], cL = Il[j];
    const double* ur = Xt + j * NP + 2 * t;
#pragma unroll
    for (int k = 0; k < 2 * NT; ++k) gk[k] = kL[k] * (uj - ur[slot_off(k)]) * cL;
    if (anyh) {
        const double wj = xg[d + j], cD = Il[d + j];
        const double* wr = Xt + (d + j) * NP + 2 * t;
#pragma unroll
        for (int k = 0; k < 2 * NT; ++k) gk[k] = fma(kD[k] * (wj - wr[slot_off(k)]), cD, gk[k]);
    }
}

// V^T = K_s^T W^T over the lower-triangular tiles of Ws [NP][WP] (zero above the diagonal): ks in the A-fragment order, v in the C order.
template <int NT>
__device__ __forceinline__ void lower_tri_v(double (&v)[2 * NT], const double (&ks)[2 * NT], const double* Ws, int g, int t) {
    constexpr int WP = w_pitch(8 * NT);
#pragma unroll
    for (int i = 0; i < NT; ++i) {
        v[2 * i] = v[2 * i + 1] = 0.0;
        const double* wr = Ws + (8 * i + g) * WP + t;
#pragma unroll
        for (int k = 0; k <= 2 * i + 1; ++k) dmma(v[2 * i], v[2 * i + 1], ks[k], wr[4 * k]);
    }
}

// The lane's part of sum_n V^2 (quad_sum completes it).
template <int NT>
__device__ __forceinline__ double sum_sq(const double (&v)[2 * NT]) {
    double ss = 0.0;
#pragma unroll
    for (int i = 0; i < NT; ++i) ss = fma(v[2 * i + 1], v[2 * i + 1], fma(v[2 * i], v[2 * i], ss));
    return ss;
}

// (c0, c1) = slots 2i, 2i + 1 of V^T F over the tiles i2 >= i, from Ft [NP][WP] staged as in the file comment.
template <int NT>
__device__ __forceinline__ void upper_tri_product(double& c0, double& c1, const double (&v)[2 * NT], const double* Ft, int i,
                                                  int g, int t) {
    constexpr int WP = w_pitch(8 * NT);
    c0 = c1 = 0.0;
    const double* fr = Ft + (8 * i + g) * WP + t;
#pragma unroll
    for (int i2 = i; i2 < NT; ++i2) {
        dmma(c0, c1, v[2 * i2], fr[8 * i2]);
        dmma(c0, c1, v[2 * i2 + 1], fr[8 * i2 + 4]);
    }
}

// (c0, c1) = slots 2i, 2i + 1 of F u = u^T F^T over the tiles i2 <= i, from the same Ft staging as upper_tri_product read
// in the other direction: F[n][m] = Ft[m][perm_slot(n)], so one staged copy serves F^T u and F u.
template <int NT>
__device__ __forceinline__ void lower_tri_product(double& c0, double& c1, const double (&u)[2 * NT], const double* Ft, int i,
                                                  int g, int t) {
    constexpr int WP = w_pitch(8 * NT);
    c0 = c1 = 0.0;
    const double* fr = Ft + (2 * t) * WP + perm_slot(8 * i + g);
#pragma unroll
    for (int i2 = 0; i2 <= i; ++i2) {
        dmma(c0, c1, u[2 * i2], fr[(8 * i2) * WP]);
        dmma(c0, c1, u[2 * i2 + 1], fr[(8 * i2 + 1) * WP]);
    }
}

// Column c of f^T T for c < P, T = table [NP][AP]: DMMA over blocks of 8 columns for P >= 8, DFMA and a quad sum below.
// store(c, value) is called, for a live point only, by the lanes that hold column c of the point.
template <int NT, class Store>
__device__ __forceinline__ void contract_table(const double (&f)[2 * NT], const double* table, int AP, int P, int g, int t,
                                               bool live, Store store) {
    if (P >= 8) {
        for (int j = 0; j < (P + 7) / 8; ++j) {
            double c0 = 0.0, c1 = 0.0;
            const double* ar = table + (2 * t) * AP + 8 * j + g;
#pragma unroll
            for (int i = 0; i < NT; ++i) {
                dmma(c0, c1, f[2 * i], ar[(8 * i) * AP]);
                dmma(c0, c1, f[2 * i + 1], ar[(8 * i + 1) * AP]);
            }
            const int col = 8 * j + 2 * t;
            if (live) {
                if (col < P) store(col, c0);
                if (col + 1 < P) store(col + 1, c1);
            }
        }
    } else {
        for (int c = 0; c < P; ++c) {
            const double* ar = table + (2 * t) * AP + c;
            double m = 0.0;
#pragma unroll
            for (int i = 0; i < NT; ++i) m = fma(f[2 * i + 1], ar[(8 * i + 1) * AP], fma(f[2 * i], ar[(8 * i) * AP], m));
            m = quad_sum(m);
            if (t == 0 && live) store(c, m);
        }
    }
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
    const RecordParams rp = record_params(th, d);

    // ---- stage the problem: W (lower triangle; zero above it and in the padding), a, scaled training inputs
    {
        const double* __restrict__ Wg = q.W + b * N * q.ld;
        for (int idx = tid; idx < NP * NP; idx += blockDim.x) {
            const int r = idx / NP, c = idx - r * NP;
            Ws[r * WP + c] = lower_entry(Wg, q.ld, N, r, c);
        }
        stage_table(As, q.a + b * N * q.Pp, q.Pp, N, P, AP, NP, tid);
        stage_points(Xt, q.X, N, NP, d, rp, tid);
    }
    __syncthreads();

    for (int grp = warp; grp < p.gpc; grp += PW) {
        const long pt0 = ((long)blockIdx.x * p.gpc + grp) * 8;
        if (pt0 >= p.Ns) break;
        // ---- this group's 8 test points (padding points beyond Ns are dead: K_s = 0, never stored)
        if (lane < 8) point_record(Xw + lane * S1, p.Xs, pt0 + lane, p.Ns, d, rp);
        __syncwarp();
        const double* xg = Xw + g * S1;

        // ---- K_s^T fragment: ks[k] = k(x_n, xs_g), n = 4k + t
        double ks[2 * NT];
        ks_fragment<NT>(ks, Xt, xg, d, t, etab);

        // ---- V^T = K_s^T W^T over the lower-triangular tiles: v[2i + e] = V^T[g][8i + 2t + e]
        double v[2 * NT];
        lower_tri_v<NT>(v, ks, Ws, g, t);

        // ---- var = k_ss - sum_n V^2
        double ss = sum_sq<NT>(v);
        ss = quad_sum(ss);
        const long ptg = pt0 + g;
        if (t == 0 && ptg < p.Ns) p.var[b * p.Ns + ptg] = xg[2 * d + 4] - ss;

        const bool live = ptg < p.Ns;
        double* mrow = p.mean + (b * p.Ns + ptg) * P;
        contract_table<NT>(v, As, AP, P, g, t, live, [&](int c, double m) { mrow[c] = m; });
        __syncwarp();  // the group's records are read by every lane before lanes 0-7 overwrite them
    }
}

template <int NT>
__global__ void __launch_bounds__(PW * 32) gpr_posterior_predict_grad_kernel(FusedArgs p) {
    constexpr int NP = 8 * NT, WP = w_pitch(NP);
    extern __shared__ __align__(16) double sm[];
    __shared__ __align__(16) double etab[512];
    const GprPosteriorData& q = p.q;
    const int N = q.N, d = q.d, P = q.P, AP = a_pitch(P), S1 = rec_len(d);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const long b = blockIdx.y;
    const double* __restrict__ th = q.theta + b * (2 * d + 3);
    double* Ws = sm;                            // [NP][WP]  W, as gpr_posterior_predict_kernel stages it
    double* Wt = Ws + NP * WP;                  // [NP][WP]  Wt[c][slot] = W[perm_n(slot)][c]
    double* As = Wt + NP * WP;                  // [NP][AP]  a
    double* Al = As + NP * AP;                  // [NP][AP]  alpha = W^T a
    double* Xt = Al + NP * AP;                  // [2d+4][NP]  training points, k-major
    double* Il = Xt + (2 * d + 4) * NP;         // [2d]  -1/ls_L, -1/ls_delta
    double* Xw = Il + 2 * d + warp * 8 * S1;    // [8][S1]  this warp's test points
    fexp512_table_fill(etab, tid, blockDim.x);
    const RecordParams rp = record_params(th, d);

    // ---- stage the problem: W twice (lower triangle, zero elsewhere), a, scaled training inputs; then alpha = W^T a
    {
        const double* __restrict__ Wg = q.W + b * N * q.ld;
        for (int idx = tid; idx < NP * NP; idx += blockDim.x) {
            const int r = idx / NP, c = idx - r * NP;
            Ws[r * WP + c] = lower_entry(Wg, q.ld, N, r, c);
            Wt[r * WP + c] = transposed_entry(Wg, q.ld, N, r, c);
        }
        stage_table(As, q.a + b * N * q.Pp, q.Pp, N, P, AP, NP, tid);
        stage_points(Xt, q.X, N, NP, d, rp, tid);
        stage_inv_ls(Il, th, d, tid);
    }
    __syncthreads();
    for (int idx = tid; idx < NP * AP; idx += blockDim.x) {
        const int r = idx / AP, c = idx - r * AP;
        double s = 0.0;
        if (r < N && c < P)
            for (int m = r; m < N; ++m) s = fma(Wt[r * WP + perm_slot(m)], As[m * AP + c], s);
        Al[idx] = s;
    }
    __syncthreads();

    for (int grp = warp; grp < p.gpc; grp += PW) {
        const long pt0 = ((long)blockIdx.x * p.gpc + grp) * 8;
        if (pt0 >= p.Ns) break;
        if (lane < 8) point_record(Xw + lane * S1, p.Xs, pt0 + lane, p.Ns, d, rp);
        __syncwarp();
        const double* xg = Xw + g * S1;
        const double sg = xg[2 * d + 2], hg = xg[2 * d + 3];
        const bool anyh = __any_sync(0xffffffffu, hg != 0.0);

        // ---- the two parts of K_s^T in predict's A-fragment layout: kL[k], kD[k] at n = 4k + t
        double kL[2 * NT], kD[2 * NT];
        {
            const double* xe = Xt + 2 * d * NP + t;
#pragma unroll
            for (int k = 0; k < 2 * NT; ++k) kL[k] = xe[4 * k] + xg[2 * d];
            for (int c = 0; c < d; ++c) {
                const double xc = xg[c];
                const double* xr = Xt + c * NP + t;
#pragma unroll
                for (int k = 0; k < 2 * NT; ++k) kL[k] = fma(xr[4 * k], xc, kL[k]);
            }
            const double* sr = Xt + (2 * d + 2) * NP + t;
#pragma unroll
            for (int k = 0; k < 2 * NT; ++k) kL[k] = fexp512(kL[k], etab) * (sr[4 * k] * sg);
#pragma unroll
            for (int k = 0; k < 2 * NT; ++k) kD[k] = 0.0;
            if (anyh) {
                const double* xf = Xt + (2 * d + 1) * NP + t;
#pragma unroll
                for (int k = 0; k < 2 * NT; ++k) kD[k] = xf[4 * k] + xg[2 * d + 1];
                for (int c = 0; c < d; ++c) {
                    const double xc = xg[d + c];
                    const double* xr = Xt + (d + c) * NP + t;
#pragma unroll
                    for (int k = 0; k < 2 * NT; ++k) kD[k] = fma(xr[4 * k], xc, kD[k]);
                }
                const double* hr = Xt + (2 * d + 3) * NP + t;
#pragma unroll
                for (int k = 0; k < 2 * NT; ++k) kD[k] = hr[4 * k] * hg != 0.0 ? fexp512(kD[k], etab) : 0.0;
            }
        }

        // ---- V^T = K_s^T W^T over the lower-triangular tiles: v[2i + e] = V^T[g][8i + 2t + e]
        double v[2 * NT];
        {
            double ks[2 * NT];
#pragma unroll
            for (int k = 0; k < 2 * NT; ++k) ks[k] = __dadd_rn(kL[k], kD[k]);  // predict's K_s, not contracted
            lower_tri_v<NT>(v, ks, Ws, g, t);
        }

        // ---- var = k_ss - sum_n V^2, mean = V^T a  (as gpr_posterior_predict_kernel)
        double ss = sum_sq<NT>(v);
        ss = quad_sum(ss);
        const long ptg = pt0 + g;
        const bool live = ptg < p.Ns;
        if (t == 0 && live) p.var[b * p.Ns + ptg] = xg[2 * d + 4] - ss;
        double* mrow = p.mean + (b * p.Ns + ptg) * P;
        contract_table<NT>(v, As, AP, P, g, t, live, [&](int c, double m) { mrow[c] = m; });

        // ---- kL, kD to the C-fragment order
        to_c_order<NT>(kL, lane, t);
        if (anyh) to_c_order<NT>(kD, lane, t);

        // ---- beta^T = V^T W over the tiles m >= n: be[2i + e] = beta[8i + 2t + e], the n of kL[2i + e] / kD[2i + e]
        double be[2 * NT];
#pragma unroll
        for (int i = 0; i < NT; ++i) upper_tri_product<NT>(be[2 * i], be[2 * i + 1], v, Wt, i, g, t);

        // ---- per coordinate j: gk = dk_s/dx*_j, dvar_j = -2 beta . gk, dmean_:j = alpha^T gk
        double* dmrow = p.dmean + (b * p.Ns + ptg) * P * d;
        for (int j = 0; j < d; ++j) {
            double gk[2 * NT];
            gk_fragment<NT>(gk, kL, kD, Xt, xg, Il, d, j, t, anyh);
            double sv = 0.0;
#pragma unroll
            for (int k = 0; k < 2 * NT; ++k) sv = fma(be[k], gk[k], sv);
            sv = quad_sum(sv);
            if (t == 0 && live) p.dvar[(b * p.Ns + ptg) * d + j] = -2.0 * sv;
            contract_table<NT>(gk, Al, AP, P, g, t, live, [&](int c, double m) { dmrow[c * d + j] = m; });
        }
        __syncwarp();
    }
}

template <int NT>
__global__ void __launch_bounds__(PW * 32) svgp_posterior_predict_kernel(SvgpFusedArgs p) {
    constexpr int NP = 8 * NT, WP = w_pitch(NP);
    extern __shared__ __align__(16) double sm[];
    __shared__ __align__(16) double etab[512];
    const SvgpPosteriorData& q = p.q;
    const int M = q.M, d = q.d, S1 = rec_len(d);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const long l = blockIdx.y;
    const double* __restrict__ th = q.theta + l * (2 * d + 3);
    double* Ws = sm;                                  // [NP][WP]  Wm, as gpr_posterior_predict_kernel stages W
    double* Lt = Ws + NP * WP;                        // [NP][WP]  Lt[c][slot] = Lq[perm_n(slot)][c]
    double* Qs = Lt + NP * WP;                        // [NP]      q_mu[:, l]
    double* Xt = Qs + NP;                             // [2d+4][NP]  inducing points, k-major
    double* Xw = Xt + (2 * d + 4) * NP + warp * 8 * S1;  // [8][S1]  this warp's test points
    fexp512_table_fill(etab, tid, blockDim.x);
    const RecordParams rp = record_params(th, d);

    // ---- stage the latent: Wm and Lq^T (lower triangles; zero elsewhere), q_mu, scaled inducing points
    {
        const double* __restrict__ Wg = q.Wm + l * M * q.ld;
        const double* __restrict__ Lg = q.Lq + l * M * q.ld;
        for (int idx = tid; idx < NP * NP; idx += blockDim.x) {
            const int r = idx / NP, c = idx - r * NP;
            Ws[r * WP + c] = lower_entry(Wg, q.ld, M, r, c);
            Lt[r * WP + c] = transposed_entry(Lg, q.ld, M, r, c);
        }
        stage_table(Qs, q.q_mu + l, q.L, M, 1, 1, NP, tid);
        stage_points(Xt, q.Z, M, NP, d, rp, tid);
    }
    __syncthreads();

    for (int grp = warp; grp < p.gpc; grp += PW) {
        const long pt0 = ((long)blockIdx.x * p.gpc + grp) * 8;
        if (pt0 >= p.Ns) break;
        // ---- this group's 8 test points (padding points beyond Ns are dead: K_s = 0, never stored)
        if (lane < 8) point_record(Xw + lane * S1, p.Xs, pt0 + lane, p.Ns, d, rp);
        __syncwarp();
        const double* xg = Xw + g * S1;

        // ---- K_s^T fragment: ks[k] = k(z_m, xs_g), m = 4k + t
        double ks[2 * NT];
        ks_fragment<NT>(ks, Xt, xg, d, t, etab);

        // ---- V^T = K_s^T Wm^T over the lower-triangular tiles: v[2i + e] = V^T[g][8i + 2t + e]
        double v[2 * NT];
        lower_tri_v<NT>(v, ks, Ws, g, t);

        // ---- sum V^2, and sum U^2 with U^T = V^T Lq over the tiles m >= n (U never leaves the accumulators)
        double ss = sum_sq<NT>(v);
        double su = 0.0;
#pragma unroll
        for (int i = 0; i < NT; ++i) {
            double c0, c1;
            upper_tri_product<NT>(c0, c1, v, Lt, i, g, t);
            su = fma(c1, c1, fma(c0, c0, su));
        }
        ss = quad_sum(ss);
        su = quad_sum(su);
        const long ptg = pt0 + g;
        const bool live = ptg < p.Ns;
        const long o = l * p.ls + ptg * p.ns;
        if (t == 0 && live) p.var[o] = xg[2 * d + 4] - ss + su;

        // ---- mean = V^T q_mu: q_mu as a table with one column
        contract_table<NT>(v, Qs, 1, 1, g, t, live, [&](int, double m) { p.mean[o] = m; });
        __syncwarp();  // the group's records are read by every lane before lanes 0-7 overwrite them
    }
}

template <int NT>
__global__ void __launch_bounds__(PW * 32, 1) svgp_posterior_predict_grad_kernel(SvgpFusedGradArgs p) {
    constexpr int NP = 8 * NT, WP = w_pitch(NP);
    extern __shared__ __align__(16) double sm[];
    __shared__ __align__(16) double etab[512];
    const SvgpPosteriorData& q = p.q;
    const int M = q.M, d = q.d, S1 = rec_len(d);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const long l = blockIdx.y;
    const double* __restrict__ th = q.theta + l * (2 * d + 3);
    double* Ws = sm;                            // [NP][WP]  Wm, as svgp_posterior_predict_kernel stages it
    double* Lt = Ws + NP * WP;                  // [NP][WP]  Lt[c][slot] = Lq[perm_n(slot)][c], as predict
    double* Wt = Lt + NP * WP;                  // [NP][WP]  Wt[c][slot] = Wm[perm_n(slot)][c]
    double* Qs = Wt + NP * WP;                  // [NP]      q_mu[:, l]
    double* Al = Qs + NP;                       // [NP]      alpha = Wm^T q_mu[:, l]
    double* Xt = Al + NP;                       // [2d+4][NP]  inducing points, k-major
    double* Il = Xt + (2 * d + 4) * NP;         // [2d]  -1/ls_L, -1/ls_delta
    double* Xw = Il + 2 * d + warp * 8 * S1;    // [8][S1]  this warp's test points
    fexp512_table_fill(etab, tid, blockDim.x);
    const RecordParams rp = record_params(th, d);

    // ---- stage the latent: Wm (twice), Lq^T (lower triangles; zero elsewhere), q_mu, scaled inducing points; then alpha
    {
        const double* __restrict__ Wg = q.Wm + l * M * q.ld;
        const double* __restrict__ Lg = q.Lq + l * M * q.ld;
        for (int idx = tid; idx < NP * NP; idx += blockDim.x) {
            const int r = idx / NP, c = idx - r * NP;
            Ws[r * WP + c] = lower_entry(Wg, q.ld, M, r, c);
            Lt[r * WP + c] = transposed_entry(Lg, q.ld, M, r, c);
            Wt[r * WP + c] = transposed_entry(Wg, q.ld, M, r, c);
        }
        stage_table(Qs, q.q_mu + l, q.L, M, 1, 1, NP, tid);
        stage_points(Xt, q.Z, M, NP, d, rp, tid);
        stage_inv_ls(Il, th, d, tid);
    }
    __syncthreads();
    for (int n = tid; n < NP; n += blockDim.x) {
        double s = 0.0;
        for (int m = n; m < M; ++m) s = fma(Ws[m * WP + n], Qs[m], s);
        Al[n] = s;
    }
    __syncthreads();

    for (int grp = warp; grp < p.gpc; grp += PW) {
        const long pt0 = ((long)blockIdx.x * p.gpc + grp) * 8;
        if (pt0 >= p.Ns) break;
        if (lane < 8) point_record(Xw + lane * S1, p.Xs, pt0 + lane, p.Ns, d, rp);
        __syncwarp();
        const double* xg = Xw + g * S1;
        const double sg = xg[2 * d + 2], hg = xg[2 * d + 3];
        const bool anyh = __any_sync(0xffffffffu, hg != 0.0);

        // ---- the two parts of K_s^T in predict's A-fragment layout: kL[k], kD[k] at m = 4k + t
        double kL[2 * NT], kD[2 * NT];
        {
            const double* xe = Xt + 2 * d * NP + t;
#pragma unroll
            for (int k = 0; k < 2 * NT; ++k) kL[k] = xe[4 * k] + xg[2 * d];
            for (int c = 0; c < d; ++c) {
                const double xc = xg[c];
                const double* xr = Xt + c * NP + t;
#pragma unroll
                for (int k = 0; k < 2 * NT; ++k) kL[k] = fma(xr[4 * k], xc, kL[k]);
            }
            const double* sr = Xt + (2 * d + 2) * NP + t;
#pragma unroll
            for (int k = 0; k < 2 * NT; ++k) kL[k] = fexp512(kL[k], etab) * (sr[4 * k] * sg);
#pragma unroll
            for (int k = 0; k < 2 * NT; ++k) kD[k] = 0.0;
            if (anyh) {
                const double* xf = Xt + (2 * d + 1) * NP + t;
#pragma unroll
                for (int k = 0; k < 2 * NT; ++k) kD[k] = xf[4 * k] + xg[2 * d + 1];
                for (int c = 0; c < d; ++c) {
                    const double xc = xg[d + c];
                    const double* xr = Xt + (d + c) * NP + t;
#pragma unroll
                    for (int k = 0; k < 2 * NT; ++k) kD[k] = fma(xr[4 * k], xc, kD[k]);
                }
                const double* hr = Xt + (2 * d + 3) * NP + t;
#pragma unroll
                for (int k = 0; k < 2 * NT; ++k) kD[k] = hr[4 * k] * hg != 0.0 ? fexp512(kD[k], etab) : 0.0;
            }
        }

        // ---- V^T = K_s^T Wm^T over the lower-triangular tiles: v[2i + e] = V^T[g][8i + 2t + e]
        double v[2 * NT];
        {
            double ks[2 * NT];
#pragma unroll
            for (int k = 0; k < 2 * NT; ++k) ks[k] = __dadd_rn(kL[k], kD[k]);  // predict's K_s, not contracted
            lower_tri_v<NT>(v, ks, Ws, g, t);
        }

        // ---- U^T = V^T Lq over the tiles m >= n; var = k_ss - sum V^2 + sum U^2, mean = V^T q_mu  (as predict)
        double u[2 * NT];
        double ss = sum_sq<NT>(v);
        double su = 0.0;
#pragma unroll
        for (int i = 0; i < NT; ++i) {
            upper_tri_product<NT>(u[2 * i], u[2 * i + 1], v, Lt, i, g, t);
            su = fma(u[2 * i + 1], u[2 * i + 1], fma(u[2 * i], u[2 * i], su));
        }
        ss = quad_sum(ss);
        su = quad_sum(su);
        const long ptg = pt0 + g;
        const bool live = ptg < p.Ns;
        const long o = l * p.ls + ptg * p.ns;
        if (t == 0 && live) p.var[o] = xg[2 * d + 4] - ss + su;
        contract_table<NT>(v, Qs, 1, 1, g, t, live, [&](int, double m) { p.mean[o] = m; });

        // ---- r = V - Lq U over the tiles m <= n (Lt read transposed), then beta^T = r^T Wm over the tiles m >= n:
        //      be[2i + e] = beta[8i + 2t + e]
        {
            double r[2 * NT];
#pragma unroll
            for (int i = 0; i < NT; ++i) {
                double c0, c1;
                lower_tri_product<NT>(c0, c1, u, Lt, i, g, t);
                r[2 * i] = v[2 * i] - c0;
                r[2 * i + 1] = v[2 * i + 1] - c1;
            }
#pragma unroll
            for (int i = 0; i < NT; ++i) upper_tri_product<NT>(v[2 * i], v[2 * i + 1], r, Wt, i, g, t);
        }
        const double(&be)[2 * NT] = v;

        // ---- kL, kD to the C-fragment order
        to_c_order<NT>(kL, lane, t);
        if (anyh) to_c_order<NT>(kD, lane, t);

        // ---- per coordinate j: gk = dk_s/dx*_j, dvar_j = -2 beta . gk, dmean_j = alpha . gk
        const double* ar = Al + 2 * t;
        const long od = o * d;
        for (int j = 0; j < d; ++j) {
            double gk[2 * NT];
            gk_fragment<NT>(gk, kL, kD, Xt, xg, Il, d, j, t, anyh);
            double sv = 0.0, sa = 0.0;
#pragma unroll
            for (int i = 0; i < NT; ++i) {
                sv = fma(be[2 * i + 1], gk[2 * i + 1], fma(be[2 * i], gk[2 * i], sv));
                sa = fma(gk[2 * i + 1], ar[8 * i + 1], fma(gk[2 * i], ar[8 * i], sa));
            }
            sv = quad_sum(sv);
            sa = quad_sum(sa);
            if (t == 0 && live) {
                p.dmean[od + j] = sa;
                p.dvar[od + j] = -2.0 * sv;
            }
        }
        __syncwarp();
    }
}

// ---- joint posterior (mfgp_gpr_posterior_predict_cov / _sample), Ns <= 64 test points.  One CTA per (chunk of sample
//      columns, problem); every CTA of a problem rebuilds Sigma and its factor the same way, so no result depends on the
//      chunking.  Shared memory (doubles), regions reused once their first tenant is dead:
//        RA  W [NP][WP]                       -> Sigma, then L  [NSP][SPp]
//        As  a [NP][AP]     Xt [2d+4][NP]     Xr  records of all test points [NSP][S1]
//        RB  V^T [NSP][WP]                    -> z tile [NSP][JZP]   (_sample)
//        Dg  predict's var, then diag(L) [NSP]     Lc  column of L being formed [NSP]     Ms  mean [NSP][P] (_sample)
constexpr int JZC = 64;        // z columns per shared-memory tile
constexpr int JZP = JZC + 4;   // its pitch: 4 mod 16 keeps the B-fragment loads Zs[4k + t][8j + g] free of bank conflicts
constexpr int JL = 8;          // z loads in flight per thread
constexpr int JOINT_MAX_NS = 64;
constexpr long JOINT_MIN_COLS = 256;  // sample columns per CTA at least: the CTA's rebuild of Sigma and L stays small
__host__ __device__ constexpr int s_pitch(int NSP) { return NSP + 4; }

struct JointSmem {
    int ra, as, xt, xr, rb, dg, lc, ms, total;  // offsets in doubles
    __host__ __device__ JointSmem(int NT, int NST, int d, int P, bool sample) {
        const int NP = 8 * NT, NSP = 8 * NST;
        const int wsz = NP * w_pitch(NP), ssz = NSP * s_pitch(NSP), vsz = NSP * w_pitch(NP), zsz = sample ? NSP * JZP : 0;
        int o = 0;
        ra = o; o += wsz > ssz ? wsz : ssz;
        as = o; o += NP * a_pitch(P);
        xt = o; o += (2 * d + 4) * NP;
        xr = o; o += NSP * rec_len(d);
        rb = o; o += vsz > zsz ? vsz : zsz;
        dg = o; o += NSP;
        lc = o; o += NSP;
        ms = o; o += sample ? NSP * P : 0;
        total = o;
    }
};

struct JointArgs {
    GprPosteriorData q;
    const double* Xs;
    int Ns;
    long SP;       // S * P sample columns per test point; 0: _predict_cov
    long cpc;      // sample columns per CTA (a multiple of JZC)
    double jitter;
    const double* z;  // [B][Ns][SP]
    double* samples;  // [B][Ns][SP]
    int* info;        // [B]
    int* d_info;
    double* mean;     // _predict_cov: [B][Ns][P]
    double* cov;      //               [B][Ns][Ns]
};

// k(x_i, x_j) from two point records in K1's expanded-square form (the form ks_fragment evaluates).
__device__ __forceinline__ double kss_pair(const double* xi, const double* xj, int d, const double* etab) {
    double e = xj[2 * d] + xi[2 * d];
    for (int c = 0; c < d; ++c) e = fma(xj[c], xi[c], e);
    double k = fexp512(e, etab) * (xj[2 * d + 2] * xi[2 * d + 2]);
    if (xj[2 * d + 3] * xi[2 * d + 3] != 0.0) {
        double e2 = xj[2 * d + 1] + xi[2 * d + 1];
        for (int c = 0; c < d; ++c) e2 = fma(xj[d + c], xi[d + c], e2);
        k += fexp512(e2, etab);
    }
    return k;
}

template <int NT>
__global__ void __launch_bounds__(PW * 32) gpr_posterior_joint_kernel(JointArgs p) {
    constexpr int NP = 8 * NT, WP = w_pitch(NP);
    extern __shared__ __align__(16) double sm[];
    __shared__ __align__(16) double etab[512];
    __shared__ int fail;
    const GprPosteriorData& q = p.q;
    const int N = q.N, d = q.d, P = q.P, AP = a_pitch(P), S1 = rec_len(d), Ns = p.Ns;
    const int NST = (Ns + 7) / 8, NSP = 8 * NST, SPp = s_pitch(NSP);
    const bool sample = p.SP > 0;
    const JointSmem lay(NT, NST, d, P, sample);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const long b = blockIdx.y;
    const double* __restrict__ th = q.theta + b * (2 * d + 3);
    double* Ws = sm + lay.ra;
    double* Sg = Ws;  // Sigma, then L, once W is dead
    double* As = sm + lay.as;
    double* Xt = sm + lay.xt;
    double* Xr = sm + lay.xr;
    double* Vt = sm + lay.rb;
    double* Zs = Vt;  // z tiles, once V is dead
    double* Dg = sm + lay.dg;
    double* Lc = sm + lay.lc;
    double* Ms = sm + lay.ms;
    fexp512_table_fill(etab, tid, blockDim.x);
    const RecordParams rp = record_params(th, d);

    // ---- stage the problem as gpr_posterior_predict_kernel does, and the records of every test point (padding: dead)
    {
        const double* __restrict__ Wg = q.W + b * N * q.ld;
        for (int idx = tid; idx < NP * NP; idx += blockDim.x) {
            const int r = idx / NP, c = idx - r * NP;
            Ws[r * WP + c] = lower_entry(Wg, q.ld, N, r, c);
        }
        stage_table(As, q.a + b * N * q.Pp, q.Pp, N, P, AP, NP, tid);
        stage_points(Xt, q.X, N, NP, d, rp, tid);
        for (int i = tid; i < NSP; i += blockDim.x) point_record(Xr + i * S1, p.Xs, i, Ns, d, rp);
    }
    __syncthreads();

    // ---- per 8-point group: K_s, V, var and mean with predict's code (so mean and diag(Sigma) are predict's bits); V^T
    //      to shared memory
    for (int grp = warp; grp < NST; grp += PW) {
        const int i = 8 * grp + g;
        const double* xg = Xr + i * S1;
        double ks[2 * NT];
        ks_fragment<NT>(ks, Xt, xg, d, t, etab);
        double v[2 * NT];
        lower_tri_v<NT>(v, ks, Ws, g, t);
        double ss = sum_sq<NT>(v);
        ss = quad_sum(ss);
        if (t == 0) Dg[i] = xg[2 * d + 4] - ss;
#pragma unroll
        for (int k = 0; k < NT; ++k) {
            Vt[i * WP + 8 * k + 2 * t] = v[2 * k];
            Vt[i * WP + 8 * k + 2 * t + 1] = v[2 * k + 1];
        }
        const bool live = i < Ns;
        if (sample) {
            contract_table<NT>(v, As, AP, P, g, t, live, [&](int c, double m) { Ms[i * P + c] = m; });
        } else {
            double* mrow = p.mean + (b * Ns + i) * P;
            contract_table<NT>(v, As, AP, P, g, t, live, [&](int c, double m) { mrow[c] = m; });
        }
    }
    __syncthreads();

    // ---- Sigma = K_ss - V^T V on the lower 8x8 tiles (DMMA over the NP training indices), predict's var on the diagonal,
    //      each entry also stored mirrored: Sigma is exactly symmetric.  Padding rows and columns: identity.
    for (int tt = warp; tt < NST * (NST + 1) / 2; tt += PW) {
        int I = 0;
        while ((I + 1) * (I + 2) / 2 <= tt) ++I;
        const int J = tt - I * (I + 1) / 2;
        double c0 = 0.0, c1 = 0.0;
        const double* ar = Vt + (8 * I + g) * WP + t;
        const double* br = Vt + (8 * J + g) * WP + t;
#pragma unroll
        for (int k = 0; k < 2 * NT; ++k) dmma(c0, c1, ar[4 * k], br[4 * k]);
        const int i = 8 * I + g;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int j = 8 * J + 2 * t + e;
            if (j > i) continue;
            double s;
            if (i >= Ns || j >= Ns) s = i == j ? 1.0 : 0.0;
            else if (i == j) s = Dg[i];
            else s = kss_pair(Xr + i * S1, Xr + j * S1, d, etab) - (e ? c1 : c0);
            Sg[i * SPp + j] = s;
            Sg[j * SPp + i] = s;
        }
    }
    __syncthreads();

    if (!sample) {
        double* cb = p.cov + b * Ns * Ns;
        for (long idx = tid; idx < (long)Ns * Ns; idx += blockDim.x) {
            const int i = (int)(idx / Ns), j = (int)(idx - (long)i * Ns);
            cb[idx] = Sg[i * SPp + j];
        }
        return;
    }

    // ---- L L^T = Sigma + jitter I in place, one column per step (right-looking).  Every thread reads the same pivot, so
    //      the exit at a pivot that is not > 0 (NaN included) is uniform.  diag(L) goes to Dg, the column to Lc.
    if (tid == 0) fail = 0;
    for (int i = tid; i < Ns; i += blockDim.x) Sg[i * SPp + i] += p.jitter;
    __syncthreads();
    for (int j = 0; j < Ns; ++j) {
        const double piv = Sg[j * SPp + j];
        if (!(piv > 0.0)) {
            if (tid == 0) fail = j + 1;
            break;
        }
        const double ljj = sqrt(piv);
        for (int i = j + 1 + tid; i < Ns; i += blockDim.x) {
            const double l = Sg[i * SPp + j] / ljj;
            Lc[i] = l;
            Sg[i * SPp + j] = l;
        }
        if (tid == 0) Dg[j] = ljj;
        __syncthreads();
        for (int i = j + 1 + warp; i < Ns; i += PW) {
            const double li = Lc[i];
            for (int k = j + 1 + lane; k <= i; k += 32) Sg[i * SPp + k] = fma(-li, Lc[k], Sg[i * SPp + k]);
        }
        __syncthreads();
    }
    __syncthreads();
    const int bad = fail;
    for (int idx = tid; idx < NSP * NSP; idx += blockDim.x) {  // L: diagonal from Dg, zero above it
        const int i = idx / NSP, k = idx - i * NSP;
        if (k > i) Sg[i * SPp + k] = 0.0;
        else if (k == i && i < Ns) Sg[i * SPp + k] = Dg[i];
    }
    if (blockIdx.x == 0 && tid == 0) {
        p.info[b] = bad;
        if (bad) atomicCAS(p.d_info, 0, bad);
    }
    __syncthreads();

    // ---- samples = mean + L z over this CTA's columns, JZC at a time: z rows through shared memory (coalesced along the
    //      S * P axis), L's lower tiles on DMMA (k-steps 0 .. 2I + 1 for row tile I), stores 64 contiguous bytes per row
    const double qnan = __longlong_as_double(0x7ff8000000000000ll);
    const long c_beg = blockIdx.x * p.cpc, c_end = c_beg + p.cpc < p.SP ? c_beg + p.cpc : p.SP;
    const double* __restrict__ zb = p.z + b * Ns * p.SP;
    double* __restrict__ ob = p.samples + b * Ns * p.SP;
    for (long c0 = c_beg; c0 < c_end; c0 += JZC) {
        const int nc = c_end - c0 < JZC ? (int)(c_end - c0) : JZC;
        if (!bad)  // JL independent loads in flight per thread before the stores
            for (int base = tid; base < NSP * JZC; base += JL * PW * 32) {
                double zv[JL];
#pragma unroll
                for (int u = 0; u < JL; ++u) {
                    const int idx = base + u * PW * 32, r = idx / JZC, cc = idx % JZC;
                    zv[u] = (idx < NSP * JZC && r < Ns && cc < nc) ? zb[(long)r * p.SP + c0 + cc] : 0.0;
                }
#pragma unroll
                for (int u = 0; u < JL; ++u) {
                    const int idx = base + u * PW * 32;
                    if (idx < NSP * JZC) Zs[(idx / JZC) * JZP + idx % JZC] = zv[u];
                }
            }
        __syncthreads();
        for (int tt = warp; tt < NST * (JZC / 8); tt += PW) {
            const int I = tt / (JZC / 8), Jc = tt % (JZC / 8);
            double c0v = 0.0, c1v = 0.0;
            if (!bad) {
                const double* lr = Sg + (8 * I + g) * SPp + t;
                const double* zr = Zs + t * JZP + 8 * Jc + g;
                for (int k = 0; k <= 2 * I + 1; ++k) dmma(c0v, c1v, lr[4 * k], zr[4 * k * JZP]);
            }
            const int i = 8 * I + g, cc = 8 * Jc + 2 * t;
            if (i < Ns) {
                double* orow = ob + (long)i * p.SP + c0;
                if (cc < nc) orow[cc] = bad ? qnan : Ms[i * P + (int)((c0 + cc) % P)] + c0v;
                if (cc + 1 < nc) orow[cc + 1] = bad ? qnan : Ms[i * P + (int)((c0 + cc + 1) % P)] + c1v;
            }
        }
        __syncthreads();
    }
}

// ---- joint covariance of the SVGP latents (mfgp_svgp_posterior_predict_cov / _sample), Ns <= 64 test points.  One CTA
//      per latent, all latents in one launch: predict's staging of Wm, Lq^T and Z, the records of every test point, then
//      per 8-point group predict's K_s, V and U with V^T and U^T to shared memory, then Sigma_l = K_ss - V^T V + U^T U on
//      the lower 8x8 tiles (DMMA over the inducing index, K_ss from the point records), each entry also stored mirrored.
//      The diagonal is written too; the caller replaces it with predict's var.
size_t svgp_joint_smem_bytes(int NT, int NST, int d) {
    const int NP = 8 * NT, NSP = 8 * NST;
    return sizeof(double) * (2 * (size_t)NP * w_pitch(NP) + (size_t)(2 * d + 4) * NP + (size_t)NSP * rec_len(d) +
                             2 * (size_t)NSP * w_pitch(NP));
}

struct SvgpJointArgs {
    SvgpPosteriorData q;
    const double* Xs;
    int Ns;
    double* Sl;  // [L][Ns][lds]
    long lds;
};

template <int NT>
__global__ void __launch_bounds__(PW * 32, 1) svgp_posterior_joint_kernel(SvgpJointArgs p) {
    constexpr int NP = 8 * NT, WP = w_pitch(NP);
    extern __shared__ __align__(16) double sm[];
    __shared__ __align__(16) double etab[512];
    const SvgpPosteriorData& q = p.q;
    const int M = q.M, d = q.d, S1 = rec_len(d), Ns = p.Ns, NST = (Ns + 7) / 8, NSP = 8 * NST;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const long l = blockIdx.y;
    const double* __restrict__ th = q.theta + l * (2 * d + 3);
    double* Ws = sm;                     // [NP][WP]    Wm, as svgp_posterior_predict_kernel stages it
    double* Lt = Ws + NP * WP;           // [NP][WP]    Lt[c][slot] = Lq[perm_n(slot)][c], as predict
    double* Xt = Lt + NP * WP;           // [2d+4][NP]  inducing points, k-major
    double* Xr = Xt + (2 * d + 4) * NP;  // [NSP][S1]   records of all test points (padding: dead)
    double* Vt = Xr + NSP * S1;          // [NSP][WP]   V^T
    double* Ut = Vt + NSP * WP;          // [NSP][WP]   U^T
    fexp512_table_fill(etab, tid, blockDim.x);

    {
        const RecordParams rp = record_params(th, d);
        const double* __restrict__ Wg = q.Wm + l * M * q.ld;
        const double* __restrict__ Lg = q.Lq + l * M * q.ld;
        for (int idx = tid; idx < NP * NP; idx += blockDim.x) {
            const int r = idx / NP, c = idx - r * NP;
            Ws[r * WP + c] = lower_entry(Wg, q.ld, M, r, c);
            Lt[r * WP + c] = transposed_entry(Lg, q.ld, M, r, c);
        }
        stage_points(Xt, q.Z, M, NP, d, rp, tid);
        for (int i = tid; i < NSP; i += blockDim.x) point_record(Xr + i * S1, p.Xs, i, Ns, d, rp);
    }
    __syncthreads();

    // ---- per 8-point group: K_s, V^T = K_s^T Wm^T and U^T = V^T Lq as predict forms them, to shared memory in the
    //      natural inducing order (slot 2k + e of lane t is m = 8k + 2t + e)
    for (int grp = warp; grp < NST; grp += PW) {
        const int i = 8 * grp + g;
        double ks[2 * NT];
        ks_fragment<NT>(ks, Xt, Xr + i * S1, d, t, etab);
        double v[2 * NT];
        lower_tri_v<NT>(v, ks, Ws, g, t);
#pragma unroll
        for (int k = 0; k < NT; ++k) {
            Vt[i * WP + 8 * k + 2 * t] = v[2 * k];
            Vt[i * WP + 8 * k + 2 * t + 1] = v[2 * k + 1];
        }
#pragma unroll
        for (int k = 0; k < NT; ++k) upper_tri_product<NT>(Ut[i * WP + 8 * k + 2 * t], Ut[i * WP + 8 * k + 2 * t + 1], v, Lt, k, g, t);
    }
    __syncthreads();

    // ---- Sigma_l on the lower 8x8 tiles, as gpr_posterior_joint_kernel forms K_ss - V^T V, plus U^T U
    double* __restrict__ So = p.Sl + l * Ns * p.lds;
    for (int tt = warp; tt < NST * (NST + 1) / 2; tt += PW) {
        int I = 0;
        while ((I + 1) * (I + 2) / 2 <= tt) ++I;
        const int J = tt - I * (I + 1) / 2;
        double c0 = 0.0, c1 = 0.0, e0 = 0.0, e1 = 0.0;
        const double* va = Vt + (8 * I + g) * WP + t;
        const double* vb = Vt + (8 * J + g) * WP + t;
        const double* ua = Ut + (8 * I + g) * WP + t;
        const double* ub = Ut + (8 * J + g) * WP + t;
#pragma unroll
        for (int k = 0; k < 2 * NT; ++k) {
            dmma(c0, c1, va[4 * k], vb[4 * k]);
            dmma(e0, e1, ua[4 * k], ub[4 * k]);
        }
        const int i = 8 * I + g;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int j = 8 * J + 2 * t + e;
            if (j > i || i >= Ns) continue;
            const double s = kss_pair(Xr + i * S1, Xr + j * S1, d, etab) - (e ? c1 : c0) + (e ? e1 : e0);
            So[(long)i * p.lds + j] = s;
            So[(long)j * p.lds + i] = s;
        }
    }
}

// Input gradient of the blocked route (launch_posterior_dx): one CTA per (tile of TS test points, chunk of PC columns,
// problem), walking the training points in tiles of TN.  Per tile it evaluates kL and kD from the scaled inputs (as K5
// recomputes dK: nothing N x Ns is stored), forms G[j][s][n] = dk_sn/dx_sj in shared memory and adds G alpha (thread =
// (point, column)) and G beta (thread = (point, coordinate)) to accumulators in shared memory.  Each sum runs over n in
// a fixed order and involves only its own test point: no atomics, no cross-point reduction.
constexpr int DX_TS = 8, DX_PC = 32, DX_TN = 16, DX_THREADS = DX_TS * DX_PC;

size_t posterior_dx_smem_bytes(int d) {
    const int R = 2 * d + 4;
    return sizeof(double) * ((size_t)DX_TS * R + (size_t)R * DX_TN + 2 * DX_TS * DX_TN + (size_t)d * DX_TS * DX_TN +
                             DX_TN * DX_PC + DX_TN * DX_TS + (size_t)DX_TS * d * DX_PC + (size_t)DX_TS * d + 2 * d);
}

__global__ void __launch_bounds__(DX_THREADS) posterior_dx_kernel(GprPosteriorData q, const double* __restrict__ Xs, int Ns,
                                                                const double* __restrict__ alpha,
                                                                const double* __restrict__ beta, long ldb,
                                                                double* __restrict__ dmean, double* __restrict__ dvar) {
    extern __shared__ __align__(16) double sm[];
    const int N = q.N, d = q.d, P = q.P, R = 2 * d + 4, tid = threadIdx.x;
    const long b = blockIdx.z;
    const int s0 = blockIdx.x * DX_TS, p0 = blockIdx.y * DX_PC;
    const bool want_var = blockIdx.y == 0;
    const double* __restrict__ th = q.theta + b * (2 * d + 3);
    double* xs = sm;                       // [TS][R]   test points
    double* xn = xs + DX_TS * R;           // [R][TN]   training points of the tile
    double* kl = xn + R * DX_TN;           // [TS][TN]
    double* kd = kl + DX_TS * DX_TN;       // [TS][TN]
    double* G = kd + DX_TS * DX_TN;        // [d][TS][TN]
    double* al = G + d * DX_TS * DX_TN;    // [TN][PC]
    double* be = al + DX_TN * DX_PC;       // [TN][TS]
    double* acc = be + DX_TN * DX_TS;      // [TS][d][PC]
    double* dv = acc + DX_TS * d * DX_PC;  // [TS][d]
    double* il = dv + DX_TS * d;           // [2d]  -1/ls_L, -1/ls_delta
    const double hlL = 0.5 * log(th[1 + d]), hlD = 0.5 * log(th[2 + 2 * d]), vL = th[1 + d], vD = th[2 + 2 * d];
    if (tid < DX_TS) prescale_point(Xs + (long)(s0 + tid < Ns ? s0 + tid : 0) * (d + 1), s0 + tid < Ns, d, th, hlL, hlD,
                                    xs + tid * R, 1);
    for (int k = tid; k < d; k += DX_THREADS) {
        il[k] = -1.0 / th[1 + k];
        il[d + k] = -1.0 / th[2 + d + k];
    }
    for (int i = tid; i < DX_TS * d * DX_PC; i += DX_THREADS) acc[i] = 0.0;
    for (int i = tid; i < DX_TS * d; i += DX_THREADS) dv[i] = 0.0;
    const double* __restrict__ ab = alpha + b * N * q.Pp;
    const double* __restrict__ bb = beta + b * N * ldb;
    const int ts = tid / DX_PC, tp = tid % DX_PC;

    for (int n0 = 0; n0 < N; n0 += DX_TN) {
        if (tid < DX_TN) prescale_point(q.X + (long)(n0 + tid < N ? n0 + tid : 0) * (d + 1), n0 + tid < N, d, th, hlL, hlD,
                                        xn + tid, DX_TN);
        for (int i = tid; i < DX_TN * DX_PC; i += DX_THREADS) {
            const int n = n0 + i / DX_PC, c = p0 + i % DX_PC;
            al[i] = (n < N && c < P) ? ab[(long)n * q.Pp + c] : 0.0;
        }
        for (int i = tid; i < DX_TN * DX_TS; i += DX_THREADS) {
            const int n = n0 + i / DX_TS, c = s0 + i % DX_TS;
            be[i] = (n < N && c < Ns) ? bb[(long)n * ldb + c] : 0.0;
        }
        __syncthreads();
        for (int i = tid; i < DX_TS * DX_TN; i += DX_THREADS) {
            const int si = i / DX_TN, n = i % DX_TN;
            const double* x = xs + si * R;
            double rL = 0.0, rD = 0.0;
            for (int c = 0; c < d; ++c) {
                const double eL = x[c] - xn[c * DX_TN + n], eD = x[d + c] - xn[(d + c) * DX_TN + n];
                rL = fma(eL, eL, rL);
                rD = fma(eD, eD, rD);
            }
            kl[i] = (x[2 * d + 2] * xn[(2 * d + 2) * DX_TN + n]) * (vL * exp(-0.5 * rL));
            kd[i] = x[2 * d + 3] * xn[(2 * d + 3) * DX_TN + n] != 0.0 ? vD * exp(-0.5 * rD) : 0.0;
        }
        __syncthreads();
        for (int i = tid; i < d * DX_TS * DX_TN; i += DX_THREADS) {
            const int j = i / (DX_TS * DX_TN), si = (i / DX_TN) % DX_TS, n = i % DX_TN, sn = si * DX_TN + n;
            const double* x = xs + si * R;
            G[i] = fma(kd[sn] * (x[d + j] - xn[(d + j) * DX_TN + n]), il[d + j], kl[sn] * (x[j] - xn[j * DX_TN + n]) * il[j]);
        }
        __syncthreads();
        for (int j = 0; j < d; ++j) {
            const double* gr = G + (j * DX_TS + ts) * DX_TN;
            double a = 0.0;
#pragma unroll
            for (int n = 0; n < DX_TN; ++n) a = fma(gr[n], al[n * DX_PC + tp], a);
            acc[(ts * d + j) * DX_PC + tp] += a;
        }
        if (want_var)
            for (int i = tid; i < DX_TS * d; i += DX_THREADS) {
                const int si = i / d, j = i % d;
                const double* gr = G + (j * DX_TS + si) * DX_TN;
                double a = 0.0;
#pragma unroll
                for (int n = 0; n < DX_TN; ++n) a = fma(gr[n], be[n * DX_TS + si], a);
                dv[i] += a;
            }
        __syncthreads();
    }
    for (int i = tid; i < DX_TS * DX_PC * d; i += DX_THREADS) {
        const int si = i / (DX_PC * d), r = i % (DX_PC * d), c = r / d, j = r % d;
        if (s0 + si < Ns && p0 + c < P) dmean[((b * Ns + s0 + si) * P + p0 + c) * d + j] = acc[(si * d + j) * DX_PC + c];
    }
    if (want_var)
        for (int i = tid; i < DX_TS * d; i += DX_THREADS)
            if (s0 + i / d < Ns) dvar[(b * Ns + s0) * d + i] = -2.0 * dv[i];
}

// 8-point groups per CTA: enough CTAs for ~8 per SM, and no more than 256 groups (chunks of <= 2048 points) so that a CTA's
// staging of the factors (read once per CTA) stays small against its arithmetic.  The split never changes a result (see
// the file comment).
int groups_per_cta(int Ns, int batch) {
    const long G = (Ns + 7) / 8;
    const long target = (long)mfgp_current_dev_info().sms * 8;
    long gpc = (G * batch + target - 1) / target;
    if (gpc > 256) gpc = 256;
    if (gpc > G) gpc = G;
    if (gpc < 1) gpc = 1;
    return (int)gpc;
}

// f(std::integral_constant<int, NT>{}) for NT = 1 .. 8 (larger NT as 8): the fused kernels are instantiated per tile count.
template <class F>
int with_nt(int NT, F f) {
    switch (NT) {
        case 1: return f(std::integral_constant<int, 1>{});
        case 2: return f(std::integral_constant<int, 2>{});
        case 3: return f(std::integral_constant<int, 3>{});
        case 4: return f(std::integral_constant<int, 4>{});
        case 5: return f(std::integral_constant<int, 5>{});
        case 6: return f(std::integral_constant<int, 6>{});
        case 7: return f(std::integral_constant<int, 7>{});
        default: return f(std::integral_constant<int, 8>{});
    }
}

// CTAs along grid x of a predict kernel: the 8-point groups of Ns, gpc per CTA.
long point_chunks(int Ns, int gpc) {
    const long G = (Ns + 7) / 8;
    return (G + gpc - 1) / gpc;
}

// One launch of a fused kernel over `batch` problems (grid y) and gx CTAs along grid x.
template <auto Kernel, class Args>
int launch_fused(cudaStream_t s, const Args& a, long gx, int batch, size_t smem) {
    static SmemOptIn optin;
    if (!optin.ensure(Kernel, smem)) return -2;
    Kernel<<<dim3((unsigned)gx, (unsigned)batch), PW * 32, smem, s>>>(a);
    return cudaGetLastError() == cudaSuccess ? 0 : -2;
}

// f(qs, b0) for the problems of q in slices of at most 65 535 (the grid-y limit): qs describes problems b0 .. b0 + qs.B - 1
// as a batch of their own.  Stops at the first nonzero return.
template <class F>
int for_batch_slices(const GprPosteriorData& q, F f) {
    constexpr int MAX_GRID_Y = 65535;
    for (int b0 = 0; b0 < q.B; b0 += MAX_GRID_Y) {
        GprPosteriorData qs = q;
        qs.B = q.B - b0 < MAX_GRID_Y ? q.B - b0 : MAX_GRID_Y;
        qs.theta = q.theta + (long)b0 * (2 * q.d + 3);
        qs.noise = q.noise + b0;
        qs.W = q.W + (long)b0 * q.N * q.ld;
        qs.a = q.a + (long)b0 * q.N * q.Pp;
        const int rc = f(qs, (long)b0);
        if (rc) return rc;
    }
    return 0;
}

}  // namespace

bool gpr_posterior_fused_ok(int N, int d, int P) {
    return N >= 1 && N <= MFGP_SMALL_MAX_N && d >= 1 && d <= MFGP_SMALL_MAX_D && P >= 1 && P <= MAX_P;
}

int gpr_posterior_predict_fused(cudaStream_t s, const GprPosteriorData& q, const double* Xs, int Ns, double* mean,
                                double* var, double* dmean, double* dvar) {
    if (!gpr_posterior_fused_ok(q.N, q.d, q.P)) return -1;
    if (Ns <= 0 || q.B <= 0) return 0;
    const bool grad = dmean != nullptr;
    const int NT = (q.N + 7) / 8;
    const size_t smem = grad ? fused_grad_smem_bytes(NT, q.d, q.P) : fused_smem_bytes(NT, q.d, q.P);
    const int gpc = groups_per_cta(Ns, q.B);
    const long gx = point_chunks(Ns, gpc);
    return for_batch_slices(q, [&](const GprPosteriorData& qs, long b0) {
        FusedArgs a{};
        a.q = qs;
        a.Xs = Xs; a.Ns = Ns; a.gpc = gpc;
        a.mean = mean + b0 * Ns * q.P;
        a.var = var + b0 * Ns;
        if (grad) {
            a.dmean = dmean + b0 * Ns * q.P * q.d;
            a.dvar = dvar + b0 * Ns * q.d;
        }
        return with_nt(NT, [&](auto nt) {
            constexpr int K = decltype(nt)::value;
            return grad ? launch_fused<gpr_posterior_predict_grad_kernel<K>>(s, a, gx, qs.B, smem)
                        : launch_fused<gpr_posterior_predict_kernel<K>>(s, a, gx, qs.B, smem);
        });
    });
}

bool gpr_posterior_joint_fused_ok(int N, int d, int P, int Ns) { return gpr_posterior_fused_ok(N, d, P) && Ns <= JOINT_MAX_NS; }

int gpr_posterior_joint_fused(cudaStream_t s, const GprPosteriorData& q, const double* Xs, int Ns, double* mean,
                              const GprJointOut& j, int* d_info) {
    if (!gpr_posterior_joint_fused_ok(q.N, q.d, q.P, Ns)) return -1;
    if (Ns <= 0 || q.B <= 0) return 0;
    const bool sample = j.SP > 0;
    const int NT = (q.N + 7) / 8, NST = (Ns + 7) / 8;
    const size_t smem = sizeof(double) * (size_t)JointSmem(NT, NST, q.d, q.P, sample).total;
    // sample columns per CTA: about 4 CTAs per SM over the whole call, at least JOINT_MIN_COLS (a multiple of JZC)
    long cpc = 0, chunks = 1;
    if (sample) {
        const long target = (long)mfgp_current_dev_info().sms * 4;
        const long tot = (long)q.B * j.SP;
        cpc = round_up((tot + target - 1) / target, JZC);
        if (cpc < JOINT_MIN_COLS) cpc = JOINT_MIN_COLS;
        if (cpc > round_up(j.SP, JZC)) cpc = round_up(j.SP, JZC);
        chunks = (j.SP + cpc - 1) / cpc;
    }
    return for_batch_slices(q, [&](const GprPosteriorData& qs, long b0) {
        JointArgs a{};
        a.q = qs;
        a.Xs = Xs; a.Ns = Ns; a.SP = j.SP; a.cpc = cpc; a.jitter = j.jitter; a.d_info = d_info;
        if (sample) {
            a.z = j.z + b0 * Ns * j.SP;
            a.samples = j.samples + b0 * Ns * j.SP;
            a.info = j.info + b0;
        } else {
            a.mean = mean + b0 * Ns * q.P;
            a.cov = j.cov + b0 * Ns * Ns;
        }
        return with_nt(NT, [&](auto nt) {
            return launch_fused<gpr_posterior_joint_kernel<decltype(nt)::value>>(s, a, chunks, qs.B, smem);
        });
    });
}

int launch_posterior_dx(cudaStream_t s, const GprPosteriorData& q, int nb, const double* Xs, int Ns, const double* alpha,
                        const double* beta, long ldb, double* dmean, double* dvar) {
    static SmemOptIn optin;
    const size_t smem = posterior_dx_smem_bytes(q.d);
    if (!optin.ensure(posterior_dx_kernel, smem)) return -2;
    dim3 grid((unsigned)((Ns + DX_TS - 1) / DX_TS), (unsigned)((q.P + DX_PC - 1) / DX_PC), (unsigned)nb);
    posterior_dx_kernel<<<grid, DX_THREADS, smem, s>>>(q, Xs, Ns, alpha, beta, ldb, dmean, dvar);
    return cudaGetLastError() == cudaSuccess ? 0 : -2;
}

bool svgp_posterior_fused_ok(int L, int M, int d) {
    return L >= 1 && L <= 65535 && M >= 1 && M <= MFGP_SMALL_MAX_N && d >= 1 && d <= MFGP_SMALL_MAX_D;
}

int svgp_posterior_predict_fused(cudaStream_t s, const SvgpPosteriorData& q, const double* Xs, int Ns, double* mean,
                                 double* var, long ls, long ns, double* dmean, double* dvar) {
    if (!svgp_posterior_fused_ok(q.L, q.M, q.d)) return -1;
    if (Ns <= 0) return 0;
    const int NT = (q.M + 7) / 8;
    const SvgpFusedArgs a{q, Xs, Ns, groups_per_cta(Ns, q.L), mean, var, ls, ns};
    const long gx = point_chunks(Ns, a.gpc);
    if (dmean) {
        const SvgpFusedGradArgs ag{a, dmean, dvar};
        const size_t smem = svgp_fused_grad_smem_bytes(NT, q.d);
        return with_nt(NT, [&](auto nt) {
            return launch_fused<svgp_posterior_predict_grad_kernel<decltype(nt)::value>>(s, ag, gx, q.L, smem);
        });
    }
    const size_t smem = svgp_fused_smem_bytes(NT, q.d);
    return with_nt(NT, [&](auto nt) {
        return launch_fused<svgp_posterior_predict_kernel<decltype(nt)::value>>(s, a, gx, q.L, smem);
    });
}

bool svgp_posterior_joint_fused_ok(int L, int M, int d, int Ns) { return svgp_posterior_fused_ok(L, M, d) && Ns <= JOINT_MAX_NS; }

int svgp_posterior_cov_fused(cudaStream_t s, const SvgpPosteriorData& q, const double* Xs, int Ns, double* Sl, long lds) {
    if (!svgp_posterior_joint_fused_ok(q.L, q.M, q.d, Ns)) return -1;
    if (Ns <= 0) return 0;
    const int NT = (q.M + 7) / 8;
    const size_t smem = svgp_joint_smem_bytes(NT, (Ns + 7) / 8, q.d);
    const SvgpJointArgs a{q, Xs, Ns, Sl, lds};
    return with_nt(NT, [&](auto nt) {
        return launch_fused<svgp_posterior_joint_kernel<decltype(nt)::value>>(s, a, 1, q.L, smem);
    });
}
