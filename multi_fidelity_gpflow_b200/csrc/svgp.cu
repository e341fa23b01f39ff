// svgp.cu -- K7/K8: whitened sparse variational GP (shared inducing points) -- ELBO, its
// hand-derived gradient and predict_f, batched over the L latent GPs.
//
// Replaces gpflow SVGP.elbo / prior_kl / predict_f and the GradientTape backward pass as
// driven by the reference (singlebin_svgp.py:79-85 with SeparateIndependent kernels;
// linear_svgp.py:181-190 with LinearCoregionalization).  SURVEY App. A.4-A.6.
//
// Forward (per latent l, all L in one batched launch sequence):
//   Kmm = K_l(Z,Z)+jitter I -> Lm (potrf) -> Wm = Lm^-1 (trtri);  Kmn = K_l(Z,X)
//   A = Wm Kmn;  C = Lq^T A;  g_mean = A^T q_mu,  g_var = knn - colsum(A^2) + colsum(C^2)
//   f = mix(g, W);  VE = Gaussian variational expectations;  ELBO = scale VE - KL
// Backward (loss = -ELBO + (kl_mult-1) KL):
//   fbar -> gbar (and Wbar, likbar) ;  C' = C diag(gbar_var)
//   qmubar = A gbar_mean + kl q_mu ;  Lqbar = tril(2 A C'^T) + kl (Lq - diag(1/Lq_ii))
//   Abar = 2 Lq C' - 2 A diag(gbar_var) + q_mu gbar_mean^T ;  Kmnbar = Wm^T Abar
//   Lmbar = -tril(Kmnbar A^T) ;  Kmmbar = sym( Wm^T Phi(Lm^T Lmbar) Wm )   (Cholesky adjoint)
//   theta/Z gradients: K5 contraction of Kmmbar, Kmnbar, gbar_var with dK recomputed on the fly.
// Every O(M^2 B) / O(M^3) product is a DMMA GEMM (gemm.cu); the rest are streaming kernels.
#include "svgp.cuh"

#include "chol.cuh"
#include "cov.cuh"
#include "gemm.cuh"
#include "gpr.cuh"

namespace {

constexpr double LOG2PI = 1.8378770664093454835606594728112;

__device__ inline double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ inline double block_sum256(double v, double* sh) {  // result valid on thread 0
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x == 0)
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += sh[w];
    __syncthreads();
    return t;
}

// Lq[l][i][j] = tril(q_sqrt[l])  (ld = ldM, zero padded)
__global__ void tril_copy_kernel(const double* __restrict__ q, int M, long ldM, double* __restrict__ Lq) {
    const int l = blockIdx.y;
    const long tot = (long)M * ldM;
    for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < tot; idx += (long)gridDim.x * blockDim.x) {
        const int i = (int)(idx / ldM), j = (int)(idx % ldM);
        Lq[(long)l * tot + idx] = (j <= i && j < M) ? q[((long)l * M + i) * M + j] : 0.0;
    }
}

// g_mean[l][n] = sum_m A[m][n] q_mu[m][l];  g_var[l][n] = knn - sum A^2 + sum C^2
__global__ void col_reduce_kernel(const double* __restrict__ A, const double* __restrict__ Cm, int M, int B, long ldB,
                                  const double* __restrict__ q_mu, int L, const double* __restrict__ knn,
                                  double* __restrict__ g_mean, double* __restrict__ g_var) {
    const int l = blockIdx.y;
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= B) return;
    const double* Al = A + (long)l * M * ldB;
    const double* Cl = Cm + (long)l * M * ldB;
    double sa = 0.0, sc = 0.0, gm = 0.0;
    for (int m = 0; m < M; ++m) {
        const double a = Al[(long)m * ldB + n], c = Cl[(long)m * ldB + n];
        sa = fma(a, a, sa);
        sc = fma(c, c, sc);
        gm = fma(a, q_mu[(long)m * L + l], gm);
    }
    g_mean[(long)l * B + n] = gm;
    g_var[(long)l * B + n] = knn[(long)l * B + n] - sa + sc;
}

// One thread per (n, p).  mode 0: ELBO (writes adjoints fbm/fbv [P][B] + per-block partial sums),
// mode 1: predict (writes mean/var [B][P]).  Likelihood epilogues (cfg->hetero / masked / lik_per_output):
//   Gaussian                 var_eff = lik_var[0]                                   (gpflow Gaussian)
//   HeteroscedasticGaussian  var_eff = lik_var[0] + Y_unc^2, Y = [Y_obs | Y_unc]    (linear_svgp.py:243-267)
//   MaskedGaussian           var_eff = lik_var[p]; entries with Y = NaN contribute nothing
//                            (reference notebooks/"demo: missing output.ipynb" cell 2, class MaskedGaussian)
// lbuf (per-output variances only): d(-ve)/d var_eff per entry, reduced per output by lik_grad_kernel.
__global__ void mix_ve_kernel(int mode, const double* __restrict__ g_mean, const double* __restrict__ g_var, int L,
                              int B, int P, const double* __restrict__ W, const double* __restrict__ Y, int hetero,
                              int masked, const double* __restrict__ lik_var, int per_out, double scale,
                              double* __restrict__ fbm, double* __restrict__ fbv, double* __restrict__ part,
                              double* __restrict__ lbuf, double* __restrict__ mean, double* __restrict__ var) {
    __shared__ double sh[8];
    const long idx = blockIdx.x * (long)blockDim.x + threadIdx.x;
    double ve = 0.0, lb = 0.0;
    if (idx < (long)B * P) {
        const int p = (int)(idx / B), n = (int)(idx % B);
        double fm, fv;
        if (W) {
            fm = 0.0;
            fv = 0.0;
            for (int l = 0; l < L; ++l) {
                const double w = W[(long)p * L + l];
                fm = fma(g_mean[(long)l * B + n], w, fm);
                fv = fma(g_var[(long)l * B + n], w * w, fv);
            }
        } else {
            fm = g_mean[(long)p * B + n];
            fv = g_var[(long)p * B + n];
        }
        if (mode == 1) {
            mean[(long)n * P + p] = fm;
            var[(long)n * P + p] = fv;
        } else {
            const long ldy = hetero ? 2L * P : P;
            const double y = Y[(long)n * ldy + p];
            double bm = 0.0, bv = 0.0;
            if (!(masked && isnan(y))) {
                double ev = lik_var[per_out ? p : 0];
                if (hetero) {
                    const double u = Y[(long)n * ldy + P + p];
                    ev = fma(u, u, ev);
                }
                const double r = y - fm;
                const double q = fma(r, r, fv);
                ve = -0.5 * LOG2PI - 0.5 * log(ev) - 0.5 * q / ev;
                lb = 0.5 / ev - 0.5 * q / (ev * ev);  // d(-ve)/d lik_var
                bm = -scale * r / ev;
                bv = scale * 0.5 / ev;
            }
            fbm[(long)p * B + n] = bm;
            fbv[(long)p * B + n] = bv;
            if (lbuf) lbuf[(long)p * B + n] = lb;
        }
    }
    if (mode == 0) {
        const double a = block_sum256(ve, sh), b = block_sum256(lb, sh);
        if (threadIdx.x == 0) {
            part[2 * blockIdx.x] = a;
            part[2 * blockIdx.x + 1] = b;
        }
    }
}

// dmean[n][p][j] = sum_l W[p][l] gm[l][n][j], dvar[n][p][j] = sum_l W[p][l]^2 gv[l][n][j] (l ascending, as mix_ve_kernel);
// without W output p is latent p.  One thread per (n, p, j).
__global__ void mix_grad_kernel(const double* __restrict__ gm, const double* __restrict__ gv, int L, int B, int P, int d,
                                const double* __restrict__ W, double* __restrict__ dmean, double* __restrict__ dvar) {
    const long idx = blockIdx.x * (long)blockDim.x + threadIdx.x;
    if (idx >= (long)B * P * d) return;
    const int j = (int)(idx % d), p = (int)((idx / d) % P);
    const long n = idx / ((long)d * P);
    double fm, fv;
    if (W) {
        fm = 0.0;
        fv = 0.0;
        for (int l = 0; l < L; ++l) {
            const double w = W[(long)p * L + l];
            const long o = ((long)l * B + n) * d + j;
            fm = fma(gm[o], w, fm);
            fv = fma(gv[o], w * w, fv);
        }
    } else {
        const long o = ((long)p * B + n) * d + j;
        fm = gm[o];
        fv = gv[o];
    }
    dmean[idx] = fm;
    dvar[idx] = fv;
}

// alpha[l][n][0] = sum_{m >= n} Wm[l][m][n] q_mu[m][l] (Wm lower triangular), alpha[l][n][1] = 0: the [L][M][2] table
// posterior_dx_kernel reads as a with P = 1, Pp = 2.
__global__ void svgp_alpha_kernel(const double* __restrict__ Wm, long ldM, const double* __restrict__ q_mu, int M, int L,
                                  double* __restrict__ alpha) {
    const int l = blockIdx.y, n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= M) return;
    const double* W = Wm + (long)l * M * ldM;
    double s = 0.0;
    for (int m = n; m < M; ++m) s = fma(W[(long)m * ldM + n], q_mu[(long)m * L + l], s);
    alpha[((long)l * M + n) * 2] = s;
    alpha[((long)l * M + n) * 2 + 1] = 0.0;
}

// glik[p] = scale * sum_n lbuf[p][n]   (per-output likelihood variances; one block per output, fixed summation order)
__global__ void lik_grad_kernel(const double* __restrict__ lbuf, int B, double scale, double* __restrict__ glik) {
    __shared__ double sh[8];
    const int p = blockIdx.x;
    double s = 0.0;
    for (int n = threadIdx.x; n < B; n += blockDim.x) s += lbuf[(long)p * B + n];
    s = block_sum256(s, sh);
    if (threadIdx.x == 0) glik[p] = scale * s;
}

// gbar_mean[l][n] = sum_p fbm[p][n] W[p][l];  gbar_var[l][n] = sum_p fbv[p][n] W[p][l]^2
__global__ void gbar_kernel(const double* __restrict__ fbm, const double* __restrict__ fbv, int L, int B, int P,
                            const double* __restrict__ W, double* __restrict__ gbm, double* __restrict__ gbv) {
    const int l = blockIdx.y;
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= B) return;
    double a = 0.0, b = 0.0;
    for (int p = 0; p < P; ++p) {
        const double w = W[(long)p * L + l];
        a = fma(fbm[(long)p * B + n], w, a);
        b = fma(fbv[(long)p * B + n], w * w, b);
    }
    gbm[(long)l * B + n] = a;
    gbv[(long)l * B + n] = b;
}

// Wbar[p][l] = sum_n fbm[p][n] g_mean[l][n] + 2 W[p][l] fbv[p][n] g_var[l][n]   (one warp per (p,l))
__global__ void wbar_kernel(const double* __restrict__ fbm, const double* __restrict__ fbv,
                            const double* __restrict__ g_mean, const double* __restrict__ g_var, int L, int B, int P,
                            const double* __restrict__ W, double* __restrict__ gW) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= P * L) return;
    const int p = warp / L, l = warp % L;
    double a = 0.0, b = 0.0;
    for (int n = lane; n < B; n += 32) {
        a = fma(fbm[(long)p * B + n], g_mean[(long)l * B + n], a);
        b = fma(fbv[(long)p * B + n], g_var[(long)l * B + n], b);
    }
    a = warp_sum(a);
    b = warp_sum(b);
    if (lane == 0) gW[(long)p * L + l] = a + 2.0 * W[(long)p * L + l] * b;
}

// Cm[l][m][n] *= gbv[l][n]
__global__ void scale_cols_kernel(double* __restrict__ Cm, int M, int B, long ldB, const double* __restrict__ gbv) {
    const int l = blockIdx.y;
    const long tot = (long)M * ldB;
    for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < tot; idx += (long)gridDim.x * blockDim.x) {
        const int n = (int)(idx % ldB);
        if (n < B) Cm[(long)l * tot + idx] *= gbv[(long)l * B + n];
    }
}

// gqmu[m][l] = klm q_mu[m][l] + sum_n A[l][m][n] gbm[l][n]      (one warp per (m, l))
__global__ void qmu_grad_kernel(const double* __restrict__ A, int M, int B, long ldB, int L,
                                const double* __restrict__ gbm, const double* __restrict__ q_mu, double klm,
                                double* __restrict__ gqmu) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= M * L) return;
    const int l = warp / M, m = warp % M;
    const double* row = A + ((long)l * M + m) * ldB;
    double s = 0.0;
    for (int n = lane; n < B; n += 32) s = fma(row[n], gbm[(long)l * B + n], s);
    s = warp_sum(s);
    if (lane == 0) gqmu[(long)m * L + l] = fma(klm, q_mu[(long)m * L + l], s);
}

// Abar[m][n] += -2 A[m][n] gbv[n] + q_mu[m][l] gbm[n]
__global__ void abar_fix_kernel(double* __restrict__ Abar, const double* __restrict__ A, int M, int B, long ldB, int L,
                                const double* __restrict__ gbm, const double* __restrict__ gbv,
                                const double* __restrict__ q_mu) {
    const int l = blockIdx.y;
    const long tot = (long)M * ldB;
    for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < tot; idx += (long)gridDim.x * blockDim.x) {
        const int m = (int)(idx / ldB), n = (int)(idx % ldB);
        if (n < B) {
            const long o = (long)l * tot + idx;
            Abar[o] += -2.0 * A[o] * gbv[(long)l * B + n] + q_mu[(long)m * L + l] * gbm[(long)l * B + n];
        }
    }
}

// gqsqrt[l][i][j] = tril(2 S1) + klm (Lq - diag(1/Lq_ii))
__global__ void qsqrt_grad_kernel(const double* __restrict__ S1, const double* __restrict__ Lq, int M, long ldM,
                                  double klm, double* __restrict__ gq) {
    const int l = blockIdx.y;
    const long tot = (long)M * M;
    for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < tot; idx += (long)gridDim.x * blockDim.x) {
        const int i = (int)(idx / M), j = (int)(idx % M);
        double v = 0.0;
        if (j <= i) {
            const long o = ((long)l * M + i) * ldM + j;
            const double lq = Lq[o];
            v = 2.0 * S1[o] + klm * (lq - (i == j ? 1.0 / lq : 0.0));
        }
        gq[(long)l * tot + idx] = v;
    }
}

// mode 0: S <- -tril(S);  mode 1: S <- Phi(S) (lower, halved diagonal)
__global__ void tri_mask_kernel(double* __restrict__ S, int M, long ldM, int mode) {
    const int l = blockIdx.y;
    const long tot = (long)M * ldM;
    for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < tot; idx += (long)gridDim.x * blockDim.x) {
        const int i = (int)(idx / ldM), j = (int)(idx % ldM);
        const long o = (long)l * tot + idx;
        double v = 0.0;
        if (j <= i && j < M) {
            v = S[o];
            if (mode == 0) v = -v;
            else if (i == j) v *= 0.5;
        }
        S[o] = v;
    }
}

// Gs = 0.5 (T + T^T)
__global__ void symmetrize_kernel(const double* __restrict__ T, int M, long ldM, double* __restrict__ Gs) {
    const int l = blockIdx.y;
    const long tot = (long)M * ldM;
    for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < tot; idx += (long)gridDim.x * blockDim.x) {
        const int i = (int)(idx / ldM), j = (int)(idx % ldM);
        if (j < M) Gs[(long)l * tot + idx] = 0.5 * (T[(long)l * tot + idx] + T[(long)l * tot + (long)j * ldM + i]);
    }
}

// theta gradient through K_diag(X): knn = [f=0] vL + [f=1] (rho^2 vL + vD)
__global__ void knn_grad_kernel(const double* __restrict__ X, int B, int d, const double* __restrict__ theta,
                                const double* __restrict__ gbv, double* __restrict__ gth /*[L][2d+4]*/) {
    __shared__ double sh[8];
    const int l = blockIdx.x;
    const double* th = theta + (long)l * (2 * d + 3);
    double s0 = 0.0, s1 = 0.0;  // sums of gbv over LF / HF rows
    for (int n = threadIdx.x; n < B; n += blockDim.x) {
        const double fid = X[(long)n * (d + 1) + d];
        const double g = gbv[(long)l * B + n];
        if (fid == 0.0) s0 += g;
        else if (fid == 1.0) s1 += g;
    }
    s0 = block_sum256(s0, sh);
    s1 = block_sum256(s1, sh);
    if (threadIdx.x == 0) {
        const double rho = th[0], vL = th[1 + d];
        double* o = gth + (long)l * (2 * d + 4);
        o[0] += s1 * 2.0 * rho * vL;
        o[1 + d] += s0 + s1 * rho * rho;
        o[2 + 2 * d] += s1;
    }
}

// klpart[l] = 0.5 (sum q_mu[:,l]^2 - M - sum log Lq_ii^2 + sum Lq^2)
__global__ void kl_kernel(const double* __restrict__ q_mu, const double* __restrict__ Lq, int M, long ldM, int L,
                          double* __restrict__ klpart) {
    __shared__ double sh[8];
    const int l = blockIdx.x;
    double s = 0.0;
    for (int m = threadIdx.x; m < M; m += blockDim.x) {
        const double q = q_mu[(long)m * L + l];
        const double dg = Lq[((long)l * M + m) * ldM + m];
        s += q * q - 1.0 - log(dg * dg);
    }
    const long tot = (long)M * ldM;
    for (long idx = threadIdx.x; idx < tot; idx += blockDim.x) {
        const double v = Lq[(long)l * tot + idx];
        s = fma(v, v, s);
    }
    s = block_sum256(s, sh);
    if (threadIdx.x == 0) klpart[l] = 0.5 * s;
}

__global__ void finalize_kernel(const double* __restrict__ part, int nblocks, const double* __restrict__ klpart, int L,
                                double scale, double* elbo, double* kl, double* glik, const double* __restrict__ gth_ws,
                                int d, double* __restrict__ gtheta) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        double ve = 0.0, lb = 0.0, k = 0.0;
        for (int i = 0; i < nblocks; ++i) {
            ve += part[2 * i];
            lb += part[2 * i + 1];
        }
        for (int l = 0; l < L; ++l) k += klpart[l];
        *elbo = scale * ve - k;
        *kl = k;
        if (glik) *glik = scale * lb;
    }
    if (gtheta) {
        const int nq = 2 * d + 3;
        for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < L * nq; idx += gridDim.x * blockDim.x)
            gtheta[idx] = gth_ws[(long)(idx / nq) * (nq + 1) + idx % nq];
    }
}

inline dim3 g2(long total, int L) { return dim3((unsigned)((total + 255) / 256 > 4096 ? 4096 : (total + 255) / 256), L); }

}  // namespace

int svgp_factor(mfgp_handle* h, Scope& sc, int L, int M, int d, double jitter, const double* Z, const double* theta,
                const double* q_sqrt, int* info_vec, Fwd& f) {
    cudaStream_t s = h->stream;
    f.Kmm = sc.alloc<double>((size_t)L * f.sMM);
    f.S = sc.alloc<double>((size_t)L * f.sMM);
    f.dinv = sc.alloc<double>((size_t)chol_dinv_count(M, L));
    f.logd = sc.alloc<double>((size_t)L * M);
    if (!sc.ok) return MFGP_ERR_CUDA;

    CovArgs c{};
    c.Xa = Z; c.Na = M; c.Xb = Z; c.Nb = M; c.d = d;
    c.theta = theta; c.theta_stride = 2 * d + 3;
    c.K = f.Kmm; c.ldk = f.ldM; c.strideK = f.sMM;
    c.symmetric = 1; c.mirror = 0; c.diag_add = jitter;
    c.batch = L;
    if (launch_cov(s, c)) return mfgp_fail(h, MFGP_ERR_CUDA, "svgp: cov(Z,Z) failed");
    CholArgs ch{};
    ch.A = f.Kmm; ch.N = M; ch.lda = f.ldM; ch.strideA = f.sMM; ch.batch = L;
    ch.dinv = f.dinv; ch.logd = f.logd; ch.d_info = h->d_info; ch.aux = h->aux_stream; ch.ev = h->ev; ch.info_vec = info_vec;
    if (launch_potrf(s, ch)) return mfgp_fail(h, MFGP_ERR_CUDA, "svgp: potrf failed");
    if (launch_trtri(s, ch, f.Wm, f.ldM, f.sMM, f.S)) return mfgp_fail(h, MFGP_ERR_CUDA, "svgp: trtri failed");
    tril_copy_kernel<<<g2(f.sMM, L), 256, 0, s>>>(q_sqrt, M, f.ldM, f.Lq);
    return 0;
}

int svgp_conditional(mfgp_handle* h, Scope& sc, int L, int M, int B, int d, const double* X, const double* Z,
                     const double* theta, const double* q_mu, Fwd& f) {
    cudaStream_t s = h->stream;
    f.ldB = round_up(B, 2);
    f.sMB = (long)M * f.ldB;
    f.Kmn = sc.alloc<double>((size_t)L * f.sMB);
    f.A = sc.alloc<double>((size_t)L * f.sMB);
    f.C = sc.alloc<double>((size_t)L * f.sMB);
    f.knn = sc.alloc<double>((size_t)L * B);
    f.g_mean = sc.alloc<double>((size_t)L * B);
    f.g_var = sc.alloc<double>((size_t)L * B);
    if (!sc.ok) return MFGP_ERR_CUDA;

    CovArgs cn{};
    cn.Xa = Z; cn.Na = M; cn.Xb = X; cn.Nb = B; cn.d = d;
    cn.theta = theta; cn.theta_stride = 2 * d + 3;
    cn.K = f.Kmn; cn.ldk = f.ldB; cn.strideK = f.sMB;
    cn.batch = L;
    if (launch_cov(s, cn)) return mfgp_fail(h, MFGP_ERR_CUDA, "svgp: cov(Z,X) failed");
    if (launch_cov_diag(s, X, B, d, theta, 2 * d + 3, f.knn, B, L)) return mfgp_fail(h, MFGP_ERR_CUDA, "svgp: cov_diag failed");

    GemmArgs a;  // A = Wm Kmn
    a.M = M; a.N = B; a.K = M;
    a.A = f.Wm; a.lda = f.ldM; a.strideA = f.sMM;
    a.B = f.Kmn; a.ldb = f.ldB; a.strideB = f.sMB;
    a.C = f.A; a.ldc = f.ldB; a.strideC = f.sMB;
    a.batch = L; a.krange = KR_HI_I;
    if (launch_gemm(s, a)) return mfgp_fail(h, MFGP_ERR_CUDA, "svgp: gemm A failed");
    GemmArgs cc;  // C = Lq^T A
    cc.transA = true;
    cc.M = M; cc.N = B; cc.K = M;
    cc.A = f.Lq; cc.lda = f.ldM; cc.strideA = f.sMM;
    cc.B = f.A; cc.ldb = f.ldB; cc.strideB = f.sMB;
    cc.C = f.C; cc.ldc = f.ldB; cc.strideC = f.sMB;
    cc.batch = L; cc.krange = KR_LO_I;
    if (launch_gemm(s, cc)) return mfgp_fail(h, MFGP_ERR_CUDA, "svgp: gemm C failed");
    col_reduce_kernel<<<dim3((B + 127) / 128, L), 128, 0, s>>>(f.A, f.C, M, B, f.ldB, q_mu, L, f.knn, f.g_mean, f.g_var);
    return 0;
}

int launch_svgp_mix(cudaStream_t s, const double* g_mean, const double* g_var, int L, int B, int P, const double* W,
                    double* mean, double* var) {
    const int nblk = (int)(((long)B * P + 255) / 256);
    mix_ve_kernel<<<nblk, 256, 0, s>>>(1, g_mean, g_var, L, B, P, W, nullptr, 0, 0, nullptr, 0, 1.0, nullptr, nullptr,
                                       nullptr, nullptr, mean, var);
    return cudaGetLastError() == cudaSuccess ? 0 : MFGP_ERR_CUDA;
}

int launch_svgp_grad_mix(cudaStream_t s, const double* gm, const double* gv, int L, int B, int P, int d, const double* W,
                         double* dmean, double* dvar) {
    const long tot = (long)B * P * d;
    if (tot == 0) return 0;
    mix_grad_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, s>>>(gm, gv, L, B, P, d, W, dmean, dvar);
    return cudaGetLastError() == cudaSuccess ? 0 : MFGP_ERR_CUDA;
}

// Cached-posterior prediction for any M, d: per chunk of test points svgp_conditional from the cached Wm and Lq, then the
// mix.  Chunked so that the chunk's Kmn, A and C (and the latent gradients) take at most half of the free device memory.
// The same kernels on the same factors as mfgp_svgp_predict.  With dmean / dvar the chunk goes on from V = f.A and
// U = f.C: R = V - Lq U (into f.A), beta = Wm^T R (into f.Kmn, free by then), and posterior_dx_kernel contracts
// dK_s/dx* with beta and alpha = Wm^T q_mu (formed once per call), one latent per problem; then the gradient mix.
int svgp_posterior_predict_blocked(mfgp_handle* h, const SvgpPosteriorData& q, const double* Xs, int Ns, double* mean,
                                   double* var, double* dmean, double* dvar) {
    cudaStream_t s = h->stream;
    Scope outer(h);
    double* alpha = nullptr;
    if (dmean) {
        alpha = outer.alloc<double>((size_t)q.L * q.M * 2);
        if (!outer.ok) return outer.finish();
        svgp_alpha_kernel<<<dim3((q.M + 127) / 128, q.L), 128, 0, s>>>(q.Wm, q.ld, q.q_mu, q.M, q.L, alpha);
    }
    // the latents as posterior_dx_kernel's problems: inducing points in the place of X, one column of alpha
    const GprPosteriorData ql{q.M, q.d, 1, 2, q.L, q.ld, q.Z, q.theta, nullptr, nullptr, nullptr};
    const size_t per = ((size_t)3 * q.L * q.M + (size_t)3 * q.L + (dmean ? (size_t)2 * q.L * q.d : 0)) * sizeof(double);
    const long chunk = chunk_by_free_memory(per, 2, LONG_MAX);
    for (long n0 = 0; n0 < Ns; n0 += chunk) {
        const int nb = (int)((Ns - n0) < chunk ? (Ns - n0) : chunk);
        Scope inner(h);
        Fwd f{};
        f.Wm = const_cast<double*>(q.Wm);  // read only: svgp_conditional does not write the factors
        f.Lq = const_cast<double*>(q.Lq);
        f.ldM = q.ld;
        f.sMM = (long)q.M * q.ld;
        const double* Xc = Xs + n0 * (q.d + 1);
        MFGP_TRY(svgp_conditional(h, inner, q.L, q.M, nb, q.d, Xc, q.Z, q.theta, q.q_mu, f));
        if (launch_svgp_mix(s, f.g_mean, f.g_var, q.L, nb, q.P, q.W, mean + n0 * q.P, var + n0 * q.P))
            return mfgp_fail(h, MFGP_ERR_CUDA, "svgp posterior: mix launch failed");
        if (!dmean) continue;
        double* gm = inner.alloc<double>((size_t)2 * q.L * nb * q.d);  // latent gradients [L][nb][d], mean then var
        if (!inner.ok) return inner.finish();
        double* gv = gm + (size_t)q.L * nb * q.d;
        GemmArgs r;  // R = V - Lq U, in place of V
        r.M = q.M; r.N = nb; r.K = q.M;
        r.alpha = -1.0; r.beta = 1.0;
        r.A = f.Lq; r.lda = f.ldM; r.strideA = f.sMM;
        r.B = f.C; r.ldb = f.ldB; r.strideB = f.sMB;
        r.C = f.A; r.ldc = f.ldB; r.strideC = f.sMB;
        r.batch = q.L; r.krange = KR_HI_I;
        if (launch_gemm(s, r)) return mfgp_fail(h, MFGP_ERR_CUDA, "svgp posterior: gemm (R) failed");
        GemmArgs bt;  // beta = Wm^T R, into the K_s buffer
        bt.transA = true;
        bt.M = q.M; bt.N = nb; bt.K = q.M;
        bt.A = f.Wm; bt.lda = f.ldM; bt.strideA = f.sMM;
        bt.B = f.A; bt.ldb = f.ldB; bt.strideB = f.sMB;
        bt.C = f.Kmn; bt.ldc = f.ldB; bt.strideC = f.sMB;
        bt.batch = q.L; bt.krange = KR_LO_I;
        if (launch_gemm(s, bt)) return mfgp_fail(h, MFGP_ERR_CUDA, "svgp posterior: gemm (beta) failed");
        if (launch_posterior_dx(s, ql, q.L, Xc, nb, alpha, f.Kmn, f.ldB, gm, gv) ||
            launch_svgp_grad_mix(s, gm, gv, q.L, nb, q.P, q.d, q.W, dmean + n0 * q.P * q.d, dvar + n0 * q.P * q.d))
            return mfgp_fail(h, MFGP_ERR_CUDA, "svgp posterior: gradient launch failed");
    }
    return 0;
}

namespace {

int svgp_forward(mfgp_handle* h, Scope& sc, int L, int M, int B, int d, double jitter, const double* X,
                 const double* Z, const double* theta, const double* q_mu, const double* q_sqrt, Fwd& f) {
    f.ldM = round_up(M, 2);
    f.sMM = (long)M * f.ldM;
    f.Wm = sc.alloc<double>((size_t)L * f.sMM);
    f.Lq = sc.alloc<double>((size_t)L * f.sMM);
    if (!sc.ok) return MFGP_ERR_CUDA;
    MFGP_TRY(svgp_factor(h, sc, L, M, d, jitter, Z, theta, q_sqrt, nullptr, f));
    return svgp_conditional(h, sc, L, M, B, d, X, Z, theta, q_mu, f);
}

}  // namespace

extern "C" {

int mfgp_svgp_elbo_grad(mfgp_handle* h, const mfgp_svgp_cfg* cfg, const double* X, const double* Y, const double* Z,
                        const double* theta, const double* W, const double* q_mu, const double* q_sqrt,
                        double lik_var, double* elbo, double* kl, double* gZ, double* gtheta, double* gW,
                        double* gqmu, double* gqsqrt, double* glik) {
    if (!h) return MFGP_ERR_ARG;
    if (cfg && cfg->lik_per_output)
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_svgp_elbo_grad: per-output likelihood variances need mfgp_svgp_elbo_grad_v");
    return mfgp_svgp_elbo_grad_v(h, cfg, X, Y, Z, theta, W, q_mu, q_sqrt, &lik_var, elbo, kl, gZ, gtheta, gW, gqmu, gqsqrt, glik);
}

int mfgp_svgp_elbo_grad_v(mfgp_handle* h, const mfgp_svgp_cfg* cfg, const double* X, const double* Y, const double* Z,
                          const double* theta, const double* W, const double* q_mu, const double* q_sqrt,
                          const double* lik_var, double* elbo, double* kl, double* gZ, double* gtheta, double* gW,
                          double* gqmu, double* gqsqrt, double* glik) {
    if (!h) return MFGP_ERR_ARG;
    if (!cfg || !X || !Y || !Z || !theta || !q_mu || !q_sqrt || !lik_var || !elbo || !kl)
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_svgp_elbo_grad: NULL argument");
    if (cfg->hetero && cfg->masked)
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_svgp_elbo_grad: hetero and masked likelihoods are exclusive");
    const int L = cfg->L, M = cfg->M, P = cfg->P, B = cfg->B, d = cfg->d;
    if (L < 1 || M < 1 || P < 1 || B < 1 || d < 1 || d > MFGP_MAX_D || (!W && L != P))
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_svgp_elbo_grad: bad configuration");
    const bool want_grad = gZ || gtheta || gqmu || gqsqrt || glik || gW;
    if (want_grad && !(gZ && gtheta && gqmu && gqsqrt && glik && (gW || !W)))
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_svgp_elbo_grad: pass all gradient outputs or none");
    cudaSetDevice(h->device);
    cudaStream_t s = h->stream;
    Scope sc(h);
    const int ycols = cfg->hetero ? 2 * P : P;
    const double* dX = sc.in(X, (size_t)B * (d + 1));
    const double* dY = sc.in(Y, (size_t)B * ycols);
    const double* dZ = sc.in(Z, (size_t)M * (d + 1));
    const double* dth = sc.in(theta, (size_t)L * (2 * d + 3));
    const double* dW = W ? sc.in(W, (size_t)P * L) : nullptr;
    const double* dqm = sc.in(q_mu, (size_t)M * L);
    const double* dqs = sc.in(q_sqrt, (size_t)L * M * M);
    double* delbo = sc.out(elbo, 1);
    double* dkl = sc.out(kl, 1);
    double* dgZ = want_grad ? sc.out(gZ, (size_t)M * (d + 1), true) : nullptr;
    double* dgth = want_grad ? sc.out(gtheta, (size_t)L * (2 * d + 3)) : nullptr;
    double* dgW = (want_grad && W) ? sc.out(gW, (size_t)P * L) : nullptr;
    double* dgqm = want_grad ? sc.out(gqmu, (size_t)M * L) : nullptr;
    double* dgqs = want_grad ? sc.out(gqsqrt, (size_t)L * M * M) : nullptr;
    const int per_out = cfg->lik_per_output ? 1 : 0, nlik = per_out ? P : 1;
    const double* dlv = sc.in(lik_var, nlik);
    double* dglik = want_grad ? sc.out(glik, nlik) : nullptr;
    if (!sc.ok) return sc.finish();

    Fwd f;
    MFGP_TRY(svgp_forward(h, sc, L, M, B, d, cfg->jitter, dX, dZ, dth, dqm, dqs, f));

    const int nblk = (int)(((long)B * P + 255) / 256);
    double* fbm = sc.alloc<double>((size_t)P * B);
    double* fbv = sc.alloc<double>((size_t)P * B);
    double* part = sc.alloc<double>((size_t)2 * nblk);
    double* klpart = sc.alloc<double>(L);
    double* gth_ws = sc.alloc<double>((size_t)L * (2 * d + 4), true);
    double* lbuf = (per_out && want_grad) ? sc.alloc<double>((size_t)P * B) : nullptr;
    if (!sc.ok) return sc.finish();
    mix_ve_kernel<<<nblk, 256, 0, s>>>(0, f.g_mean, f.g_var, L, B, P, dW, dY, cfg->hetero, cfg->masked, dlv, per_out,
                                       cfg->scale, fbm, fbv, part, lbuf, nullptr, nullptr);
    if (lbuf) lik_grad_kernel<<<P, 256, 0, s>>>(lbuf, B, cfg->scale, dglik);
    kl_kernel<<<L, 256, 0, s>>>(dqm, f.Lq, M, f.ldM, L, klpart);

    if (want_grad) {
        const double klm = cfg->kl_mult;
        double *gbm = fbm, *gbv = fbv;  // SeparateIndependent: gbar == fbar (L == P)
        if (dW) {
            gbm = sc.alloc<double>((size_t)L * B);
            gbv = sc.alloc<double>((size_t)L * B);
            if (!sc.ok) return sc.finish();
            gbar_kernel<<<dim3((B + 127) / 128, L), 128, 0, s>>>(fbm, fbv, L, B, P, dW, gbm, gbv);
            wbar_kernel<<<(P * L * 32 + 255) / 256, 256, 0, s>>>(fbm, fbv, f.g_mean, f.g_var, L, B, P, dW, dgW);
        }
        double* Abar = sc.alloc<double>((size_t)L * f.sMB);
        double* Kmnbar = sc.alloc<double>((size_t)L * f.sMB);
        double* S1 = sc.alloc<double>((size_t)L * f.sMM);
        double* S2 = sc.alloc<double>((size_t)L * f.sMM);
        double* T1 = sc.alloc<double>((size_t)L * f.sMM);
        if (!sc.ok) return sc.finish();

        qmu_grad_kernel<<<(M * L * 32 + 255) / 256, 256, 0, s>>>(f.A, M, B, f.ldB, L, gbm, dqm, klm, dgqm);
        scale_cols_kernel<<<g2(f.sMB, L), 256, 0, s>>>(f.C, M, B, f.ldB, gbv);  // C' = C diag(gbar_var)

        GemmArgs g1;  // S1 = A C'^T  (lower tiles)
        g1.transB = true;
        g1.M = M; g1.N = M; g1.K = B;
        g1.A = f.A; g1.lda = f.ldB; g1.strideA = f.sMB;
        g1.B = f.C; g1.ldb = f.ldB; g1.strideB = f.sMB;
        g1.C = S1; g1.ldc = f.ldM; g1.strideC = f.sMM;
        g1.batch = L; g1.lower_only = 1;
        if (launch_gemm(s, g1)) return mfgp_fail(h, MFGP_ERR_CUDA, "svgp: gemm S1 failed");
        qsqrt_grad_kernel<<<g2((long)M * M, L), 256, 0, s>>>(S1, f.Lq, M, f.ldM, klm, dgqs);

        GemmArgs g2a;  // Abar = 2 Lq C'
        g2a.M = M; g2a.N = B; g2a.K = M; g2a.alpha = 2.0;
        g2a.A = f.Lq; g2a.lda = f.ldM; g2a.strideA = f.sMM;
        g2a.B = f.C; g2a.ldb = f.ldB; g2a.strideB = f.sMB;
        g2a.C = Abar; g2a.ldc = f.ldB; g2a.strideC = f.sMB;
        g2a.batch = L; g2a.krange = KR_HI_I;
        if (launch_gemm(s, g2a)) return mfgp_fail(h, MFGP_ERR_CUDA, "svgp: gemm Abar failed");
        abar_fix_kernel<<<g2(f.sMB, L), 256, 0, s>>>(Abar, f.A, M, B, f.ldB, L, gbm, gbv, dqm);

        GemmArgs g3;  // Kmnbar = Wm^T Abar
        g3.transA = true;
        g3.M = M; g3.N = B; g3.K = M;
        g3.A = f.Wm; g3.lda = f.ldM; g3.strideA = f.sMM;
        g3.B = Abar; g3.ldb = f.ldB; g3.strideB = f.sMB;
        g3.C = Kmnbar; g3.ldc = f.ldB; g3.strideC = f.sMB;
        g3.batch = L; g3.krange = KR_LO_I;
        if (launch_gemm(s, g3)) return mfgp_fail(h, MFGP_ERR_CUDA, "svgp: gemm Kmnbar failed");

        GemmArgs g4;  // S2 = Kmnbar A^T (lower tiles) ; Lmbar = -tril(S2)
        g4.transB = true;
        g4.M = M; g4.N = M; g4.K = B;
        g4.A = Kmnbar; g4.lda = f.ldB; g4.strideA = f.sMB;
        g4.B = f.A; g4.ldb = f.ldB; g4.strideB = f.sMB;
        g4.C = S2; g4.ldc = f.ldM; g4.strideC = f.sMM;
        g4.batch = L; g4.lower_only = 1;
        if (launch_gemm(s, g4)) return mfgp_fail(h, MFGP_ERR_CUDA, "svgp: gemm S2 failed");
        tri_mask_kernel<<<g2(f.sMM, L), 256, 0, s>>>(S2, M, f.ldM, 0);

        GemmArgs g5;  // T1 = Lm^T Lmbar (lower tiles) ; Phi
        g5.transA = true;
        g5.M = M; g5.N = M; g5.K = M;
        g5.A = f.Kmm; g5.lda = f.ldM; g5.strideA = f.sMM;  // Kmm buffer holds Lm
        g5.B = S2; g5.ldb = f.ldM; g5.strideB = f.sMM;
        g5.C = T1; g5.ldc = f.ldM; g5.strideC = f.sMM;
        g5.batch = L; g5.krange = KR_LO_MAXIJ; g5.lower_only = 1;
        if (launch_gemm(s, g5)) return mfgp_fail(h, MFGP_ERR_CUDA, "svgp: gemm T1 failed");
        tri_mask_kernel<<<g2(f.sMM, L), 256, 0, s>>>(T1, M, f.ldM, 1);

        GemmArgs g6;  // S1 = Phi Wm   (S1 reused as T2)
        g6.M = M; g6.N = M; g6.K = M;
        g6.A = T1; g6.lda = f.ldM; g6.strideA = f.sMM;
        g6.B = f.Wm; g6.ldb = f.ldM; g6.strideB = f.sMM;
        g6.C = S1; g6.ldc = f.ldM; g6.strideC = f.sMM;
        g6.batch = L; g6.krange = KR_HI_I | KR_LO_J;
        if (launch_gemm(s, g6)) return mfgp_fail(h, MFGP_ERR_CUDA, "svgp: gemm T2 failed");
        GemmArgs g7;  // S2 = Wm^T T2   (S2 reused as T3)
        g7.transA = true;
        g7.M = M; g7.N = M; g7.K = M;
        g7.A = f.Wm; g7.lda = f.ldM; g7.strideA = f.sMM;
        g7.B = S1; g7.ldb = f.ldM; g7.strideB = f.sMM;
        g7.C = S2; g7.ldc = f.ldM; g7.strideC = f.sMM;
        g7.batch = L; g7.krange = KR_LO_I;
        if (launch_gemm(s, g7)) return mfgp_fail(h, MFGP_ERR_CUDA, "svgp: gemm T3 failed");
        symmetrize_kernel<<<g2(f.sMM, L), 256, 0, s>>>(S2, M, f.ldM, T1);  // T1 <- Kmmbar (symmetric)

        // theta / Z gradients
        CovGradArgs cg{};
        cg.Xa = dZ; cg.Na = M; cg.Xb = dZ; cg.Nb = M; cg.d = d;
        cg.theta = dth; cg.theta_stride = 2 * d + 3;
        cg.G = T1; cg.ldg = f.ldM; cg.strideG = f.sMM;
        cg.sym_lower = 0;
        cg.out = gth_ws; cg.out_stride = 2 * d + 4; cg.out_scale = 1.0; cg.accumulate = 0;
        cg.rowgrad = dgZ; cg.rowgrad_stride = 0; cg.rowgrad_scale = 2.0;
        cg.batch = L;
        CovGradArgs cn = cg;
        cn.Xb = dX; cn.Nb = B;
        cn.G = Kmnbar; cn.ldg = f.ldB; cn.strideG = f.sMB;
        cn.accumulate = 1; cn.rowgrad_scale = 1.0;
        const long pc = cov_grad_partial_count(cg) > cov_grad_partial_count(cn) ? cov_grad_partial_count(cg)
                                                                                  : cov_grad_partial_count(cn);
        double* partial = sc.alloc<double>((size_t)pc);
        if (!sc.ok) return sc.finish();
        cg.partial = partial;
        cn.partial = partial;
        if (launch_cov_grad(s, cg)) return mfgp_fail(h, MFGP_ERR_CUDA, "svgp: cov_grad(Z,Z) failed");
        if (launch_cov_grad(s, cn)) return mfgp_fail(h, MFGP_ERR_CUDA, "svgp: cov_grad(Z,X) failed");
        knn_grad_kernel<<<L, 256, 0, s>>>(dX, B, d, dth, gbv, gth_ws);
    }
    finalize_kernel<<<(L * (2 * d + 3) + 255) / 256, 256, 0, s>>>(part, nblk, klpart, L, cfg->scale, delbo, dkl,
                                                                  per_out ? nullptr : dglik, gth_ws, d, dgth);
    return sc.finish();
}

int mfgp_svgp_predict(mfgp_handle* h, const mfgp_svgp_cfg* cfg, const double* Xs, int Ns, const double* Z,
                      const double* theta, const double* W, const double* q_mu, const double* q_sqrt, double* mean,
                      double* var) {
    if (!h) return MFGP_ERR_ARG;
    if (!cfg || !Xs || !Z || !theta || !q_mu || !q_sqrt || !mean || !var)
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_svgp_predict: NULL argument");
    const int L = cfg->L, M = cfg->M, P = cfg->P, d = cfg->d;
    if (L < 1 || M < 1 || P < 1 || Ns < 1 || d < 1 || d > MFGP_MAX_D || (!W && L != P))
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_svgp_predict: bad configuration");
    cudaSetDevice(h->device);
    cudaStream_t s = h->stream;
    Scope sc(h);
    const double* dX = sc.in(Xs, (size_t)Ns * (d + 1));
    const double* dZ = sc.in(Z, (size_t)M * (d + 1));
    const double* dth = sc.in(theta, (size_t)L * (2 * d + 3));
    const double* dW = W ? sc.in(W, (size_t)P * L) : nullptr;
    const double* dqm = sc.in(q_mu, (size_t)M * L);
    const double* dqs = sc.in(q_sqrt, (size_t)L * M * M);
    double* dmean = sc.out(mean, (size_t)Ns * P);
    double* dvar = sc.out(var, (size_t)Ns * P);
    if (!sc.ok) return sc.finish();
    Fwd f;
    MFGP_TRY(svgp_forward(h, sc, L, M, Ns, d, cfg->jitter, dX, dZ, dth, dqm, dqs, f));
    if (launch_svgp_mix(s, f.g_mean, f.g_var, L, Ns, P, dW, dmean, dvar))
        return mfgp_fail(h, MFGP_ERR_CUDA, "mfgp_svgp_predict: mix launch failed");
    return sc.finish();
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// Device-resident Adam loop for the SVGP models (SURVEY 8(f) rank 1): the optimize() loops of
// mfgpflow/singlebin_svgp.py:64-97 and mfgpflow/linear_svgp.py:153-203 (full-batch, Adam + CosineDecay, loss =
// -ELBO + (kl_multiplier - 1) KL) without a host round trip per step.
namespace {
__device__ __forceinline__ double sp_fwd(double u) { return u > 0.0 ? u + log1p(exp(-u)) : log1p(exp(u)); }
// segments of the flat layout: [0, n_theta) softplus; [n_theta, o_lik) identity; [o_lik, n) lik_lower + softplus
__global__ void svgp_constrain_kernel(const double* __restrict__ u, double* __restrict__ c, long n, long n_theta, long o_lik,
                                      double lik_lower) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double x = u[i];
    c[i] = i < n_theta ? sp_fwd(x) : (i >= o_lik ? lik_lower + sp_fwd(x) : x);
}
__global__ void svgp_adam_kernel(double* __restrict__ u, double* __restrict__ m, double* __restrict__ v,
                                 const double* __restrict__ c, const double* __restrict__ g, const unsigned char* __restrict__ mask,
                                 long n, long n_theta, long o_lik, double lik_lower, const double* __restrict__ lr_t,
                                 const int* __restrict__ step_ptr, double b1, double b2, double eps,
                                 const double* __restrict__ elbo_kl, double kl_mult, double* __restrict__ loss_hist,
                                 double* __restrict__ kl_hist) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    const int step = *step_ptr;  // device-side step counter: the same captured graph is replayed for every step
    if (i == 0) {
        if (loss_hist) loss_hist[step] = -elbo_kl[0] + (kl_mult - 1.0) * elbo_kl[1];
        if (kl_hist) kl_hist[step] = elbo_kl[1];
    }
    if (i >= n || (mask && !mask[i])) return;
    double gu = g[i];
    if (i < n_theta) gu *= 1.0 - exp(-c[i]);                       // d softplus
    else if (i >= o_lik) gu *= 1.0 - exp(-(c[i] - lik_lower));     // positive(lower): 1e-6 Gaussian, 0 Heteroscedastic
    double mi = m[i], vi = v[i];
    mi += (gu - mi) * (1.0 - b1);
    vi += (gu * gu - vi) * (1.0 - b2);
    u[i] -= lr_t[step] * mi / (sqrt(vi) + eps);
    m[i] = mi;
    v[i] = vi;
}
__global__ void svgp_step_inc_kernel(int* step) { ++*step; }

// data-parallel bookkeeping after one rank's evaluation: eg[0] <- elbo + kl = scale * VE_local, eg[1] <- kl / nranks, so that
// an all-reduce(sum) over the ranks leaves [scale * VE, KL, gradient of -ELBO + (kl_mult - 1) KL]
__global__ void svgp_dp_fix_kernel(double* eg, double inv_ranks) {
    const double e = eg[0], k = eg[1];
    eg[0] = e + k;
    eg[1] = k * inv_ranks;
}
// loss / KL history from the all-reduced pair: -ELBO + (kl_mult - 1) KL with ELBO = eg[0] - eg[1]
__global__ void svgp_dp_hist_kernel(const double* __restrict__ eg, double* __restrict__ ek) {
    ek[0] = eg[0] - eg[1];
    ek[1] = eg[1];
}

struct FlatLayout {
    long n_theta, o_Z, o_W, o_qm, o_qs, o_lv, n;
    FlatLayout(const mfgp_svgp_cfg* c, int has_W) {
        n_theta = (long)c->L * (2 * c->d + 3);
        o_Z = n_theta;
        o_W = o_Z + (long)c->M * (c->d + 1);
        o_qm = o_W + (has_W ? (long)c->P * c->L : 0);
        o_qs = o_qm + (long)c->M * c->L;
        o_lv = o_qs + (long)c->L * c->M * c->M;
        n = o_lv + (c->lik_per_output ? c->P : 1);
    }
};

struct WorkspaceGuard {  // the loop's workspace mode ends on every exit path (mfgp_workspace, include/mfgp.h)
    mfgp_handle* h;
    bool mine;
    explicit WorkspaceGuard(mfgp_handle* hh) : h(hh), mine(hh->ws.mode == MFGP_WS_POOL) {
        if (mine) mfgp_workspace(h, MFGP_WS_MEASURE, nullptr);  // a caller-chosen mode is left alone
    }
    bool fix() {
        if (!mine) return false;
        if (mfgp_workspace(h, MFGP_WS_FIXED, nullptr) == 0) return true;
        cudaGetLastError();  // no arena (out of memory): the loop goes on with pool allocations, the error must not stick
        h->err[0] = 0;
        return false;
    }
    ~WorkspaceGuard() {
        if (mine) mfgp_workspace(h, MFGP_WS_POOL, nullptr);
    }
};
struct AsyncGuard {  // nested library calls only enqueue; the caller's mode comes back on every exit path
    mfgp_handle* h;
    int was;
    explicit AsyncGuard(mfgp_handle* hh) : h(hh), was(hh->async) { h->async = 1; }
    ~AsyncGuard() { h->async = was; }
};
}  // namespace

namespace {
// The loop of mfgp_svgp_adam and mfgp_svgp_adam_minibatch.  Without a stream (mb == nullptr) every step evaluates the cfg->B
// rows of X, Y; with one, X, Y hold the N = mb->N rows of the data set and each step first gathers its cfg->B rows of the
// shuffled stream into batch buffers (positions mb->pos0 + step * B ...), reading the device step counter.
int svgp_adam_loop(mfgp_handle* h, const char* who, const mfgp_svgp_cfg* cfg, const double* X, const double* Y,
                   const MinibatchStream* mb, int has_W, double* u, double* m, double* v, const unsigned char* mask,
                   const double* lr_t, double beta1, double beta2, double eps, int nsteps, double* loss_hist, double* kl_hist) {
    if (!h) return MFGP_ERR_ARG;
    if (!cfg || !X || !Y || !u || !m || !v || !lr_t || nsteps < 0) return mfgp_fail(h, MFGP_ERR_ARG, "%s: NULL argument", who);
    const int L = cfg->L, M = cfg->M, P = cfg->P, B = cfg->B, d = cfg->d;
    if (L < 1 || M < 1 || P < 1 || B < 1 || d < 1 || d > MFGP_MAX_D || (!has_W && L != P))
        return mfgp_fail(h, MFGP_ERR_ARG, "%s: bad configuration", who);
    if (mb && (mb->N < B || mb->pos0 < 0)) return mfgp_fail(h, MFGP_ERR_ARG, "%s: need 1 <= B <= N and pos0 >= 0", who);
    if (nsteps == 0) return 0;
    cudaSetDevice(h->device);
    cudaStream_t s = h->stream;
    const long n_theta = (long)L * (2 * d + 3), n_Z = (long)M * (d + 1), n_W = has_W ? (long)P * L : 0, n_qm = (long)M * L,
               n_qs = (long)L * M * M, n_lv = cfg->lik_per_output ? P : 1;
    const long o_Z = n_theta, o_W = o_Z + n_Z, o_qm = o_W + n_W, o_qs = o_qm + n_qm, o_lv = o_qs + n_qs, n = o_lv + n_lv;
    const int ycols = cfg->hetero ? 2 * P : P;
    int rc = 0;
    Scope sc(h);
    const size_t rows = mb ? (size_t)mb->N : (size_t)B;
    const double* dX = sc.in(X, rows * (d + 1));
    const double* dY = sc.in(Y, rows * ycols);
    double* Xb = mb ? sc.alloc<double>((size_t)B * (d + 1)) : nullptr;  // the step's batch, filled by the gather
    double* Yb = mb ? sc.alloc<double>((size_t)B * ycols) : nullptr;
    const double* dlr = sc.in(lr_t, nsteps);
    const unsigned char* dmask = mask ? sc.in(mask, (size_t)n) : nullptr;
    double* du = sc.inout(u, (size_t)n);
    double* dm = sc.inout(m, (size_t)n);
    double* dv = sc.inout(v, (size_t)n);
    double* dl = loss_hist ? sc.out(loss_hist, nsteps) : nullptr;
    double* dk = kl_hist ? sc.out(kl_hist, nsteps) : nullptr;
    double* c = sc.alloc<double>((size_t)n);
    double* g = sc.alloc<double>((size_t)n, true);
    double* ek = sc.alloc<double>(2);
    int* dstep = sc.alloc<int>(1, true);
    if (!sc.ok) return sc.finish();
    const int tb = 256;
    const unsigned gb = (unsigned)((n + tb - 1) / tb);
    {
        AsyncGuard guard(h);  // the nested evaluations only enqueue: all their pointers are device memory
        WorkspaceGuard wsg(h);  // step 0 measures the step's temporaries; the captured step takes them from one arena
        const MinibatchStream ds = mb ? MinibatchStream{dX, d + 1, dY, ycols, mb->N, mb->seed, mb->pos0} : MinibatchStream{};
        auto one_step = [&]() -> int {
            if (mb && launch_minibatch_gather(s, ds, dstep, B, 0, B, Xb, Yb))
                return mfgp_fail(h, MFGP_ERR_CUDA, "%s: gather launch failed", who);
            svgp_constrain_kernel<<<gb, tb, 0, s>>>(du, c, n, n_theta, o_lv, cfg->lik_lower);
            int r = mfgp_svgp_elbo_grad_v(h, cfg, mb ? Xb : dX, mb ? Yb : dY, c + o_Z, c, has_W ? c + o_W : nullptr, c + o_qm,
                                          c + o_qs, c + o_lv, ek, ek + 1, g + o_Z, g, has_W ? g + o_W : nullptr, g + o_qm,
                                          g + o_qs, g + o_lv);
            svgp_adam_kernel<<<gb, tb, 0, s>>>(du, dm, dv, c, g, dmask, n, n_theta, o_lv, cfg->lik_lower, dlr, dstep, beta1, beta2,
                                               eps, ek, cfg->kl_mult, dl, dk);
            svgp_step_inc_kernel<<<1, 1, 0, s>>>(dstep);
            return r;
        };
        // Step 0 runs eagerly (first-call attribute settings, pool growth).  The remaining steps replay ONE captured CUDA
        // graph of a whole step (~60 kernels for the small models, where launch latency dominates); if anything in the
        // step is not capturable the loop falls back to eager launches.
        rc = one_step();
        int done = 1;
        if (rc == 0 && nsteps > 2) {
            cudaGraph_t graph = nullptr;
            cudaGraphExec_t exec = nullptr;
            wsg.fix();  // no allocation nodes in the graph (if the arena cannot be had the capture still works, see below)
            bool ok = cudaStreamBeginCapture(s, cudaStreamCaptureModeRelaxed) == cudaSuccess;
            if (ok) {
                const int r = one_step();
                ok = (cudaStreamEndCapture(s, &graph) == cudaSuccess) && r == 0 && graph != nullptr;
            }
            if (ok) ok = cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess;
            if (ok) {
                for (; done < nsteps && ok; ++done) ok = cudaGraphLaunch(exec, s) == cudaSuccess;
                if (!ok) rc = mfgp_fail(h, MFGP_ERR_CUDA, "%s: graph launch failed", who);
            } else {
                cudaGetLastError();  // capture not possible: clear the error, run eagerly
            }
            if (exec) cudaGraphExecDestroy(exec);
            if (graph) cudaGraphDestroy(graph);
            // Temporaries that did not come from the arena were captured as graph-owned allocations, which the driver keeps
            // reserved after the graph is destroyed (include/mfgp.h: mfgp_workspace).  Hand them back once the replays
            // have drained.
            if ((exec || graph) && (h->ws.mode != MFGP_WS_FIXED || h->ws.spilled)) {
                cudaStreamSynchronize(s);
                cudaDeviceGraphMemTrim(h->device);
            }
        }
        for (; done < nsteps && rc == 0; ++done) rc = one_step();
    }
    if (rc) return rc;
    return sc.finish();
}
}  // namespace

extern "C" int mfgp_svgp_adam(mfgp_handle* h, const mfgp_svgp_cfg* cfg, const double* X, const double* Y, int has_W, double* u,
                              double* m, double* v, const unsigned char* mask, const double* lr_t, double beta1, double beta2,
                              double eps, int nsteps, double* loss_hist, double* kl_hist) {
    return svgp_adam_loop(h, "mfgp_svgp_adam", cfg, X, Y, nullptr, has_W, u, m, v, mask, lr_t, beta1, beta2, eps, nsteps,
                          loss_hist, kl_hist);
}

extern "C" int mfgp_svgp_adam_minibatch(mfgp_handle* h, const mfgp_svgp_cfg* cfg, const double* X, const double* Y, int N,
                                        unsigned long long seed, long long pos0, int has_W, double* u, double* m, double* v,
                                        const unsigned char* mask, const double* lr_t, double beta1, double beta2, double eps,
                                        int nsteps, double* loss_hist, double* kl_hist) {
    MinibatchStream mb{};  // the stream's data pointers and column counts are the loop's device copies of X and Y
    mb.N = N;
    mb.seed = seed;
    mb.pos0 = pos0;
    return svgp_adam_loop(h, "mfgp_svgp_adam_minibatch", cfg, X, Y, &mb, has_W, u, m, v, mask, lr_t, beta1, beta2, eps, nsteps,
                          loss_hist, kl_hist);
}

// ---------------------------------------------------------------------------------------------
// Building blocks of the DATA-PARALLEL device loop (SURVEY 8(e) row 2; reference loops singlebin_svgp.py:79-85,
// linear_svgp.py:181-190): rows of the minibatch shard across ranks, every rank runs
//     mfgp_svgp_constrain -> mfgp_svgp_elbo_grad_flat -> [all-reduce(sum) of eg, in place, by the caller] -> mfgp_svgp_adam_update
// on device memory only; nothing is staged through the host and none of the three calls synchronises.
extern "C" long mfgp_svgp_flat_size(const mfgp_svgp_cfg* cfg, int has_W) { return cfg ? FlatLayout(cfg, has_W).n : -1; }

static int svgp_dp_check(mfgp_handle* h, const mfgp_svgp_cfg* cfg, int has_W, const char* who) {
    if (!cfg) return mfgp_fail(h, MFGP_ERR_ARG, "%s: NULL cfg", who);
    if (cfg->L < 1 || cfg->M < 1 || cfg->P < 1 || cfg->B < 1 || cfg->d < 1 || cfg->d > MFGP_MAX_D || (!has_W && cfg->L != cfg->P))
        return mfgp_fail(h, MFGP_ERR_ARG, "%s: bad configuration", who);
    return 0;
}

extern "C" int mfgp_svgp_constrain(mfgp_handle* h, const mfgp_svgp_cfg* cfg, int has_W, const double* u, double* c) {
    if (!h) return MFGP_ERR_ARG;
    MFGP_TRY(svgp_dp_check(h, cfg, has_W, "mfgp_svgp_constrain"));
    if (!u || !c || !mfgp_is_device_ptr(u) || !mfgp_is_device_ptr(c))
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_svgp_constrain: u and c must be device pointers");
    cudaSetDevice(h->device);
    const FlatLayout f(cfg, has_W);
    svgp_constrain_kernel<<<(unsigned)((f.n + 255) / 256), 256, 0, h->stream>>>(u, c, f.n, f.n_theta, f.o_lv, cfg->lik_lower);
    CUDA_TRY(h, cudaGetLastError());
    return 0;
}

extern "C" int mfgp_svgp_elbo_grad_flat(mfgp_handle* h, const mfgp_svgp_cfg* cfg, const double* X, const double* Y, int has_W,
                                        const double* c, int nranks, double* eg) {
    if (!h) return MFGP_ERR_ARG;
    MFGP_TRY(svgp_dp_check(h, cfg, has_W, "mfgp_svgp_elbo_grad_flat"));
    if (!X || !Y || !c || !eg || nranks < 1 || !mfgp_is_device_ptr(X) || !mfgp_is_device_ptr(Y) || !mfgp_is_device_ptr(c) ||
        !mfgp_is_device_ptr(eg))
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_svgp_elbo_grad_flat: X, Y, c, eg must be device pointers, nranks >= 1");
    const FlatLayout f(cfg, has_W);
    mfgp_svgp_cfg local = *cfg;
    local.kl_mult = cfg->kl_mult / nranks;  // sum over ranks of (-scale VE_r + kl_mult / nranks KL) = -scale VE + kl_mult KL
    double* g = eg + 2;
    int rc;
    {
        AsyncGuard guard(h);
        rc = mfgp_svgp_elbo_grad_v(h, &local, X, Y, c + f.o_Z, c, has_W ? c + f.o_W : nullptr, c + f.o_qm, c + f.o_qs, c + f.o_lv,
                                   eg, eg + 1, g + f.o_Z, g, has_W ? g + f.o_W : nullptr, g + f.o_qm, g + f.o_qs, g + f.o_lv);
    }
    if (rc) return rc;
    svgp_dp_fix_kernel<<<1, 1, 0, h->stream>>>(eg, 1.0 / nranks);
    CUDA_TRY(h, cudaGetLastError());
    return 0;
}

extern "C" int mfgp_svgp_adam_update(mfgp_handle* h, const mfgp_svgp_cfg* cfg, int has_W, double* u, double* m, double* v,
                                     const unsigned char* mask, const double* c, const double* eg, const double* lr_t, int* step,
                                     double beta1, double beta2, double eps, double* loss_hist, double* kl_hist, double* scratch2) {
    if (!h) return MFGP_ERR_ARG;
    MFGP_TRY(svgp_dp_check(h, cfg, has_W, "mfgp_svgp_adam_update"));
    if (!u || !m || !v || !c || !eg || !lr_t || !step || !scratch2)
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_svgp_adam_update: NULL argument");
    cudaSetDevice(h->device);
    const FlatLayout f(cfg, has_W);
    cudaStream_t s = h->stream;
    svgp_dp_hist_kernel<<<1, 1, 0, s>>>(eg, scratch2);
    svgp_adam_kernel<<<(unsigned)((f.n + 255) / 256), 256, 0, s>>>(u, m, v, c, eg + 2, mask, f.n, f.n_theta, f.o_lv, cfg->lik_lower,
                                                                  lr_t, step, beta1, beta2, eps, scratch2, cfg->kl_mult, loss_hist,
                                                                  kl_hist);
    svgp_step_inc_kernel<<<1, 1, 0, s>>>(step);
    CUDA_TRY(h, cudaGetLastError());
    return 0;
}
