// gpr.cuh -- exact GPR device-side drivers (all pointers are device pointers).
#pragma once
#include "common.cuh"

// batch problems; problem b: RHS = Y[:, c : c + P] with c = ((b_off + b) * per_batch_cols) % ycols (row stride
// ldy; ycols == 0: c = 0), theta_d[b, 2d+3], noise_d[b].  nlml_d [batch]; grad_d [batch, 2d+4] or nullptr.
int gpr_nlml_grad_device(mfgp_handle* h, Scope& sc, const double* X, const double* Y, long ldy, int per_batch_cols,
                         int b_off, int ycols, int N, int d, int P, int batch, const double* theta_d, const double* noise_d,
                         double* nlml_d, double* grad_d, int* info_vec, long route_batch = 0);
int gpr_predict_device(mfgp_handle* h, Scope& sc, const double* X, const double* Y, int N, int d, int P,
                       const double* Xs, int Ns, const double* theta_d, const double* noise_d, double* mean_d,
                       double* var_d);

// Pieces of the pipeline, shared with the graph-kernel model (graph.cu): workspaces of `batch` problems of size N ...
struct GprFactor {
    double *K, *W, *G, *dinv, *logd, *Yw, *a;
    long ld, strideM;
    int Pp;
};
// want_W = false (value only): no W / G buffers (2 N^2 doubles less), and gpr_factor_from_K skips the triangular inverse.
int gpr_factor_alloc(mfgp_handle* h, Scope& sc, int N, int P, int batch, GprFactor& f, bool want_W = true);
// ... K (lower triangle valid, noise included) -> L, W = L^-1, a = W Y; without W: a = L^-1 Y by blocked forward
// substitution over the 128-blocks with the diagonal-block inverses potrf leaves behind (N^2 P flops instead of N^3 / 3) ...
int gpr_factor_from_K(mfgp_handle* h, const double* Y, long ldy, int per_batch_cols, int b_off, int ycols, int N, int P,
                      int batch, int* info_vec, GprFactor& f);
// out <- L^-1 rhs (rhs destroyed) by blocked forward substitution; see gpr.cu.
int gpr_forward_subst(mfgp_handle* h, const GprFactor& f, int N, int batch, double* rhs, double* out, int cols, long ld,
                      long stride);
// ... nlml = 1/2 |a|^2 + P sum log L_ii + N P / 2 log 2 pi ...
void gpr_nlml_from_factor(mfgp_handle* h, const GprFactor& f, int N, int P, int batch, double* nlml_d);
// ... and f.G (lower tiles) <- alpha alpha^T - P K^-1.
int gpr_build_G(mfgp_handle* h, Scope& sc, int N, int P, int batch, GprFactor& f);
// Assemble (K1 + noise) -> factor -> (want_W) W = L^-1 -> a = W Y for `batch` problems, RHS columns as in
// gpr_nlml_grad_device.  theta_d [batch, 2d+3] and noise_d [batch] are device arrays; buffers come from `sc`.  A call
// chunked over problems passes its whole problem count as route_batch (CovArgs::route_batch).
int gpr_factor(mfgp_handle* h, Scope& sc, const double* X, const double* Y, long ldy, int per_batch_cols, int b_off,
               int ycols, int N, int d, int P, int batch, const double* theta_d, const double* noise_d, int* info_vec,
               GprFactor& f, bool want_W = true, long route_batch = 0);

// Cached posterior of B exact GPs that share X (mfgp_gpr_posterior_* in include/mfgp.h).  The storage format both predict
// routes read; every pointer is device memory owned by the posterior.
//   W [B][N][ld]  W = L^-1 of K + noise I: lower triangle; zero above the diagonal and in the padding column (ld even)
//   a [B][N][Pp]  a = W Y (Pp = round_up(P, 2), padding column zero)
// A problem whose factorisation failed holds NaN on the diagonal of W and in all of a, so both routes predict NaN for it.
struct GprPosteriorData {
    int N, d, P, Pp, B;
    long ld;
    const double* X;      // [N, d+1]
    const double* theta;  // [B, 2d+3]
    const double* noise;  // [B]
    const double* W;
    const double* a;
};
// mean [B][Ns][P], var [B][Ns]; with dmean [B][Ns][P][d] and dvar [B][Ns][d] (both or neither) also the gradients with
// respect to the d continuous coordinates of each test point (mfgp_gpr_posterior_predict_grad).  All device pointers.
// Fused route (posterior.cu): one kernel, N <= 64, d <= 16, P <= 64 (gpr_posterior_fused_ok).
bool gpr_posterior_fused_ok(int N, int d, int P);
int gpr_posterior_predict_fused(cudaStream_t s, const GprPosteriorData& q, const double* Xs, int Ns, double* mean,
                                double* var, double* dmean = nullptr, double* dvar = nullptr);
// Joint outputs (mfgp_gpr_posterior_predict_cov / _sample), device pointers.  SP == 0: cov [B][Ns][Ns].  SP = S * P > 0:
// samples [B][Ns][SP] = mean + L z with L L^T = Sigma + jitter I, z [B][Ns][SP], info [B] zeroed by the caller.
struct GprJointOut {
    double* cov;
    long SP;
    double jitter;
    const double* z;
    double* samples;
    int* info;
    bool mean_var_given;  // mean and var were computed by _predict's own route (the fused kernel): the chunks only read them
};
// Fused joint route (posterior.cu): gpr_posterior_fused_ok and Ns <= 64, one kernel.  mean [B][Ns][P] is written for
// _predict_cov only; a failed factor is also CAS'ed into d_info.
bool gpr_posterior_joint_fused_ok(int N, int d, int P, int Ns);
int gpr_posterior_joint_fused(cudaStream_t s, const GprPosteriorData& q, const double* Xs, int Ns, double* mean,
                              const GprJointOut& j, int* d_info);
// Blocked route (gpr.cu): any size, built from K1 / cov_diag / the batched GEMM, chunked over problems.  With `joint` the
// chunk goes on to the joint outputs; mean and var are then required, full-size workspaces or outputs.
int gpr_posterior_predict_blocked(mfgp_handle* h, const GprPosteriorData& q, const double* Xs, int Ns, double* mean,
                                  double* var, double* dmean = nullptr, double* dvar = nullptr,
                                  const GprJointOut* joint = nullptr);
// The tail of the blocked joint route, shared with the SVGP posterior (api.cu), for nb problems of Sigma [nb][Ns][lds]
// whose lower triangle is valid off the diagonal.  launch_joint_diag: the diagonal <- var [nb][Ns] + jitter; with cov
// [nb][Ns][Ns], cov <- Sigma with var on the diagonal, the lower triangle mirrored (Sigma itself keeps its diagonal).
// gpr_joint_sample: the diagonal <- var + jitter, L L^T = Sigma (potrf, in place), samples [nb][Ns][SP] = L z + mean for
// z [nb][Ns][SP] and mean [nb][Ns][P] (column c takes mean column c % P).  info [nb], zeroed by the caller, gets each
// problem's 1-based failed pivot, whose samples are then NaN; the first failure also reaches h->d_info.
int launch_joint_diag(cudaStream_t s, double* Sg, int Ns, long lds, int nb, const double* var, double jitter, double* cov);
int gpr_joint_sample(mfgp_handle* h, Scope& sc, double* Sg, int Ns, long lds, int nb, const double* var, double jitter,
                     const double* z, long SP, int P, const double* mean, double* samples, int* info);
// The input-gradient contraction of the blocked route (posterior.cu) for nb problems of q (theta from q.theta):
// dmean[b][s][p][j] = sum_n alpha[b][n][p] dk_sn/dx_sj, dvar[b][s][j] = -2 sum_n beta[b][n][s] dk_sn/dx_sj, with
// alpha [nb][N][q.Pp] = W^T a and beta [nb][N][ldb] = K^-1 K_s.
int launch_posterior_dx(cudaStream_t s, const GprPosteriorData& q, int nb, const double* Xs, int Ns, const double* alpha,
                        const double* beta, long ldb, double* dmean, double* dvar);
