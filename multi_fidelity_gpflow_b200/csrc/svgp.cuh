// svgp.cuh -- K7/K8 sparse variational GP drivers.
#pragma once
#include "common.cuh"

// Workspaces of the whitened SVGP forward pass for L latents, M inducing points and B rows (svgp.cu).  [L][M][ldM]
// matrices: Kmm (Lm after potrf), Wm = Lm^-1, S (trtri scratch), Lq = tril(q_sqrt); [L][M][ldB]: Kmn, A = Wm Kmn,
// C = Lq^T A; [L][B]: knn, g_mean, g_var.
struct Fwd {
    double *Kmm, *Wm, *S, *dinv, *logd, *Kmn, *A, *C, *Lq, *knn, *g_mean, *g_var;
    long ldM, ldB, sMM, sMB;
};
// K_l(Z,Z) + jitter I -> Lm (potrf; per-latent status in info_vec [L] when given) -> f.Wm = Lm^-1 (trtri), and
// f.Lq = tril(q_sqrt).  f.Wm, f.Lq, f.ldM and f.sMM are the caller's; Kmm, S, dinv and logd come from sc.
int svgp_factor(mfgp_handle* h, Scope& sc, int L, int M, int d, double jitter, const double* Z, const double* theta,
                const double* q_sqrt, int* info_vec, Fwd& f);
// From f.Wm and f.Lq: Kmn = K_l(Z,X), knn, A = Wm Kmn, C = Lq^T A and the latent marginals g_mean / g_var [L][B]
// (col_reduce_kernel).  q_mu [M][L].  Buffers of B rows come from sc.
int svgp_conditional(mfgp_handle* h, Scope& sc, int L, int M, int B, int d, const double* X, const double* Z,
                     const double* theta, const double* q_mu, Fwd& f);
// mean / var [B][P] from the latent marginals g_mean / g_var [L][B]: f = g W^T, f_var = g_var (W o W)^T, or f = g when
// W == NULL (L == P).  A fixed l order per output, as the ELBO's mixing.
int launch_svgp_mix(cudaStream_t s, const double* g_mean, const double* g_var, int L, int B, int P, const double* W,
                    double* mean, double* var);

// Cached SVGP posterior (mfgp_svgp_posterior_* in include/mfgp.h).  Every pointer is device memory owned by the posterior.
//   Wm [L][M][ld]  Lm^-1 of K_l(Z,Z) + jitter I: lower triangle, zero above it and in the padding column (ld even)
//   Lq [L][M][ld]  tril(q_sqrt[l]), zero above the diagonal and in the padding column
//   q_mu [M][L]    as the caller passes it (col_reduce_kernel reads it in this layout)
// A latent whose factorisation failed holds NaN on the diagonal of Wm, so both routes predict NaN for it.
struct SvgpPosteriorData {
    int L, M, P, d;
    long ld;
    const double* Z;      // [M, d+1]
    const double* theta;  // [L, 2d+3]
    const double* W;      // [P, L] or nullptr (SeparateIndependent, L == P)
    const double* Wm;
    const double* Lq;
    const double* q_mu;
};
// Fused route (posterior.cu): one kernel for M <= 64, d <= 16.  Writes the latent marginals of point n and latent l
// to mean[l * ls + n * ns] and var[l * ls + n * ns]: (ls, ns) = (1, P) is the [Ns][P] output itself when W == NULL,
// (Ns, 1) the [L][Ns] input of launch_svgp_mix.  With dmean / dvar (both or neither; svgp_posterior_predict_grad_kernel)
// also the latent input gradients d mean / dx*_j and d var / dx*_j at (l * ls + n * ns) * d + j.
bool svgp_posterior_fused_ok(int L, int M, int d);
int svgp_posterior_predict_fused(cudaStream_t s, const SvgpPosteriorData& q, const double* Xs, int Ns, double* mean,
                                 double* var, long ls, long ns, double* dmean = nullptr, double* dvar = nullptr);
// Blocked route (svgp.cu): any size, svgp_conditional and the mix from the cached factors, chunked over Ns.
// mean / var [Ns][P]; with dmean / dvar [Ns][P][d] (both or neither) also the input gradients.
int svgp_posterior_predict_blocked(mfgp_handle* h, const SvgpPosteriorData& q, const double* Xs, int Ns, double* mean,
                                   double* var, double* dmean = nullptr, double* dvar = nullptr);
// dmean / dvar [B][P][d] from the latent gradients gm / gv [L][B][d] as launch_svgp_mix mixes the marginals:
// dmean = sum_l W_pl gm_l, dvar = sum_l W_pl^2 gv_l in a fixed l order, or the gather of latent p when W == NULL.
int launch_svgp_grad_mix(cudaStream_t s, const double* gm, const double* gv, int L, int B, int P, int d, const double* W,
                         double* dmean, double* dvar);

// The shuffled-epoch row stream over a device-resident data set (include/mfgp.h: minibatch stream): X [N][xcols],
// Y [N][ycols] or nullptr.
struct MinibatchStream {
    const double* X;
    int xcols;
    const double* Y;
    int ycols;
    long long N;
    unsigned long long seed;
    long long pos0;
};
// minibatch.cu: Xb [count][xcols] (and Yb) <- the rows of positions pos0 + (*step) B + lo + j, j < count (step nullptr: 0).
int launch_minibatch_gather(cudaStream_t s, const MinibatchStream& ms, const int* step, int B, int lo, int count, double* Xb,
                            double* Yb);
