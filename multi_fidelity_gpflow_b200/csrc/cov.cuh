// cov.cuh -- K1 covariance assembly and K5 gradient contraction (declarations).
#pragma once
#include <cuda_runtime.h>

#define MFGP_MAX_D 32
#define COV_TILE 64

struct CovArgs {
    const double* Xa;  // [Na, d+1]
    int Na;
    const double* Xb;  // [Nb, d+1]
    int Nb;
    int d;
    const double* theta;  // [batch, theta_stride]
    long theta_stride;
    double* K;  // [batch][Na, ldk]
    long ldk;
    long strideK;
    int symmetric;  // Xa == Xb: only tiles I >= J are computed
    int mirror;     // symmetric only: also write the transposed tile
    double diag_add;                // added on global i == j (symmetric only)
    const double* diag_add_vec;     // optional per-batch value (overrides diag_add)
    int batch;
    // problem count that picks the kernel (streaming or tiled; their results differ in the last bits): the whole call's
    // count when a call is chunked over problems, so that a problem's result does not depend on its chunk.  0: batch
    long route_batch;
};
int launch_cov(cudaStream_t s, const CovArgs& a);
int launch_cov_diag(cudaStream_t s, const double* X, int N, int d, const double* theta, long theta_stride,
                    double* out, long out_stride, int batch);

struct CovGradArgs {
    const double* Xa;
    int Na;
    const double* Xb;
    int Nb;
    int d;
    const double* theta;
    long theta_stride;
    const double* G;  // [batch][Na, ldg] weights: out = sum_ij G_ij dK_ij/dtheta
    long ldg;
    long strideG;
    int sym_lower;    // Xa == Xb, G symmetric with valid LOWER triangle: tiles I>=J, off-diagonal counted twice
    double* partial;  // workspace [batch][ntiles][2d+4]
    double* out;      // [batch][2d+4]: dtheta (2d+3) and sum_i G_ii (sym_lower only, else 0)
    long out_stride;
    double out_scale;   // multiplies every output
    int accumulate;     // out += instead of out =
    double* rowgrad;    // optional [batch][Na, d+1]: += rowgrad_scale * sum_j G_ij dk(a_i,b_j)/da_i   (atomicAdd)
    long rowgrad_stride;
    double rowgrad_scale;
    int batch;
};
long cov_grad_partial_count(const CovGradArgs& a);  // doubles needed in `partial`
int launch_cov_grad(cudaStream_t s, const CovGradArgs& a);
