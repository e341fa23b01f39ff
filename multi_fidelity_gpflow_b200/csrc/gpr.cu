// gpr.cu -- exact multi-fidelity GPR drivers: NLML, analytic gradient, prediction.
//
// Pipeline (all fp64, batched over independent problems):
//   K1 cov (lower tiles + noise)  ->  K2 potrf  ->  K4 trtri: W = L^-1
//   a = W Y, nlml = 1/2 |a|^2 + P sum log L_ii + NP/2 log 2pi          (GPflow logdensities.multivariate_normal)
//   alpha = W^T a,  G = alpha alpha^T - P W^T W  (lower tiles)  ->  K5 contraction with dK/dtheta
// Replaces GPR.log_marginal_likelihood / tape.gradient / predict_f behind
// MultiFidelityGPModel (reference mfgpflow/linear.py:148-156, :203-209; SURVEY App. A.2-A.3).
#include "gpr.cuh"

#include "chol.cuh"
#include "cov.cuh"
#include "gemm.cuh"

namespace {

constexpr double LOG2PI = 1.8378770664093454835606594728112;

// Yw[b][i][p] = Y[i*ldy + col0(b) + p]  (zero padded to Pp columns); col0(b) = ((b_off + b) * per_batch_cols) % ycols
__global__ void pack_rhs_kernel(const double* __restrict__ Y, long ldy, int N, int P, int Pp, int per_batch_cols,
                                int b_off, int ycols, double* __restrict__ Yw) {
    const int b = blockIdx.y;
    const long col0 = ycols > 0 ? ((long)(b_off + b) * per_batch_cols) % ycols : 0;
    const long tot = (long)N * Pp;
    for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < tot; idx += (long)gridDim.x * blockDim.x) {
        const int i = (int)(idx / Pp), pcol = (int)(idx % Pp);
        Yw[(long)b * tot + idx] = pcol < P ? Y[(long)i * ldy + col0 + pcol] : 0.0;
    }
}

__device__ inline double block_sum(double v, double* sh) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x == 0)
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += sh[w];
    __syncthreads();
    return t;  // valid on thread 0
}

__global__ void nlml_kernel(const double* __restrict__ a, int N, int Pp, int P, const double* __restrict__ logd,
                            double* __restrict__ out) {
    __shared__ double sh[8];
    const int b = blockIdx.x;
    double q = 0.0, ld = 0.0;
    const double* ab = a + (long)b * N * Pp;
    for (long i = threadIdx.x; i < (long)N * Pp; i += blockDim.x) q = fma(ab[i], ab[i], q);
    for (int i = threadIdx.x; i < N; i += blockDim.x) ld += logd[(long)b * N + i];
    q = block_sum(q, sh);
    ld = block_sum(ld, sh);
    if (threadIdx.x == 0) out[b] = 0.5 * q + P * ld + 0.5 * (double)N * P * LOG2PI;
}

// var[b][j] = kss[b][j] - sum_i As[b][i][j]^2  (problem b = blockIdx.y; As stride strideA, kss / var stride Ns)
__global__ void predict_var_kernel(const double* __restrict__ As, int N, int Ns, long ld, const double* __restrict__ kss,
                                   double* __restrict__ var, long strideA) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= Ns) return;
    const long b = blockIdx.y;
    As += b * strideA;
    double s = 0.0;
    for (int i = 0; i < N; ++i) {
        const double v = As[(long)i * ld + j];
        s = fma(v, v, s);
    }
    var[b * Ns + j] = kss[b * Ns + j] - s;
}

// Sigma's diagonal <- var (+ jitter for the factorisation); with cov, the whole matrix out: the lower triangle, mirrored.
__global__ void joint_diag_kernel(double* __restrict__ Sg, int Ns, long lds, const double* __restrict__ var, double jitter,
                                  double* __restrict__ cov) {
    const long b = blockIdx.y;
    double* S = Sg + b * Ns * lds;
    const double* v = var + b * Ns;
    if (!cov) {
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < Ns; i += gridDim.x * blockDim.x) S[(long)i * lds + i] = v[i] + jitter;
        return;
    }
    double* c = cov + b * Ns * Ns;
    for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < (long)Ns * Ns; idx += (long)gridDim.x * blockDim.x) {
        const long i = idx / Ns, j = idx - i * Ns;
        c[idx] = i == j ? v[i] : (i > j ? S[i * lds + j] : S[j * lds + i]);
    }
}

// samples [nb][Ns][SP] (holding L z) += mean [nb][Ns][P] broadcast over the S draws; NaN for a problem whose factor failed.
__global__ void joint_sample_epilogue_kernel(double* __restrict__ out, int Ns, long SP, int P, const double* __restrict__ mean,
                                             const int* __restrict__ info) {
    const long b = blockIdx.y, per = (long)Ns * SP;
    const bool bad = info[b] != 0;
    const double qnan = __longlong_as_double(0x7ff8000000000000ll);
    double* o = out + b * per;
    const double* m = mean + b * Ns * P;
    for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < per; idx += (long)gridDim.x * blockDim.x) {
        const long i = idx / SP, col = idx - i * SP;
        o[idx] = bad ? qnan : o[idx] + m[i * P + col % P];
    }
}

// The joint outputs of nb problems (from b0) of the blocked route, from the chunk's A_s = W K_s [nb][N][lds], var and mean:
// K_ss (K1, symmetric), Sigma = K_ss - A_s^T A_s (lower tiles), diag <- var.  _predict_cov mirrors Sigma into cov;
// _sample goes on in gpr_joint_sample.
int joint_chunk(mfgp_handle* h, Scope& sc, const GprPosteriorData& q, long b0, int nb, const double* Xs, int Ns,
                const double* th, const double* As, long lds, const double* var, const double* mean, const GprJointOut& j) {
    cudaStream_t s = h->stream;
    const int np = 2 * q.d + 3, N = q.N;    double* Sg = sc.alloc<double>((size_t)nb * Ns * lds, true);
    if (!sc.ok) return sc.finish();
    CovArgs k{};
    k.Xa = Xs; k.Na = Ns; k.Xb = Xs; k.Nb = Ns; k.d = q.d;
    k.theta = th; k.theta_stride = np;
    k.K = Sg; k.ldk = lds; k.strideK = (long)Ns * lds;
    k.symmetric = 1;
    k.batch = nb; k.route_batch = q.B;
    if (launch_cov(s, k)) return mfgp_fail(h, MFGP_ERR_CUDA, "cov launch (K_ss) failed");
    GemmArgs g;  // Sigma = K_ss - A_s^T A_s
    g.transA = true;
    g.M = Ns; g.N = Ns; g.K = N;
    g.alpha = -1.0; g.beta = 1.0;
    g.A = As; g.lda = lds; g.strideA = (long)N * lds;
    g.B = As; g.ldb = lds; g.strideB = (long)N * lds;
    g.C = Sg; g.ldc = lds; g.strideC = (long)Ns * lds;
    g.batch = nb;
    g.lower_only = 1;
    if (launch_gemm(s, g)) return mfgp_fail(h, MFGP_ERR_CUDA, "gemm (Sigma) failed");
    if (!j.SP) {
        if (launch_joint_diag(s, Sg, Ns, lds, nb, var, 0.0, j.cov + b0 * Ns * Ns))
            return mfgp_fail(h, MFGP_ERR_CUDA, "joint_diag_kernel launch failed");
        return 0;
    }
    return gpr_joint_sample(h, sc, Sg, Ns, lds, nb, var, j.jitter, j.z + b0 * Ns * j.SP, j.SP, q.P, mean,
                            j.samples + b0 * Ns * j.SP, j.info + b0);
}

}  // namespace

int launch_joint_diag(cudaStream_t s, double* Sg, int Ns, long lds, int nb, const double* var, double jitter, double* cov) {
    const long work = cov ? (long)Ns * Ns : Ns;
    const dim3 dgrid((unsigned)((work + 255) / 256 < 64 ? (work + 255) / 256 : 64), (unsigned)nb);
    joint_diag_kernel<<<dgrid, 256, 0, s>>>(Sg, Ns, lds, var, jitter, cov);
    return cudaGetLastError() == cudaSuccess ? 0 : MFGP_ERR_CUDA;
}

int gpr_joint_sample(mfgp_handle* h, Scope& sc, double* Sg, int Ns, long lds, int nb, const double* var, double jitter,
                     const double* z, long SP, int P, const double* mean, double* samples, int* info) {
    cudaStream_t s = h->stream;
    if (launch_joint_diag(s, Sg, Ns, lds, nb, var, jitter, nullptr))
        return mfgp_fail(h, MFGP_ERR_CUDA, "joint_diag_kernel launch failed");
    CholArgs ch{};
    ch.A = Sg; ch.N = Ns; ch.lda = lds; ch.strideA = (long)Ns * lds; ch.batch = nb;
    ch.dinv = sc.alloc<double>((size_t)chol_dinv_count(Ns, nb));
    ch.logd = sc.alloc<double>((size_t)nb * Ns);
    const long ldz = round_up(SP, 2);
    double* Zw = sc.alloc<double>((size_t)nb * Ns * ldz);
    if (!sc.ok) return sc.finish();
    ch.d_info = h->d_info; ch.aux = h->aux_stream; ch.ev = h->ev; ch.info_vec = info;
    if (launch_potrf(s, ch)) return mfgp_fail(h, MFGP_ERR_CUDA, "potrf launch (Sigma) failed");
    // the GEMM's TMA operands need an even leading dimension: stage z with ld = round_up(SP, 2)
    CUDA_TRY(h, cudaMemcpy2DAsync(Zw, ldz * sizeof(double), z, SP * sizeof(double), SP * sizeof(double), (size_t)nb * Ns,
                                  cudaMemcpyDeviceToDevice, s));
    constexpr long MAX_COLS = 1L << 30;  // GemmArgs::N is an int
    for (long c0 = 0; c0 < SP; c0 += MAX_COLS) {
        GemmArgs lz;  // samples = L Z (L lower triangular)
        lz.M = Ns; lz.N = (int)(SP - c0 < MAX_COLS ? SP - c0 : MAX_COLS); lz.K = Ns;
        lz.A = Sg; lz.lda = lds; lz.strideA = (long)Ns * lds;
        lz.B = Zw + c0; lz.ldb = ldz; lz.strideB = (long)Ns * ldz;
        lz.C = samples + c0; lz.ldc = SP; lz.strideC = (long)Ns * SP;
        lz.batch = nb;
        lz.krange = KR_HI_I;
        lz.small_tiles = 1;  // one tile shape whatever SP: a column's value does not depend on S
        if (launch_gemm(s, lz)) return mfgp_fail(h, MFGP_ERR_CUDA, "gemm (L Z) failed");
    }
    const long per = (long)Ns * SP;
    const unsigned ex = (unsigned)((per + 255) / 256 < 1024 ? (per + 255) / 256 : 1024);
    joint_sample_epilogue_kernel<<<dim3(ex, (unsigned)nb), 256, 0, s>>>(samples, Ns, SP, P, mean, info);
    return cudaGetLastError() == cudaSuccess ? 0 : mfgp_fail(h, MFGP_ERR_CUDA, "joint_sample_epilogue_kernel launch failed");
}

using Factor = GprFactor;

// Assemble + factor + invert + a = W Y for `batch` problems.  theta_d/noise_d are device arrays.
int gpr_factor(mfgp_handle* h, Scope& sc, const double* X, const double* Y, long ldy, int per_batch_cols, int b_off,
               int ycols, int N, int d, int P, int batch, const double* theta_d, const double* noise_d, int* info_vec,
               Factor& f, bool want_W, long route_batch) {
    MFGP_TRY(gpr_factor_alloc(h, sc, N, P, batch, f, want_W));
    CovArgs c{};
    c.Xa = X; c.Na = N; c.Xb = X; c.Nb = N; c.d = d;
    c.theta = theta_d; c.theta_stride = 2 * d + 3;
    c.K = f.K; c.ldk = f.ld; c.strideK = f.strideM;
    c.symmetric = 1; c.mirror = 0;
    c.diag_add = 0.0; c.diag_add_vec = noise_d;
    c.batch = batch; c.route_batch = route_batch;
    if (launch_cov(h->stream, c)) return mfgp_fail(h, MFGP_ERR_CUDA, "cov launch failed");
    return gpr_factor_from_K(h, Y, ldy, per_batch_cols, b_off, ycols, N, P, batch, info_vec, f);
}

int gpr_factor_alloc(mfgp_handle* h, Scope& sc, int N, int P, int batch, GprFactor& f, bool want_W) {
    f.ld = round_up(N, 2);
    f.strideM = (long)N * f.ld;
    f.Pp = (int)round_up(P, 2);
    f.K = sc.alloc<double>((size_t)batch * f.strideM);
    f.W = want_W ? sc.alloc<double>((size_t)batch * f.strideM) : nullptr;
    f.G = want_W ? sc.alloc<double>((size_t)batch * f.strideM) : nullptr;  // trtri scratch, then G
    f.dinv = sc.alloc<double>((size_t)chol_dinv_count(N, batch));
    f.logd = sc.alloc<double>((size_t)batch * N);
    f.Yw = sc.alloc<double>((size_t)batch * N * f.Pp);
    f.a = sc.alloc<double>((size_t)batch * N * f.Pp);
    (void)h;
    return sc.ok ? 0 : MFGP_ERR_CUDA;
}

// out[batch][N, ld] (cols columns) <- L^-1 rhs, block row by block row: out_k = inv(L_kk) rhs_k with the diagonal-block
// inverses potrf left in f.dinv, then rhs_{k+1:} -= L_{k+1:, k} out_k.  rhs is destroyed; L is read once (4.3 GB at
// N = 32 768).  ld even, both arrays 16-byte aligned (the TMA-fed GEMM's contract).
int gpr_forward_subst(mfgp_handle* h, const GprFactor& f, int N, int batch, double* rhs, double* out, int cols, long ld,
                      long stride) {
    cudaStream_t s = h->stream;
    const long strideD = (long)chol_nblk(N) * CHOL_NB * CHOL_NB;
    for (int k0 = 0; k0 < N; k0 += CHOL_NB) {
        const int nb = N - k0 < CHOL_NB ? N - k0 : CHOL_NB, k1 = k0 + nb;
        GemmArgs t;  // out_k = inv(L_kk) rhs_k
        t.M = nb; t.N = cols; t.K = nb;
        t.A = f.dinv + (long)(k0 / CHOL_NB) * CHOL_NB * CHOL_NB; t.lda = CHOL_NB; t.strideA = strideD;
        t.B = rhs + (long)k0 * ld; t.ldb = ld; t.strideB = stride;
        t.C = out + (long)k0 * ld; t.ldc = ld; t.strideC = stride;
        t.batch = batch;
        if (launch_gemm(s, t)) return mfgp_fail(h, MFGP_ERR_CUDA, "gemm (inv(L_kk) rhs_k) failed");
        if (k1 >= N) break;
        GemmArgs u;  // rhs_{k+1:} -= L_{k+1:, k} out_k
        u.M = N - k1; u.N = cols; u.K = nb;
        u.alpha = -1.0; u.beta = 1.0;
        u.A = f.K + (long)k1 * f.ld + k0; u.lda = f.ld; u.strideA = f.strideM;
        u.B = out + (long)k0 * ld; u.ldb = ld; u.strideB = stride;
        u.C = rhs + (long)k1 * ld; u.ldc = ld; u.strideC = stride;
        u.batch = batch;
        if (launch_gemm(s, u)) return mfgp_fail(h, MFGP_ERR_CUDA, "gemm (forward substitution update) failed");
    }
    return 0;
}

// f.K holds the (lower triangle of the) noisy covariance: potrf -> W = L^-1 -> a = W Y.
int gpr_factor_from_K(mfgp_handle* h, const double* Y, long ldy, int per_batch_cols, int b_off, int ycols, int N, int P,
                      int batch, int* info_vec, GprFactor& f) {
    cudaStream_t s = h->stream;
    CholArgs ch{};
    ch.A = f.K; ch.N = N; ch.lda = f.ld; ch.strideA = f.strideM; ch.batch = batch;
    ch.dinv = f.dinv; ch.logd = f.logd; ch.d_info = h->d_info; ch.aux = h->aux_stream; ch.ev = h->ev; ch.info_vec = info_vec;
    if (launch_potrf(s, ch)) return mfgp_fail(h, MFGP_ERR_CUDA, "potrf launch failed");
    pack_rhs_kernel<<<dim3(64, batch), 256, 0, s>>>(Y, ldy, N, P, f.Pp, per_batch_cols, b_off, ycols, f.Yw);
    if (!f.W)  // value only: a = L^-1 Yw without the N^3 / 3 inverse and without the W and G buffers
        return gpr_forward_subst(h, f, N, batch, f.Yw, f.a, f.Pp, f.Pp, (long)N * f.Pp);
    if (launch_trtri(s, ch, f.W, f.ld, f.strideM, f.G)) return mfgp_fail(h, MFGP_ERR_CUDA, "trtri launch failed");

    GemmArgs g;  // a = W Yw
    g.transA = false; g.transB = false;
    g.M = N; g.N = f.Pp; g.K = N;
    g.A = f.W; g.lda = f.ld; g.strideA = f.strideM;
    g.B = f.Yw; g.ldb = f.Pp; g.strideB = (long)N * f.Pp;
    g.C = f.a; g.ldc = f.Pp; g.strideC = (long)N * f.Pp;
    g.batch = batch;
    g.krange = KR_HI_I;
    if (launch_gemm(s, g)) return mfgp_fail(h, MFGP_ERR_CUDA, "gemm (a = W Y) failed");
    return 0;
}

void gpr_nlml_from_factor(mfgp_handle* h, const GprFactor& f, int N, int P, int batch, double* nlml_d) {
    nlml_kernel<<<batch, 256, 0, h->stream>>>(f.a, N, f.Pp, P, f.logd, nlml_d);
}

// f.G (lower tiles) <- alpha alpha^T - P K^-1 with alpha = W^T a, K^-1 = W^T W
int gpr_build_G(mfgp_handle* h, Scope& sc, int N, int P, int batch, GprFactor& f) {
    cudaStream_t s = h->stream;
    const long strideV = (long)N * f.Pp;
    double* alpha = sc.alloc<double>((size_t)batch * strideV);
    if (!sc.ok) return MFGP_ERR_CUDA;
    GemmArgs g;  // alpha = W^T a
    g.transA = true; g.transB = false;
    g.M = N; g.N = f.Pp; g.K = N;
    g.A = f.W; g.lda = f.ld; g.strideA = f.strideM;
    g.B = f.a; g.ldb = f.Pp; g.strideB = strideV;
    g.C = alpha; g.ldc = f.Pp; g.strideC = strideV;
    g.batch = batch;
    g.krange = KR_LO_I;
    if (launch_gemm(s, g)) return mfgp_fail(h, MFGP_ERR_CUDA, "gemm (alpha) failed");

    GemmArgs o;  // G = alpha alpha^T  (lower tiles)
    o.transA = false; o.transB = true;
    o.M = N; o.N = N; o.K = f.Pp;
    o.A = alpha; o.lda = f.Pp; o.strideA = strideV;
    o.B = alpha; o.ldb = f.Pp; o.strideB = strideV;
    o.C = f.G; o.ldc = f.ld; o.strideC = f.strideM;
    o.batch = batch;
    o.lower_only = 1;
    if (launch_gemm(s, o)) return mfgp_fail(h, MFGP_ERR_CUDA, "gemm (alpha alpha^T) failed");

    GemmArgs k;  // G -= P * W^T W   (K^-1 = L^-T L^-1)
    k.transA = true; k.transB = false;
    k.M = N; k.N = N; k.K = N;
    k.alpha = -(double)P; k.beta = 1.0;
    k.A = f.W; k.lda = f.ld; k.strideA = f.strideM;
    k.B = f.W; k.ldb = f.ld; k.strideB = f.strideM;
    k.C = f.G; k.ldc = f.ld; k.strideC = f.strideM;
    k.batch = batch;
    k.krange = KR_LO_MAXIJ;
    k.lower_only = 1;
    if (launch_gemm(s, k)) return mfgp_fail(h, MFGP_ERR_CUDA, "gemm (W^T W) failed");
    return 0;
}

int gpr_nlml_grad_device(mfgp_handle* h, Scope& sc, const double* X, const double* Y, long ldy, int per_batch_cols,
                         int b_off, int ycols, int N, int d, int P, int batch, const double* theta_d, const double* noise_d,
                         double* nlml_d, double* grad_d, int* info_vec, long route_batch) {
    cudaStream_t s = h->stream;
    Factor f;
    MFGP_TRY(gpr_factor(h, sc, X, Y, ldy, per_batch_cols, b_off, ycols, N, d, P, batch, theta_d, noise_d, info_vec, f, grad_d != nullptr,
                        route_batch));
    gpr_nlml_from_factor(h, f, N, P, batch, nlml_d);
    if (!grad_d) return 0;
    MFGP_TRY(gpr_build_G(h, sc, N, P, batch, f));

    CovGradArgs cg{};
    cg.Xa = X; cg.Na = N; cg.Xb = X; cg.Nb = N; cg.d = d;
    cg.theta = theta_d; cg.theta_stride = 2 * d + 3;
    cg.G = f.G; cg.ldg = f.ld; cg.strideG = f.strideM;
    cg.sym_lower = 1;
    cg.out = grad_d; cg.out_stride = 2 * d + 4;
    cg.out_scale = -0.5;  // d(nlml)/dtheta = -1/2 sum_ij G_ij dK_ij/dtheta
    cg.accumulate = 0;
    cg.rowgrad = nullptr;
    cg.batch = batch;
    cg.partial = sc.alloc<double>((size_t)cov_grad_partial_count(cg));
    if (!sc.ok) return MFGP_ERR_CUDA;
    if (launch_cov_grad(s, cg)) return mfgp_fail(h, MFGP_ERR_CUDA, "cov_grad launch failed");
    return 0;
}

int gpr_predict_device(mfgp_handle* h, Scope& sc, const double* X, const double* Y, int N, int d, int P,
                       const double* Xs, int Ns, const double* theta_d, const double* noise_d, double* mean_d,
                       double* var_d) {
    cudaStream_t s = h->stream;
    Factor f;
    // A_s = L^-1 K_s by forward substitution (N^2 Ns flops in k = 128 updates) beats building W = L^-1 first (N^3 / 3 more
    // flops) for as long as Ns < N: measured at N = 16 384 (scripts/predict_once.py) 61 + 0.0098 Ns ms against
    // 100 + 0.0077 Ns ms for W + one full-rate GEMM.
    const bool want_W = Ns > N;
    MFGP_TRY(gpr_factor(h, sc, X, Y, P, 0, 0, 0, N, d, P, 1, theta_d, noise_d, nullptr, f, want_W));
    const long lds = round_up(Ns, 2);
    double* Ks = sc.alloc<double>((size_t)N * lds);
    double* As = sc.alloc<double>((size_t)N * lds);
    double* kss = sc.alloc<double>((size_t)Ns);
    if (!sc.ok) return MFGP_ERR_CUDA;
    CovArgs c{};
    c.Xa = X; c.Na = N; c.Xb = Xs; c.Nb = Ns; c.d = d;
    c.theta = theta_d; c.theta_stride = 2 * d + 3;
    c.K = Ks; c.ldk = lds; c.strideK = 0;
    c.batch = 1;
    if (launch_cov(s, c)) return mfgp_fail(h, MFGP_ERR_CUDA, "cov launch failed");
    if (launch_cov_diag(s, Xs, Ns, d, theta_d, 0, kss, 0, 1)) return mfgp_fail(h, MFGP_ERR_CUDA, "cov_diag failed");
    if (want_W) {
        GemmArgs g;  // As = W Ks
        g.transA = false; g.transB = false;
        g.M = N; g.N = Ns; g.K = N;
        g.A = f.W; g.lda = f.ld;
        g.B = Ks; g.ldb = lds;
        g.C = As; g.ldc = lds;
        g.krange = KR_HI_I;
        if (launch_gemm(s, g)) return mfgp_fail(h, MFGP_ERR_CUDA, "gemm (As) failed");
    } else {
        MFGP_TRY(gpr_forward_subst(h, f, N, 1, Ks, As, Ns, lds, 0));
    }
    predict_var_kernel<<<(Ns + 127) / 128, 128, 0, s>>>(As, N, Ns, lds, kss, var_d, 0);
    GemmArgs m;  // mean = As^T a
    m.transA = true; m.transB = false;
    m.M = Ns; m.N = P; m.K = N;
    m.A = As; m.lda = lds;
    m.B = f.a; m.ldb = f.Pp;
    m.C = mean_d; m.ldc = P;
    if (launch_gemm(s, m)) return mfgp_fail(h, MFGP_ERR_CUDA, "gemm (mean) failed");
    return 0;
}

// Cached-posterior prediction for any N, d, P: per chunk of problems  K_s = K(X, Xs) (K1, batched rectangular), k_ss,
// A_s = W K_s, var = k_ss - colsum(A_s^2), mean = A_s^T a.  Chunked so that K_s and A_s of a chunk take at most half of
// the free device memory.  With dmean / dvar the chunk goes on from the same A_s: beta = W^T A_s = K^-1 K_s (into the
// K_s buffer, which is free by then), alpha = W^T a, and posterior_dx_kernel contracts dK_s/dx* with both.
int gpr_posterior_predict_blocked(mfgp_handle* h, const GprPosteriorData& q, const double* Xs, int Ns, double* mean,
                                  double* var, double* dmean, double* dvar, const GprJointOut* joint) {
    cudaStream_t s = h->stream;
    const int np = 2 * q.d + 3, N = q.N;
    const long lds = round_up(Ns, 2);
    size_t per = ((size_t)2 * N * lds + Ns + (dmean ? (size_t)N * q.Pp : 0)) * sizeof(double);
    if (joint)  // Sigma, and for _sample potrf's workspaces and the staged z
        per += ((size_t)Ns * lds + (joint->SP ? (size_t)chol_dinv_count(Ns, 1) + Ns + (size_t)Ns * round_up(joint->SP, 2) : 0)) *
               sizeof(double);
    const long chunk = chunk_by_free_memory(per, 1, 16384);  // 16384: grid z of the batched kernels
    for (long b0 = 0; b0 < q.B; b0 += chunk) {
        const int nb = (int)((q.B - b0) < chunk ? (q.B - b0) : chunk);
        Scope inner(h);
        double* Ks = inner.alloc<double>((size_t)nb * N * lds);
        double* As = inner.alloc<double>((size_t)nb * N * lds);
        double* kss = inner.alloc<double>((size_t)nb * Ns);
        double* alpha = dmean ? inner.alloc<double>((size_t)nb * N * q.Pp) : nullptr;
        if (!inner.ok) return inner.finish();
        const double* th = q.theta + b0 * np;
        CovArgs c{};
        c.Xa = q.X; c.Na = N; c.Xb = Xs; c.Nb = Ns; c.d = q.d;
        c.theta = th; c.theta_stride = np;
        c.K = Ks; c.ldk = lds; c.strideK = (long)N * lds;
        c.batch = nb; c.route_batch = q.B;
        if (launch_cov(s, c)) return mfgp_fail(h, MFGP_ERR_CUDA, "cov launch failed");
        if (launch_cov_diag(s, Xs, Ns, q.d, th, np, kss, Ns, nb)) return mfgp_fail(h, MFGP_ERR_CUDA, "cov_diag failed");
        GemmArgs g;  // A_s = W K_s
        g.M = N; g.N = Ns; g.K = N;
        g.A = q.W + b0 * N * q.ld; g.lda = q.ld; g.strideA = (long)N * q.ld;
        g.B = Ks; g.ldb = lds; g.strideB = (long)N * lds;
        g.C = As; g.ldc = lds; g.strideC = (long)N * lds;
        g.batch = nb;
        g.krange = KR_HI_I;
        if (launch_gemm(s, g)) return mfgp_fail(h, MFGP_ERR_CUDA, "gemm (As) failed");
        GemmArgs m;  // mean = A_s^T a
        m.transA = true;
        m.M = Ns; m.N = q.P; m.K = N;
        m.A = As; m.lda = lds; m.strideA = (long)N * lds;
        m.B = q.a + b0 * N * q.Pp; m.ldb = q.Pp; m.strideB = (long)N * q.Pp;
        m.C = mean + b0 * Ns * q.P; m.ldc = q.P; m.strideC = (long)Ns * q.P;
        m.batch = nb;
        if (!(joint && joint->mean_var_given)) {
            predict_var_kernel<<<dim3((Ns + 127) / 128, nb), 128, 0, s>>>(As, N, Ns, lds, kss, var + b0 * Ns, (long)N * lds);
            if (launch_gemm(s, m)) return mfgp_fail(h, MFGP_ERR_CUDA, "gemm (mean) failed");
        }
        if (joint) {
            MFGP_TRY(joint_chunk(h, inner, q, b0, nb, Xs, Ns, th, As, lds, var + b0 * Ns, m.C, *joint));
            continue;
        }
        if (!dmean) continue;
        GemmArgs bt;  // beta = W^T A_s, into the K_s buffer
        bt.transA = true;
        bt.M = N; bt.N = Ns; bt.K = N;
        bt.A = g.A; bt.lda = q.ld; bt.strideA = g.strideA;
        bt.B = As; bt.ldb = lds; bt.strideB = (long)N * lds;
        bt.C = Ks; bt.ldc = lds; bt.strideC = (long)N * lds;
        bt.batch = nb;
        bt.krange = KR_LO_I;
        if (launch_gemm(s, bt)) return mfgp_fail(h, MFGP_ERR_CUDA, "gemm (beta) failed");
        GemmArgs at;  // alpha = W^T a
        at.transA = true;
        at.M = N; at.N = q.Pp; at.K = N;
        at.A = g.A; at.lda = q.ld; at.strideA = g.strideA;
        at.B = m.B; at.ldb = q.Pp; at.strideB = m.strideB;
        at.C = alpha; at.ldc = q.Pp; at.strideC = (long)N * q.Pp;
        at.batch = nb;
        at.krange = KR_LO_I;
        if (launch_gemm(s, at)) return mfgp_fail(h, MFGP_ERR_CUDA, "gemm (alpha) failed");
        GprPosteriorData qc = q;
        qc.theta = th;
        if (launch_posterior_dx(s, qc, nb, Xs, Ns, alpha, Ks, lds, dmean + b0 * Ns * q.P * q.d, dvar + b0 * Ns * q.d))
            return mfgp_fail(h, MFGP_ERR_CUDA, "posterior_dx_kernel launch failed");
    }
    return 0;
}
