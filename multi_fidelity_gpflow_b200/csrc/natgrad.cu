// natgrad.cu -- natural-gradient step for the SVGP variational distributions q(u) = N(m, Lq Lq^T): GPflow's
// NaturalGradient (XiNat) for all L latents in one batched launch sequence (include/mfgp.h: mfgp_svgp_natgrad).
//
// Per latent l (m = q_mu[:, l], Lq = tril(q_sqrt[l]), gm = g_q_mu[:, l], G = tril(g_q_sqrt[l])):
//   Wq = Lq^-1 (trtri)                          g_S = sym( Wq^T Phi(Lq^T G) Wq )   (Cholesky adjoint, as K7's Kmmbar)
//   Lam = Wq^T Wq                               theta1' = Lam m - gamma (gm - 2 g_S m),  Lam' = Lam + 2 gamma g_S
//   R = chol(Lam') (potrf), R^-1 (trtri)        S' = R^-T R^-1,  m' = S' theta1',  Lq' = chol(S') (potrf)
// Every O(M^3) product is a DMMA GEMM on a triangular k-range, the factorisations are K2 / K4; the kernels below are the
// glue.  A latent whose R or Lq' factorisation fails keeps its m and Lq bit for bit.
#include "svgp.cuh"

#include "chol.cuh"
#include "gemm.cuh"

namespace {

// dinv[l][kb] <- inverse of the kb-th CHOL_NB x CHOL_NB diagonal block of the lower-triangular A[l], in the layout
// launch_potrf leaves for launch_trtri (lower, zero elsewhere).  Forward substitution, thread j solves column j; the
// k loop runs over all earlier rows (column j is zero above row j) so that every thread reads the same A entries.
__global__ void tri_block_inv_kernel(const double* __restrict__ A, int N, long lda, long strideA, double* __restrict__ dinv) {
    const int kb = blockIdx.x, l = blockIdx.y, j = threadIdx.x;
    const int k0 = kb * CHOL_NB, nb = min(CHOL_NB, N - k0);
    const double* Ab = A + (long)l * strideA + (long)k0 * lda + k0;
    double* D = dinv + ((long)l * gridDim.x + kb) * CHOL_NB * CHOL_NB;
    for (int i = 0; i < CHOL_NB; ++i) {
        double x = 0.0;
        if (i < nb && j <= i) {
            const double* row = Ab + (long)i * lda;
            double s0 = (i == j) ? 1.0 : 0.0, s1 = 0.0;
            int k = 0;
#pragma unroll 4
            for (; k + 1 < i; k += 2) {
                s0 = fma(-row[k], D[k * CHOL_NB + j], s0);
                s1 = fma(-row[k + 1], D[(k + 1) * CHOL_NB + j], s1);
            }
            if (k < i) s0 = fma(-row[k], D[k * CHOL_NB + j], s0);
            x = (s0 + s1) / row[i];
        }
        D[i * CHOL_NB + j] = x;
    }
}

__device__ inline double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// One warp per (latent l, row i): th1[l][i] = sum_j Lam_ij m_j - gamma (gm_i - 2 sum_j gS_ij m_j), and, in place,
// Lam_ij <- Lam_ij + 2 gamma gS_ij for j <= i (the triangle potrf reads).  Lam and gS hold full rows; each warp reads and
// writes its own row only.
__global__ void natgrad_theta_kernel(double* __restrict__ Lam, const double* __restrict__ gS, int M, long ld, int L,
                                     const double* __restrict__ q_mu, const double* __restrict__ g_q_mu, double gamma,
                                     const double* __restrict__ gamma_t, const int* __restrict__ step,
                                     double* __restrict__ th1) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= M * L) return;
    const int l = warp / M, i = warp % M;
    const double g = gamma_t ? gamma_t[*step] : gamma;
    double* lr = Lam + ((long)l * M + i) * ld;
    const double* gr = gS + ((long)l * M + i) * ld;
    double a = 0.0, b = 0.0;
    for (int j = lane; j < M; j += 32) {
        const double mj = q_mu[(long)j * L + l], lij = lr[j], gij = gr[j];
        a = fma(lij, mj, a);
        b = fma(gij, mj, b);
        if (j <= i) lr[j] = fma(2.0 * g, gij, lij);
    }
    a = warp_sum(a);
    b = warp_sum(b);
    if (lane == 0) th1[(long)l * M + i] = a - g * fma(-2.0, b, g_q_mu[(long)i * L + l]);
}

// One warp per (latent l, row i): mn[l][i] = sum_j S_ij th1[l][j]  (S holds full rows)
__global__ void natgrad_mean_kernel(const double* __restrict__ S, int M, long ld, int L, const double* __restrict__ th1,
                                    double* __restrict__ mn) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= M * L) return;
    const int l = warp / M, i = warp % M;
    const double* sr = S + ((long)l * M + i) * ld;
    double a = 0.0;
    for (int j = lane; j < M; j += 32) a = fma(sr[j], th1[(long)l * M + j], a);
    a = warp_sum(a);
    if (lane == 0) mn[(long)l * M + i] = a;
}

// Per-latent status select: st = infoR[l], or infoS[l] when R factored.  st == 0: q_mu[:, l] <- mn[l], q_sqrt[l] <- Lq'
// (strictly upper part zero); otherwise both stay as they are.  info[l] keeps its first failure.
__global__ void natgrad_select_kernel(const double* __restrict__ Lqn, const double* __restrict__ mn, int M, long ld, int L,
                                      const int* __restrict__ infoR, const int* __restrict__ infoS, double* __restrict__ q_mu,
                                      double* __restrict__ q_sqrt, int* __restrict__ info) {
    const int l = blockIdx.y;
    const int st = infoR[l] ? infoR[l] : infoS[l];
    if (blockIdx.x == 0 && threadIdx.x == 0 && info && !info[l]) info[l] = st;
    if (st) return;
    const long tot = (long)M * M;
    for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < tot; idx += (long)gridDim.x * blockDim.x) {
        const int i = (int)(idx / M), j = (int)(idx % M);
        q_sqrt[(long)l * tot + idx] = j <= i ? Lqn[((long)l * M + i) * ld + j] : 0.0;
        if (j == 0) q_mu[(long)i * L + l] = mn[(long)l * M + i];
    }
}

inline dim3 g2(long total, int L) { return dim3((unsigned)((total + 255) / 256 > 4096 ? 4096 : (total + 255) / 256), L); }

}  // namespace

int svgp_natgrad_step(mfgp_handle* h, int L, int M, double* q_mu, double* q_sqrt, const double* g_q_mu, const double* g_q_sqrt,
                      double gamma, const double* gamma_t, const int* step, int* info) {
    cudaStream_t s = h->stream;
    Scope sc(h);
    const long ld = round_up(M, 2), sMM = (long)M * ld;
    const size_t mat = (size_t)L * sMM;
    double* Lq = sc.alloc<double>(mat);   // tril(q_sqrt), later g_S
    double* G = sc.alloc<double>(mat);    // tril(g_q_sqrt), later Wq^T Phi Wq, later S'
    double* Wq = sc.alloc<double>(mat);   // Lq^-1, later R^-1
    double* T = sc.alloc<double>(mat);    // trtri scratch, Phi(Lq^T G)
    double* Lam = sc.alloc<double>(mat);  // Phi Wq, later Lam, Lam', R
    double* dinv = sc.alloc<double>((size_t)chol_dinv_count(M, L));
    double* logd = sc.alloc<double>((size_t)L * M);
    double* th1 = sc.alloc<double>((size_t)L * M);
    double* mn = sc.alloc<double>((size_t)L * M);
    int* infoR = sc.alloc<int>((size_t)L, true);
    int* infoS = sc.alloc<int>((size_t)L, true);
    if (!sc.ok) return sc.finish();
    const char* who = "mfgp_svgp_natgrad";

    tril_copy_kernel<<<g2(sMM, L), 256, 0, s>>>(q_sqrt, M, ld, Lq);
    tril_copy_kernel<<<g2(sMM, L), 256, 0, s>>>(g_q_sqrt, M, ld, G);
    CholArgs ch{};
    ch.A = Lq; ch.N = M; ch.lda = ld; ch.strideA = sMM; ch.batch = L;
    ch.dinv = dinv; ch.logd = logd; ch.d_info = h->d_info; ch.aux = h->aux_stream; ch.ev = h->ev;
    tri_block_inv_kernel<<<dim3(chol_nblk(M), L), CHOL_NB, 0, s>>>(Lq, M, ld, sMM, dinv);
    if (launch_trtri(s, ch, Wq, ld, sMM, T)) return mfgp_fail(h, MFGP_ERR_CUDA, "%s: trtri (Lq) failed", who);

    GemmArgs g1;  // T = Lq^T G (lower tiles) ; Phi
    g1.transA = true;
    g1.M = M; g1.N = M; g1.K = M;
    g1.A = Lq; g1.lda = ld; g1.strideA = sMM;
    g1.B = G; g1.ldb = ld; g1.strideB = sMM;
    g1.C = T; g1.ldc = ld; g1.strideC = sMM;
    g1.batch = L; g1.krange = KR_LO_MAXIJ; g1.lower_only = 1;
    if (launch_gemm(s, g1)) return mfgp_fail(h, MFGP_ERR_CUDA, "%s: gemm (Lq^T G) failed", who);
    tri_mask_kernel<<<g2(sMM, L), 256, 0, s>>>(T, M, ld, 1);
    GemmArgs g2a;  // Lam <- Phi Wq
    g2a.M = M; g2a.N = M; g2a.K = M;
    g2a.A = T; g2a.lda = ld; g2a.strideA = sMM;
    g2a.B = Wq; g2a.ldb = ld; g2a.strideB = sMM;
    g2a.C = Lam; g2a.ldc = ld; g2a.strideC = sMM;
    g2a.batch = L; g2a.krange = KR_HI_I | KR_LO_J;
    if (launch_gemm(s, g2a)) return mfgp_fail(h, MFGP_ERR_CUDA, "%s: gemm (Phi Wq) failed", who);
    GemmArgs g3;  // G <- Wq^T (Phi Wq) ; g_S = sym(G) into Lq
    g3.transA = true;
    g3.M = M; g3.N = M; g3.K = M;
    g3.A = Wq; g3.lda = ld; g3.strideA = sMM;
    g3.B = Lam; g3.ldb = ld; g3.strideB = sMM;
    g3.C = G; g3.ldc = ld; g3.strideC = sMM;
    g3.batch = L; g3.krange = KR_LO_I;
    if (launch_gemm(s, g3)) return mfgp_fail(h, MFGP_ERR_CUDA, "%s: gemm (Wq^T Phi Wq) failed", who);
    symmetrize_kernel<<<g2(sMM, L), 256, 0, s>>>(G, M, ld, Lq);
    double* gS = Lq;

    GemmArgs g4;  // Lam = Wq^T Wq (full rows: the row kernel reads them)
    g4.transA = true;
    g4.M = M; g4.N = M; g4.K = M;
    g4.A = Wq; g4.lda = ld; g4.strideA = sMM;
    g4.B = Wq; g4.ldb = ld; g4.strideB = sMM;
    g4.C = Lam; g4.ldc = ld; g4.strideC = sMM;
    g4.batch = L; g4.krange = KR_LO_MAXIJ;
    if (launch_gemm(s, g4)) return mfgp_fail(h, MFGP_ERR_CUDA, "%s: gemm (Lam) failed", who);
    const unsigned rows_grid = (unsigned)(((long)M * L * 32 + 255) / 256);
    natgrad_theta_kernel<<<rows_grid, 256, 0, s>>>(Lam, gS, M, ld, L, q_mu, g_q_mu, gamma, gamma_t, step, th1);

    CholArgs cr = ch;  // R = chol(Lam'), R^-1 into Wq
    cr.A = Lam; cr.info_vec = infoR;
    if (launch_potrf(s, cr)) return mfgp_fail(h, MFGP_ERR_CUDA, "%s: potrf (R) failed", who);
    if (launch_trtri(s, cr, Wq, ld, sMM, T)) return mfgp_fail(h, MFGP_ERR_CUDA, "%s: trtri (R) failed", who);
    GemmArgs g5;  // S' = R^-T R^-1 into G (full rows)
    g5.transA = true;
    g5.M = M; g5.N = M; g5.K = M;
    g5.A = Wq; g5.lda = ld; g5.strideA = sMM;
    g5.B = Wq; g5.ldb = ld; g5.strideB = sMM;
    g5.C = G; g5.ldc = ld; g5.strideC = sMM;
    g5.batch = L; g5.krange = KR_LO_MAXIJ;
    if (launch_gemm(s, g5)) return mfgp_fail(h, MFGP_ERR_CUDA, "%s: gemm (S') failed", who);
    natgrad_mean_kernel<<<rows_grid, 256, 0, s>>>(G, M, ld, L, th1, mn);
    CholArgs cs = ch;  // Lq' = chol(S') in place
    cs.A = G; cs.info_vec = infoS;
    if (launch_potrf(s, cs)) return mfgp_fail(h, MFGP_ERR_CUDA, "%s: potrf (Lq') failed", who);
    natgrad_select_kernel<<<g2((long)M * M, L), 256, 0, s>>>(G, mn, M, ld, L, infoR, infoS, q_mu, q_sqrt, info);
    CUDA_TRY(h, cudaGetLastError());
    return sc.finish();
}

extern "C" int mfgp_svgp_natgrad(mfgp_handle* h, const mfgp_svgp_cfg* cfg, double gamma, double* q_mu, double* q_sqrt,
                                 const double* g_q_mu, const double* g_q_sqrt, int* info) {
    if (!h) return MFGP_ERR_ARG;
    if (!cfg || !q_mu || !q_sqrt || !g_q_mu || !g_q_sqrt) return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_svgp_natgrad: NULL argument");
    const int L = cfg->L, M = cfg->M;
    if (L < 1 || M < 1 || !(gamma == gamma))
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_svgp_natgrad: need L >= 1, M >= 1 and gamma not NaN");
    cudaSetDevice(h->device);
    Scope sc(h);
    double* dqm = sc.inout(q_mu, (size_t)M * L);
    double* dqs = sc.inout(q_sqrt, (size_t)L * M * M);
    const double* dgm = sc.in(g_q_mu, (size_t)M * L);
    const double* dgs = sc.in(g_q_sqrt, (size_t)L * M * M);
    int* dinfo = info ? sc.out(info, (size_t)L, true) : nullptr;
    if (!sc.ok) return sc.finish();
    int rc;
    {
        const int was = h->async;  // the step only enqueues; this call's finish() decides about synchronising
        h->async = 1;
        rc = svgp_natgrad_step(h, L, M, dqm, dqs, dgm, dgs, gamma, nullptr, nullptr, dinfo);
        h->async = was;
    }
    if (rc) return rc;
    return sc.finish();
}
