/* mfgp.h -- C-ABI of libmfgp.so: the B200 (sm_100a) implementation of the Kennedy-O'Hagan
 * linear multi-fidelity GP objective, its gradient and its predictive equations.
 *
 * Drop-in boundary.  The reference (qezlou/multi_fidelity_gpflow, pure Python) reaches
 * this arithmetic through GPflow's operator API; each entry point below names the
 * reference interface it replaces (file:line in /root/reference).  INTEGRATION.md shows
 * the ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *  - All matrices are dense, row-major, float64.  `X` arrays are [N, d+1] with the
 *    fidelity indicator (exactly 0.0 or 1.0) in the last column (linear.py:67-70); rows
 *    with any other fidelity value have all-zero covariance (linear.py:82,99-102).
 *  - theta (per kernel) = [rho, ls_L[0..d-1], var_L, ls_delta[0..d-1], var_delta],
 *    length 2d+3, CONSTRAINED values (the softplus chain rule lives in the host shim).
 *  - Every pointer argument may be a HOST pointer or a DEVICE pointer of the handle's
 *    device; the library detects which (cudaPointerGetAttributes) and stages host
 *    buffers through the handle's stream.  Caller owns all buffers.
 *  - Return value: 0 ok; >0 = LAPACK-style info (1-based index of the first non-positive
 *    Cholesky pivot; for batched calls the first failing problem's info, per-problem
 *    values in `info[]`); <0 = bad argument (-1), CUDA error (-2), not supported (-3).
 *    mfgp_last_error() returns the message.
 *  - A handle is not thread-safe: one handle per GPU per thread.  Calls are ordered on
 *    the handle's stream and, unless async mode is on, synchronous on return.
 */
#ifndef MFGP_H
#define MFGP_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mfgp_handle mfgp_handle;

/* ---- lifetime / control ------------------------------------------------------------ */
int mfgp_version(void);
int mfgp_create(int device, mfgp_handle** out);
int mfgp_destroy(mfgp_handle* h);
/* Run on a caller-owned CUDA stream (cudaStream_t passed as void*; NULL is the legacy default
 * stream).  mfgp_reset_stream() returns to the handle's own non-blocking stream. */
int mfgp_set_stream(mfgp_handle* h, void* cuda_stream);
int mfgp_reset_stream(mfgp_handle* h);
/* async != 0: calls whose outputs are all device pointers return without synchronising;
 * non-PD status is then collected by mfgp_sync(). */
int mfgp_set_async(mfgp_handle* h, int async);
int mfgp_sync(mfgp_handle* h, int* info_out);
const char* mfgp_last_error(mfgp_handle* h);
int mfgp_sm_count(mfgp_handle* h);

/* ---- K1: covariance assembly ---------------------------------------------------------
 * replaces LinearMultiFidelityKernel.K (mfgpflow/linear.py:55-104) and K_diag (:106-136)
 * X2 == NULL -> X2 = X (linear.py:59-60): the symmetric fast path computes the lower
 * triangle of tiles once and mirrors it.  K is [N, N2] with leading dimension ldk. */
int mfgp_cov(mfgp_handle* h, const double* X, int N, const double* X2, int N2, int d,
             const double* theta, double* K, long ldk);
int mfgp_cov_diag(mfgp_handle* h, const double* X, int N, int d, const double* theta, double* out);

/* K5: out[q] = scale * sum_ij G_ij dK_ij/dtheta_q (q < 2d+3) with K = K(X, X; theta) and dK recomputed on the fly (never
 * stored); out[2d+3] = scale * sum_i G_ii (derivative of the noise term).  G [N, ldg] is symmetric and only its LOWER triangle
 * is read (off-diagonal entries count twice).  This is the contraction of tape.gradient through K (linear.py:207) exposed for
 * callers that build G = alpha alpha^T - K^-1 themselves (the distributed exact-GP gradient, dist_chol.py). */
int mfgp_cov_grad(mfgp_handle* h, const double* X, int N, int d, const double* theta, const double* G, long ldg, double scale,
                  double* out /* [2d+4] */);

/* ---- K2..K5: exact multi-fidelity GPR -------------------------------------------------
 * replaces gpflow GPR.log_marginal_likelihood as called at linear.py:206,227 (model built
 * at linear.py:148-156: zero mean, Gaussian noise `noise`, ONE kernel/Cholesky shared by
 * all P columns of Y [N, P]).  *nlml = -log_marginal_likelihood. */
int mfgp_gpr_nlml(mfgp_handle* h, const double* X, const double* Y, int N, int d, int P,
                  const double* theta, double noise, double* nlml);
/* + analytic gradient of nlml w.r.t. [theta (2d+3), noise] -- replaces
 * tape.gradient(loss, trainable_variables) at linear.py:207 (constrained space). */
int mfgp_gpr_nlml_grad(mfgp_handle* h, const double* X, const double* Y, int N, int d, int P,
                       const double* theta, double noise, double* nlml, double* grad /* [2d+4] */);
/* replaces gpflow GPR.predict_f(Xnew) (tests/test_ho2021_multibin.py:83, tests/test_scipy.py:48):
 * mean [Ns, P], var [Ns] (identical for every output column). */
int mfgp_gpr_predict(mfgp_handle* h, const double* X, const double* Y, int N, int d, int P,
                     const double* Xs, int Ns, const double* theta, double noise,
                     double* mean, double* var);
/* K6: "one GP per k-bin" (gpemulator_singlebin.py:1-14 design; BASELINE config 2): problem
 * b uses y = Y[:, b % ycols] (Y is [N, ycols] row-major with leading dimension ldy),
 * theta[b, :], noise[b]; B > ycols evaluates several hyper-parameter sets (restarts) per
 * bin in one launch.  nlml [B]; grad [B, 2d+4] or NULL; info [B] (int) or NULL.
 * N <= 64 runs one CTA per problem entirely in shared memory. */
int mfgp_gpr_batched_nlml_grad(mfgp_handle* h, const double* X, int N, int d, const double* Y,
                               long ldy, int ycols, int B, const double* theta, const double* noise,
                               double* nlml, double* grad, int* info);

/* Cached posterior of B independent exact GPs (GPflow model.posterior() with PrecomputeCacheType.TENSOR): factor once,
 * predict many times.  X [N, d+1] is shared.  Problem b uses theta[b, 2d+3], noise[b] and the RHS columns
 * Y[:, c : c + P] with c = (b * P) % ycols (row stride ldy; requires ycols % P == 0).  P = 1, ycols = #bins gives the
 * per-bin convention of mfgp_gpr_batched_nlml_grad (b = r * bins + p); B = 1, P = ycols gives MultiFidelityGPModel.
 *  - Snapshot: the posterior owns device copies of X, theta and noise and the factors W = L^-1 [B][N][ld] and
 *    a = W Y [B][N][round_up(P, 2)]; later changes to the caller's buffers do not reach it.
 *  - Memory: plain cudaMalloc on the handle's device (not the per-call pool, not the mfgp_workspace arena).  The posterior
 *    belongs to that device, not to the handle: any handle on the same device may predict with it, and it may be
 *    destroyed before or after the handle that created it.
 *  - info [B] or NULL.  With info, a non-PD problem is that problem's status (1-based pivot in info[b]), it predicts NaN,
 *    *out is set and the call returns the first failure's pivot like the other batched calls.  Without info, a non-PD
 *    problem makes the call return its pivot with *out = NULL.  Creation always synchronises (it decides what is returned;
 *    mfgp_gpr_batched_lbfgs does too, because when it ends depends on the data).
 *  - Cost: the blocked batched factorisation (K1 -> potrf -> trtri -> a = W Y), chunked over B by free memory.
 * mfgp_gpr_posterior_predict: mean [B, Ns, P], var [B, Ns] (the same for every column, like mfgp_gpr_predict); host or
 * device pointers, async mode as for every call.  N <= 64, d <= 16, P <= 64 run ONE fused kernel for all problems and
 * points (gpr_posterior_predict_kernel); anything larger the blocked route (K1, cov_diag, two batched GEMMs), chunked over
 * B.  A point's result does not depend on the other points or problems of the call. */
typedef struct mfgp_gpr_posterior mfgp_gpr_posterior;
int mfgp_gpr_posterior_create(mfgp_handle* h, const double* X, int N, int d, const double* Y, long ldy, int ycols, int P,
                              int B, const double* theta, const double* noise, int* info, mfgp_gpr_posterior** out);
int mfgp_gpr_posterior_predict(mfgp_handle* h, const mfgp_gpr_posterior* post, const double* Xs, int Ns,
                               double* mean, double* var);
/* mfgp_gpr_posterior_predict_grad: mean [B, Ns, P] and var [B, Ns] as mfgp_gpr_posterior_predict, and their gradients
 * with respect to the d continuous coordinates of each test point, dmean [B, Ns, P, d] = d mean / d Xs[s, j] and
 * dvar [B, Ns, d] = d var / d Xs[s, j] (the fidelity column has no gradient: it enters the kernel only through equality
 * masks).  All four outputs are required.  A test row with fidelity not in {0, 1} has zero gradients; a problem whose
 * factorisation failed gives NaN in all four.  Pointers, async mode, the device check and Ns == 0 as for _predict.  The
 * fused route (N <= 64, d <= 16, P <= 64) is one kernel, gpr_posterior_predict_grad_kernel; the blocked route adds
 * beta = K^-1 K_s and alpha = W^T a (two batched GEMMs) and posterior_dx_kernel to the _predict pipeline.  A point's
 * results do not depend on the other points or problems of the call. */
int mfgp_gpr_posterior_predict_grad(mfgp_handle* h, const mfgp_gpr_posterior* post, const double* Xs, int Ns,
                                    double* mean, double* var, double* dmean, double* dvar);
/* Joint posterior over the Ns test points (GPflow GPR.predict_f(full_cov=True) and predict_f_samples):
 * Sigma_b = K(Xs, Xs) - V^T V with V = W K(X, Xs), the same for every output column of problem b.
 * mfgp_gpr_posterior_predict_cov: mean [B, Ns, P] and the joint covariance cov [B, Ns, Ns] (both triangles, exactly
 * symmetric).  mean is _predict's mean bit for bit and the diagonal of cov is _predict's var bit for bit.
 * mfgp_gpr_posterior_sample: samples[b, i, k, c] = mean[b, i, c] + sum_j L_b[i, j] z[b, j, k, c] with
 * L_b L_b^T = Sigma_b + jitter I, Sigma_b exactly the matrix _predict_cov returns (GPflow sample_mvn, full_cov=True).
 * z and samples are [B, Ns, S, P]: each test point's S * P draws are contiguous, and z and samples must not overlap.
 *  - Failures: info[b] (info [B] or NULL) is the 1-based first pivot of Sigma_b + jitter I that is not > 0 (NaN counts),
 *    so a problem whose factorisation failed at creation reports 1.  All samples of a failing problem are NaN.  The call
 *    returns the first failure's pivot with or without info; with info that is the problem's status.  _predict_cov gives
 *    NaN mean and cov for a problem that failed at creation, as _predict does, and returns 0.
 *  - A test row with fidelity not in {0, 1} has a zero row and column in cov and a zero mean.  With jitter > 0 its row of
 *    L is sqrt(jitter) e_i, so its samples are sqrt(jitter) z; with jitter == 0 it is a failed pivot.
 *  - jitter finite and >= 0, S >= 0, no NULL pointer except info: otherwise -1.  Ns == 0 or S == 0 returns 0.  Pointers,
 *    async mode (a non-PD status then reaches mfgp_sync) and the device check as for _predict.
 *  - A problem's results do not depend on the other problems of the call, and a sample column's values do not depend on S
 *    or on how the work is split.  Indices are 64-bit: B * Ns * S * P may exceed 2^31.
 *  - Routes as for _predict.  N <= 64, d <= 16, P <= 64 and Ns <= 64 run ONE kernel (gpr_posterior_joint_kernel: each CTA
 *    rebuilds Sigma on DMMA, factors it in shared memory and streams its chunk of z); anything else extends the blocked
 *    route with K1 for K(Xs, Xs), one GEMM for Sigma, potrf and one GEMM for L Z. */
int mfgp_gpr_posterior_predict_cov(mfgp_handle* h, const mfgp_gpr_posterior* post, const double* Xs, int Ns,
                                   double* mean, double* cov);
int mfgp_gpr_posterior_sample(mfgp_handle* h, const mfgp_gpr_posterior* post, const double* Xs, int Ns, int S,
                              double jitter, const double* z, double* samples, int* info);
int mfgp_gpr_posterior_destroy(mfgp_gpr_posterior* post);

/* Training loop on the device (SURVEY 8(f) rank 1): the Adam branch of MultiFidelityGPModel.optimize (mfgpflow/linear.py:
 * 190-221: loss = -log_marginal_likelihood, tape.gradient w.r.t. the UNCONSTRAINED variables, Keras Adam, noise fixed) for
 * B independent per-bin GPs, nsteps steps without a host round trip.  Per step: theta = softplus(u) -> K6 NLML + gradient
 * -> chain rule (1 - exp(-theta)) -> m, v, u update (ResourceApplyAdam: m += (g-m)(1-beta1), v += (g^2-v)(1-beta2),
 * u -= lr_t m / (sqrt(v) + eps)).  u, m, v are [B, 2d+3] and updated in place (m = v = 0 to start); lr_t [nsteps] holds
 * the per-step factor lr(step) sqrt(1-beta2^t)/(1-beta1^t), computed by the host shim so that the float32-rounded
 * hyper-parameters and the CosineDecay schedule of the reference (quirk Q8) stay in one place.  fix_rho != 0 freezes rho
 * (use_rho=False, linear.py:51-52).  loss_hist [nsteps, B] (or NULL) receives the NLML evaluated BEFORE each update (the
 * reference's loss_history); theta_out [B, 2d+3] (or NULL) the constrained values after the last update.
 * N <= 64 only (the K6 kernel).  Returns >0 if a Cholesky failed at any step (per-problem first failure in info[B]). */
int mfgp_gpr_batched_adam(mfgp_handle* h, const double* X, int N, int d, const double* Y, long ldy, int ycols, int B,
                          double* u, double* m, double* v, const double* noise, const double* lr_t, double beta1,
                          double beta2, double eps, int fix_rho, int nsteps, double* loss_hist, double* theta_out, int* info);

/* Multi-start L-BFGS on the device: the SciPy branch of MultiFidelityGPModel.optimize (mfgpflow/linear.py:222-234,
 * gpflow.optimizers.Scipy -> scipy.optimize.minimize(method="L-BFGS-B")) for B independent per-bin GPs in one loop.
 * Problem indexing, Y, X and the limits (N <= 64, d <= 16) are those of mfgp_gpr_batched_nlml_grad (b = r * bins + p).
 *  - Variables: u [B, 2d+3] in/out, theta = softplus(u) as in mfgp_gpr_batched_adam.  fix_rho != 0 keeps rho out of the
 *    variable vector (u[b, 0] is left bit for bit).  train_noise == 0 uses noise [B] exactly as passed (then the objective
 *    is Adam's, bit for bit); train_noise != 0 adds the variable v, noise = 1e-6 + softplus(v) (gpflow Gaussian's lower
 *    bound), started at v = softplus^-1(noise - 1e-6) and written back to noise at the end.
 *  - Algorithm: SciPy's L-BFGS-B on unbounded variables, written out: two-loop direction over the last m pairs, MINPACK-2
 *    dcsrch line search (ftol 1e-3, gtol 0.9, xtol 0.1), stp = min(1/||d||, 1e10) on iteration 0.  After an accepted step
 *    the tests run in SciPy's order: nit >= maxiter, nfev > maxfun, ||g||_inf <= gtol, relative reduction of f <= ftol.
 *    One deliberate deviation: a trial point whose covariance is not positive definite, or whose objective or gradient is
 *    not finite, fails that problem's trial only (GPflow's closure would abort the whole minimize).  It counts as an
 *    evaluation and against maxls, and the search restarts from its base point with stp = 0.1 x the failed step and
 *    stpmax = 0.5 x the failed step.
 *  - opts NULL = SciPy's defaults {m 10, maxiter 15000, maxfun 15000, maxls 20, ftol 2.220446049250313e-09, gtol 1e-5};
 *    1 <= m <= MFGP_LBFGS_MAX_M, maxiter, maxfun, maxls >= 1, ftol, gtol >= 0.
 *  - Outputs [B]: f (final loss, NaN for MFGP_LBFGS_NOT_PD), nit, nfev, status (MFGP_LBFGS_*), info or NULL.  A problem
 *    whose START point fails stops with MFGP_LBFGS_NOT_PD, its 1-based pivot in info[b] (0 when the factor exists but the
 *    objective is not finite) and its u and noise unchanged.  The call returns the pivot of the lowest-index such
 *    problem: with info that is the problems' status, without info the call's error, as for the other batched calls.
 *  - Cost: one round = one K6 launch over all B problems at their current trial points + one lbfgs_step_kernel.  Finished
 *    problems stay in the K6 launch at their last point.  The host reads the number of active problems every 16 rounds.
 *  - A problem's results do not depend on the other problems of the call.  Host or device pointers.  The call always
 *    synchronises: when it ends depends on the data (as for mfgp_gpr_posterior_create). */
#define MFGP_LBFGS_PGTOL 1    /* ||g||_inf <= gtol */
#define MFGP_LBFGS_FTOL 2     /* (f_old - f) <= ftol * max(|f_old|, |f|, 1) */
#define MFGP_LBFGS_MAXITER 3  /* nit reached maxiter */
#define MFGP_LBFGS_MAXFUN 4   /* nfev exceeded maxfun */
#define MFGP_LBFGS_ABNORMAL 5 /* the line search failed with an empty memory ("ABNORMAL_TERMINATION_IN_LNSRCH") */
#define MFGP_LBFGS_NOT_PD 6   /* the start point is not positive definite or not finite */
#define MFGP_LBFGS_MAX_M 32
typedef struct { int m, maxiter, maxfun, maxls; double ftol, gtol; } mfgp_lbfgs_opts;
int mfgp_gpr_batched_lbfgs(mfgp_handle* h, const double* X, int N, int d, const double* Y, long ldy, int ycols, int B,
                           double* u, double* noise, int fix_rho, int train_noise, const mfgp_lbfgs_opts* opts,
                           double* f, int* nit, int* nfev, int* status, int* info);

/* ---- Graph-structured multi-fidelity kernel (SURVEY 8(f) rank 3) ---------------------------------------------------
 * replaces GraphMultiFidelityKernel.K / K_diag (mfgpflow/graph.py:39-93, :96-115) and, for GraphMultiFidelityGPModel
 * (graph.py:118-188), GPR.log_marginal_likelihood + tape.gradient.  num_lf low-fidelity sources (fidelity column value
 * i in [0, num_lf)) and one high-fidelity level (value num_lf); rows with any other value have zero covariance.
 * gtheta (constrained values), length mfgp_graph_nparams(num_lf, d) = m + m^2 + (m + 1)(d + 1):
 *   [rho (m)] [rho_LF (m x m, row-major, diagonal unused)] [ls_Li (d), var_Li] for i < m, [ls_delta (d), var_delta].
 * Only K(X, X) exists: the reference's rectangular call is not shape-consistent (graph.py:76-79, :91).  K is the FULL
 * N x N matrix including the 1e-6 jitter of graph.py:91; like the reference it is not symmetric once the low-fidelity
 * kernels differ (graph.py:63 uses the row's kernel).  The objective factors the lower triangle of K + noise I and
 * contracts the symmetric sensitivity with the derivative of every entry -- TensorFlow's Cholesky / gradient semantics.
 * grad [nparams + 1] (or NULL): d nlml / d [gtheta, noise]; the entries of the unused rho_LF diagonal are 0. */
int mfgp_graph_nparams(int num_lf, int d);
int mfgp_graph_cov(mfgp_handle* h, const double* X, int N, int d, int num_lf, const double* gtheta, double* K, long ldk);
int mfgp_graph_cov_diag(mfgp_handle* h, const double* X, int N, int d, int num_lf, const double* gtheta, double* out);
int mfgp_graph_gpr_nlml_grad(mfgp_handle* h, const double* X, const double* Y, int N, int d, int P, int num_lf,
                             const double* gtheta, double noise, double* nlml, double* grad);

/* ---- K7/K8: sparse variational GP (whitened, shared inducing points) -------------------
 * replaces gpflow SVGP.elbo / prior_kl / predict_f as called at singlebin_svgp.py:83,97 and
 * linear_svgp.py:177,184,188,199 with kernels SeparateIndependent (W == NULL, L == P,
 * singlebin_svgp.py:39-47) or LinearCoregionalization (W [P, L], linear_svgp.py:121-122). */
typedef struct {
    int L;          /* latent GPs */
    int M;          /* inducing points */
    int P;          /* outputs */
    int B;          /* rows in this (mini)batch */
    int d;          /* input dimension without the fidelity column */
    int hetero;     /* 1: Y is [B, 2P] = [Y_obs | Y_unc], var_eff = lik_var + Y_unc^2 (linear_svgp.py:259) */
    double scale;   /* num_data / B, or 1 (singlebin_svgp.py passes no num_data) */
    double kl_mult; /* loss = -ELBO + (kl_mult - 1) KL   (linear_svgp.py:188) */
    double jitter;  /* gpflow default_jitter() = 1e-6 */
    double lik_lower; /* lower bound of the likelihood-variance transform, used by mfgp_svgp_adam only: gpflow Gaussian
                       * positive(lower=1e-6); HeteroscedasticGaussian positive() = 0 (linear_svgp.py:240) */
    int masked;     /* 1: entries of Y that are NaN are missing outputs and contribute nothing (MaskedGaussian,
                     * notebooks/"demo: missing output.ipynb" cell 2); exclusive with hetero */
    int lik_per_output; /* 1: the likelihood variance is a [P] vector, one per output (same notebook: variance=np.ones(P)) */
} mfgp_svgp_cfg;

/* Forward + hand-derived backward.  Outputs (any grad pointer may be NULL to skip all
 * gradients): elbo, kl (scalars); gradients of loss w.r.t. CONSTRAINED values:
 * gZ [M, d+1] (fidelity column == 0, quirk Q5), gtheta [L, 2d+3], gW [P, L] (NULL if W is
 * NULL), gqmu [M, L], gqsqrt [L, M, M] (lower triangle, rest 0), glik (scalar). */
int mfgp_svgp_elbo_grad(mfgp_handle* h, const mfgp_svgp_cfg* cfg, const double* X, const double* Y,
                        const double* Z, const double* theta, const double* W, const double* q_mu,
                        const double* q_sqrt, double lik_var, double* elbo, double* kl,
                        double* gZ, double* gtheta, double* gW, double* gqmu, double* gqsqrt,
                        double* glik);
/* Same with the likelihood variance passed by pointer (host or device): lik_var and glik hold 1 value, or P values when
 * cfg->lik_per_output is set.  mfgp_svgp_elbo_grad is the scalar-by-value convenience form of this call. */
int mfgp_svgp_elbo_grad_v(mfgp_handle* h, const mfgp_svgp_cfg* cfg, const double* X, const double* Y,
                          const double* Z, const double* theta, const double* W, const double* q_mu,
                          const double* q_sqrt, const double* lik_var, double* elbo, double* kl,
                          double* gZ, double* gtheta, double* gW, double* gqmu, double* gqsqrt,
                          double* glik);
/* mean [Ns, P], var [Ns, P]  (cfg->B is ignored, Ns rows are predicted). */
int mfgp_svgp_predict(mfgp_handle* h, const mfgp_svgp_cfg* cfg, const double* Xs, int Ns,
                      const double* Z, const double* theta, const double* W, const double* q_mu,
                      const double* q_sqrt, double* mean, double* var);

/* Cached SVGP posterior (GPflow SVGP.posterior()): factor the inducing covariances of the L latents once, then predict
 * every latent in one launch, with the results of mfgp_svgp_predict.
 *  - cfg supplies L, M, P, d and jitter as for mfgp_svgp_predict; B and the likelihood fields are ignored.  W [P, L] or
 *    NULL (SeparateIndependent, L == P).  Only the lower triangle of q_sqrt [L, M, M] is read; q_mu is [M, L].
 *  - Snapshot: the posterior owns device copies of Z, theta, W, q_mu, Wm = Lm^-1 of K_l(Z,Z) + jitter I and
 *    Lq = tril(q_sqrt) (the factors mfgp_svgp_predict computes); later changes to the caller's buffers do not reach it.
 *  - Memory: one plain cudaMalloc block on the handle's device, owned by the device (not the handle): any handle on that
 *    device may predict with it, and it outlives the handle that created it.  Free it with mfgp_svgp_posterior_destroy.
 *  - Status: creation always synchronises.  Without info a non-positive-definite latent makes the call return its pivot
 *    (> 0) with *out = NULL.  With info [L] (host or device) info[l] holds latent l's pivot (0 = ok), the call returns the
 *    first pivot and the posterior exists: latent l predicts NaN, so with W every output reads NaN (NaN * 0 = NaN).
 * mfgp_svgp_posterior_predict: mean [Ns, P], var [Ns, P] as mfgp_svgp_predict; host or device pointers, async mode, Ns == 0
 * returns at once, and the handle must be on the posterior's device.  M <= 64 and d <= 16 run one sm_100a kernel
 * (svgp_posterior_predict_kernel: V = Wm K_s and U = Lq^T V on DMMA) plus the mix when W is given; anything larger runs
 * the second half of mfgp_svgp_predict (K1, cov_diag, two batched GEMMs, col_reduce, mix) chunked over Ns.  A point's
 * result does not depend on the other points of the call. */
typedef struct mfgp_svgp_posterior mfgp_svgp_posterior;
int mfgp_svgp_posterior_create(mfgp_handle* h, const mfgp_svgp_cfg* cfg, const double* Z, const double* theta,
                               const double* W, const double* q_mu, const double* q_sqrt, int* info,
                               mfgp_svgp_posterior** out);
int mfgp_svgp_posterior_predict(mfgp_handle* h, const mfgp_svgp_posterior* post, const double* Xs, int Ns,
                                double* mean, double* var);
/* mfgp_svgp_posterior_predict_grad: mean [Ns, P] and var [Ns, P] as mfgp_svgp_posterior_predict, and their gradients
 * with respect to the d continuous coordinates of each test point, dmean [Ns, P, d] = d mean / d Xs[s, j] and
 * dvar [Ns, P, d] = d var / d Xs[s, j] (the fidelity column has no gradient).  All four outputs are required.  A test row
 * with fidelity not in {0, 1} has zero gradients, dead inducing points contribute nothing, and a failed latent gives NaN
 * in its outputs (with W in all of them).  Pointers, async mode, the device check and Ns == 0 as for _predict.  The
 * fused route (M <= 64, d <= 16) is one kernel, svgp_posterior_predict_grad_kernel, plus the two mixes when W is given;
 * the blocked route adds R = V - Lq U and beta = Wm^T R (two batched GEMMs), alpha = Wm^T q_mu and posterior_dx_kernel to
 * the _predict pipeline.  A point's results do not depend on the other points of the call. */
int mfgp_svgp_posterior_predict_grad(mfgp_handle* h, const mfgp_svgp_posterior* post, const double* Xs, int Ns,
                                     double* mean, double* var, double* dmean, double* dvar);
int mfgp_svgp_posterior_destroy(mfgp_svgp_posterior* post);

/* Training loop on the device for the SVGP models (SURVEY 8(f) rank 1): the optimize() loops of mfgpflow/singlebin_svgp.py:
 * 64-97 and mfgpflow/linear_svgp.py:153-203 -- full-batch, Keras Adam (+ CosineDecay folded into lr_t, see
 * mfgp_gpr_batched_adam), loss = -ELBO + (kl_mult - 1) KL -- nsteps steps without a host round trip.
 * Flat parameter layout (doubles): [theta L*(2d+3)] [Z M*(d+1)] [W P*L, only if has_W] [q_mu M*L] [q_sqrt L*M*M] [lik_var 1, or P with
 * cfg->lik_per_output].
 * u holds the UNCONSTRAINED values in that layout (theta = softplus(u), lik_var = cfg->lik_lower + softplus(u), the rest identity;
 * the strictly upper part of every q_sqrt matrix must be zero and stays zero); u, m, v are updated in place.
 * mask (n bytes or NULL): 0 freezes an entry (not in trainable_variables).  loss_hist / kl_hist [nsteps] or NULL receive
 * the loss and KL evaluated BEFORE each update (the reference's loss_history / kl_history). */
int mfgp_svgp_adam(mfgp_handle* h, const mfgp_svgp_cfg* cfg, const double* X, const double* Y, int has_W, double* u,
                   double* m, double* v, const unsigned char* mask, const double* lr_t, double beta1, double beta2,
                   double eps, int nsteps, double* loss_hist, double* kl_hist);

/* Minibatch stream: the rows the minibatch SVGP loops train on, one endless sequence of shuffled epochs over a data set of
 * N rows, defined by an integer-only stateless rule (the GPU evaluates it inside a captured graph from the device step
 * counter; every rank of a data-parallel run computes its slice of the same global batch without communicating).
 *  - Stream position p >= 0 (64-bit) is epoch e = p / N, offset i = p mod N, row pi_{seed,e}(i).
 *  - pi_{seed,e} is a balanced Feistel network on 2k-bit values, k the smallest integer with 4^k >= N, cycle-walked (the
 *    network is applied again until the value is below N).  A value x splits into l = x >> k, r = x & (2^k - 1); each of
 *    8 rounds j = 0..7 does (l, r) <- (r, l ^ (mix32(r ^ key_j) & (2^k - 1))); x = (l << k) | r.
 *  - key_j = low 32 bits of splitmix64(splitmix64(splitmix64(seed) ^ e) ^ j), all arithmetic modulo 2^64.
 *    splitmix64(z): z += 0x9E3779B97F4A7C15; z = (z ^ z >> 30) * 0xBF58476D1CE4E5B9; z = (z ^ z >> 27) * 0x94D049BB133111EB;
 *    z ^ z >> 31.  mix32(x) (32-bit): x ^= x >> 16; x *= 0x7FEB352D; x ^= x >> 15; x *= 0x846CA68B; x ^ x >> 16.
 *  - Step t of a loop that starts at position pos0 with batch size B reads positions pos0 + t B ... pos0 + t B + B - 1:
 *    batches cross epoch boundaries and B need not divide N.
 * The rule is fixed: changing any constant above changes every minibatch trajectory.
 *
 * mfgp_svgp_adam_minibatch: mfgp_svgp_adam on minibatches of that stream.  X [N, d+1] and Y [N, ycols] are the whole data
 * set (copied to the device once per call when they are host memory); cfg->B is the batch size, 1 <= B <= N, and
 * cfg->scale what the caller wants (num_data / B).  Each step gathers its B rows (minibatch_gather_kernel) and then runs
 * the step of mfgp_svgp_adam on them; loss_hist / kl_hist receive each step's minibatch estimate.  The batch buffers are
 * allocated before the step is captured, so the graph has no allocation nodes.  pos0 >= 0; otherwise -1.
 *
 * mfgp_minibatch_gather: Xb [count, xcols] and Yb [count, ycols] <- rows X[row], Y[row] of positions
 * pos0 + (*step) B + lo + j, j < count, with 1 <= B <= N, 0 <= lo, lo + count <= B.  step is an int (host or device), or
 * NULL for 0; Y and Yb may both be NULL.  A data-parallel rank r gathers lo, count = its shard of each global batch of B
 * rows, reading the step counter mfgp_svgp_adam_update advances.  Host or device pointers; NaN entries are copied as they
 * are. */
int mfgp_svgp_adam_minibatch(mfgp_handle* h, const mfgp_svgp_cfg* cfg, const double* X, const double* Y, int N,
                             unsigned long long seed, long long pos0, int has_W, double* u, double* m, double* v,
                             const unsigned char* mask, const double* lr_t, double beta1, double beta2, double eps,
                             int nsteps, double* loss_hist, double* kl_hist);
int mfgp_minibatch_gather(mfgp_handle* h, const double* X, int xcols, const double* Y, int ycols, int N,
                          unsigned long long seed, long long pos0, const int* step, int B, int lo, int count, double* Xb,
                          double* Yb);

/* Data-parallel SVGP training step on device memory only (SURVEY 8(e) row 2: rows of the minibatch shard across one
 * process per GPU, ONE all-reduce of the flat gradient; reference loops singlebin_svgp.py:79-85, linear_svgp.py:181-190).
 * Per step every rank runs, on the handle's stream and without any host synchronisation:
 *     mfgp_svgp_constrain(u -> c);  mfgp_svgp_elbo_grad_flat(rows of this rank, c -> eg);
 *     all-reduce(sum) of eg [2 + n] in place (the caller's collective: ncclAllReduce on the same stream);
 *     mfgp_svgp_adam_update(u, m, v <- eg).
 * n = mfgp_svgp_flat_size() doubles in the flat layout of mfgp_svgp_adam.  All pointers are DEVICE pointers.
 * eg after mfgp_svgp_elbo_grad_flat: eg[0] = cfg->scale * VE of this rank's rows, eg[1] = KL / nranks, eg[2 + i] = d/d c_i of
 * (-scale VE_rank + kl_mult / nranks KL); after the all-reduce: [scale VE, KL, gradient of -ELBO + (kl_mult - 1) KL].
 * The gradient pieces are written by the kernels straight into eg: no host staging, no concatenation.
 * cfg->B is the number of rows of THIS call; cfg->scale = num_data / (global batch size). */
long mfgp_svgp_flat_size(const mfgp_svgp_cfg* cfg, int has_W);
int mfgp_svgp_constrain(mfgp_handle* h, const mfgp_svgp_cfg* cfg, int has_W, const double* u, double* c);
int mfgp_svgp_elbo_grad_flat(mfgp_handle* h, const mfgp_svgp_cfg* cfg, const double* X, const double* Y, int has_W,
                             const double* c, int nranks, double* eg /* [2 + n] */);
/* Keras-Adam update from the all-reduced eg; lr_t [nsteps] and the step counter *step live on the device (the counter is
 * incremented by the call); loss_hist / kl_hist [nsteps] (device, or NULL) receive entry *step; scratch2: 2 doubles. */
int mfgp_svgp_adam_update(mfgp_handle* h, const mfgp_svgp_cfg* cfg, int has_W, double* u, double* m, double* v,
                          const unsigned char* mask, const double* c, const double* eg, const double* lr_t, int* step,
                          double beta1, double beta2, double eps, double* loss_hist, double* kl_hist, double* scratch2);

/* ---- dense fp64 building blocks (exported for tests / bench / comparators) ------------- */
/* C[m,n] = alpha * op(A) op(B) + beta * C, row-major; transa/transb are 'N' or 'T'.
 * Runs the DMMA (mma.sync m8n8k4 f64) tile kernel; the operand tiles are fed by TMA (cp.async.bulk.tensor + mbarrier), which
 * is why A, B must be 16-byte aligned with even lda / ldb (tensor-map strides are multiples of 16 bytes). */
int mfgp_gemm(mfgp_handle* h, char transa, char transb, int m, int n, int k, double alpha,
              const double* A, long lda, const double* B, long ldb, double beta, double* C, long ldc);
/* In-place lower Cholesky A = L L^T (row-major).  Only the lower triangle is referenced; on return the
 * strictly-upper part of every 128x128 diagonal block is zeroed, upper off-diagonal blocks are untouched. */
int mfgp_potrf(mfgp_handle* h, double* A, int N, long lda);
/* Winv [N, N] = inv(L) for the lower factor produced by mfgp_potrf. */
int mfgp_potrf_inv(mfgp_handle* h, double* A, int N, long lda, double* Winv, long ldw);
/* Y[M, 0:nc] += alpha * A[M, K] X[K, 0:nc] for nc <= 2 right-hand sides (device pointers; A rows 16-byte aligned, K <= 3072).
 * The replicated forward-substitution step of the distributed Cholesky (y[k+1:] -= L[k+1:, k] a_k), HBM-bound. */
int mfgp_tall_skinny_update(mfgp_handle* h, int M, int K, int nc, double alpha, const double* A, long lda, const double* X,
                            long ldx, double* Y, long ldy);

/* One-to-many store: `count` doubles (even, 16-byte aligned) from src into ndst <= MFGP_PEER_MAX destination buffers in ONE
 * kernel on the handle's stream.  The destinations are device pointers valid in this process -- buffers of PEER GPUs mapped
 * over NVLink (symmetric memory, CUDA IPC) or local ones.  Used for the critical-path messages of the distributed Cholesky
 * (dist_chol.py: inv(L_kk) and the early block go to all peers by direct stores instead of an NCCL broadcast); the caller
 * orders the stores against the receivers with its own signal (never synchronises). */
#define MFGP_PEER_MAX 8
int mfgp_peer_store(mfgp_handle* h, const double* src, long count, int ndst, double* const* dsts);

/* Where the temporaries of the following calls on this handle come from.
 *   MFGP_WS_POOL    (default) stream-ordered allocations from the device's default memory pool, per call;
 *   MFGP_WS_MEASURE the same, and the library records the largest number of bytes one call takes;
 *   MFGP_WS_FIXED   one arena of the measured size is allocated NOW (call it outside any stream capture) and every
 *                   following call carves its temporaries out of it, starting again at its beginning (the predecessor's
 *                   temporaries are dead in stream order: keep the calls on one stream).  A call that needs more than was
 *                   measured takes the excess from the pool.
 * Back to MFGP_WS_POOL releases the arena (stream-ordered).  *bytes (may be NULL) receives the measured size (MEASURE ->
 * FIXED or POOL) or 0.  Purpose: library calls captured into a CUDA graph in FIXED mode contain NO allocation nodes, so the
 * graph owns no memory.  Captured in POOL mode the temporaries become graph-owned memory (1.3 GB for the Goku single-bin
 * SVGP step), which the driver keeps reserved after the graph is destroyed until mfgp_graph_mem_trim -- and once trimmed,
 * the next capture pays for reserving it again (measured: 1.0 s instead of 0.07 s per mfgp_svgp_adam call).
 * mfgp_svgp_adam does MEASURE (its eager first step) -> FIXED -> capture -> POOL itself; dist.py does the same around
 * torch.cuda.graph.  Not thread safe per handle, like everything else. */
#define MFGP_WS_POOL 0
#define MFGP_WS_MEASURE 1
#define MFGP_WS_FIXED 2
int mfgp_workspace(mfgp_handle* h, int mode, long* bytes);

/* Give the memory that DESTROYED CUDA graphs of the handle's device still reserve back to the driver
 * (cudaDeviceGraphMemTrim).  Only graphs that captured library calls in MFGP_WS_POOL mode own memory (see mfgp_workspace,
 * which avoids that at its root); call it after destroying such a graph.  Synchronises the stream. */
int mfgp_graph_mem_trim(mfgp_handle* h);

/* FP64 pipe microbenchmarks (bench.py: measured FP64 peak).  kind 0: DFMA, 1: DMMA m8n8k4, 2: both interleaved with equal
 * pipe time (tells whether the two share one datapath: same FLOP/s as either alone, or not: up to twice).
 * Returns achieved FLOP/s in *flops. */
int mfgp_fp64_peak(mfgp_handle* h, int kind, int iters, double* flops);

#ifdef __cplusplus
}
#endif
#endif /* MFGP_H */
