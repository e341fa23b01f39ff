// lbfgs.cu -- device-resident multi-start L-BFGS for the batched per-bin exact GPs (include/mfgp.h:
// mfgp_gpr_batched_lbfgs).  SciPy's L-BFGS-B on unbounded variables, one resumable state machine per problem: every round
// is one K6 launch over all problems at their current trial points and one lbfgs_step_kernel that consumes those values,
// advances each problem (line-search step, accept, termination, memory update, new direction) and writes its next trial
// point into the buffers K6 reads.  tests/_lbfgs_twin.py is the scalar NumPy statement of the same algorithm.
#include <cuda_runtime.h>

#include <climits>
#include <cmath>

#include "common.cuh"
#include "gpr_small.cuh"
#include "mathx.cuh"

namespace {

constexpr int LB_G = 32;             // lanes per problem: a warp, lanes over the n <= 36 variables
constexpr int LB_POLL = 16;          // rounds between two reads of the active-problem counter
constexpr double LB_STPMAX = 1e10;   // L-BFGS-B's stpmax for unbounded problems
constexpr double LB_NOISE_LOWER = 1e-6;
enum { ACT_NEW_ITER, ACT_TRIAL, ACT_ACCEPT, ACT_FAIL, ACT_DONE };
enum { TASK_FG, TASK_CONV, TASK_WARN, TASK_ERROR };

// MINPACK-2 dcsrch state (the dsave / isave of the Fortran) plus the step bounds of the current search.
struct Dcsrch {
    double stp, stpmax, finit, ginit, gtest, stx, fx, gx, sty, fy, gy, stmin, stmax, width, width1;
    int brackt, stage;
};

struct ProbState {
    Dcsrch ls;
    double f, fold, gdold;
    int phase;   // 0: the start point is being evaluated, 1: a line-search trial point is
    int status;  // 0 while running, then MFGP_LBFGS_*
    int nit, nfev, ifun, col, head, info;
};

struct LbArgs {
    int B, n, np, m, fix_rho, train_noise;
    int maxiter, maxfun, maxls;
    double ftol, gtol;
    ProbState* st;
    double* vec;  // per problem: x, g, t, r, d, z [n each], S [m][n], Y [m][n], dr [m]
    long per;     // doubles per problem in vec
    double* theta;        // [B, np]   what K6 reads
    double* noise;        // [B]
    const double* nlml;   // [B]       what K6 wrote
    const double* grad;   // [B, np+1]
    const int* kinfo;     // [B]
    int* active;          // problems still running
    int* first_bad;       // min over not_pd start points of b * 128 + pivot
};

// ---- MINPACK-2 dcstep / dcsrch (tests/_lbfgs_twin.py: dcstep, Dcsrch) -----------------------------------------
__device__ double sgn(double v) { return v > 0.0 ? 1.0 : (v < 0.0 ? -1.0 : 0.0); }

__device__ void dcstep(double& stx, double& fx, double& dx, double& sty, double& fy, double& dy, double& stp, double fp,
                       double dp, int& brackt, double stpmin, double stpmax) {
    const double sgnd = sgn(dp) * sgn(dx);
    double stpf;
    if (fp > fx) {
        const double theta = 3.0 * (fx - fp) / (stp - stx) + dx + dp;
        const double s = fmax(fabs(theta), fmax(fabs(dx), fabs(dp)));
        double gamma = s * sqrt((theta / s) * (theta / s) - (dx / s) * (dp / s));
        if (stp < stx) gamma = -gamma;
        const double p = (gamma - dx) + theta, q = ((gamma - dx) + gamma) + dp;
        const double stpc = stx + (p / q) * (stp - stx);
        const double stpq = stx + ((dx / ((fx - fp) / (stp - stx) + dx)) / 2.0) * (stp - stx);
        stpf = fabs(stpc - stx) <= fabs(stpq - stx) ? stpc : stpc + (stpq - stpc) / 2.0;
        brackt = 1;
    } else if (sgnd < 0.0) {
        const double theta = 3.0 * (fx - fp) / (stp - stx) + dx + dp;
        const double s = fmax(fabs(theta), fmax(fabs(dx), fabs(dp)));
        double gamma = s * sqrt((theta / s) * (theta / s) - (dx / s) * (dp / s));
        if (stp > stx) gamma = -gamma;
        const double p = (gamma - dp) + theta, q = ((gamma - dp) + gamma) + dx;
        const double stpc = stp + (p / q) * (stx - stp);
        const double stpq = stp + (dp / (dp - dx)) * (stx - stp);
        stpf = fabs(stpc - stp) > fabs(stpq - stp) ? stpc : stpq;
        brackt = 1;
    } else if (fabs(dp) < fabs(dx)) {
        const double theta = 3.0 * (fx - fp) / (stp - stx) + dx + dp;
        const double s = fmax(fabs(theta), fmax(fabs(dx), fabs(dp)));
        double gamma = s * sqrt(fmax(0.0, (theta / s) * (theta / s) - (dx / s) * (dp / s)));
        if (stp > stx) gamma = -gamma;
        const double p = (gamma - dp) + theta, q = (gamma + (dx - dp)) + gamma;
        const double r = p / q;
        double stpc;
        if (r < 0.0 && gamma != 0.0) stpc = stp + r * (stx - stp);
        else if (stp > stx) stpc = stpmax;
        else stpc = stpmin;
        const double stpq = stp + (dp / (dp - dx)) * (stx - stp);
        if (brackt) {
            stpf = fabs(stpc - stp) < fabs(stpq - stp) ? stpc : stpq;
            stpf = stp > stx ? fmin(stp + 0.66 * (sty - stp), stpf) : fmax(stp + 0.66 * (sty - stp), stpf);
        } else {
            stpf = fabs(stpc - stp) > fabs(stpq - stp) ? stpc : stpq;
            stpf = fmin(stpmax, fmax(stpmin, stpf));
        }
    } else {
        if (brackt) {
            const double theta = 3.0 * (fp - fy) / (sty - stp) + dy + dp;
            const double s = fmax(fabs(theta), fmax(fabs(dy), fabs(dp)));
            double gamma = s * sqrt((theta / s) * (theta / s) - (dy / s) * (dp / s));
            if (stp > sty) gamma = -gamma;
            const double p = (gamma - dp) + theta, q = ((gamma - dp) + gamma) + dy;
            stpf = stp + (p / q) * (sty - stp);
        } else {
            stpf = stp > stx ? stpmax : stpmin;
        }
    }
    if (fp > fx) {
        sty = stp; fy = fp; dy = dp;
    } else {
        if (sgnd < 0.0) { sty = stx; fy = fx; dy = dx; }
        stx = stp; fx = fp; dx = dp;
    }
    stp = stpf;
}

__device__ int dcsrch_start(Dcsrch& s, double stp, double f, double g, double stpmax) {
    s.stp = stp;
    s.stpmax = stpmax;
    if (stp < 0.0 || stp > stpmax || g >= 0.0) return TASK_ERROR;
    s.brackt = 0;
    s.stage = 1;
    s.finit = f;
    s.ginit = g;
    s.gtest = 1e-3 * g;
    s.width = stpmax;
    s.width1 = stpmax / 0.5;
    s.stx = 0.0; s.fx = f; s.gx = g;
    s.sty = 0.0; s.fy = f; s.gy = g;
    s.stmin = 0.0;
    s.stmax = stp + 4.0 * stp;
    return TASK_FG;
}

// f, g: the value and directional derivative at s.stp.  On TASK_FG s.stp is the next trial step.
__device__ int dcsrch_step(Dcsrch& s, double f, double g) {
    constexpr double gtol = 0.9, xtol = 0.1, stpmin = 0.0;  // with ftol = 1e-3 (gtest): L-BFGS-B's line-search constants
    double stp = s.stp;
    const double ftest = s.finit + stp * s.gtest;
    if (s.stage == 1 && f <= ftest && g >= 0.0) s.stage = 2;
    int task = TASK_FG;
    if (s.brackt && (stp <= s.stmin || stp >= s.stmax)) task = TASK_WARN;
    if (s.brackt && s.stmax - s.stmin <= xtol * s.stmax) task = TASK_WARN;
    if (stp == s.stpmax && f <= ftest && g <= s.gtest) task = TASK_WARN;
    if (stp == stpmin && (f > ftest || g >= s.gtest)) task = TASK_WARN;
    if (f <= ftest && fabs(g) <= gtol * -s.ginit) task = TASK_CONV;
    if (task != TASK_FG) return task;
    if (s.stage == 1 && f <= s.fx && f > ftest) {
        const double gt = s.gtest;
        double fxm = s.fx - s.stx * gt, fym = s.fy - s.sty * gt, gxm = s.gx - gt, gym = s.gy - gt;
        dcstep(s.stx, fxm, gxm, s.sty, fym, gym, stp, f - stp * gt, g - gt, s.brackt, s.stmin, s.stmax);
        s.fx = fxm + s.stx * gt;
        s.fy = fym + s.sty * gt;
        s.gx = gxm + gt;
        s.gy = gym + gt;
    } else {
        dcstep(s.stx, s.fx, s.gx, s.sty, s.fy, s.gy, stp, f, g, s.brackt, s.stmin, s.stmax);
    }
    if (s.brackt) {
        if (fabs(s.sty - s.stx) >= 0.66 * s.width1) stp = s.stx + 0.5 * (s.sty - s.stx);
        s.width1 = s.width;
        s.width = fabs(s.sty - s.stx);
        s.stmin = fmin(s.stx, s.sty);
        s.stmax = fmax(s.stx, s.sty);
    } else {
        s.stmin = stp + 1.1 * (stp - s.stx);
        s.stmax = stp + 4.0 * (stp - s.stx);
    }
    stp = fmin(s.stpmax, fmax(stpmin, stp));
    if ((s.brackt && (stp <= s.stmin || stp >= s.stmax)) || (s.brackt && s.stmax - s.stmin <= xtol * s.stmax)) stp = s.stx;
    s.stp = stp;
    return TASK_FG;
}

// ---- group reductions: the G lanes of one problem; a fixed xor tree, so every lane holds the same bits ----------
template <int G>
__device__ __forceinline__ double group_sum(double v) {
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o, G);
    return v;
}
template <int G>
__device__ __forceinline__ double group_max(double v) {
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o, G));
    return v;
}
template <int G>
__device__ __forceinline__ double dot(const double* a, const double* b, int n, int lane) {
    double s = 0.0;
    for (int j = lane; j < n; j += G) s = fma(a[j], b[j], s);
    return group_sum<G>(s);
}

// variable j -> index into theta [0, np) or np for the noise
__device__ __forceinline__ int var_slot(int j, int fix_rho) { return j + (fix_rho ? 1 : 0); }

__global__ void lbfgs_init_kernel(LbArgs a, const double* __restrict__ u, const double* __restrict__ noise_in) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= a.B) return;
    for (int q = 0; q < a.np; ++q) a.theta[(long)b * a.np + q] = softplus_fwd(u[(long)b * a.np + q]);
    double* x = a.vec + (long)b * a.per;
    for (int j = 0; j < a.n; ++j) {
        const int q = var_slot(j, a.fix_rho);
        x[j] = q < a.np ? u[(long)b * a.np + q] : 0.0;
    }
    if (a.train_noise) {
        const double s = noise_in[b] - LB_NOISE_LOWER;
        const double v = s + log(-expm1(-s));  // softplus^-1 (base.Transform.inverse); NaN for noise <= 1e-6: not_pd
        x[a.n - 1] = v;
        a.noise[b] = LB_NOISE_LOWER + softplus_fwd(v);
    } else {
        a.noise[b] = noise_in[b];
    }
    ProbState s{};
    a.st[b] = s;
    if (b == 0) {
        *a.active = a.B;
        *a.first_bad = INT_MAX;
    }
}

// One round for every problem: consume K6's value and gradient at the point in x, advance the state machine, and write
// the next trial point (or nothing, once the problem has finished).
template <int G>
__global__ void __launch_bounds__(256) lbfgs_step_kernel(LbArgs a) {
    const int lane = threadIdx.x % G;
    const int b = (int)(((long)blockIdx.x * blockDim.x + threadIdx.x) / G);
    if (b >= a.B) return;
    ProbState st = a.st[b];
    if (st.status) return;
    const int n = a.n, np = a.np, m = a.m;
    double* x = a.vec + (long)b * a.per;
    double *g = x + n, *t = x + 2 * n, *r = x + 3 * n, *d = x + 4 * n, *z = x + 5 * n;
    double *S = x + 6 * n, *Yv = S + (long)m * n, *DR = Yv + (long)m * n;

    // u-space gradient at x: d nlml / d theta * d theta / d u, d theta / d u = sigmoid(u) = 1 - exp(-softplus(u))
    const double fnew = a.nlml[b];
    bool ok = a.kinfo[b] == 0 && isfinite(fnew);
    for (int j = lane; j < n; j += G) {
        const int q = var_slot(j, a.fix_rho);
        const double th = q < np ? a.theta[(long)b * np + q] : softplus_fwd(x[j]);
        const double gj = a.grad[(long)b * (np + 1) + q] * (1.0 - exp(-th));
        g[j] = gj;
        ok = ok && isfinite(gj);
    }
    if (G > 1) ok = __all_sync(0xffffffffu, ok);
    st.nfev += 1;

    int act;
    if (st.phase == 0) {
        if (!ok) {
            st.status = MFGP_LBFGS_NOT_PD;
            st.info = a.kinfo[b];
            st.f = nan("");
            if (lane == 0 && st.info) atomicMin(a.first_bad, b * 128 + st.info);
            act = ACT_DONE;
        } else {
            st.f = fnew;
            double gm = 0.0;
            for (int j = lane; j < n; j += G) gm = fmax(gm, fabs(g[j]));
            if (group_max<G>(gm) <= a.gtol) {
                st.status = MFGP_LBFGS_PGTOL;
                act = ACT_DONE;
            } else {
                act = ACT_NEW_ITER;
            }
        }
    } else if (!ok) {  // a failed trial: a fresh search from the base point, short of the failed step
        const double bad = st.ls.stp;
        act = dcsrch_start(st.ls, 0.1 * bad, st.fold, st.gdold, 0.5 * bad) == TASK_FG ? ACT_TRIAL : ACT_FAIL;
    } else {
        st.f = fnew;
        const int task = dcsrch_step(st.ls, fnew, dot<G>(g, d, n, lane));
        act = task == TASK_CONV || task == TASK_WARN ? ACT_ACCEPT : (task == TASK_FG ? ACT_TRIAL : ACT_FAIL);
    }

    double al[MFGP_LBFGS_MAX_M];
    while (act != ACT_DONE) {
        if (act == ACT_ACCEPT) {
            st.nit += 1;
            double gm = 0.0;
            for (int j = lane; j < n; j += G) gm = fmax(gm, fabs(g[j]));
            gm = group_max<G>(gm);
            if (st.nit >= a.maxiter) st.status = MFGP_LBFGS_MAXITER;
            else if (st.nfev > a.maxfun) st.status = MFGP_LBFGS_MAXFUN;
            else if (gm <= a.gtol) st.status = MFGP_LBFGS_PGTOL;
            else if (st.fold - st.f <= a.ftol * fmax(fmax(fabs(st.fold), fabs(st.f)), 1.0)) st.status = MFGP_LBFGS_FTOL;
            if (st.status) { act = ACT_DONE; break; }
            // memory update: y = g - r, s = stp d, s^T y = dr from the directional derivatives (L-BFGS-B's matupd)
            const double stp = st.ls.stp;
            const double gd = dot<G>(g, d, n, lane);
            double dr = gd - st.gdold, ddum = -st.gdold;
            if (stp != 1.0) { dr *= stp; ddum *= stp; }
            if (!(dr <= 2.220446049250313e-16 * ddum)) {
                int slot;
                if (st.col < m) { slot = (st.head + st.col) % m; st.col += 1; }
                else { slot = st.head; st.head = (st.head + 1) % m; }
                for (int j = lane; j < n; j += G) {
                    S[(long)slot * n + j] = stp == 1.0 ? d[j] : stp * d[j];
                    Yv[(long)slot * n + j] = g[j] - r[j];
                }
                if (lane == 0) DR[slot] = dr;
                __syncwarp();
            }
            act = ACT_NEW_ITER;
        }
        if (act == ACT_FAIL) {  // restore the base point; clear the memory or stop
            for (int j = lane; j < n; j += G) { x[j] = t[j]; g[j] = r[j]; }
            st.f = st.fold;
            if (st.col == 0) {
                st.nit += 1;
                st.status = MFGP_LBFGS_ABNORMAL;
                act = ACT_DONE;
                break;
            }
            st.col = 0;
            st.head = 0;
            act = ACT_NEW_ITER;
        }
        if (act == ACT_NEW_ITER) {
            // d = -H g by the two-loop recursion, newest pair first; H0 = dr / y^T y of the newest pair
            for (int j = lane; j < n; j += G) d[j] = -g[j];
            if (st.col > 0) {
                __syncwarp();
                for (int k = st.col - 1; k >= 0; --k) {
                    const int i = (st.head + k) % m;
                    const double ai = dot<G>(S + (long)i * n, d, n, lane) / DR[i];
                    al[k] = ai;
                    for (int j = lane; j < n; j += G) d[j] -= ai * Yv[(long)i * n + j];
                }
                const int nw = (st.head + st.col - 1) % m;
                const double h0 = DR[nw] / dot<G>(Yv + (long)nw * n, Yv + (long)nw * n, n, lane);
                for (int j = lane; j < n; j += G) d[j] *= h0;
                for (int k = 0; k < st.col; ++k) {
                    const int i = (st.head + k) % m;
                    const double bi = dot<G>(Yv + (long)i * n, d, n, lane) / DR[i];
                    for (int j = lane; j < n; j += G) d[j] += (al[k] - bi) * S[(long)i * n + j];
                }
            }
            for (int j = lane; j < n; j += G) {
                z[j] = x[j] + d[j];
                d[j] = z[j] - x[j];
                t[j] = x[j];
                r[j] = g[j];
            }
            const double stp = st.nit == 0 ? fmin(1.0 / sqrt(dot<G>(d, d, n, lane)), LB_STPMAX) : 1.0;
            st.fold = st.f;
            st.ifun = 0;
            const double gd = dot<G>(g, d, n, lane);
            st.gdold = gd;
            act = gd < 0.0 && dcsrch_start(st.ls, stp, st.f, gd, LB_STPMAX) == TASK_FG ? ACT_TRIAL : ACT_FAIL;
        }
        if (act == ACT_TRIAL) {
            st.ifun += 1;
            if (st.ifun > a.maxls) { act = ACT_FAIL; continue; }
            const double stp = st.ls.stp;
            for (int j = lane; j < n; j += G) {
                const double v = stp == 1.0 ? z[j] : stp * d[j] + t[j];
                x[j] = v;
                const int q = var_slot(j, a.fix_rho);
                if (q < np) a.theta[(long)b * np + q] = softplus_fwd(v);
                else a.noise[b] = LB_NOISE_LOWER + softplus_fwd(v);
            }
            st.phase = 1;
            break;
        }
    }
    __syncwarp();
    if (lane == 0) {
        if (st.status) atomicSub(a.active, 1);
        a.st[b] = st;
    }
}

// Results: u and noise from x (not for a not_pd start: left as passed), f, nit, nfev, status, info.
__global__ void lbfgs_finish_kernel(LbArgs a, double* __restrict__ u, double* __restrict__ noise, double* __restrict__ f,
                                    int* __restrict__ nit, int* __restrict__ nfev, int* __restrict__ status,
                                    int* __restrict__ info) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= a.B) return;
    const ProbState st = a.st[b];
    const int s = st.status ? st.status : MFGP_LBFGS_MAXFUN;  // only past the round cap, which the loop does not reach
    if (s != MFGP_LBFGS_NOT_PD) {
        const double* x = a.vec + (long)b * a.per;
        for (int j = 0; j < a.n; ++j) {
            const int q = var_slot(j, a.fix_rho);
            if (q < a.np) u[(long)b * a.np + q] = x[j];
            else noise[b] = LB_NOISE_LOWER + softplus_fwd(x[j]);
        }
    }
    f[b] = st.f;
    nit[b] = st.nit;
    nfev[b] = st.nfev;
    status[b] = s;
    if (info) info[b] = st.info;
}

}  // namespace

extern "C" int mfgp_gpr_batched_lbfgs(mfgp_handle* h, const double* X, int N, int d, const double* Y, long ldy, int ycols,
                                      int B, double* u, double* noise, int fix_rho, int train_noise,
                                      const mfgp_lbfgs_opts* opts, double* f, int* nit, int* nfev, int* status, int* info) {
    if (!h) return MFGP_ERR_ARG;
    mfgp_lbfgs_opts o{10, 15000, 15000, 20, 2.220446049250313e-09, 1e-5};
    if (opts) o = *opts;
    if (!X || !Y || !u || !noise || !f || !nit || !nfev || !status || N < 1 || B < 0 || B > INT_MAX / 128 || d < 1 ||
        ycols < 1 || ldy < ycols || o.m < 1 || o.m > MFGP_LBFGS_MAX_M || o.maxiter < 1 || o.maxfun < 1 || o.maxls < 1 ||
        !(o.ftol >= 0.0) || !(o.gtol >= 0.0))
        return mfgp_fail(h, MFGP_ERR_ARG, "mfgp_gpr_batched_lbfgs: bad argument");
    if (N > MFGP_SMALL_MAX_N || d > MFGP_SMALL_MAX_D)
        return mfgp_fail(h, MFGP_ERR_UNSUPPORTED, "mfgp_gpr_batched_lbfgs: N <= 64 and d <= 16 only");
    cudaSetDevice(h->device);
    if (B == 0) return 0;
    const int np = 2 * d + 3;
    const int n = np - (fix_rho ? 1 : 0) + (train_noise ? 1 : 0);
    Scope sc(h);
    const double* dX = sc.in(X, (size_t)N * (d + 1));
    const double* dY = sc.in(Y, (size_t)N * ldy);
    double* du = sc.inout(u, (size_t)B * np);
    double* dnz = train_noise ? sc.inout(noise, B) : const_cast<double*>(sc.in(noise, B));
    double* df = sc.out(f, B);
    int* dnit = sc.out(nit, B);
    int* dnfev = sc.out(nfev, B);
    int* dstat = sc.out(status, B);
    int* dinfo = info ? sc.out(info, B) : nullptr;
    LbArgs a{};
    a.B = B; a.n = n; a.np = np; a.m = o.m; a.fix_rho = fix_rho ? 1 : 0; a.train_noise = train_noise ? 1 : 0;
    a.maxiter = o.maxiter; a.maxfun = o.maxfun; a.maxls = o.maxls; a.ftol = o.ftol; a.gtol = o.gtol;
    a.per = (long)(6 + 2 * o.m) * n + o.m;
    a.st = sc.alloc<ProbState>(B);
    a.vec = sc.alloc<double>((size_t)B * a.per);
    a.theta = sc.alloc<double>((size_t)B * np);
    a.noise = sc.alloc<double>(B);
    double* dnl = sc.alloc<double>(B);
    double* dg = sc.alloc<double>((size_t)B * (np + 1));
    int* dki = sc.alloc<int>(B);
    int* ctl = sc.alloc<int>(3, true);  // active, first_bad, and K6's first failure (not the handle's: failed trials are expected)
    int* hctl = nullptr;
    if (!sc.ok) return sc.finish();
    a.nlml = dnl; a.grad = dg; a.kinfo = dki; a.active = ctl; a.first_bad = ctl + 1;
    CUDA_TRY(h, cudaMallocHost(&hctl, 2 * sizeof(int)));
    int rc = 0;
    SmallArgs k{};
    k.X = dX; k.N = N; k.d = d; k.Y = dY; k.ldy = ldy; k.ycols = ycols; k.B = B;
    k.theta = a.theta; k.noise = a.noise; k.nlml = dnl; k.grad = dg; k.info = dki; k.d_info = ctl + 2;
    const int tb1 = 128, gb1 = (B + tb1 - 1) / tb1;
    const int tbs = 256, gbs = (int)(((long)B * LB_G + tbs - 1) / tbs);
    lbfgs_init_kernel<<<gb1, tb1, 0, h->stream>>>(a, du, dnz);
    // Every active problem makes one evaluation per round; past maxfun evaluations a problem ends within two line searches
    // (one that fails and clears the memory, one more), so the cap below is never the reason a loop stops.
    const long max_rounds = (long)o.maxfun + 2L * o.maxls + 2;
    for (long round = 0; !rc && round < max_rounds; ++round) {
        if (launch_gpr_small(h->stream, k)) { rc = mfgp_fail(h, MFGP_ERR_CUDA, "gpr_small launch failed"); break; }
        lbfgs_step_kernel<LB_G><<<gbs, tbs, 0, h->stream>>>(a);
        if ((round + 1) % LB_POLL == 0) {
            if (cudaMemcpyAsync(hctl, ctl, 2 * sizeof(int), cudaMemcpyDeviceToHost, h->stream) != cudaSuccess ||
                cudaStreamSynchronize(h->stream) != cudaSuccess) {
                rc = mfgp_fail(h, MFGP_ERR_CUDA, "mfgp_gpr_batched_lbfgs: %s", cudaGetErrorString(cudaGetLastError()));
                break;
            }
            if (hctl[0] == 0) break;
        }
    }
    if (!rc) {
        lbfgs_finish_kernel<<<gb1, tb1, 0, h->stream>>>(a, du, dnz, df, dnit, dnfev, dstat, dinfo);
        if (cudaMemcpyAsync(hctl, ctl, 2 * sizeof(int), cudaMemcpyDeviceToHost, h->stream) != cudaSuccess)
            rc = mfgp_fail(h, MFGP_ERR_CUDA, "mfgp_gpr_batched_lbfgs: copy failed");
    }
    sc.host_out = true;  // synchronise in finish(): the first-failure word is read below
    const int fin = sc.finish();
    const int first_bad = hctl[1];
    cudaFreeHost(hctl);
    if (rc) return rc;
    if (fin) return fin;
    if (first_bad != INT_MAX) {
        snprintf(h->err, sizeof(h->err), "Cholesky decomposition was not successful (problem %d, pivot %d not positive)",
                 first_bad / 128, first_bad % 128);
        return first_bad % 128;
    }
    return 0;
}
