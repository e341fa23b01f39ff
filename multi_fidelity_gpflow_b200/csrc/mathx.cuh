// mathx.cuh -- branch-free fp64 exp for the SE-kernel exponent (arguments <= ~0), and the FP64 tensor-core warp primitives.
#pragma once

// One mma.sync.m8n8k4.f64 (SASS: DMMA.8x8x4): C[8x8] += A[8x4] B[4x8].  Lane (g, t) = (lane / 4, lane % 4) holds
// A[g][t], B[t][g] and C[g][2t], C[g][2t + 1].
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

// Round-to-nearest range reduction, degree-13 Taylor/Horner on |r| <= ln2/2 (truncation 4e-18), exponent spliced
// into the high word.  Arguments below -700 are clamped (result ~1e-304 instead of a denormal / 0).
__device__ __forceinline__ double fexp(double x) {
    x = fmax(x, -700.0);
    const double t = fma(x, 1.4426950408889634074, 6755399441055744.0);
    const int n = __double2loint(t);
    const double nf = t - 6755399441055744.0;
    double r = fma(nf, -6.93147180369123816490e-01, x);
    r = fma(nf, -1.90821492927058770002e-10, r);
    double p = 1.6059043836821613e-10;            // 1/13!
    p = fma(p, r, 2.08767569878681e-09);          // 1/12!
    p = fma(p, r, 2.505210838544172e-08);         // 1/11!
    p = fma(p, r, 2.755731922398589e-07);         // 1/10!
    p = fma(p, r, 2.7557319223985893e-06);        // 1/9!
    p = fma(p, r, 2.48015873015873e-05);          // 1/8!
    p = fma(p, r, 1.984126984126984e-04);         // 1/7!
    p = fma(p, r, 1.388888888888889e-03);         // 1/6!
    p = fma(p, r, 8.333333333333333e-03);         // 1/5!
    p = fma(p, r, 4.1666666666666664e-02);        // 1/4!
    p = fma(p, r, 1.6666666666666666e-01);        // 1/3!
    p = fma(p, r, 0.5);
    p = fma(p, r, 1.0);
    p = fma(p, r, 1.0);
    return __hiloint2double(__double2hiint(p) + (n << 20), __double2loint(p));
}

// ---- table-driven exp: exp(x) = 2^k * 2^(j/64) * e^r, |r| <= ln2/128, degree-5 polynomial (truncation 3.5e-17) ----
// `tab` holds 2^(j/64), j = 0..63 (shared memory, filled by fexp_table_fill).  10 FP64-pipe instructions instead of 18.
// Returns exactly 0 below -700 (true value < 1e-304).
__device__ __forceinline__ void fexp_table_fill(double* tab, int tid, int nthreads) {
    for (int j = tid; j < 64; j += nthreads) tab[j] = exp2((double)j * (1.0 / 64.0));
}
__device__ __forceinline__ double fexp_tab(double x, const double* tab) {
    const double t = fma(x, 92.33248261689366, 6755399441055744.0);  // 64 / ln 2
    const int n = __double2loint(t);
    const double nf = t - 6755399441055744.0;
    double r = fma(nf, -0.01083042469326756, x);   // ln2/64, high part (trailing bits zero)
    r = fma(nf, -2.9815858269852933e-12, r);          // ln2/64, low part
    const double T = tab[n & 63];
    double q = fma(r, 8.3333333333333332e-03, 4.1666666666666664e-02);
    q = fma(q, r, 1.6666666666666666e-01);
    q = fma(q, r, 0.5);
    const double p = fma(q, r * r, r);
    double v = fma(T, p, T);
    v = __hiloint2double(__double2hiint(v) + ((n >> 6) << 20), __double2loint(v));
    return (x < -700.0) ? 0.0 : v;
}

// ---- 512-entry variant for the streaming covariance kernel (K1), where every non-FP64 instruction counts too ----
// exp(x) = 2^k * 2^(j/512) * e^r, n = 512 k + j = round(x * 512 / ln 2), |r| <= ln2/1024, degree-4 polynomial
// (truncation 1.6e-18; measured against a long-double exp: < 1 ulp).  Arguments below -700 are clamped with ONE unsigned
// integer min on the high word (negative doubles order like unsigned integers) instead of a compare and two selects on
// the result: the value is then ~1e-304, not 0.  9 FP64-pipe + 6 integer/LDS instructions, against 11 + 9 for fexp_tab.
// `tab` = 2^(j/512), 4 KB; declare it as a static __shared__ array so that its address is an immediate of the lookup.
__device__ __forceinline__ void fexp512_table_fill(double* tab, int tid, int nthreads) {
    for (int j = tid; j < 512; j += nthreads) tab[j] = exp2((double)j * (1.0 / 512.0));
}
__device__ __forceinline__ double fexp512(double x, const double* tab) {
    {
        const unsigned hi = min((unsigned)__double2hiint(x), 0xC085E000u);  // hi word of -700.0
        x = __hiloint2double((int)hi, __double2loint(x));
    }
    const double t = fma(x, 738.6598609351493, 6755399441055744.0);     // 512 / ln 2, 1.5 * 2^52
    const int n = __double2loint(t);
    const double nf = t - 6755399441055744.0;
    double r = fma(nf, -0.001353803086658445, x);                       // ln2/512, high part (21 trailing zero bits)
    r = fma(nf, -3.7269822837316166e-13, r);                            // ln2/512, low part
    const double T = tab[n & 511];
    double q = fma(r, 4.1666666666666664e-02, 1.6666666666666666e-01);
    q = fma(q, r, 0.5);
    const double p = fma(q, r * r, r);
    const double v = fma(T, p, T);
    return __hiloint2double(__double2hiint(v) + ((n >> 9) << 20), __double2loint(v));
}

// gpflow.utilities.positive(): tfp Softplus, lower = 0.  The device training loops (Adam, L-BFGS) share it, so that they
// optimise the same objective bit for bit.
__device__ __forceinline__ double softplus_fwd(double u) {
    return u > 0.0 ? u + log1p(exp(-u)) : log1p(exp(u));
}

// 1/sqrt(x) for positive normal x: hardware seed (rsqrt.approx.ftz.f64, ~2^-22) + two Newton steps (8 instructions
// against 13 for the CUDA library call, no special-case branch: x <= 0 / NaN give NaN or inf, which the caller detects).
__device__ __forceinline__ double frsqrt(double x) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    const double h = 0.5 * x;
    double e = fma(-(h * y), y, 0.5);
    y = fma(y, e, y);
    e = fma(-(h * y), y, 0.5);
    y = fma(y, e, y);
    return y;
}
