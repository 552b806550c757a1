// glg_math.h -- branch-free fp64 elementary functions for the GreenLight RHS.
//
// Why not libdevice: exp/log/cbrt/sqrt/div from libdevice carry a special-case test and an out-of-line slow path
// each (~70 BSSY/BSYNC regions and 34 CALLs per RHS in the first build, ncu: branch_resolving + no_instruction
// stalls), which chops the 2.5k-instruction RHS into small basic blocks so ptxas cannot interleave the ~30
// independent transcendental chains, and their polynomial coefficients are materialised with two MOVs each.
// Here every function is straight-line code, so the whole RHS is ONE basic block, and coefficients are
// `static const` doubles that ptxas folds into constant-bank operands of the DFMA.
//
// Accuracy (checked in tests/test_math_host.py against libm on 1e6 points each): <= 4e-16 relative, i.e. within
// a couple of ulp of the oracle's libm; the parity gate is 1e-9 per env-step.
// Domain: the arguments the model can produce.  Out-of-range inputs saturate instead of trapping:
//   glg_exp  : saturates at 2^-1021 / 2^1023 (never returns inf/0; 1/(1+exp(709)) flushes to 0, which
//              is the IEEE behaviour the reference's cond() relies on, aux_states.hpp:60-63)
//   glg_rcp / glg_sqrt / glg_cbrt / glg_log : positive normal arguments (the model adds 1e-10-type epsilons);
//              NaN propagates, so a diverged env still ends up flagged non-finite.
// Host build (tests only): same algorithms, seeds from libm.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <type_traits>

#if defined(__CUDACC__)
#define GLG_HD __host__ __device__ __forceinline__
#else
#define GLG_HD inline
#endif

// Polynomial coefficients live in the constant bank on the device: a DFMA can take one c[bank][offset] operand, so
// no instruction is spent on materialising 64-bit immediates (the first build spent ~400 IMAD.MOV/UMOV per RHS on
// that, which also pushed the RK4 loop past the 32 KB instruction cache of an SM).
#if defined(__CUDA_ARCH__)
#define GLG_COEF __constant__
#else
#define GLG_COEF static const
#endif
// Table-driven exp: x = (128 m + j) ln2/128 + r, |r| <= ln2/256; exp(x) = 2^m T[j] (1 + expm1(r)) with a degree-4 Taylor
// polynomial (remainder r^5/120 < 1.3e-15) and a one-constant argument reduction (error 1.2e-16 |x| relative): 8 FP64
// instructions per exp -- exp is the largest single item of the FP64 instruction stream of the RHS (25 per evaluation).
// Accuracy: <= 2e-15 + 1.2e-16 |x| relative (the model's arguments that matter stay below |x| ~ 40; the parity gate is 1e-9
// per env-step).  T[j] = 2^(j/128) is per-lane indexed: it lives in global memory and is read through the L1 (8 cache
// lines; the load is issued right after the reduction and consumed by the last FMA).
GLG_COEF double glg_kExpT[5] = {0x1.71547652b82fep+7 /*128/ln2*/, -0x1.62e42fefa39efp-8 /*-(ln2/128)*/,
                                0x1.5555555555555p-5 /*1/24*/, 0x1.5555555555555p-3 /*1/6*/, 0x1.0000000000000p-1};
#define GLG_EXP_TABLE_VALUES \
    0x1.0000000000000p+0, 0x1.0163da9fb3335p+0, 0x1.02c9a3e778061p+0, 0x1.04315e86e7f85p+0, \
    0x1.059b0d3158574p+0, 0x1.0706b29ddf6dep+0, 0x1.0874518759bc8p+0, 0x1.09e3ecac6f383p+0, \
    0x1.0b5586cf9890fp+0, 0x1.0cc922b7247f7p+0, 0x1.0e3ec32d3d1a2p+0, 0x1.0fb66affed31bp+0, \
    0x1.11301d0125b51p+0, 0x1.12abdc06c31ccp+0, 0x1.1429aaea92de0p+0, 0x1.15a98c8a58e51p+0, \
    0x1.172b83c7d517bp+0, 0x1.18af9388c8deap+0, 0x1.1a35beb6fcb75p+0, 0x1.1bbe084045cd4p+0, \
    0x1.1d4873168b9aap+0, 0x1.1ed5022fcd91dp+0, 0x1.2063b88628cd6p+0, 0x1.21f49917ddc96p+0, \
    0x1.2387a6e756238p+0, 0x1.251ce4fb2a63fp+0, 0x1.26b4565e27cddp+0, 0x1.284dfe1f56381p+0, \
    0x1.29e9df51fdee1p+0, 0x1.2b87fd0dad990p+0, 0x1.2d285a6e4030bp+0, 0x1.2ecafa93e2f56p+0, \
    0x1.306fe0a31b715p+0, 0x1.32170fc4cd831p+0, 0x1.33c08b26416ffp+0, 0x1.356c55f929ff1p+0, \
    0x1.371a7373aa9cbp+0, 0x1.38cae6d05d866p+0, 0x1.3a7db34e59ff7p+0, 0x1.3c32dc313a8e5p+0, \
    0x1.3dea64c123422p+0, 0x1.3fa4504ac801cp+0, 0x1.4160a21f72e2ap+0, 0x1.431f5d950a897p+0, \
    0x1.44e086061892dp+0, 0x1.46a41ed1d0057p+0, 0x1.486a2b5c13cd0p+0, 0x1.4a32af0d7d3dep+0, \
    0x1.4bfdad5362a27p+0, 0x1.4dcb299fddd0dp+0, 0x1.4f9b2769d2ca7p+0, 0x1.516daa2cf6642p+0, \
    0x1.5342b569d4f82p+0, 0x1.551a4ca5d920fp+0, 0x1.56f4736b527dap+0, 0x1.58d12d497c7fdp+0, \
    0x1.5ab07dd485429p+0, 0x1.5c9268a5946b7p+0, 0x1.5e76f15ad2148p+0, 0x1.605e1b976dc09p+0, \
    0x1.6247eb03a5585p+0, 0x1.6434634ccc320p+0, 0x1.6623882552225p+0, 0x1.68155d44ca973p+0, \
    0x1.6a09e667f3bcdp+0, 0x1.6c012750bdabfp+0, 0x1.6dfb23c651a2fp+0, 0x1.6ff7df9519484p+0, \
    0x1.71f75e8ec5f74p+0, 0x1.73f9a48a58174p+0, 0x1.75feb564267c9p+0, 0x1.780694fde5d3fp+0, \
    0x1.7a11473eb0187p+0, 0x1.7c1ed0130c132p+0, 0x1.7e2f336cf4e62p+0, 0x1.80427543e1a12p+0, \
    0x1.82589994cce13p+0, 0x1.8471a4623c7adp+0, 0x1.868d99b4492edp+0, 0x1.88ac7d98a6699p+0, \
    0x1.8ace5422aa0dbp+0, 0x1.8cf3216b5448cp+0, 0x1.8f1ae99157736p+0, 0x1.9145b0b91ffc6p+0, \
    0x1.93737b0cdc5e5p+0, 0x1.95a44cbc8520fp+0, 0x1.97d829fde4e50p+0, 0x1.9a0f170ca07bap+0, \
    0x1.9c49182a3f090p+0, 0x1.9e86319e32323p+0, 0x1.a0c667b5de565p+0, 0x1.a309bec4a2d33p+0, \
    0x1.a5503b23e255dp+0, 0x1.a799e1330b358p+0, 0x1.a9e6b5579fdbfp+0, 0x1.ac36bbfd3f37ap+0, \
    0x1.ae89f995ad3adp+0, 0x1.b0e07298db666p+0, 0x1.b33a2b84f15fbp+0, 0x1.b59728de5593ap+0, \
    0x1.b7f76f2fb5e47p+0, 0x1.ba5b030a1064ap+0, 0x1.bcc1e904bc1d2p+0, 0x1.bf2c25bd71e09p+0, \
    0x1.c199bdd85529cp+0, 0x1.c40ab5fffd07ap+0, 0x1.c67f12e57d14bp+0, 0x1.c8f6d9406e7b5p+0, \
    0x1.cb720dcef9069p+0, 0x1.cdf0b555dc3fap+0, 0x1.d072d4a07897cp+0, 0x1.d2f87080d89f2p+0, \
    0x1.d5818dcfba487p+0, 0x1.d80e316c98398p+0, 0x1.da9e603db3285p+0, 0x1.dd321f301b460p+0, \
    0x1.dfc97337b9b5fp+0, 0x1.e264614f5a129p+0, 0x1.e502ee78b3ff6p+0, 0x1.e7a51fbc74c83p+0, \
    0x1.ea4afa2a490dap+0, 0x1.ecf482d8e67f1p+0, 0x1.efa1bee615a27p+0, 0x1.f252b376bba97p+0, \
    0x1.f50765b6e4540p+0, 0x1.f7bfdad9cbe14p+0, 0x1.fa7c1819e90d8p+0, 0x1.fd3c22b8f71f1p+0
#if defined(__CUDACC__)
__device__ const double glg_exp_tbl_dev[128] = {GLG_EXP_TABLE_VALUES};
// Per-CTA copy of the table in shared memory (a 32-bit address and an LDS instead of a 64-bit address and an L1 load: two integer
// instructions fewer per exp).  Every kernel that evaluates an exp calls glg_exp_tbl_fill() before its first use.
__shared__ double glg_exp_tbl_sh[128];
__device__ __forceinline__ void glg_exp_tbl_fill() {
    for (int i = threadIdx.x; i < 128; i += blockDim.x) glg_exp_tbl_sh[i] = glg_exp_tbl_dev[i];
    __syncthreads();
}
#endif
static const double glg_exp_tbl_host[128] = {GLG_EXP_TABLE_VALUES};
GLG_COEF double glg_kLog[9] = {
    0x1.2b584aae78a57p-3, 0x1.39fe606542ddep-3, 0x1.7462b4ab2ef6bp-3, 0x1.c71c62e5800a1p-3, 0x1.2492492df148dp-2,
    0x1.99999999952e2p-2, 0x1.5555555555558p-1, 0x1.62e42fee00000p-1 /*ln2_hi*/, 0x1.a39ef35793c76p-33 /*ln2_lo*/};

GLG_HD double glg_bits2d(long long b) {
#if defined(__CUDA_ARCH__)
    return __longlong_as_double(b);
#else
    double d;
    memcpy(&d, &b, 8);
    return d;
#endif
}
GLG_HD long long glg_d2bits(double d) {
#if defined(__CUDA_ARCH__)
    return __double_as_longlong(d);
#else
    long long b;
    memcpy(&b, &d, 8);
    return b;
#endif
}
GLG_HD double glg_fma(double a, double b, double c) {
#if defined(__CUDA_ARCH__)
    return __fma_rn(a, b, c);
#else
    return fma(a, b, c);
#endif
}

// ---- reciprocal: ~20-bit hardware seed (MUFU.RCP64H) + one cubic correction: r = r0 (1 + e + e^2), e = 1 - x r0
GLG_HD double glg_rcp(double x) {
#if defined(__CUDA_ARCH__)
    double r0;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r0) : "d"(x));
    const double e = __fma_rn(-x, r0, 1.0);
    const double t = __fma_rn(e, e, e);
    return __fma_rn(r0, t, r0);  // seed error 2^-20 -> e^3 = 2^-60
#else
    return 1.0 / x;
#endif
}
GLG_HD double glg_div(double a, double b) { return a * glg_rcp(b); }

// ---- sqrt for x > 0: rsqrt seed (MUFU.RSQ64H, ~2^-20) + one coupled Goldschmidt step (2^-40) + a residual correction
GLG_HD double glg_sqrt(double x) {
#if defined(__CUDA_ARCH__)
    double r;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    double g = x * r, h = 0.5 * r;
    const double e = __fma_rn(-h, g, 0.5);
    g = __fma_rn(g, e, g);
    h = __fma_rn(h, e, h);
    const double d = __fma_rn(-g, g, x);
    return __fma_rn(d, h, g);
#else
    return sqrt(x);
#endif
}

// ---- exp (table-driven, see glg_kExpT).  2^m goes through the exponent field; m is clamped on the integer pipe so the
//      result stays a normal number and the function saturates (~1e-308 / ~1e308) instead of wrapping for |x| > 708.
GLG_HD double glg_exp_tbl(int j) {
#if defined(__CUDA_ARCH__)
    // address = base + 8 j as ONE multiply-add (left to itself the compiler emits shift, mask and add), 32-bit shared-window load
    unsigned a;
    double T;
    asm("mad.lo.u32 %0, %1, 8, %2;" : "=r"(a) : "r"(j), "r"((unsigned)__cvta_generic_to_shared(glg_exp_tbl_sh)));
    asm("ld.shared.f64 %0, [%1];" : "=d"(T) : "r"(a));
    return T;
#else
    return glg_exp_tbl_host[j];
#endif
}
// y 2^m for y in [1, 2) and m in [-1021, 1023]: m goes into the exponent field -- of the high word alone on the device (a 64-bit
// integer add costs a second instruction for a carry that cannot happen)
GLG_HD double glg_scale2(double y, int m) {
#if defined(__CUDA_ARCH__)
    return __hiloint2double(__double2hiint(y) + (m << 20), __double2loint(y));
#else
    return glg_bits2d(glg_d2bits(y) + ((long long)m << 52));
#endif
}
GLG_HD double glg_exp(double x) {
    const double MAGIC = 6755399441055744.0;  // 1.5 * 2^52: adding it rounds to nearest integer in the low word
    const double t = glg_fma(x, glg_kExpT[0], MAGIC);
    const double kf = t - MAGIC;
    const int k = (int)(uint32_t)(uint64_t)glg_d2bits(t);  // two's complement in the low word, valid for |x| < 2^23
    const double T = glg_exp_tbl(k & 127);
    const double r = glg_fma(kf, glg_kExpT[1], x);
    const double r2 = r * r;
    double q = glg_fma(r, glg_kExpT[2], glg_kExpT[3]);
    q = glg_fma(r, q, glg_kExpT[4]);
    const double p = glg_fma(r2, q, r);  // expm1(r)
    const double y = glg_fma(T, p, T);   // in [1, 2)
    int m = k >> 7;
    m = m < -1021 ? -1021 : (m > 1023 ? 1023 : m);
    return glg_scale2(y, m);
}

// ---- accurate exp (<= 4e-16 relative): two-constant argument reduction, degree-5 polynomial.  For once-per-env-step code
//      whose closed loop amplifies rounding differences (rule-based controller, glg_controller.h); not used by the RHS.
GLG_HD double glg_exp_acc(double x) {
    const double MAGIC = 6755399441055744.0;
    const double t = glg_fma(x, glg_kExpT[0], MAGIC);
    const double kf = t - MAGIC;
    const int k = (int)(uint32_t)(uint64_t)glg_d2bits(t);
    const double T = glg_exp_tbl(k & 127);
    double r = glg_fma(kf, -0x1.62e42fef80000p-8 /*-(ln2/128)_hi, 34 bits*/, x);
    r = glg_fma(kf, -0x1.1cf79abc9e3b4p-43 /*-(ln2/128)_lo*/, r);
    double q = glg_fma(r, 0x1.1111111111111p-7 /*1/120*/, glg_kExpT[2]);
    q = glg_fma(r, q, glg_kExpT[3]);
    q = glg_fma(r, q, glg_kExpT[4]);
    const double y = glg_fma(T, glg_fma(r * r, q, r), T);
    int m = k >> 7;
    m = m < -1021 ? -1021 : (m > 1023 ? 1023 : m);
    return glg_scale2(y, m);
}

// ---- N independent exps with their dependency chains interleaved in SOURCE order.  The hardware issues in order and
//      ptxas does not interleave independent chains by itself; writing the steps "step-major" gives a lone warp N-way
//      ILP at zero extra instructions.
template <int N>
GLG_HD void glg_exp_n(const double (&x)[N], double (&y)[N]) {
    const double MAGIC = 6755399441055744.0;
    double t[N], r[N], T[N], r2[N], q[N];
    int k[N];
#pragma unroll
    for (int i = 0; i < N; ++i) t[i] = glg_fma(x[i], glg_kExpT[0], MAGIC);
#pragma unroll
    for (int i = 0; i < N; ++i) {
        k[i] = (int)(uint32_t)(uint64_t)glg_d2bits(t[i]);
        T[i] = glg_exp_tbl(k[i] & 127);
    }
#pragma unroll
    for (int i = 0; i < N; ++i) r[i] = glg_fma(t[i] - MAGIC, glg_kExpT[1], x[i]);
#pragma unroll
    for (int i = 0; i < N; ++i) { r2[i] = r[i] * r[i]; q[i] = glg_fma(r[i], glg_kExpT[2], glg_kExpT[3]); }
#pragma unroll
    for (int i = 0; i < N; ++i) q[i] = glg_fma(r[i], q[i], glg_kExpT[4]);
#pragma unroll
    for (int i = 0; i < N; ++i) q[i] = glg_fma(r2[i], q[i], r[i]);
#pragma unroll
    for (int i = 0; i < N; ++i) {
        const double v = glg_fma(T[i], q[i], T[i]);
        int m = k[i] >> 7;
        m = m < -1021 ? -1021 : (m > 1023 ? 1023 : m);
        y[i] = glg_scale2(v, m);
    }
}
// N independent reciprocals, interleaved the same way
template <int N>
GLG_HD void glg_rcp_n(const double (&x)[N], double (&y)[N]) {
#if defined(__CUDA_ARCH__)
    double r0[N], e[N];
#pragma unroll
    for (int i = 0; i < N; ++i) asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r0[i]) : "d"(x[i]));
#pragma unroll
    for (int i = 0; i < N; ++i) e[i] = __fma_rn(-x[i], r0[i], 1.0);
#pragma unroll
    for (int i = 0; i < N; ++i) e[i] = __fma_rn(e[i], e[i], e[i]);
#pragma unroll
    for (int i = 0; i < N; ++i) y[i] = __fma_rn(r0[i], e[i], r0[i]);
#else
    for (int i = 0; i < N; ++i) y[i] = 1.0 / x[i];
#endif
}

// N independent square roots / cube roots, interleaved
template <int N>
GLG_HD void glg_sqrt_n(const double (&x)[N], double (&y)[N]) {
#if defined(__CUDA_ARCH__)
    double g[N], h[N], e[N];
#pragma unroll
    for (int i = 0; i < N; ++i) asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(h[i]) : "d"(x[i]));
#pragma unroll
    for (int i = 0; i < N; ++i) { g[i] = x[i] * h[i]; h[i] = 0.5 * h[i]; }
#pragma unroll
    for (int i = 0; i < N; ++i) e[i] = __fma_rn(-h[i], g[i], 0.5);
#pragma unroll
    for (int i = 0; i < N; ++i) { g[i] = __fma_rn(g[i], e[i], g[i]); h[i] = __fma_rn(h[i], e[i], h[i]); }
#pragma unroll
    for (int i = 0; i < N; ++i) e[i] = __fma_rn(-g[i], g[i], x[i]);
#pragma unroll
    for (int i = 0; i < N; ++i) y[i] = __fma_rn(e[i], h[i], g[i]);
#else
    for (int i = 0; i < N; ++i) y[i] = sqrt(x[i]);
#endif
}
template <int N>
GLG_HD void glg_cbrt_n(const double (&x)[N], double (&y)[N]) {  // see glg_cbrt
    const double third = 0x1.5555555555555p-2;
    double r[N], s[N], d[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
#if defined(__CUDA_ARCH__)
        const float xf = fmaxf(__double2float_rn(x[i]), 1e-36f);
        float lg, sd;
        asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(xf));
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(sd) : "f"(-0.33333334f * lg));
        r[i] = (double)sd;
#else
        r[i] = (double)(float)(1.0 / cbrt(fmax(x[i], 1e-36))) * (1.0 + 1e-7);
#endif
    }
#pragma unroll
    for (int i = 0; i < N; ++i) r[i] = r[i] * r[i];
#pragma unroll
    for (int i = 0; i < N; ++i) { y[i] = x[i] * r[i]; s[i] = r[i] * third; }
#pragma unroll
    for (int it = 0; it < 2; ++it) {
#pragma unroll
        for (int i = 0; i < N; ++i) d[i] = y[i] * y[i];
#pragma unroll
        for (int i = 0; i < N; ++i) d[i] = glg_fma(-d[i], y[i], x[i]);
#pragma unroll
        for (int i = 0; i < N; ++i) y[i] = glg_fma(d[i], s[i], y[i]);
    }
}

// ---- 1/(1+exp(z)) -- the model's ubiquitous sigmoid building block
GLG_HD double glg_inv1pexp(double z) { return glg_rcp(1.0 + glg_exp(z)); }

// ---- natural log for positive normal x: x = m 2^e, m in [sqrt(1/2), sqrt(2)); f = (m-1)/(m+1);
//      log m = 2f + f^3 P(f^2), P degree 6 (abs err 3e-16 on P => < 2e-18 on the log)
GLG_HD double glg_log(double x) {
    const long long SQRT_HALF_BITS = 0x3FE6A09E667F3BCDLL;  // bits of sqrt(1/2)
    long long b = glg_d2bits(x);
    // exponent such that the remaining mantissa lies in [sqrt(1/2), sqrt(2))
    const long long eb = (b - SQRT_HALF_BITS) >> 52;
    b -= eb << 52;
    const double m = glg_bits2d(b);
    const double e = (double)(int)eb;
    const double f = (m - 1.0) * glg_rcp(m + 1.0);
    const double s = f * f;
    double p = glg_kLog[0];
    p = glg_fma(p, s, glg_kLog[1]);
    p = glg_fma(p, s, glg_kLog[2]);
    p = glg_fma(p, s, glg_kLog[3]);
    p = glg_fma(p, s, glg_kLog[4]);
    p = glg_fma(p, s, glg_kLog[5]);
    p = glg_fma(p, s, glg_kLog[6]);
    const double lm = glg_fma(f * s, p, 2.0 * f);
    return glg_fma(e, glg_kLog[7], glg_fma(e, glg_kLog[8], lm));
}
GLG_HD double glg_pow(double b, double e) { return glg_exp(e * glg_log(b)); }  // b > 0

// ---- cube root for x > 0: fp32 seed r ~ x^(-1/3) (MUFU.LG2/EX2, relative error d ~ 2^-21), y0 = x r^2, then two steps of
//      y <- y + (x - y^3) s with the FIXED slope s = r^2/3 ~ 1/(3 y^2): the error goes d -> d^2 -> d^3 (2^-63), at 3 FP64
//      instructions per step and no division: 9 FP64 instructions in all.
GLG_HD double glg_cbrt(double x) {
#if defined(__CUDA_ARCH__)
    // seed in fp32 on the MUFU pipe; clamped so x = 0 gives a finite r (and then cbrt = 0 * r^2 = 0)
    const float xf = fmaxf(__double2float_rn(x), 1e-36f);
    float lg, sd;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(xf));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(sd) : "f"(-0.33333334f * lg));
    const double r = (double)sd;
#else
    const double r = (double)(float)(1.0 / cbrt(fmax(x, 1e-36))) * (1.0 + 1e-7);  // deliberately imperfect seed, like the device's
#endif
    const double r2 = r * r;
    const double s = r2 * 0x1.5555555555555p-2;
    double y = x * r2;
    y = glg_fma(glg_fma(-(y * y), y, x), s, y);
    y = glg_fma(glg_fma(-(y * y), y, x), s, y);
    return y;
}

// ---- x^(1/3) (cube = true) or x^(1/4) (cube = false) for x > 0, selected per lane WITHOUT divergence: fp32 seed of
//      r = x^(-1/n) (MUFU.LG2/EX2), two Newton steps r <- r + r (1 - x r^n)/n (quadratic: 2^-22 -> 2^-44 -> rounding), then
//      x^(1/n) = x r^(n-1).  Used where the model switches between the two roots on a state comparison (floor <-> air
//      free convection, aux_states.hpp:876): a warp whose lanes disagree would otherwise execute both root routines in turn.
GLG_HD double glg_root34(double x, bool cube) {
    const double invn = cube ? 0x1.5555555555555p-2 : 0.25;
#if defined(__CUDA_ARCH__)
    const float xf = fmaxf(__double2float_rn(x), 1e-36f);
    float lg, sd;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(xf));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(sd) : "f"((cube ? -0.33333334f : -0.25f) * lg));
    double r = (double)sd;
#else
    double r = (double)(float)pow(fmax(x, 1e-36), cube ? -1.0 / 3.0 : -0.25) * (1.0 + 1e-7);  // deliberately imperfect seed
#endif
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int it = 0; it < 2; ++it) {
        const double r2 = r * r;
        const double rn = r2 * (cube ? r : r2);
        const double e = glg_fma(-x, rn, 1.0);
        r = glg_fma(r * invn, e, r);
    }
    const double r2 = r * r;
    return x * (cube ? r2 : r2 * r);
}

// dispatcher used by the accuracy tests (host build and the glg_debug_math kernel)
GLG_HD double glg_math_eval(int op, double v) {
    switch (op) {
        case 0: return glg_exp(v);
        case 1: return glg_log(v);
        case 2: return glg_rcp(v);
        case 3: return glg_sqrt(v);
        case 4: return glg_cbrt(v);
        case 5: return glg_pow(v, 0.66);
        case 6: return glg_pow(v, 0.32);
        case 7: return glg_inv1pexp(v);
        case 8: return glg_root34(v, true);
        case 9: return glg_root34(v, false);
        case 10: return glg_exp_acc(v);
        default: return v;
    }
}

// =========================================================================================================
// fp32 versions (throughput mode, glg_config.precision = 1): the hardware's approximate MUFU functions are already at
// fp32 accuracy (2^-22 .. 2^-23 relative), so each elementary function is 1-3 instructions and needs no interleaving.
// inf/0 semantics are IEEE-like: exp saturates to +inf / 0, rcp(inf) = 0 -- cond()'s 1/(1+exp(big)) = 0 holds
// (aux_states.hpp:60-63 overflows fp32 routinely, SURVEY.md 7.3 item 4).
// =========================================================================================================
GLG_HD float glg_rcp(float x) {
#if defined(__CUDA_ARCH__)
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#else
    return 1.0f / x;
#endif
}
GLG_HD float glg_sqrt(float x) {
#if defined(__CUDA_ARCH__)
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#else
    return sqrtf(x);
#endif
}
GLG_HD float glg_exp(float x) {
#if defined(__CUDA_ARCH__)
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x * 1.4426950408889634f));
    return r;
#else
    return expf(x);
#endif
}
GLG_HD float glg_log(float x) {
#if defined(__CUDA_ARCH__)
    float r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r * 0.6931471805599453f;
#else
    return logf(x);
#endif
}
GLG_HD float glg_pow(float b, float e) {
#if defined(__CUDA_ARCH__)
    float l, r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(b));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e * l));
    return r;
#else
    return powf(b, e);
#endif
}
GLG_HD float glg_cbrt(float x) {
#if defined(__CUDA_ARCH__)
    const float xc = fmaxf(x, 1e-36f);
    float l, y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(xc));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(0.33333334f * l));
    // one Newton step on y^3 = x:  y <- y - (y^3 - x) / (3 y^2)
    const float y2 = y * y;
    return x == 0.0f ? 0.0f : y - (y2 * y - x) * glg_rcp(3.0f * y2);
#else
    return cbrtf(x);
#endif
}
GLG_HD float glg_root34(float x, bool cube) {
#if defined(__CUDA_ARCH__)
    const float xc = fmaxf(x, 1e-36f);
    float l, y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(xc));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"((cube ? 0.33333334f : 0.25f) * l));
    return x == 0.0f ? 0.0f : y;
#else
    return cube ? cbrtf(x) : sqrtf(sqrtf(x));
#endif
}
GLG_HD float glg_inv1pexp(float z) { return glg_rcp(1.0f + glg_exp(z)); }
template <int N>
GLG_HD void glg_exp_n(const float (&x)[N], float (&y)[N]) {
#pragma unroll
    for (int i = 0; i < N; ++i) y[i] = glg_exp(x[i]);
}
template <int N>
GLG_HD void glg_rcp_n(const float (&x)[N], float (&y)[N]) {
#pragma unroll
    for (int i = 0; i < N; ++i) y[i] = glg_rcp(x[i]);
}
template <int N>
GLG_HD void glg_sqrt_n(const float (&x)[N], float (&y)[N]) {
#pragma unroll
    for (int i = 0; i < N; ++i) y[i] = glg_sqrt(x[i]);
}
template <int N>
GLG_HD void glg_cbrt_n(const float (&x)[N], float (&y)[N]) {
#pragma unroll
    for (int i = 0; i < N; ++i) y[i] = glg_cbrt(x[i]);
}

// =========================================================================================================
// Forward-mode tangents (glg_tangent.cuh): GlgDual<N> is an fp64 value and N fp64 tangent directions.  The flux units, the hoist
// and the RK4 tangent are templates over their scalar type, so instantiating them with GlgDual<N> gives the exact derivative of
// the same arithmetic: every value part goes through exactly the double function above, so it is what the double code computes.
// Derivatives are formed from the primal result where possible (exp' = y, rcp' = -y^2, sqrt' = 0.5/y, cbrt' = y/(3x),
// pow(b, e)' = e y / b, inv1pexp' = -y (1 - y)).
// Conventions at non-smooth points:
//   fabs'(0) = 0 (CasADi's sign(0) = 0);
//   fmin / fmax / ?: carry the derivative of the branch the primal takes (the first argument on a tie);
//   exponents of glg_pow / pow are constants: their tangent is not propagated (every call site passes a literal);
//   step-count decisions (harvest micro-steps, the graded integrator's splits) are taken on value parts only, so a tangent is
//   the exact derivative of the discrete map on the grid that was executed.
// Operators with a plain double exist so constants (K, C, p) cost no tangent arithmetic: 0 * x cannot be folded under IEEE rules.
// =========================================================================================================
template <int N>
struct GlgDual {
    double v;
    double t[N];
    GlgDual() = default;
    GLG_HD GlgDual(double a) : v(a) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (int i = 0; i < N; ++i) t[i] = 0.0;
    }
    GLG_HD GlgDual &operator+=(const GlgDual &b) { return *this = *this + b; }
    GLG_HD GlgDual &operator-=(const GlgDual &b) { return *this = *this - b; }
    GLG_HD GlgDual &operator*=(const GlgDual &b) { return *this = *this * b; }
    GLG_HD GlgDual &operator+=(double b) { v += b; return *this; }
    GLG_HD GlgDual &operator-=(double b) { v -= b; return *this; }
};
template <class T>
struct glg_is_dual : std::false_type {};
template <int N>
struct glg_is_dual<GlgDual<N>> : std::true_type {};

GLG_HD double glg_value(double a) { return a; }
GLG_HD float glg_value(float a) { return a; }
template <int N>
GLG_HD double glg_value(const GlgDual<N> &a) { return a.v; }

// y with tangent s * a.t: the chain rule of a unary function whose derivative at a.v is s
template <int N>
GLG_HD GlgDual<N> glg_chain(double y, double s, const GlgDual<N> &a) {
    GlgDual<N> r;
    r.v = y;
#pragma unroll
    for (int i = 0; i < N; ++i) r.t[i] = s * a.t[i];
    return r;
}

template <int N>
GLG_HD GlgDual<N> operator-(const GlgDual<N> &a) { return glg_chain(-a.v, -1.0, a); }
template <int N>
GLG_HD GlgDual<N> operator+(const GlgDual<N> &a, const GlgDual<N> &b) {
    GlgDual<N> r;
    r.v = a.v + b.v;
#pragma unroll
    for (int i = 0; i < N; ++i) r.t[i] = a.t[i] + b.t[i];
    return r;
}
template <int N>
GLG_HD GlgDual<N> operator-(const GlgDual<N> &a, const GlgDual<N> &b) {
    GlgDual<N> r;
    r.v = a.v - b.v;
#pragma unroll
    for (int i = 0; i < N; ++i) r.t[i] = a.t[i] - b.t[i];
    return r;
}
template <int N>
GLG_HD GlgDual<N> operator*(const GlgDual<N> &a, const GlgDual<N> &b) {
    GlgDual<N> r;
    r.v = a.v * b.v;
#pragma unroll
    for (int i = 0; i < N; ++i) r.t[i] = a.t[i] * b.v + a.v * b.t[i];
    return r;
}
template <int N>
GLG_HD GlgDual<N> operator/(const GlgDual<N> &a, const GlgDual<N> &b) {
    GlgDual<N> r;
    r.v = a.v / b.v;
    const double ib = 1.0 / b.v;
#pragma unroll
    for (int i = 0; i < N; ++i) r.t[i] = (a.t[i] - r.v * b.t[i]) * ib;
    return r;
}
template <int N>
GLG_HD GlgDual<N> operator+(const GlgDual<N> &a, double b) {
    GlgDual<N> r = a;
    r.v = a.v + b;
    return r;
}
template <int N>
GLG_HD GlgDual<N> operator+(double a, const GlgDual<N> &b) {
    GlgDual<N> r = b;
    r.v = a + b.v;
    return r;
}
template <int N>
GLG_HD GlgDual<N> operator-(const GlgDual<N> &a, double b) {
    GlgDual<N> r = a;
    r.v = a.v - b;
    return r;
}
template <int N>
GLG_HD GlgDual<N> operator-(double a, const GlgDual<N> &b) { return glg_chain(a - b.v, -1.0, b); }
template <int N>
GLG_HD GlgDual<N> operator*(const GlgDual<N> &a, double b) { return glg_chain(a.v * b, b, a); }
template <int N>
GLG_HD GlgDual<N> operator*(double a, const GlgDual<N> &b) { return glg_chain(a * b.v, a, b); }
template <int N>
GLG_HD GlgDual<N> operator/(const GlgDual<N> &a, double b) { return glg_chain(a.v / b, 1.0 / b, a); }
template <int N>
GLG_HD GlgDual<N> operator/(double a, const GlgDual<N> &b) {
    const double y = a / b.v;
    return glg_chain(y, -y / b.v, b);
}
#define GLG_DUAL_CMP(OP)                                                                                   \
    template <int N>                                                                                       \
    GLG_HD bool operator OP(const GlgDual<N> &a, const GlgDual<N> &b) { return a.v OP b.v; }             \
    template <int N>                                                                                       \
    GLG_HD bool operator OP(const GlgDual<N> &a, double b) { return a.v OP b; }                           \
    template <int N>                                                                                       \
    GLG_HD bool operator OP(double a, const GlgDual<N> &b) { return a OP b.v; }
GLG_DUAL_CMP(<)
GLG_DUAL_CMP(>)
GLG_DUAL_CMP(<=)
GLG_DUAL_CMP(>=)
GLG_DUAL_CMP(==)
GLG_DUAL_CMP(!=)
#undef GLG_DUAL_CMP

template <int N>
GLG_HD GlgDual<N> fabs(const GlgDual<N> &a) { return glg_chain(fabs(a.v), a.v > 0.0 ? 1.0 : (a.v < 0.0 ? -1.0 : 0.0), a); }
template <int N>
GLG_HD GlgDual<N> fmin(const GlgDual<N> &a, const GlgDual<N> &b) {
    GlgDual<N> r = b.v < a.v ? b : a;
    r.v = fmin(a.v, b.v);
    return r;
}
template <int N>
GLG_HD GlgDual<N> fmax(const GlgDual<N> &a, const GlgDual<N> &b) {
    GlgDual<N> r = b.v > a.v ? b : a;
    r.v = fmax(a.v, b.v);
    return r;
}
template <int N>
GLG_HD GlgDual<N> sqrt(const GlgDual<N> &a) {
    const double y = sqrt(a.v);
    return glg_chain(y, 0.5 / y, a);
}
template <int N>
GLG_HD GlgDual<N> exp(const GlgDual<N> &a) {
    const double y = exp(a.v);
    return glg_chain(y, y, a);
}
template <int N>
GLG_HD GlgDual<N> pow(const GlgDual<N> &b, double e) {
    const double y = pow(b.v, e);
    return glg_chain(y, e * y / b.v, b);
}

template <int N>
GLG_HD GlgDual<N> glg_exp(const GlgDual<N> &a) {
    const double y = glg_exp(a.v);
    return glg_chain(y, y, a);
}
template <int N>
GLG_HD GlgDual<N> glg_rcp(const GlgDual<N> &a) {
    const double y = glg_rcp(a.v);
    return glg_chain(y, -(y * y), a);
}
template <int N>
GLG_HD GlgDual<N> glg_sqrt(const GlgDual<N> &a) {
    const double y = glg_sqrt(a.v);
    return glg_chain(y, 0.5 / y, a);
}
template <int N>
GLG_HD GlgDual<N> glg_cbrt(const GlgDual<N> &a) {
    const double y = glg_cbrt(a.v);
    return glg_chain(y, y / (3.0 * a.v), a);
}
template <int N>
GLG_HD GlgDual<N> glg_pow(const GlgDual<N> &b, double e) {
    const double y = glg_pow(b.v, e);
    return glg_chain(y, e * y / b.v, b);
}
template <int N>
GLG_HD GlgDual<N> glg_pow(const GlgDual<N> &b, const GlgDual<N> &e) { return glg_pow(b, e.v); }  // constant exponent
template <int N>
GLG_HD GlgDual<N> glg_root34(const GlgDual<N> &a, bool cube) {
    const double y = glg_root34(a.v, cube);
    return glg_chain(y, y * (cube ? 0x1.5555555555555p-2 : 0.25) / a.v, a);
}
template <int N>
GLG_HD GlgDual<N> glg_inv1pexp(const GlgDual<N> &z) {
    const double y = glg_inv1pexp(z.v);
    return glg_chain(y, -(y * (1.0 - y)), z);
}
#if defined(__CUDA_ARCH__)
#define GLG_UNROLL _Pragma("unroll")
#else
#define GLG_UNROLL
#endif
// interleaved batches: the value parts go through the double batch functions, so they are bit-identical to them
#define GLG_DUAL_BATCH(NAME, DERIV)                                                      \
    template <int M, int N>                                                              \
    GLG_HD void NAME(const GlgDual<N>(&x)[M], GlgDual<N>(&y)[M]) {                       \
        double xv[M], yv[M];                                                             \
        GLG_UNROLL for (int i = 0; i < M; ++i) xv[i] = x[i].v;                           \
        NAME<M>(xv, yv);                                                                 \
        GLG_UNROLL for (int i = 0; i < M; ++i) {                                         \
            const double yy = yv[i], xx = xv[i];                                         \
            (void)xx;                                                                    \
            y[i] = glg_chain(yy, DERIV, x[i]);                                           \
        }                                                                                \
    }
GLG_DUAL_BATCH(glg_exp_n, yy)
GLG_DUAL_BATCH(glg_rcp_n, -(yy * yy))
GLG_DUAL_BATCH(glg_sqrt_n, 0.5 / yy)
GLG_DUAL_BATCH(glg_cbrt_n, yy / (3.0 * xx))
#undef GLG_DUAL_BATCH
