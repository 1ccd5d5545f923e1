// lz_exact_math.h -- fp32 expf that reproduces glibc's float expf bit-for-bit, usable from CUDA
// device code and from plain C/C++ host code (tests/ compile it on the host against libm).
//
// Why: the reference tree computes child priors with `exp(logit - max)` on floats
// (lzero/mcts/ctree/ctree_muzero/lib/cnode.cpp:127-132), which binds to glibc's expf.  glibc >= 2.27
// implements expf with the ARM "optimized routines" algorithm: the argument is promoted to double,
// reduced with a 32-entry table of 2^(i/32) and a cubic polynomial, and the double result is
// rounded to float once.  That result is NOT always the correctly rounded exp (max error 0.502 ULP),
// so neither CUDA's expf nor (float)exp((double)x) matches it on every input.  Restating the same
// double-precision operation sequence does: IEEE double add/mul/fma are exact-rounded on both x86
// and sm_100, so the device reproduces the host bit pattern.  tests/test_exact_math.py checks this
// restatement against libm expf for EVERY float in [-104, +0] (1.12e9 inputs) on the host.
//
// Published algorithm restated: glibc 2.39 sysdeps/ieee754/flt-32/e_expf.c + e_exp2f_data.c
// (N = 32, InvLn2N = 0x1.71547652b82fep+0 * N, SHIFT = 0x1.8p+52,
//  poly = {0x1.c6af84b912394p-5, 0x1.ebfce50fac4f3p-3, 0x1.62e42ff0c52d6p-1} scaled by 1/N^3, 1/N^2, 1/N).
// Variant: on every x86-64 CPU with FMA3 (all hosts this runs beside) glibc's ifunc selects
// __expf_fma, i.e. e_expf.c compiled with -mfma -ffp-contract=fast, where the compiler fuses
// kd = z + SHIFT and r = z - kd (z = InvLn2N*x has only add/sub uses) as well as the polynomial.
// The fused reduction differs from the unfused one on 1 input in 1.12e9 (x = -0x1.f8cbb2p+5), so
// the fused sequence is the one restated here.
// The table below is T[i] = bits(round_to_double(2^(i/32))) - (i << 47), regenerated from
// exp2l(i/32) (not copied); the exhaustive test is what certifies it.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define LZ_HD __host__ __device__ __forceinline__
#else
#define LZ_HD static inline
#include <math.h>
#include <string.h>
#endif

#define LZ_EXP2F_TAB_INIT { \
    0x3ff0000000000000ULL, 0x3fefd9b0d3158574ULL, 0x3fefb5586cf9890fULL, 0x3fef9301d0125b51ULL, \
    0x3fef72b83c7d517bULL, 0x3fef54873168b9aaULL, 0x3fef387a6e756238ULL, 0x3fef1e9df51fdee1ULL, \
    0x3fef06fe0a31b715ULL, 0x3feef1a7373aa9cbULL, 0x3feedea64c123422ULL, 0x3feece086061892dULL, \
    0x3feebfdad5362a27ULL, 0x3feeb42b569d4f82ULL, 0x3feeab07dd485429ULL, 0x3feea47eb03a5585ULL, \
    0x3feea09e667f3bcdULL, 0x3fee9f75e8ec5f74ULL, 0x3feea11473eb0187ULL, 0x3feea589994cce13ULL, \
    0x3feeace5422aa0dbULL, 0x3feeb737b0cdc5e5ULL, 0x3feec49182a3f090ULL, 0x3feed503b23e255dULL, \
    0x3feee89f995ad3adULL, 0x3feeff76f2fb5e47ULL, 0x3fef199bdd85529cULL, 0x3fef3720dcef9069ULL, \
    0x3fef5818dcfba487ULL, 0x3fef7c97337b9b5fULL, 0x3fefa4afa2a490daULL, 0x3fefd0765b6e4540ULL, }
#if defined(__CUDACC__)
static __device__ __constant__ uint64_t lz_exp2f_tab_dev[32] = LZ_EXP2F_TAB_INIT;
#endif
static const uint64_t lz_exp2f_tab_host[32] = LZ_EXP2F_TAB_INIT;

// expf for x <= 0 and moderate positive x, glibc-bit-exact.  Out-of-range handling mirrors
// e_expf.c: x < -0x1.9fe368p6 underflows to +0, x > 0x1.62e42ep6 overflows to +inf.
LZ_HD float lz_expf_exact(float x)
{
    if (x < -0x1.9fe368p6f) return 0.0f;
    if (x > 0x1.62e42ep6f) return __builtin_huge_valf();
    const double InvLn2N = 0x1.71547652b82fep+0 * 32.0;
    const double Shift = 0x1.8p+52;
    const double C0 = 0x1.c6af84b912394p-5 / 32.0 / 32.0 / 32.0;
    const double C1 = 0x1.ebfce50fac4f3p-3 / 32.0 / 32.0;
    const double C2 = 0x1.62e42ff0c52d6p-1 / 32.0;
    double xd = (double)x;
#if defined(__CUDA_ARCH__)
    double kd = __fma_rn(InvLn2N, xd, Shift);
    uint64_t ki = (uint64_t)__double_as_longlong(kd);
    kd = __dsub_rn(kd, Shift);
    double r = __fma_rn(InvLn2N, xd, -kd);
    uint64_t t = lz_exp2f_tab_dev[ki & 31] + (ki << 47);
    double s = __longlong_as_double((long long)t);
    double zz = __fma_rn(C0, r, C1);
    double r2 = __dmul_rn(r, r);
    double y = __fma_rn(C2, r, 1.0);
    y = __fma_rn(zz, r2, y);
    y = __dmul_rn(y, s);
    return __double2float_rn(y);
#else
    double kd = fma(InvLn2N, xd, Shift);
    uint64_t ki;
    memcpy(&ki, &kd, 8);
    kd -= Shift;
    double r = fma(InvLn2N, xd, -kd);
    uint64_t t = lz_exp2f_tab_host[ki & 31] + (ki << 47);
    double s;
    memcpy(&s, &t, 8);
    double zz = fma(C0, r, C1);
    double r2 = r * r;
    double y = fma(C2, r, 1.0);
    y = fma(zz, r2, y);
    y = y * s;
    return (float)y;
#endif
}

// ---- logf -------------------------------------------------------------------------------------------
// The Gumbel MuZero tree's softmax (ctree_gumbel_muzero/lib/cnode.cpp:903-932) subtracts log(sum) with sum a float,
// which binds to glibc's logf.  Published algorithm restated: glibc 2.39 sysdeps/ieee754/flt-32/e_logf.c +
// e_logf_data.c (ARM optimized routines): x = 2^k z with z in [OFF, 2 OFF), a 16-entry table of (1/c, log c) for the
// subinterval of z, r = z/c - 1 and a degree-3 polynomial for log1p(r), all in double, rounded to float once.
// Variant: as for expf, glibc's ifunc selects __logf_fma on FMA3 hosts (e_logf.c built with -mfma -ffp-contract=fast),
// so r = z*invc - 1, y0 = logc + k*Ln2 and the three polynomial steps are fused multiply-adds.
// tests/csrc/check_logf.c compares this against libm logf on every float in [1, 64] (LZ_EXHAUSTIVE=1: every
// positive finite float).  Only positive finite inputs are handled (a softmax sum lies in [1, n]); 0 gives -inf.
#define LZ_LOGF_TAB_INIT { \
    0x1.661ec79f8f3bep+0, -0x1.57bf7808caadep-2, 0x1.571ed4aaf883dp+0, -0x1.2bef0a7c06ddbp-2, \
    0x1.49539f0f010bp+0,  -0x1.01eae7f513a67p-2, 0x1.3c995b0b80385p+0, -0x1.b31d8a68224e9p-3, \
    0x1.30d190c8864a5p+0, -0x1.6574f0ac07758p-3, 0x1.25e227b0b8eap+0,  -0x1.1aa2bc79c81p-3,   \
    0x1.1bb4a4a1a343fp+0, -0x1.a4e76ce8c0e5ep-4, 0x1.12358f08ae5bap+0, -0x1.1973c5a611cccp-4, \
    0x1.0953f419900a7p+0, -0x1.252f438e10c1ep-5, 0x1p+0,               0x0p+0,                \
    0x1.e608cfd9a47acp-1, 0x1.aa5aa5df25984p-5,  0x1.ca4b31f026aap-1,  0x1.c5e53aa362eb4p-4,  \
    0x1.b2036576afce6p-1, 0x1.526e57720db08p-3,  0x1.9c2d163a1aa2dp-1, 0x1.bc2860d22477p-3,   \
    0x1.886e6037841edp-1, 0x1.1058bc8a07ee1p-2,  0x1.767dcf5534862p-1, 0x1.4043057b6ee09p-2, }
#if defined(__CUDACC__)
static __device__ __constant__ double lz_logf_tab_dev[32] = LZ_LOGF_TAB_INIT;   // {invc, logc} x 16
#endif
static const double lz_logf_tab_host[32] = LZ_LOGF_TAB_INIT;

LZ_HD float lz_logf_exact(float x)
{
    const double Ln2 = 0x1.62e42fefa39efp-1;
    const double P0 = -0x1.00ea348b88334p-2, P1 = 0x1.5575b0be00b6ap-2, P2 = -0x1.ffffef20a4123p-2;
    const uint32_t OFF = 0x3f330000u;
#if defined(__CUDA_ARCH__)
    uint32_t ix = __float_as_uint(x);
#else
    uint32_t ix;
    memcpy(&ix, &x, 4);
#endif
    if (ix == 0x3f800000u) return 0.0f;
    if (ix - 0x00800000u >= 0x7f800000u - 0x00800000u) {   // zero, subnormal, inf (negative / NaN are not inputs here)
        if (ix * 2 == 0) return -__builtin_huge_valf();
        if (ix == 0x7f800000u) return x;
        float xs = x * 0x1p23f;                             // subnormal: normalise
#if defined(__CUDA_ARCH__)
        ix = __float_as_uint(xs);
#else
        memcpy(&ix, &xs, 4);
#endif
        ix -= 23u << 23;
    }
    const uint32_t tmp = ix - OFF;
    const int i = (int)((tmp >> (23 - 4)) % 16);
    const int k = (int32_t)tmp >> 23;
    const uint32_t iz = ix - (tmp & 0xff800000u);
#if defined(__CUDA_ARCH__)
    const double invc = lz_logf_tab_dev[2 * i], logc = lz_logf_tab_dev[2 * i + 1];
    const double z = (double)__uint_as_float(iz);
    const double r = __fma_rn(z, invc, -1.0);
    const double y0 = __fma_rn((double)k, Ln2, logc);
    const double r2 = __dmul_rn(r, r);
    double y = __fma_rn(P1, r, P2);
    y = __fma_rn(P0, r2, y);
    y = __fma_rn(y, r2, __dadd_rn(y0, r));
    return __double2float_rn(y);
#else
    const double invc = lz_logf_tab_host[2 * i], logc = lz_logf_tab_host[2 * i + 1];
    float zf;
    memcpy(&zf, &iz, 4);
    const double z = (double)zf;
    const double r = fma(z, invc, -1.0);
    const double y0 = fma((double)k, Ln2, logc);
    const double r2 = r * r;
    double y = fma(P1, r, P2);
    y = fma(P0, r2, y);
    y = fma(y, r2, y0 + r);
    return (float)y;
#endif
}
