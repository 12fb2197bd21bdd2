// polya_math.cuh — expf and logf as glibc computes them (x86-64, glibc >= 2.28), for host and device.
//
// The poly(A) segmentation HMM (polya.cu) evaluates five expf and three logf per raw sample, and its scores must equal
// the reference's bit for bit.  CUDA's expf/logf are not the host's libm, so both are restated here from the published
// table-driven algorithms that glibc ships (sysdeps/ieee754/flt-32/e_expf.c, e_logf.c), which come from ARM's
// optimized-routines (math/expf.c, math/logf.c, math/exp2f_data.c, math/logf_data.c):
//
//   expf: x*N/ln2 = k + r, 2^(k/N) from a 32-entry table, a cubic in r, all in double.  glibc's x86-64 build picks the
//         FMA variant at run time on CPUs with FMA, where the compiler contracts the polynomial; the contracted form is
//         restated (without it one input in [-103, 0], -0x1.f8cbb2p+5, differs).
//   logf: x = 2^k z, z/c - 1 from a 16-entry {1/c, log c} table, a quadratic-plus in r, all in double.  Contraction does
//         not change any result, so it is written without.
//
// Every double operation is spelled with its rounding (__dmul_rn / __dadd_rn / __fma_rn on the device; plain C on the
// host, built without contraction, and std::fma where the FMA variant fuses).  tests/cuda/check_polya_math.cu compares
// both functions with the libm of the machine it runs on over every float of their domain here (expf: x <= 0, logf: x >= 0).
#pragma once
#include <cstdint>
#include <cstring>
#include <cmath>

#if defined(__CUDACC__)
#define NPH_PM_HD __host__ __device__ __forceinline__
#else
#define NPH_PM_HD inline
#endif

namespace nph_polya_math {

// exp2f_data.c: tab[i] = bits(RN(2^(i/32))) - (i << 47), so that adding k << 47 gives the bits of 2^(k/32) for any k
#define NPH_PM_EXP2F_TAB {                                                                                           \
    0x3ff0000000000000ull, 0x3fefd9b0d3158574ull, 0x3fefb5586cf9890full, 0x3fef9301d0125b51ull,                     \
    0x3fef72b83c7d517bull, 0x3fef54873168b9aaull, 0x3fef387a6e756238ull, 0x3fef1e9df51fdee1ull,                     \
    0x3fef06fe0a31b715ull, 0x3feef1a7373aa9cbull, 0x3feedea64c123422ull, 0x3feece086061892dull,                     \
    0x3feebfdad5362a27ull, 0x3feeb42b569d4f82ull, 0x3feeab07dd485429ull, 0x3feea47eb03a5585ull,                     \
    0x3feea09e667f3bcdull, 0x3fee9f75e8ec5f74ull, 0x3feea11473eb0187ull, 0x3feea589994cce13ull,                     \
    0x3feeace5422aa0dbull, 0x3feeb737b0cdc5e5ull, 0x3feec49182a3f090ull, 0x3feed503b23e255dull,                     \
    0x3feee89f995ad3adull, 0x3feeff76f2fb5e47ull, 0x3fef199bdd85529cull, 0x3fef3720dcef9069ull,                     \
    0x3fef5818dcfba487ull, 0x3fef7c97337b9b5full, 0x3fefa4afa2a490daull, 0x3fefd0765b6e4540ull,                     \
}

// logf_data.c (ARM optimized-routines __logf_data, identical in glibc's e_logf_data.c): {invc, logc} per subinterval
#define NPH_PM_LOGF_TAB {                                                                                            \
    { 0x1.661ec79f8f3bep+0, -0x1.57bf7808caadep-2 },                                                                \
    { 0x1.571ed4aaf883dp+0, -0x1.2bef0a7c06ddbp-2 },                                                                \
    { 0x1.49539f0f010bp+0, -0x1.01eae7f513a67p-2 },                                                                 \
    { 0x1.3c995b0b80385p+0, -0x1.b31d8a68224e9p-3 },                                                                \
    { 0x1.30d190c8864a5p+0, -0x1.6574f0ac07758p-3 },                                                                \
    { 0x1.25e227b0b8eap+0, -0x1.1aa2bc79c81p-3 },                                                                   \
    { 0x1.1bb4a4a1a343fp+0, -0x1.a4e76ce8c0e5ep-4 },                                                                \
    { 0x1.12358f08ae5bap+0, -0x1.1973c5a611cccp-4 },                                                                \
    { 0x1.0953f419900a7p+0, -0x1.252f438e10c1ep-5 },                                                                \
    { 0x1p+0, 0x0p+0 },                                                                                             \
    { 0x1.e608cfd9a47acp-1, 0x1.aa5aa5df25984p-5 },                                                                 \
    { 0x1.ca4b31f026aap-1, 0x1.c5e53aa362eb4p-4 },                                                                  \
    { 0x1.b2036576afce6p-1, 0x1.526e57720db08p-3 },                                                                 \
    { 0x1.9c2d163a1aa2dp-1, 0x1.bc2860d22477p-3 },                                                                  \
    { 0x1.886e6037841edp-1, 0x1.1058bc8a07ee1p-2 },                                                                 \
    { 0x1.767dcf5534862p-1, 0x1.4043057b6ee09p-2 },                                                                 \
}

#if defined(__CUDACC__)
__device__ __constant__ uint64_t kExp2fTabDev[32] = NPH_PM_EXP2F_TAB;
__device__ __constant__ double kLogfTabDev[16][2] = NPH_PM_LOGF_TAB;
#endif
static const uint64_t kExp2fTabHost[32] = NPH_PM_EXP2F_TAB;
static const double kLogfTabHost[16][2] = NPH_PM_LOGF_TAB;

#if defined(__CUDA_ARCH__)
#define NPH_PM_TAB(name) name##Dev
#else
#define NPH_PM_TAB(name) name##Host
#endif

NPH_PM_HD uint32_t f2u(float x) { uint32_t u; memcpy(&u, &x, 4); return u; }
NPH_PM_HD float u2f(uint32_t u) { float x; memcpy(&x, &u, 4); return x; }
NPH_PM_HD uint64_t d2u(double x) { uint64_t u; memcpy(&u, &x, 8); return u; }
NPH_PM_HD double u2d(uint64_t u) { double x; memcpy(&x, &u, 8); return x; }

#if defined(__CUDA_ARCH__)
NPH_PM_HD double pm_dmul(double a, double b) { return __dmul_rn(a, b); }
NPH_PM_HD double pm_dadd(double a, double b) { return __dadd_rn(a, b); }
NPH_PM_HD double pm_dsub(double a, double b) { return __dsub_rn(a, b); }
NPH_PM_HD double pm_dfma(double a, double b, double c) { return __fma_rn(a, b, c); }
NPH_PM_HD float pm_fmul(float a, float b) { return __fmul_rn(a, b); }
NPH_PM_HD float pm_fadd(float a, float b) { return __fadd_rn(a, b); }
#else
NPH_PM_HD double pm_dmul(double a, double b) { return a * b; }
NPH_PM_HD double pm_dadd(double a, double b) { return a + b; }
NPH_PM_HD double pm_dsub(double a, double b) { return a - b; }
NPH_PM_HD double pm_dfma(double a, double b, double c) { return std::fma(a, b, c); }
NPH_PM_HD float pm_fmul(float a, float b) { return a * b; }
NPH_PM_HD float pm_fadd(float a, float b) { return a + b; }
#endif

// glibc __expf (e_expf.c), FMA variant.  Results for every float: 0 below log(2^-150), +inf above log(2^128), NaN for NaN.
NPH_PM_HD float expf_glibc(float x)
{
    const double kInvLn2N = 0x1.71547652b82fep+5, kShift = 0x1.8p+52;
    const double kC0 = 0x1.c6af84b912394p-20, kC1 = 0x1.ebfce50fac4f3p-13, kC2 = 0x1.62e42ff0c52d6p-6;
    const uint32_t abstop = (f2u(x) >> 20) & 0x7ff;
    if (abstop >= (f2u(88.0f) >> 20)) {
        if (f2u(x) == 0xff800000u) return 0.0f;             // -inf
        if (abstop >= (0x7f800000u >> 20)) return pm_fadd(x, x);   // +inf, NaN
        if (x > 0x1.62e42ep6f) return u2f(0x7f800000u);     // overflow
        if (x < -0x1.9fe368p6f) return 0.0f;                // underflow
    }
    const double xd = (double)x;
    const double z = pm_dmul(kInvLn2N, xd);
    double kd = pm_dadd(z, kShift);
    const uint64_t ki = d2u(kd);
    kd = pm_dsub(kd, kShift);
    const double r = pm_dfma(kInvLn2N, xd, -kd);               // z - kd, contracted
    uint64_t t = NPH_PM_TAB(kExp2fTab)[ki % 32];
    t += ki << 47;
    const double s = u2d(t);
    const double zz = pm_dfma(kC0, r, kC1);
    const double r2 = pm_dmul(r, r);
    double y = pm_dfma(kC2, r, 1.0);
    y = pm_dfma(zz, r2, y);
    y = pm_dmul(y, s);
    return (float)y;                                        // RN double -> float (subnormals included)
}

// glibc __logf (e_logf.c).  -inf for +-0, NaN for negative and NaN inputs, +inf for +inf.
NPH_PM_HD float logf_glibc(float x)
{
    const double kLn2 = 0x1.62e42fefa39efp-1;
    const double kA0 = -0x1.00ea348b88334p-2, kA1 = 0x1.5575b0be00b6ap-2, kA2 = -0x1.ffffef20a4123p-2;
    uint32_t ix = f2u(x);
    if (ix == 0x3f800000u) return 0.0f;
    if (ix - 0x00800000u >= 0x7f800000u - 0x00800000u) {
        if (ix * 2 == 0) return u2f(0xff800000u);           // log(+-0) = -inf
        if (ix == 0x7f800000u) return x;                    // log(inf) = inf
        if ((ix & 0x80000000u) || ix * 2 >= 0xff000000u) return u2f(0x7fc00000u);   // negative or NaN
        ix = f2u(pm_fmul(x, 0x1p23f));                         // subnormal: normalise
        ix -= 23u << 23;
    }
    const uint32_t tmp = ix - 0x3f330000u;
    const int i = (int)((tmp >> (23 - 4)) % 16);
    const int k = (int32_t)tmp >> 23;
    const uint32_t iz = ix - (tmp & (0x1ffu << 23));
    const double invc = NPH_PM_TAB(kLogfTab)[i][0], logc = NPH_PM_TAB(kLogfTab)[i][1];
    const double z = (double)u2f(iz);
    const double r = pm_dsub(pm_dmul(z, invc), 1.0);
    const double y0 = pm_dadd(logc, pm_dmul((double)k, kLn2));
    const double r2 = pm_dmul(r, r);
    double y = pm_dadd(pm_dmul(kA1, r), kA2);
    y = pm_dadd(pm_dmul(kA0, r2), y);
    y = pm_dadd(pm_dmul(y, r2), pm_dadd(y0, r));
    return (float)y;
}

} // namespace nph_polya_math
