// ok_math.cuh -- device arithmetic whose results must be bit-identical to the reference's HOST
// arithmetic (x86-64, binary32, no FMA contraction, glibc libm).
//
// Rules used throughout the kernels:
//   * binary32 +,-,* go through __fadd_rn / __fsub_rn / __fmul_rn: ptxas never fuses these, so the
//     results do not depend on -fmad;
//   * division and square root are the IEEE-rounded __fdiv_rn / __fsqrt_rn;
//   * cos/sin of a float are ok::sincosf below: the glibc 2.39 algorithm (sysdeps/ieee754/flt-32/
//     s_sincosf.{c,h}, ARM optimized-routines) in binary64 with the FMA contraction pattern of
//     its x86-64 __sincosf_fma ifunc variant -- the symbol the reference's Agent.cpp:94-96,115-117
//     and CollisionChecker.cu:122-124,157-158 resolve to on this image's hosts.  B200 has
//     full-rate-class FP64 (DFMA), so this costs ~40 instructions per call.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

namespace ok
{

#define OK_DEG2RAD 0.0174532924f /* float(M_PI / 180.0), Typedefs.h:10 */

__device__ __forceinline__ float fadd(float a, float b)
{
    return __fadd_rn(a, b);
}
__device__ __forceinline__ float fsub(float a, float b)
{
    return __fsub_rn(a, b);
}
__device__ __forceinline__ float fmul(float a, float b)
{
    return __fmul_rn(a, b);
}
__device__ __forceinline__ float fdiv(float a, float b)
{
    return __fdiv_rn(a, b);
}

// cosine / sine polynomial coefficients for quadrant parity 0 (the parity-1 table is the
// same with the cosine coefficients negated)
#define OK_SC_C0 0x1p0
#define OK_SC_C1 -0x1.ffffffd0c621cp-2
#define OK_SC_C2 0x1.55553e1068f19p-5
#define OK_SC_C3 -0x1.6c087e89a359dp-10
#define OK_SC_C4 0x1.99343027bf8c3p-16
#define OK_SC_S1 -0x1.555545995a603p-3
#define OK_SC_S2 0x1.1107605230bc4p-7
#define OK_SC_S3 -0x1.994eb3774cf24p-13

// 4/pi in 32-bit limbs, overlapping windows, for |x| >= 120
__device__ __constant__ uint32_t kInvPio4[24] = {
    0xa2,       0xa2f9,     0xa2f983,   0xa2f9836e, 0xf9836e4e, 0x836e4e44, 0x6e4e4415, 0x4e441529,
    0x441529fc, 0x1529fc27, 0x29fc2757, 0xfc2757d1, 0x2757d1f5, 0x57d1f534, 0xd1f534dd, 0xf534ddc0,
    0x34ddc0db, 0xddc0db62, 0xc0db6295, 0xdb629599, 0x6295993c, 0x95993c43, 0x993c4390, 0x3c439041};

// polynomial core: x = reduced argument WITHOUT the quadrant sign, q = quadrant that selects sign and table (glibc's
// sign[q & 3] = {1,-1,-1,1} and "negated-cosine table for q & 2"), n = quadrant that swaps sine and cosine.
// glibc multiplies x by the sign and negates the cosine coefficients BEFORE the polynomials; both polynomials are
// odd / even in exactly the operands that change sign and every step rounds to nearest, so negating the two binary32
// results instead gives the same bits (a zero result, where -(+0) would differ, needs x = 0, which only the
// |y| < 2^-12 shortcut sees) -- checked against libm on all 2^32 inputs (tools/sincosf_unified_exhaustive.c).  One
// path, no binary64 selects or sign products: the warp's lanes no longer split between "|y| < pi/4" and the rest.
__device__ __forceinline__ void sincos_core(double x, int n, int q, float &sin_out, float &cos_out)
{
    const double x2 = x * x;
    const double x4 = x2 * x2;
    const double x3 = x2 * x;
    const double c2 = fma(x2, OK_SC_C4, OK_SC_C3);
    const double s1 = fma(x2, OK_SC_S3, OK_SC_S2);
    const double c1 = fma(x2, OK_SC_C1, OK_SC_C0);
    const double x5 = x3 * x2;
    const double x6 = x4 * x2;
    const double s  = fma(x3, OK_SC_S1, x);
    const double c  = fma(x4, OK_SC_C2, c1);
    const uint32_t sv = __float_as_uint(__double2float_rn(fma(x5, s1, s))) ^ ((static_cast<uint32_t>(q + 1) & 2u) << 30);
    const uint32_t cv = __float_as_uint(__double2float_rn(fma(x6, c2, c))) ^ ((static_cast<uint32_t>(q) & 2u) << 30);
    sin_out           = __uint_as_float((n & 1) ? cv : sv);
    cos_out           = __uint_as_float((n & 1) ? sv : cv);
}

__device__ __forceinline__ void sincosf(float y, float &sin_out, float &cos_out)
{
    const uint32_t top = (__float_as_uint(y) >> 20) & 0x7ffu;
    double         x   = static_cast<double>(y);
    if (top < 0x42fu)
    { // |y| < 120: n = round(x * 2/pi) via a 2^24-scaled truncation.  glibc's separate branch for |y| < 0.75 is this one
      // with n = 0 (x - 0 * pi/2 = x exactly, sign +1, table 0); its |y| < 2^-12 shortcut is applied on top.
        const double r = x * 0x1.45F306DC9C883p+23;
        const int    n = (__double2int_rz(r) + 0x800000) >> 24;
        x              = fma(-static_cast<double>(n), 0x1.921FB54442D18p0, x);
        float sv, cv;
        sincos_core(x, n, n, sv, cv);
        const bool tiny = top < 0x398u; // |y| < 2^-12
        sin_out         = tiny ? y : sv;
        cos_out         = tiny ? 1.0f : cv;
    }
    else if (top < 0x7f8u)
    { // finite, large: Payne-Hanek style reduction with 4/pi in fixed point
        uint32_t        xi    = __float_as_uint(y);
        const int       sign  = static_cast<int>(xi >> 31);
        const uint32_t *arr   = &kInvPio4[(xi >> 26) & 15];
        const int       shift = (xi >> 23) & 7;
        xi                    = (xi & 0xffffffu) | 0x800000u;
        xi <<= shift;
        uint64_t       res0 = static_cast<uint64_t>(xi * arr[0]); // 32-bit product, as in the original
        const uint64_t res1 = static_cast<uint64_t>(xi) * arr[4];
        const uint64_t res2 = static_cast<uint64_t>(xi) * arr[8];
        res0                = (res2 >> 32) | (res0 << 32);
        res0 += res1;
        const uint64_t nn = (res0 + (1ULL << 61)) >> 62;
        res0 -= nn << 62;
        x           = static_cast<double>(static_cast<int64_t>(res0)) * 0x1.921FB54442D18p-62;
        const int n = static_cast<int>(nn);
        sincos_core(x, n, n + sign, sin_out, cos_out);
    }
    else
    {
        sin_out = cos_out = __fsub_rn(y, y); // inf / nan -> nan
    }
}

// Philox4x32-10 (Salmon et al., SC'11): the synthetic action stream of SURVEY.md 8(d)
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t out[4])
{
#pragma unroll
    for (int r = 0; r < 10; ++r)
    {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0, c1 = lo1, c2 = n2, c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0, out[1] = c1, out[2] = c2, out[3] = c3;
}

} // namespace ok
