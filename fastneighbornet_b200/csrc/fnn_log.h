// fnn_log.h — natural logarithm from IEEE binary64 + - * / and bit operations only, shared by libfastnn.so (device) and
// oracle/libdist_oracle.so (host).  CUDA's log and glibc's log do not agree bit for bit; this one is the same function on both
// sides as long as neither contracts a*b+c into an FMA (nvcc --fmad=false, g++ -ffp-contract=off).
//
// Method (the reduction of fdlibm's e_log.c, with a Taylor series instead of a minimax polynomial):
//   x = 2^k * (1 + f), 1 + f in [sqrt(1/2), sqrt(2)]   (subnormal x first scaled by 2^54)
//   s = f / (2 + f), z = s^2, |s| <= 0.1716, z <= 0.02944
//   log(1 + f) = 2 atanh(s) = 2s + s R,  R = z (2/3 + z (2/5 + ... + z 2/25))    (12 terms; the first omitted term,
//                                                                                 z^13 2/27 relative to 2s, is < 2^-70)
//   2s = f - hfsq + s hfsq with hfsq = f^2 / 2, so log(1 + f) = f - (hfsq - s (hfsq + R)): s and R only enter a
//   correction term, and the leading f = (1 + f) - 1 is exact (Sterbenz).
//   log x = k ln2_hi - ((hfsq - (s (hfsq + R) + k ln2_lo)) - f)
// ln2_hi has 32 significant bits, so k ln2_hi is exact for every |k| <= 1128 that occurs.
//
// Constants, derived with Python's decimal module at 60 digits and rounded to binary64:
//   ln2    = Decimal(2).ln()
//   ln2_hi = round(ln2 * 2^32) / 2^32          = 2977044472 / 2^32   (exact)
//   ln2_lo = float(ln2 - ln2_hi)
//   C_k    = float(Decimal(2) / Decimal(2k + 1)),  k = 1..12
//   the reduction threshold is the bit pattern of float(Decimal(2).sqrt()).
// Properties held by tests/test_alignment_cpu.py: fnn_log(1.0) == +0.0, non-decreasing, within 1 ulp of numpy.log on
// (0, 1] (subnormals included) and of a 40-digit decimal log.  fnn_log(0) = -inf, fnn_log(x < 0) = NaN, fnn_log(+inf) = +inf.
#pragma once
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define FNN_LOG_HD __host__ __device__ __forceinline__
#else
#define FNN_LOG_HD inline
#endif

FNN_LOG_HD uint64_t fnn_log_bits_(double x) {
#if defined(__CUDA_ARCH__)
    return (uint64_t)__double_as_longlong(x);
#else
    uint64_t u;
    memcpy(&u, &x, sizeof(u));
    return u;
#endif
}

FNN_LOG_HD double fnn_log_from_bits_(uint64_t u) {
#if defined(__CUDA_ARCH__)
    return __longlong_as_double((long long)u);
#else
    double x;
    memcpy(&x, &u, sizeof(x));
    return x;
#endif
}

FNN_LOG_HD double fnn_log(double x) {
    if (!(x > 0.0)) return x == 0.0 ? fnn_log_from_bits_(0xFFF0000000000000ull) : fnn_log_from_bits_(0x7FF8000000000000ull);
    uint64_t u = fnn_log_bits_(x);
    if (u >= 0x7FF0000000000000ull) return x;   // +inf, NaN
    int k = 0;
    if (u < 0x0010000000000000ull) {             // subnormal: scale into the normal range
        u = fnn_log_bits_(x * 0x1p54);
        k = -54;
    }
    k += (int)(u >> 52) - 1023;
    u = (u & 0x000FFFFFFFFFFFFFull) | 0x3FF0000000000000ull;   // 1 + f in [1, 2)
    if (u > 0x3FF6A09E667F3BCDull) {                           // above sqrt(2): halve it
        u -= 0x0010000000000000ull;
        ++k;
    }
    const double f = fnn_log_from_bits_(u) - 1.0;
    const double s = f / (2.0 + f);
    const double z = s * s;
    const double R =
        z * (0x1.5555555555555p-1 +
        z * (0x1.999999999999ap-2 +
        z * (0x1.2492492492492p-2 +
        z * (0x1.c71c71c71c71cp-3 +
        z * (0x1.745d1745d1746p-3 +
        z * (0x1.3b13b13b13b14p-3 +
        z * (0x1.1111111111111p-3 +
        z * (0x1.e1e1e1e1e1e1ep-4 +
        z * (0x1.af286bca1af28p-4 +
        z * (0x1.8618618618618p-4 +
        z * (0x1.642c8590b2164p-4 +
        z * 0x1.47ae147ae147bp-4)))))))))));
    const double hfsq = 0.5 * f * f;
    const double dk = (double)k;
    const double ln2_hi = 0x1.62e42ffp-1, ln2_lo = -0x1.718432a1b0e26p-35;
    return dk * ln2_hi - ((hfsq - (s * (hfsq + R) + dk * ln2_lo)) - f);
}
