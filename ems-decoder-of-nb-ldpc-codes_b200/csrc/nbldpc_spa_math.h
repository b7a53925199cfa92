/*
 * nbldpc_spa_math.h -- the f32 exp and log of the sum-product check node (nbldpc_spa.cuh), for the device and the host.
 *
 * CUDA's expf/logf and glibc's do not agree bit for bit, so the check node uses its own: explicit range reduction and a
 * fixed polynomial of f32 +, -, * (and one division in nb_spa_log).  Every operation is one IEEE f32 operation rounded to
 * nearest, so the device build (-fmad=false, no ftz) and a host build with -ffp-contract=off give the same bits.
 *
 *   nb_spa_exp(d), d <= 0: e^d.  d < -87 (and -inf) gives 0, so no result is subnormal.
 *     k = round(d * log2 e) by the 1.5 * 2^23 trick (ties to even), r = (d - k ln2_hi) - k ln2_lo with the Cody-Waite
 *     split of ln 2 (ln2_hi has 16 significant bits, so k ln2_hi is exact), e^r by the degree-7 Taylor polynomial in
 *     Horner form on |r| <= ln2 / 2, then * 2^k.
 *     Largest error over every float d in [-87, 0] (scripts/check_spa_math.c): 1.22 ulp against the f64 exp.
 *   nb_spa_log(x), x a positive normal float: ln x.
 *     x = 2^k m with m in [sqrt(1/2), sqrt(2)), f = m - 1 (exact), s = f / (2 + f), ln m = 2s + 2s z (1/3 + z/5 + z^2/7 + z^3/9)
 *     with z = s^2, then k ln2_hi + (k ln2_lo + ln m).
 *     Largest error over every float x in [2^-24, 2^9] (scripts/check_spa_math.c): 1.97 ulp against the f64 log.
 *     The check node calls it on [2^-20 c_max, c_max] with 1 <= c_max <= q.
 */
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define NB_SPA_FN __host__ __device__ static inline
#else
#include <string.h>
#define NB_SPA_FN static inline
#endif

NB_SPA_FN uint32_t nb_spa_bits(float x)
{
#ifdef __CUDA_ARCH__
    return __float_as_uint(x);
#else
    uint32_t u; memcpy(&u, &x, 4); return u;
#endif
}
NB_SPA_FN float nb_spa_float(uint32_t u)
{
#ifdef __CUDA_ARCH__
    return __uint_as_float(u);
#else
    float x; memcpy(&x, &u, 4); return x;
#endif
}

#define NB_SPA_LN2_HI 0x1.62e400p-1f         /* 0.693145751953125 */
#define NB_SPA_LN2_LO 0x1.7f7d1cp-20f        /* ln 2 - ln2_hi, rounded */

NB_SPA_FN float nb_spa_exp(float d)
{
    if (!(d >= -87.0f)) return 0.0f;
    const float kf = (d * 0x1.715476p+0f + 12582912.0f) - 12582912.0f;      /* round(d log2 e), -126 <= k <= 0 */
    const float r = (d - kf * NB_SPA_LN2_HI) - kf * NB_SPA_LN2_LO;
    float p = 1.0f / 5040.0f;
    p = p * r + 1.0f / 720.0f;
    p = p * r + 1.0f / 120.0f;
    p = p * r + 1.0f / 24.0f;
    p = p * r + 1.0f / 6.0f;
    p = p * r + 0.5f;
    p = p * r + 1.0f;
    p = p * r + 1.0f;
    return p * nb_spa_float((uint32_t)(127 + (int)kf) << 23);
}

NB_SPA_FN float nb_spa_log(float x)
{
    const uint32_t u = nb_spa_bits(x);
    int k = (int)(u >> 23) - 127;
    float m = nb_spa_float((u & 0x7fffffu) | 0x3f800000u);                    /* [1, 2) */
    if (m > 0x1.6a09e6p+0f) { m = m * 0.5f; k += 1; }                       /* [sqrt(1/2), sqrt(2)) */
    const float f = m - 1.0f;
    const float s = f / (2.0f + f);
    const float z = s * s;
    float R = 1.0f / 9.0f;
    R = R * z + 1.0f / 7.0f;
    R = R * z + 1.0f / 5.0f;
    R = R * z + 1.0f / 3.0f;
    R = R * z;
    const float s2 = s + s;
    const float lm = s2 + s2 * R;
    const float kf = (float)k;
    return kf * NB_SPA_LN2_HI + (kf * NB_SPA_LN2_LO + lm);
}
