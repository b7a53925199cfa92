/*
 * check_spa_math.c -- exhaustive check of the f32 exp and log of the sum-product check node (csrc/nbldpc_spa_math.h)
 * against the f64 functions of libm, over every float of the domain the check node calls them on:
 *   nb_spa_exp on every float d in [-87, 0]   (the node calls it on mu - Mvc[x] <= 0; below -87 it returns 0)
 *   nb_spa_log on every float x in [2^-24, 2^9] (the node calls it on [2^-20 c_max, c_max] with 1 <= c_max <= q <= 256)
 * The error of a result y against the exact value v is |y - v| in units of the f32 ulp at v (2^(floor(log2 |v|) - 23)).
 * Prints the largest error of each function and where it occurs; the bounds quoted in the header must not be exceeded.
 *
 *   gcc -O2 -fopenmp -ffp-contract=off -I ems-decoder-of-nb-ldpc-codes_b200/csrc -o /tmp/check_spa_math scripts/check_spa_math.c -lm
 *   /tmp/check_spa_math        (about 20 seconds on 16 cores; exit status 1 if a bound is exceeded)
 */
#include "nbldpc_spa_math.h"
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#define EXP_BOUND 1.22
#define LOG_BOUND 1.97

static inline float u2f(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
static inline uint32_t f2u(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }

static double ulp_err(float y, double v)
{
    if (v == 0.0) return y == 0.0f ? 0.0 : INFINITY;
    int e;
    frexp(fabs(v), &e);                                        /* |v| in [2^(e-1), 2^e) */
    return fabs((double)y - v) / ldexp(1.0, e - 1 - 23);
}

int main(void)
{
    double emax = 0.0, lmax = 0.0;
    float earg = 0.0f, larg = 0.0f;
    const uint32_t e_lo = f2u(-0.0f), e_hi = f2u(-87.0f);      /* negative floats: bit patterns grow with |d| */
#pragma omp parallel
    {
        double m = 0.0; float a = 0.0f;
#pragma omp for schedule(static) nowait
        for (int64_t u = e_lo; u <= (int64_t)e_hi; u++) {
            const float d = u2f((uint32_t)u);
            const double err = ulp_err(nb_spa_exp(d), exp((double)d));
            if (err > m) { m = err; a = d; }
        }
        {
            const float d = 0.0f;
            const double err = ulp_err(nb_spa_exp(d), 1.0);
            if (err > m) { m = err; a = d; }
        }
#pragma omp critical
        if (m > emax) { emax = m; earg = a; }
    }
    const uint32_t l_lo = f2u(0x1p-24f), l_hi = f2u(0x1p9f);
#pragma omp parallel
    {
        double m = 0.0; float a = 0.0f;
#pragma omp for schedule(static) nowait
        for (int64_t u = l_lo; u <= (int64_t)l_hi; u++) {
            const float x = u2f((uint32_t)u);
            const double err = ulp_err(nb_spa_log(x), log((double)x));
            if (err > m) { m = err; a = x; }
        }
#pragma omp critical
        if (m > lmax) { lmax = m; larg = a; }
    }
    printf("nb_spa_exp on [-87, 0]:      largest error %.3f ulp at d = %a (bound %.2f)\n", emax, earg, EXP_BOUND);
    printf("nb_spa_log on [2^-24, 2^9]:  largest error %.3f ulp at x = %a (bound %.2f)\n", lmax, larg, LOG_BOUND);
    return (emax > EXP_BOUND || lmax > LOG_BOUND) ? 1 : 0;
}
