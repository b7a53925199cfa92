/*
 * oracle/nbldpc_oracle_spa.c -- TEST INFRASTRUCTURE ONLY: the sum-product check node (ecn_kind = 2), restated from its
 * definition in include/nbldpc_b200.h, and the decode loop of nbo_decode_frame (nbldpc_oracle.c, NB_LDPC.c:266-474) with
 * that node in place of the EMS nodes.  The reference has no such node, so this file is the specification the GPU kernel is
 * checked against bit for bit.  A library of its own (tests/spa_oracle.py builds it with -ffp-contract=off): it works on the
 * nbo_code of liboracle.so (nbldpc_oracle.h) and shares no code with the product.  Every float line below is one IEEE f32
 * operation rounded to nearest, in the order the definition gives.
 */
#include "nbldpc_oracle.h"
#include <stdlib.h>
#include <string.h>

/* E: e^d for d <= 0 (0 below -87): Cody-Waite reduction, degree-7 Taylor polynomial, scaling by 2^k */
float nbo_spa_exp(float d)
{
    if (!(d >= -87.0f)) return 0.0f;
    const float kf = (d * 0x1.715476p+0f + 12582912.0f) - 12582912.0f;
    const float r = (d - kf * 0x1.62e400p-1f) - kf * 0x1.7f7d1cp-20f;
    float p = 1.0f / 5040.0f;
    p = p * r + 1.0f / 720.0f;
    p = p * r + 1.0f / 120.0f;
    p = p * r + 1.0f / 24.0f;
    p = p * r + 1.0f / 6.0f;
    p = p * r + 0.5f;
    p = p * r + 1.0f;
    p = p * r + 1.0f;
    uint32_t sb = (uint32_t)(127 + (int)kf) << 23;
    float s;
    memcpy(&s, &sb, 4);
    return p * s;
}

/* L: ln x for a positive normal x: x = 2^k m, m in [sqrt(1/2), sqrt(2)), ln m = 2s + 2s R(s^2) with s = (m - 1) / (m + 1) */
float nbo_spa_log(float x)
{
    uint32_t u;
    memcpy(&u, &x, 4);
    int k = (int)(u >> 23) - 127;
    uint32_t mb = (u & 0x7fffffu) | 0x3f800000u;
    float m;
    memcpy(&m, &mb, 4);
    if (m > 0x1.6a09e6p+0f) { m = m * 0.5f; k += 1; }
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
    return kf * 0x1.62e400p-1f + (kf * 0x1.7f7d1cp-20f + lm);
}

/* WHT without scaling: stage s = 0 .. log2 GF - 1 pairs i < j = i | 2^s, writes (v[i] + v[j], v[i] - v[j]) */
static void spa_wht(float *v, int GF)
{
    int s, i;
    for (s = 1; s < GF; s <<= 1)
        for (i = 0; i < GF; i++)
            if (!(i & s)) { const float a = v[i], b = v[i | s]; v[i] = a + b; v[i | s] = a - b; }
}

/* image of MULGF[x][h] (bubble_decoder.c:145 rotation) */
static int spa_rot(const nbo_code *c, int x, int h)
{
    const int GF = c->GF, lg = c->logGF;
    const int y = c->mulgf[x * GF + h];
    int img = 0, l;
    for (l = 0; l < lg; l++) img |= c->bingf[y * lg + l] << l;
    return img;
}

/* steps 2-7 of include/nbldpc_b200.h: mvc[dc][GF] -> ctov[dc][GF] (symbol order); cgf[dc][GF] = identity */
void nbo_check_node_spa(const nbo_code *c, int node, const float *mvc, float *ctov, int *cgf)
{
    const int GF = c->GF, dc = c->row_deg[node];
    const int *h = c->val + c->row_ptr[node];
    float *U = malloc(sizeof(float) * (size_t)dc * GF);
    float fwd[256], bwd[256], T[256];
    int e, x, k;
    for (e = 0; e < dc; e++) {
        const float *m = mvc + (size_t)e * GF;
        float *u = U + (size_t)e * GF;
        float mu = m[0];
        for (x = 1; x < GF; x++) if (m[x] < mu) mu = m[x];
        for (x = 0; x < GF; x++)
            u[spa_rot(c, x, h[e])] = (m[x] >= 1e5f && m[x] > mu) ? 0.0f : nbo_spa_exp(mu - m[x]);
        spa_wht(u, GF);
        const float r = 1.0f / u[0];
        for (k = 0; k < GF; k++) u[k] = u[k] * r;
    }
    for (k = 0; k < GF; k++) fwd[k] = 1.0f;
    for (e = 0; e < dc; e++) {
        int j;
        for (k = 0; k < GF; k++) bwd[k] = 1.0f;
        for (j = dc - 1; j > e; j--) for (k = 0; k < GF; k++) bwd[k] = bwd[k] * U[(size_t)j * GF + k];
        for (k = 0; k < GF; k++) T[k] = fwd[k] * bwd[k];
        for (k = 0; k < GF; k++) fwd[k] = fwd[k] * U[(size_t)e * GF + k];
        spa_wht(T, GF);
        float cmax = T[0];
        for (k = 1; k < GF; k++) if (T[k] > cmax) cmax = T[k];
        const float floor_c = cmax * 0x1p-20f, lmax = nbo_spa_log(cmax);
        for (x = 0; x < GF; x++) {
            float cx = T[spa_rot(c, x, h[e])];
            if (!(cx >= floor_c)) cx = floor_c;
            ctov[(size_t)e * GF + x] = lmax - nbo_spa_log(cx);
            cgf[(size_t)e * GF + x] = x;
        }
    }
    free(U);
}

/* tools.c:312-330 */
static void spa_decision(const float *app, int N, int GF, int *decide)
{
    int n, g;
    for (n = 0; n < N; n++) {
        float best = 1e5f; int ind = 0;
        for (g = 0; g < GF; g++) if (app[(size_t)n * GF + g] < best) { best = app[(size_t)n * GF + g]; ind = g; }
        decide[n] = ind;
    }
}

/* tools.c:284-299 */
static int spa_syndrome(const nbo_code *c, const int *decide)
{
    int m, k, synd = 0;
    for (m = 0; m < c->M; m++) {
        for (k = c->row_ptr[m]; k < c->row_ptr[m + 1]; k++)
            synd = c->addgf[synd * c->GF + c->mulgf[c->val[k] * c->GF + decide[c->col[k]]]];
        if (synd != 0) break;
    }
    return synd;
}

/* nbo_decode_frame with the sum-product node: same arguments and outputs; p->n_m, nb_oper, offset and ecn are not read */
int nbo_spa_decode_frame(const nbo_code *c, const nbo_params *p, const float *llr,
                         int *decide, int *synd_out, int *iters_out,
                         int *decide_trace, int *synd_trace, float *app_out, float *ctov_out)
{
    const int N = c->N, GF = c->GF, E = c->E;
    float *APP = malloc(sizeof(float) * (size_t)N * GF);
    float *CtoV = calloc((size_t)E * GF, sizeof(float));                         /* NB_LDPC.c:273-279 */
    float *mvc = malloc(sizeof(float) * (size_t)c->dc_max * GF);
    float *cl = malloc(sizeof(float) * (size_t)c->dc_max * GF);
    int *cg = malloc(sizeof(int) * (size_t)c->dc_max * GF);
    int iter, node, i, g, synd = 0, passes = 0;
    memcpy(APP, llr, sizeof(float) * (size_t)N * GF);
    for (iter = 0; iter < p->nb_iter_max - 1; iter++) {                          /* NB_LDPC.c:314 */
        for (node = 0; node < c->M; node++) {
            const int dc = c->row_deg[node], e0 = c->row_ptr[node];
            for (i = 0; i < dc; i++) {                                            /* step 1, NB_LDPC.c:334 */
                const float *a = APP + (size_t)c->col[e0 + i] * GF;
                const float *cv = CtoV + (size_t)(e0 + i) * GF;
                for (g = 0; g < GF; g++) mvc[i * GF + g] = a[g] - cv[g];
            }
            nbo_check_node_spa(c, node, mvc, cl, cg);                             /* steps 2-7 */
            for (i = 0; i < dc; i++) {                                            /* step 8, NB_LDPC.c:438, 448 */
                float *a = APP + (size_t)c->col[e0 + i] * GF;
                float *cv = CtoV + (size_t)(e0 + i) * GF;
                for (g = 0; g < GF; g++) { cv[g] = cl[i * GF + g]; a[g] = cl[i * GF + g] + mvc[i * GF + g]; }
            }
        }
        spa_decision(APP, N, GF, decide);                                         /* NB_LDPC.c:468 */
        synd = spa_syndrome(c, decide);                                           /* NB_LDPC.c:469 */
        if (decide_trace) memcpy(decide_trace + (size_t)iter * N, decide, sizeof(int) * N);
        if (synd_trace) synd_trace[iter] = synd;
        passes++;
        if (synd == 0 && !p->force_passes) break;                                 /* NB_LDPC.c:470 */
    }
    if (synd_out) *synd_out = synd;
    if (iters_out) *iters_out = iter + 1;                                         /* NB_LDPC.c:474 */
    if (app_out) memcpy(app_out, APP, sizeof(float) * (size_t)N * GF);
    if (ctov_out) memcpy(ctov_out, CtoV, sizeof(float) * (size_t)E * GF);
    free(APP); free(CtoV); free(mvc); free(cl); free(cg);
    return passes;
}
