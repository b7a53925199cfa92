/*
 * tests/minmax_oracle.c -- TEST INFRASTRUCTURE ONLY: the Min-Max check node (ecn_kind = 4), restated from its definition in
 * include/nbldpc_b200.h with plain O(q^2) convolutions and no pruning, and the decode loop of nbo_decode_frame
 * (oracle/nbldpc_oracle.c, NB_LDPC.c:266-474) with that node in place of the EMS nodes.  The reference has no such node, so
 * this file is the specification the GPU kernel is checked against bit for bit.  A library of its own (tests/minmax_oracle.py
 * builds it with -ffp-contract=off): it works on the nbo_code of liboracle.so (oracle/nbldpc_oracle.h) and shares no code
 * with the product.  The only float arithmetic is steps 1, 2 and 6, one IEEE f32 operation each; the rest compares values.
 */
#include "nbldpc_oracle.h"
#include <stdlib.h>
#include <string.h>

/* image of MULGF[x][h] (bubble_decoder.c:145 rotation) */
static int mm_rot(const nbo_code *c, int x, int h)
{
    const int GF = c->GF, lg = c->logGF;
    const int y = c->mulgf[x * GF + h];
    int img = 0, l;
    for (l = 0; l < lg; l++) img |= c->bingf[y * lg + l] << l;
    return img;
}

/* out = A (*) B: out[z] = min_a max(A[a], B[a ^ z]) */
static void mm_conv(const float *A, const float *B, float *out, int GF)
{
    int z, a;
    for (z = 0; z < GF; z++) {
        float best = A[0] > B[z] ? A[0] : B[z];
        for (a = 1; a < GF; a++) {
            const float v = A[a] > B[a ^ z] ? A[a] : B[a ^ z];
            if (v < best) best = v;
        }
        out[z] = best;
    }
}

/* steps 2-5 of include/nbldpc_b200.h: mvc[dc][GF] -> ctov[dc][GF] (symbol order); t_e folds u_j, j != e, in edge order */
void nbo_check_node_minmax(const nbo_code *c, int node, const float *mvc, float *ctov)
{
    const int GF = c->GF, dc = c->row_deg[node];
    const int *h = c->val + c->row_ptr[node];
    float *U = malloc(sizeof(float) * (size_t)dc * GF);
    float t[256], tmp[256];
    int e, j, x;
    for (e = 0; e < dc; e++) {
        const float *m = mvc + (size_t)e * GF;
        float mu = m[0];
        for (x = 1; x < GF; x++) if (m[x] < mu) mu = m[x];
        for (x = 0; x < GF; x++) U[(size_t)e * GF + mm_rot(c, x, h[e])] = m[x] - mu;
    }
    for (e = 0; e < dc; e++) {
        int first = 1;
        for (j = 0; j < dc; j++) {
            if (j == e) continue;
            if (first) { memcpy(t, U + (size_t)j * GF, sizeof(float) * GF); first = 0; continue; }
            mm_conv(t, U + (size_t)j * GF, tmp, GF);
            memcpy(t, tmp, sizeof(float) * GF);
        }
        for (x = 0; x < GF; x++) ctov[(size_t)e * GF + x] = t[mm_rot(c, x, h[e])];
    }
    free(U);
}

/* tools.c:312-330 */
static void mm_decision(const float *app, int N, int GF, int *decide)
{
    int n, g;
    for (n = 0; n < N; n++) {
        float best = 1e5f; int ind = 0;
        for (g = 0; g < GF; g++) if (app[(size_t)n * GF + g] < best) { best = app[(size_t)n * GF + g]; ind = g; }
        decide[n] = ind;
    }
}

/* tools.c:284-299 */
static int mm_syndrome(const nbo_code *c, const int *decide)
{
    int m, k, synd = 0;
    for (m = 0; m < c->M; m++) {
        for (k = c->row_ptr[m]; k < c->row_ptr[m + 1]; k++)
            synd = c->addgf[synd * c->GF + c->mulgf[c->val[k] * c->GF + decide[c->col[k]]]];
        if (synd != 0) break;
    }
    return synd;
}

/* nbo_decode_frame with the Min-Max node: same arguments and outputs; p->n_m, nb_oper, offset and ecn are not read */
int nbo_minmax_decode_frame(const nbo_code *c, const nbo_params *p, const float *llr,
                            int *decide, int *synd_out, int *iters_out,
                            int *decide_trace, int *synd_trace, float *app_out, float *ctov_out)
{
    const int N = c->N, GF = c->GF, E = c->E;
    float *APP = malloc(sizeof(float) * (size_t)N * GF);
    float *CtoV = calloc((size_t)E * GF, sizeof(float));                         /* NB_LDPC.c:273-279 */
    float *mvc = malloc(sizeof(float) * (size_t)c->dc_max * GF);
    float *cl = malloc(sizeof(float) * (size_t)c->dc_max * GF);
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
            nbo_check_node_minmax(c, node, mvc, cl);                              /* steps 2-5 */
            for (i = 0; i < dc; i++) {                                            /* step 6, NB_LDPC.c:438, 448 */
                float *a = APP + (size_t)c->col[e0 + i] * GF;
                float *cv = CtoV + (size_t)(e0 + i) * GF;
                for (g = 0; g < GF; g++) { cv[g] = cl[i * GF + g]; a[g] = mvc[i * GF + g] + cl[i * GF + g]; }
            }
        }
        mm_decision(APP, N, GF, decide);                                          /* NB_LDPC.c:468 */
        synd = mm_syndrome(c, decide);                                            /* NB_LDPC.c:469 */
        if (decide_trace) memcpy(decide_trace + (size_t)iter * N, decide, sizeof(int) * N);
        if (synd_trace) synd_trace[iter] = synd;
        passes++;
        if (synd == 0 && !p->force_passes) break;                                 /* NB_LDPC.c:470 */
    }
    if (synd_out) *synd_out = synd;
    if (iters_out) *iters_out = iter + 1;                                         /* NB_LDPC.c:474 */
    if (app_out) memcpy(app_out, APP, sizeof(float) * (size_t)N * GF);
    if (ctov_out) memcpy(ctov_out, CtoV, sizeof(float) * (size_t)E * GF);
    free(APP); free(CtoV); free(mvc); free(cl);
    return passes;
}
