/* nbldpc_internal.h -- shared between the C host layer (nbldpc_host.c) and the CUDA layer. */
#ifndef NBLDPC_INTERNAL_H
#define NBLDPC_INTERNAL_H
#include "nbldpc_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

struct nbgpu_code {
    int N, M, K, q, logq, E, dc_max, dc_min, dialect;
    float rate;
    int *row_deg;      /* [M]   */
    int *row_ptr;      /* [M+1] */
    int *col;          /* [E]   */
    int *val;          /* [E]   */
    int *bingf;        /* [q*logq] */
    int *addgf, *mulgf, *divgf;   /* [q*q] */
    int *img;          /* [q] binary image of each symbol (bit l = bingf[s][l]) */
    int *inv;          /* [q] symbol of each binary image */
    /* encoder (lazy) */
    int  enc_ready;
    int *piv_col;      /* see nbldpc_host.c */
    int *perm;
    int *ut_ptr, *ut_col, *ut_val;   /* sparse upper-triangular rows */
};

/* schedule of one decoding pass: check nodes packed into steps of mutually independent nodes while
 * keeping the reference's update order between nodes that share a variable (NB_LDPC.c:320) */
typedef struct {
    int nsteps;
    int *step_ptr;     /* [nsteps+1] into order */
    int *order;        /* [M] check node ids grouped by step */
    int depth;         /* dependency depth (steps with unlimited width) */
} nbgpu_schedule;

int  nbgpu_build_schedule(const struct nbgpu_code *c, int cap, nbgpu_schedule *out);
void nbgpu_free_schedule(nbgpu_schedule *s);
void nbgpu_set_global_error(const char *fmt, ...);
const char *nbgpu_get_global_error(void);

/* one noisy sample, (float)(point + sigma*sqrt(-2 ln u)*cos(2 PI v)): channel.c:59 (point = 1 - 2*bit) or channel.c:234-263
 * (point = an I or Q coordinate of any table) */
float nbgpu_mapped_sample(float sigma, float point, float u, float v);
/* one faded symbol: draws d[] = u_I, v_I, u_Q, v_Q, w_I (, w_Q) of the stream, point m[2] -> rx[4] = (y_I, y_Q, rho_I, rho_Q) */
void nbgpu_faded_sample(float sigma, const float *m, const float *d, int fading, float *rx);
/* split channel: 1 if `points` points per GF(q) symbol is allowed (P >= 2 dividing log2 q), else 0 */
int nbgpu_split_points_ok(int logq, int points);
/* puncturing pattern of p variables of N: map[N] = compact index of each variable in the frames, -1 = punctured.  Returns
 * Nt = N - p, or NBGPU_EINVAL with the message of nbgpu_set_puncturing (map then partly written) */
int nbgpu_puncture_map(int N, int p, const int *vars, int *map);

/* syndrome_ems configuration table (syndrome_decoder.c:1542, 1661, 2285); returns malloc'd [size*dc] */
int *nbgpu_build_config_table(int dc, int d1, int d2, int d3, int trunc, int *size_out);

#ifdef __cplusplus
}
#endif
#endif
