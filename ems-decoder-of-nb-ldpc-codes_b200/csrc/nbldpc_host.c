/*
 * nbldpc_host.c -- host side of the B200 EMS NB-LDPC decoder, plain C (no CUDA).
 *
 * What the reference does once per run on the CPU stays on the CPU here, behind the same meaning:
 *   alist parsing            LoadCode            init.c:143-272   (both dialects, runtime switch)
 *   GF(q) tables             LoadTables          init.c:427-506   (+ Table_Add/Mul/Div_GF 37-130)
 *   systematic encoder       GaussianElimination tools.c:151-218, Encoding tools.c:232-268
 *   frame source / noise     RandomBinaryGenerator tools.c:124, ModelChannel_AWGN_BPSK channel.c:51-62
 *   statistics               NB_LDPC.c:474-507
 * plus what only the GPU path needs: the conflict-free step schedule of one decoding pass.
 */
#include "nbldpc_internal.h"
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

static __thread char g_err[512];

void nbgpu_set_global_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}
const char *nbgpu_get_global_error(void) { return g_err; }

const char *nbgpu_version(void) { return "nbldpc_b200 0.1 (sm_100a)"; }

/* ------------------------------------------------------------------------------------------------
 * GF(2^m): symbol 0 is zero, symbol k is alpha^(k-1) (struct.h:119-476 are the binary images for the
 * primitive polynomials x^4+x+1, x^6+x+1, x^8+x^4+x^3+x^2+1 with bit l = coefficient of x^l).
 * ---------------------------------------------------------------------------------------------- */
static int field_poly(int q)
{
    switch (q) { case 16: return 0x13; case 64: return 0x43; case 256: return 0x11D; default: return 0; }
}

static int make_tables(struct nbgpu_code *c, const int *bingf, const int *addgf, const int *mulgf, const int *divgf)
{
    const int q = c->q, lg = c->logq;
    int a, b, l;
    c->bingf = malloc(sizeof(int) * q * lg);
    c->addgf = malloc(sizeof(int) * q * q);
    c->mulgf = malloc(sizeof(int) * q * q);
    c->divgf = malloc(sizeof(int) * q * q);
    c->img = malloc(sizeof(int) * q);
    c->inv = malloc(sizeof(int) * q);
    if (!c->bingf || !c->addgf || !c->mulgf || !c->divgf || !c->img || !c->inv) return NBGPU_ENOMEM;
    if (bingf) {
        memcpy(c->bingf, bingf, sizeof(int) * q * lg);
    } else {
        int poly = field_poly(q), x = 1, k;
        if (!poly) { nbgpu_set_global_error("GF(%d) is not supported (16, 64, 256 only, as init.c:431)", q); return NBGPU_EINVAL; }
        for (l = 0; l < lg; l++) c->bingf[l] = 0;
        for (k = 1; k < q; k++) {
            for (l = 0; l < lg; l++) c->bingf[k * lg + l] = (x >> l) & 1;
            x <<= 1;
            if (x & q) x ^= poly;
        }
    }
    for (a = 0; a < q; a++) c->inv[a] = -1;
    for (a = 0; a < q; a++) {
        int v = 0;
        for (l = 0; l < lg; l++) v |= (c->bingf[a * lg + l] & 1) << l;
        c->img[a] = v;
        if (c->inv[v] != -1) { nbgpu_set_global_error("BINGF is not a bijection (symbols %d and %d)", c->inv[v], a); return NBGPU_EINVAL; }
        c->inv[v] = a;
    }
    if (addgf) memcpy(c->addgf, addgf, sizeof(int) * q * q);
    else for (a = 0; a < q; a++) for (b = 0; b < q; b++) c->addgf[a * q + b] = c->inv[c->img[a] ^ c->img[b]];
    if (mulgf) memcpy(c->mulgf, mulgf, sizeof(int) * q * q);
    else for (a = 0; a < q; a++) for (b = 0; b < q; b++)
        c->mulgf[a * q + b] = (a && b) ? ((a + b - 2) % (q - 1)) + 1 : 0;
    if (divgf) memcpy(c->divgf, divgf, sizeof(int) * q * q);
    else for (a = 0; a < q; a++) for (b = 0; b < q; b++)
        c->divgf[a * q + b] = (b == 0) ? -1 : (a ? ((a - b + (q - 1)) % (q - 1)) + 1 : 0);
    /* The kernels work on binary images (GF addition == XOR).  Check that whatever tables we were
     * handed really have that structure, and that MUL/DIV are consistent. */
    for (a = 0; a < q; a++) for (b = 0; b < q; b++) {
        if (c->addgf[a * q + b] != c->inv[c->img[a] ^ c->img[b]]) {
            nbgpu_set_global_error("ADDGF[%d][%d] is not the XOR of the binary images", a, b); return NBGPU_EINVAL;
        }
        int m = c->mulgf[a * q + b];
        if (m < 0 || m >= q || m != c->mulgf[b * q + a]) { nbgpu_set_global_error("MULGF[%d][%d] invalid", a, b); return NBGPU_EINVAL; }
        if (b != 0 && c->divgf[m * q + b] != a && !(a == 0 && c->divgf[m * q + b] == 0)) {
            nbgpu_set_global_error("DIVGF is not the inverse of MULGF at (%d,%d)", a, b); return NBGPU_EINVAL;
        }
    }
    return NBGPU_OK;
}

static void finish_graph(struct nbgpu_code *c)
{
    int m;
    c->row_ptr = malloc(sizeof(int) * (c->M + 1));
    c->row_ptr[0] = 0;
    c->dc_max = 0; c->dc_min = 1 << 30;
    for (m = 0; m < c->M; m++) {
        c->row_ptr[m + 1] = c->row_ptr[m] + c->row_deg[m];
        if (c->row_deg[m] > c->dc_max) c->dc_max = c->row_deg[m];
        if (c->row_deg[m] < c->dc_min) c->dc_min = c->row_deg[m];
    }
}

static int check_graph(const struct nbgpu_code *c)
{
    int e;
    for (e = 0; e < c->E; e++) {
        if (c->col[e] < 0 || c->col[e] >= c->N) { nbgpu_set_global_error("edge %d: column %d out of range", e, c->col[e]); return NBGPU_EINVAL; }
        if (c->val[e] < 1 || c->val[e] >= c->q) { nbgpu_set_global_error("edge %d: coefficient %d out of range", e, c->val[e]); return NBGPU_EINVAL; }
    }
    return NBGPU_OK;
}

/* All integers of the file.  The three layouts differ only in how the integers after "N M GF" are arranged:
 *   UBS  (init.c:195-207)  col degrees | row degrees | E columns (0-based) | E coefficients (symbols 1..q-1)
 *   KN   (init.c:211-227)  col degrees | row degrees | per row: (column 1-based, exponent 0..q-2) pairs
 *   FULL (SURVEY.md 8f.4; matrices/KN/N64800_*, which the reference cannot read)
 *                          dv_max dc_max | col degrees | row degrees | per column: (row, exponent) pairs |
 *                          per row: (column 1-based, exponent) pairs; lists may be zero-padded to the maximum degree */
static int read_ints(FILE *f, int **out, size_t *count)
{
    size_t cap = 1 << 16, n = 0;
    int *t = malloc(sizeof(int) * cap), v;
    if (!t) return NBGPU_ENOMEM;
    while (fscanf(f, "%d", &v) == 1) {
        if (n == cap) { cap *= 2; int *t2 = realloc(t, sizeof(int) * cap); if (!t2) { free(t); return NBGPU_ENOMEM; } t = t2; }
        t[n++] = v;
    }
    *out = t; *count = n;
    return NBGPU_OK;
}

/* FULL layout: returns 1 and fills row_deg/col/val when the token stream fits it, 0 otherwise */
static int parse_full_alist(struct nbgpu_code *c, const int *t, size_t T)
{
    const int N = c->N, M = c->M;
    if (T < (size_t)5 + N + M) return 0;
    const int dv = t[3], dc = t[4];
    const int *cd = t + 5, *rd = t + 5 + N;
    long Ec = 0, Er = 0;
    int n, m, k, mx;
    for (mx = 0, n = 0; n < N; n++) { if (cd[n] < 0 || cd[n] > dv) return 0; Ec += cd[n]; if (cd[n] > mx) mx = cd[n]; }
    if (mx != dv) return 0;
    for (mx = 0, m = 0; m < M; m++) { if (rd[m] < 0 || rd[m] > dc) return 0; Er += rd[m]; if (rd[m] > mx) mx = rd[m]; }
    if (mx != dc || Ec != Er) return 0;
    const size_t exact = (size_t)5 + N + M + 4 * (size_t)Er, padded = (size_t)5 + N + M + 2 * ((size_t)N * dv + (size_t)M * dc);
    if (T != exact && T != padded) return 0;
    const int pad = (T != exact);
    const int *cols = t + 5 + N + M;
    const int *rows = cols + (pad ? 2 * (size_t)N * dv : 2 * (size_t)Ec);
    {   /* the column lists must describe the same matrix as the row lists (only the row lists are kept) */
        size_t cpos = 0, rpos = 0;
        size_t *rstart = malloc(sizeof(size_t) * M);
        int ok = rstart != NULL;
        for (m = 0; ok && m < M; m++) { rstart[m] = rpos; rpos += pad ? 2 * (size_t)dc : 2 * (size_t)rd[m]; }
        for (n = 0; ok && n < N; n++) {
            const int *cl = cols + (pad ? 2 * (size_t)n * dv : cpos);
            cpos += 2 * (size_t)cd[n];
            for (k = 0; ok && k < cd[n]; k++) {
                const int r = cl[2 * k] - 1, e = cl[2 * k + 1];
                int found = 0, j;
                if (r < 0 || r >= M) { ok = 0; break; }
                for (j = 0; j < rd[r]; j++) if (rows[rstart[r] + 2 * j] == n + 1 && rows[rstart[r] + 2 * j + 1] == e) found = 1;
                if (!found) ok = 0;
            }
        }
        free(rstart);
        if (!ok) return 0;
    }
    c->row_deg = malloc(sizeof(int) * M);
    memcpy(c->row_deg, rd, sizeof(int) * M);
    finish_graph(c);
    c->E = c->row_ptr[M];
    c->col = malloc(sizeof(int) * c->E);
    c->val = malloc(sizeof(int) * c->E);
    for (m = 0; m < M; m++) {
        const int *r = rows + (pad ? 2 * (size_t)m * dc : 2 * (size_t)c->row_ptr[m]);
        for (k = 0; k < rd[m]; k++) { c->col[c->row_ptr[m] + k] = r[2 * k] - 1; c->val[c->row_ptr[m] + k] = r[2 * k + 1] + 1; }
    }
    return 1;
}

int nbgpu_code_load(nbgpu_code **out, const char *path, int dialect)
{
    *out = NULL;
    FILE *f = fopen(path, "r");
    if (!f) { nbgpu_set_global_error("cannot open matrix file '%s'", path); return NBGPU_EIO; }
    struct nbgpu_code *c = calloc(1, sizeof *c);
    int rc = NBGPU_EIO, n, k;
    int *tok = NULL;
    size_t T = 0;
    if ((rc = read_ints(f, &tok, &T)) != NBGPU_OK) { nbgpu_set_global_error("out of memory reading '%s'", path); goto fail; }
    rc = NBGPU_EIO;
    if (T < 3 || tok[0] <= 0 || tok[1] <= 0 || tok[1] > tok[0]) { nbgpu_set_global_error("'%s': bad alist header", path); goto fail; }
    c->N = tok[0]; c->M = tok[1]; c->q = tok[2];
    c->logq = (int)rint(log((double)c->q) / log(2.0));                 /* init.c:160-163 */
    if ((1 << c->logq) != c->q || !field_poly(c->q)) {
        nbgpu_set_global_error("GF(%d) is not supported (16, 64, 256 only, as init.c:431)", c->q); rc = NBGPU_EINVAL; goto fail;
    }
    c->K = c->N - c->M;
    c->rate = (float)(c->N - c->M) / c->N;                             /* init.c:167 */
    if ((dialect == NBGPU_ALIST_AUTO || dialect == NBGPU_ALIST_FULL) && parse_full_alist(c, tok, T)) dialect = NBGPU_ALIST_FULL;
    else if (dialect == NBGPU_ALIST_FULL) { nbgpu_set_global_error("'%s': not a full alist file (degree sums or length do not fit)", path); rc = NBGPU_EINVAL; goto fail; }
    else {
        if (T < (size_t)3 + c->N + c->M) { nbgpu_set_global_error("'%s': truncated degree lists", path); goto fail; }
        const int *coldeg = tok + 3;
        c->row_deg = malloc(sizeof(int) * c->M);
        for (n = 0; n < c->M; n++) { c->row_deg[n] = tok[3 + c->N + n]; if (c->row_deg[n] < 0) { nbgpu_set_global_error("'%s': negative row degree", path); goto fail; } }
        finish_graph(c);
        c->E = c->row_ptr[c->M];
        const int *rest = tok + 3 + c->N + c->M;
        if (T < (size_t)3 + c->N + c->M + 2 * (size_t)c->E) {
            nbgpu_set_global_error("'%s': truncated edge list (%zu of %d values)", path, T - 3 - c->N - c->M, 2 * c->E); goto fail;
        }
        if (dialect == NBGPU_ALIST_AUTO) {
            /* a dialect is plausible when all values are in range and the column degrees of the header are met */
            int ok_ubs = 1, ok_kn = 1;
            int *cnt = calloc(c->N, sizeof(int));
            for (k = 0; k < c->E && ok_ubs; k++) {
                if (rest[k] < 0 || rest[k] >= c->N || rest[c->E + k] < 1 || rest[c->E + k] >= c->q) ok_ubs = 0; else cnt[rest[k]]++;
            }
            for (n = 0; n < c->N && ok_ubs; n++) if (cnt[n] != coldeg[n]) ok_ubs = 0;
            memset(cnt, 0, sizeof(int) * c->N);
            for (k = 0; k < c->E && ok_kn; k++) {
                if (rest[2 * k] < 1 || rest[2 * k] > c->N || rest[2 * k + 1] < 0 || rest[2 * k + 1] > c->q - 2) ok_kn = 0; else cnt[rest[2 * k] - 1]++;
            }
            for (n = 0; n < c->N && ok_kn; n++) if (cnt[n] != coldeg[n]) ok_kn = 0;
            free(cnt);
            if (ok_ubs == ok_kn) {
                nbgpu_set_global_error("'%s': cannot tell the alist dialect (%s); pass NBGPU_ALIST_UBS, NBGPU_ALIST_KN or NBGPU_ALIST_FULL",
                                       path, ok_ubs ? "both fit" : "neither fits");
                rc = NBGPU_EINVAL; goto fail;
            }
            dialect = ok_ubs ? NBGPU_ALIST_UBS : NBGPU_ALIST_KN;
        }
        c->col = malloc(sizeof(int) * c->E);
        c->val = malloc(sizeof(int) * c->E);
        for (k = 0; k < c->E; k++) {
            if (dialect == NBGPU_ALIST_KN) { c->col[k] = rest[2 * k] - 1; c->val[k] = rest[2 * k + 1] + 1; }   /* init.c:218-221 */
            else { c->col[k] = rest[k]; c->val[k] = rest[c->E + k]; }                                          /* init.c:197-205 */
        }
    }
    c->dialect = dialect;
    if ((rc = check_graph(c)) != NBGPU_OK) goto fail;
    if ((rc = make_tables(c, NULL, NULL, NULL, NULL)) != NBGPU_OK) goto fail;
    free(tok); fclose(f);
    *out = c;
    return NBGPU_OK;
fail:
    free(tok); fclose(f);
    nbgpu_code_free(c);
    return rc;
}

int nbgpu_code_from_arrays(nbgpu_code **out, int N, int M, int q, const int *row_deg, const int *col,
                           const int *val, const int *bingf, const int *addgf, const int *mulgf, const int *divgf)
{
    if (!out) { nbgpu_set_global_error("nbgpu_code_from_arrays: NULL output pointer"); return NBGPU_EINVAL; }
    *out = NULL;
    if (N <= 0 || M <= 0 || M > N || !row_deg || !col || !val) { nbgpu_set_global_error("bad code arrays"); return NBGPU_EINVAL; }
    /* the kernels exist for the fields the reference's LoadTables knows (init.c:431-435): GF(16), GF(64), GF(256) */
    if (q != 16 && q != 64 && q != 256) { nbgpu_set_global_error("GF(%d) is not supported (16, 64 or 256)", q); return NBGPU_EINVAL; }
    struct nbgpu_code *c = calloc(1, sizeof *c);
    if (!c) { nbgpu_set_global_error("out of memory"); return NBGPU_ENOMEM; }
    int rc;
    c->N = N; c->M = M; c->K = N - M; c->q = q;
    c->logq = (int)rint(log((double)q) / log(2.0));
    if ((1 << c->logq) != q || (!bingf && !field_poly(q))) {
        nbgpu_set_global_error("GF(%d) is not supported", q); free(c); return NBGPU_EINVAL;
    }
    c->rate = (float)(N - M) / N;
    c->row_deg = malloc(sizeof(int) * M);
    memcpy(c->row_deg, row_deg, sizeof(int) * M);
    finish_graph(c);
    c->E = c->row_ptr[M];
    c->col = malloc(sizeof(int) * c->E); c->val = malloc(sizeof(int) * c->E);
    memcpy(c->col, col, sizeof(int) * c->E); memcpy(c->val, val, sizeof(int) * c->E);
    c->dialect = 0;
    if ((rc = check_graph(c)) != NBGPU_OK || (rc = make_tables(c, bingf, addgf, mulgf, divgf)) != NBGPU_OK) { nbgpu_code_free(c); return rc; }
    *out = c;
    return NBGPU_OK;
}

void nbgpu_code_free(nbgpu_code *c)
{
    if (!c) return;
    free(c->row_deg); free(c->row_ptr); free(c->col); free(c->val);
    free(c->bingf); free(c->addgf); free(c->mulgf); free(c->divgf); free(c->img); free(c->inv);
    free(c->piv_col); free(c->perm); free(c->ut_ptr); free(c->ut_col); free(c->ut_val);
    free(c);
}

void nbgpu_code_info(const nbgpu_code *c, int *info)
{
    info[0] = c->N; info[1] = c->M; info[2] = c->K; info[3] = c->q; info[4] = c->logq; info[5] = c->E;
    info[6] = c->dc_max; info[7] = c->dc_min; info[8] = c->dialect; info[9] = 0;
}
float nbgpu_code_rate(const nbgpu_code *c) { return c->rate; }
void nbgpu_code_graph(const nbgpu_code *c, int *row_deg, int *col, int *val)
{
    if (row_deg) memcpy(row_deg, c->row_deg, sizeof(int) * c->M);
    if (col) memcpy(col, c->col, sizeof(int) * c->E);
    if (val) memcpy(val, c->val, sizeof(int) * c->E);
}
void nbgpu_code_tables(const nbgpu_code *c, int *bingf, int *addgf, int *mulgf, int *divgf)
{
    if (bingf) memcpy(bingf, c->bingf, sizeof(int) * c->q * c->logq);
    if (addgf) memcpy(addgf, c->addgf, sizeof(int) * c->q * c->q);
    if (mulgf) memcpy(mulgf, c->mulgf, sizeof(int) * c->q * c->q);
    if (divgf) memcpy(divgf, c->divgf, sizeof(int) * c->q * c->q);
}

/* ------------------------------------------------------------------------------------------------
 * drand48 recurrence (glibc): X <- (0x5DEECE66D X + 0xB) mod 2^48, value X / 2^48.
 * ---------------------------------------------------------------------------------------------- */
#define RNG_A 0x5DEECE66DULL
#define RNG_C 0xBULL
#define RNG_M ((1ULL << 48) - 1)
void nbgpu_rng_reference_default(nbgpu_rng *r) { r->x = 0; }
double nbgpu_rng_drand48(nbgpu_rng *r)
{
    r->x = (RNG_A * r->x + RNG_C) & RNG_M;
    return (double)r->x * (1.0 / 281474976710656.0);
}
void nbgpu_rng_skip(nbgpu_rng *r, uint64_t n)
{
    uint64_t mul = RNG_A, add = RNG_C, accm = 1, acca = 0;
    for (; n; n >>= 1) {
        if (n & 1) { accm = (accm * mul) & RNG_M; acca = (acca * mul + add) & RNG_M; }
        add = ((mul + 1) * add) & RNG_M;
        mul = (mul * mul) & RNG_M;
    }
    r->x = (accm * r->x + acca) & RNG_M;
}

/* ------------------------------------------------------------------------------------------------
 * Encoder.  Same elimination order, pivot choice and column swaps as tools.c:151-218 so that the
 * codeword of a given information word is the reference's; the triangular matrix is kept sparse.
 * ---------------------------------------------------------------------------------------------- */
int nbgpu_code_prepare_encoder(nbgpu_code *c)
{
    if (c->enc_ready) return NBGPU_OK;
    const int N = c->N, M = c->M, q = c->q;
    unsigned char *U = calloc((size_t)M * N, 1);
    int *perm = malloc(sizeof(int) * N);
    if (!U || !perm) { free(U); free(perm); nbgpu_set_global_error("out of memory in encoder setup"); return NBGPU_ENOMEM; }
    int m, n, k, r;
    for (n = 0; n < N; n++) perm[n] = n;
    for (m = 0; m < M; m++) for (k = c->row_ptr[m]; k < c->row_ptr[m + 1]; k++) U[(size_t)m * N + c->col[k]] = (unsigned char)c->val[k];
    for (m = 0; m < M; m++) {
        unsigned char *pr = U + (size_t)m * N;
        int ind = m;
        while (ind < N && pr[ind] == 0) ind++;
        if (ind == N) { free(U); free(perm); nbgpu_set_global_error("The matrix is not full rank (%d,%d)", m, ind); return NBGPU_ERANK; }
        if (ind != m) {
            int t = perm[ind]; perm[ind] = perm[m]; perm[m] = t;
            for (r = 0; r < M; r++) { unsigned char *x = U + (size_t)r * N; unsigned char u = x[m]; x[m] = x[ind]; x[ind] = u; }
        }
        const int piv = pr[m];
        for (r = m + 1; r < M; r++) {
            unsigned char *x = U + (size_t)r * N;
            const int lead = x[m];
            if (!lead) continue;
            for (n = m; n < N; n++) {
                int v = x[n];
                if (v) v = c->divgf[v * q + lead];
                if (v) v = c->mulgf[v * q + piv];
                x[n] = (unsigned char)c->addgf[v * q + pr[n]];
            }
        }
    }
    size_t nnz = 0;
    for (m = 0; m < M; m++) for (n = m; n < N; n++) nnz += U[(size_t)m * N + n] != 0;
    c->ut_ptr = malloc(sizeof(int) * (M + 1));
    c->ut_col = malloc(sizeof(int) * nnz);
    c->ut_val = malloc(sizeof(int) * nnz);
    c->piv_col = malloc(sizeof(int) * M);
    nnz = 0;
    for (m = 0; m < M; m++) {
        c->ut_ptr[m] = (int)nnz;
        c->piv_col[m] = U[(size_t)m * N + m];
        for (n = m + 1; n < N; n++) if (U[(size_t)m * N + n]) { c->ut_col[nnz] = n; c->ut_val[nnz] = U[(size_t)m * N + n]; nnz++; }
    }
    c->ut_ptr[M] = (int)nnz;
    c->perm = perm;
    free(U);
    c->enc_ready = 1;
    return NBGPU_OK;
}

static float draw_float(nbgpu_rng *r) { return (float)nbgpu_rng_drand48(r); }      /* My_drand48, tools.c:73 */

int nbgpu_random_codeword(const nbgpu_code *c, nbgpu_rng *r, int *codeword, int *nbin)
{
    if (!c->enc_ready) { nbgpu_set_global_error("call nbgpu_code_prepare_encoder first"); return NBGPU_EINVAL; }
    const int N = c->N, M = c->M, q = c->q, lg = c->logq;
    int *ns = malloc(sizeof(int) * N);
    int k, l, m, n;
    for (k = 0; k < c->K; k++) {                       /* tools.c:129-135: bit = floor(u * 1.9999) */
        int bits = 0;
        for (l = 0; l < lg; l++) bits |= ((int)floor(draw_float(r) * 1.9999)) << l;
        ns[M + k] = c->inv[bits];
    }
    for (m = M - 1; m >= 0; m--) {                     /* tools.c:244-254 */
        int acc = 0;
        for (k = c->ut_ptr[m]; k < c->ut_ptr[m + 1]; k++)
            acc = c->addgf[acc * q + c->mulgf[c->ut_val[k] * q + ns[c->ut_col[k]]]];
        ns[m] = c->divgf[acc * q + c->piv_col[m]];
    }
    for (n = 0; n < N; n++) codeword[c->perm[n]] = ns[n];                             /* tools.c:257-258 */
    if (nbin) for (n = 0; n < N; n++) for (l = 0; l < lg; l++) nbin[n * lg + l] = c->bingf[codeword[n] * lg + l];
    free(ns);
    return NBGPU_OK;
}

float nbgpu_sigma(const nbgpu_code *c, float EbN)
{
    return (float)sqrt(1.0 / (2.0 * c->rate * pow(10, EbN / 10.0)));                    /* channel.c:51 */
}

/* noisy[nt][points][dims] of one frame: transmitted symbol t, variable n = tx[t] (tx = NULL: n = t, every symbol sent) with
 * binary image nbin[n][0..logq) (LSB first), is sent as `points` points of m = logq / points bits, point j as
 * mod[sub-image j] = mod[(img >> j*m) & (2^m - 1)], each coordinate plus Box-Muller noise from two draws in stream order:
 * channel.c:52-62 (BPSK: one point per bit, dims = 1, mod = {+1, -1}) and channel.c:234-263 (mapped: one point, dims = 2;
 * split: P points, dims = 2) */
static void awgn_points(const nbgpu_code *c, nbgpu_rng *r, const int *nbin, const int *tx, int nt, int points, int dims,
                        const float *mod, float sigma, float *noisy)
{
    const int m = c->logq / points;
    int t, b, j;
    for (t = 0; t < nt; t++) {
        const int n = tx ? tx[t] : t;
        int som = 0;
        for (b = 0; b < c->logq; b++) som += (nbin ? nbin[n * c->logq + b] : 0) << b;
        for (j = 0; j < points; j++) {
            const int sub = (som >> (j * m)) & ((1 << m) - 1);
            for (b = 0; b < dims; b++) {
                float u = draw_float(r);
                float v = draw_float(r);
                *noisy++ = nbgpu_mapped_sample(sigma, mod[dims * sub + b], u, v);
            }
        }
    }
}

static const float bpsk_points[2] = { 1.0f, -1.0f };                                   /* channel.c:59: 1 - 2*bit */

int nbgpu_awgn_bpsk_noise(const nbgpu_code *c, nbgpu_rng *r, const int *nbin, float EbN, float *noisy)
{
    awgn_points(c, r, nbin, NULL, c->N, c->logq, 1, bpsk_points, nbgpu_sigma(c, EbN), noisy);
    return NBGPU_OK;
}

/* ------------------------------------------------------------------------------------------------
 * 64-APSK over AWGN (ModelChannel_AWGN_64, channel.c:112-312): one GF(64) symbol = one point of the
 * DVB-S2X 8+16+20+20 APSK constellation, two noisy reals (I, Q) per symbol.  The host side is the constellation,
 * sigma and the noise; the LLR computation is a GPU intake kernel (nbldpc_cuda.cu).
 * ---------------------------------------------------------------------------------------------- */
#define NB_PI 3.1415926536                                     /* channel.c:18 */
/* a constellation point as the reference's initialiser writes it (channel.c:133-198): radius * cos / sin(PI * num / den),
 * evaluated in double, stored as float.  Index = binary image of the symbol (LSB first). */
#define APSK(r, num, den) { (float)((r) * cos(NB_PI * (num) / (den))), (float)((r) * sin(NB_PI * (num) / (den))) }
#define APSK1(num, den) { (float)cos(NB_PI * (num) / (den)), (float)sin(NB_PI * (num) / (den)) }
int nbgpu_apsk64_table(float *mod)
{
    /* rings of radius 1, 2.2, 3.6, 5.2 with 8, 16, 20, 20 points; the order is the bit labelling of the constellation */
    const float pts[64][2] = {
        APSK(2.2, 25, 16), APSK(2.2, 23, 16), APSK(2.2, 7, 16), APSK(2.2, 9, 16), APSK(5.2, 7, 4), APSK(5.2, 5, 4), APSK(5.2, 1, 4), APSK(5.2, 3, 4),
        APSK(2.2, 27, 16), APSK(2.2, 21, 16), APSK(2.2, 5, 16), APSK(2.2, 11, 16), APSK(3.6, 7, 4), APSK(3.6, 5, 4), APSK(3.6, 1, 4), APSK(3.6, 3, 4),
        APSK(5.2, 31, 20), APSK(5.2, 29, 20), APSK(5.2, 9, 20), APSK(5.2, 11, 20), APSK(5.2, 33, 20), APSK(5.2, 27, 20), APSK(5.2, 7, 20), APSK(5.2, 13, 20),
        APSK(3.6, 31, 20), APSK(3.6, 29, 20), APSK(3.6, 9, 20), APSK(3.6, 11, 20), APSK(3.6, 33, 20), APSK(3.6, 27, 20), APSK(3.6, 7, 20), APSK(3.6, 13, 20),
        APSK1(13, 8), APSK1(11, 8), APSK1(3, 8), APSK1(5, 8), APSK(5.2, 37, 20), APSK(5.2, 23, 20), APSK(5.2, 3, 20), APSK(5.2, 17, 20),
        APSK(2.2, 29, 16), APSK(2.2, 19, 16), APSK(2.2, 3, 16), APSK(2.2, 13, 16), APSK(3.6, 37, 20), APSK(3.6, 23, 20), APSK(3.6, 3, 20), APSK(3.6, 17, 20),
        APSK1(15, 8), APSK1(9, 8), APSK1(1, 8), APSK1(7, 8), APSK(5.2, 39, 20), APSK(5.2, 21, 20), APSK(5.2, 1, 20), APSK(5.2, 19, 20),
        APSK(2.2, 31, 16), APSK(2.2, 17, 16), APSK(2.2, 1, 16), APSK(2.2, 15, 16), APSK(3.6, 39, 20), APSK(3.6, 21, 20), APSK(3.6, 1, 20), APSK(3.6, 19, 20) };
    float norm = 0.0f;
    int i;
    if (!mod) return NBGPU_EINVAL;
    for (i = 0; i < 64; i++) norm = pts[i][0] * pts[i][0] + pts[i][1] * pts[i][1] + norm;      /* channel.c:205-211: average power 1 */
    norm = sqrt(64 / norm);
    for (i = 0; i < 64; i++) { mod[2 * i] = norm * pts[i][0]; mod[2 * i + 1] = norm * pts[i][1]; }   /* :215-222 */
    return NBGPU_OK;
}
float nbgpu_sigma_apsk64(float EbN)
{
    return (float)sqrt(1.0 / (2.0 * pow(10, EbN / 10.0)));      /* channel.c:232 (no code rate here) */
}
/* one sample of channel.c:59 (point = 1 - 2*bit) or channel.c:234-263 (point = I or Q coordinate of a constellation point),
 * for any table; also the host recomputation of the samples the device source flags (nbldpc_source.cuh) */
float nbgpu_mapped_sample(float sigma, float point, float u, float v)
{
    const double pi = NB_PI;
    return (float)(point + sigma * sqrt(-2.0 * log(u)) * cos(2.0 * pi * v));
}

/* Gray-labelled square M-QAM, M = 2^(2m), m bits per axis: mod[M][2] of average power 1 (include/nbldpc_b200.h, NBGPU_MAP_QAM) */
static void gray_qam(int m, float *mod)
{
    const int L = 1 << m, M = L * L;
    const double scale = sqrt(2.0 * (M - 1) / 3.0);             /* average power 1 */
    for (int x = 0; x < M; x++)
        for (int c = 0; c < 2; c++) {
            const int g = (x >> (c * m)) & (L - 1);                 /* I: bits [0, m), Q: bits [m, 2m) */
            int level = g;
            for (int s = g >> 1; s; s >>= 1) level ^= s;            /* inverse binary-reflected Gray code */
            mod[2 * x + c] = (float)((double)(2 * level - (L - 1)) / scale);
        }
}

int nbgpu_constellation(int kind, int q, float *mod)
{
    if (!mod) { nbgpu_set_global_error("nbgpu_constellation: NULL table"); return NBGPU_EINVAL; }
    if (kind == NBGPU_MAP_APSK64) {
        if (q != 64) { nbgpu_set_global_error("nbgpu_constellation: 64-APSK has 64 points, not q = %d", q); return NBGPU_EINVAL; }
        return nbgpu_apsk64_table(mod);
    }
    if (kind != NBGPU_MAP_QAM) { nbgpu_set_global_error("nbgpu_constellation: unknown kind %d (NBGPU_MAP_APSK64 = %d, NBGPU_MAP_QAM = %d)", kind, NBGPU_MAP_APSK64, NBGPU_MAP_QAM); return NBGPU_EINVAL; }
    if (q != 16 && q != 64 && q != 256) { nbgpu_set_global_error("nbgpu_constellation: square QAM for q = 16, 64 or 256, not %d", q); return NBGPU_EINVAL; }
    gray_qam(q == 16 ? 2 : q == 64 ? 3 : 4, mod);
    return NBGPU_OK;
}

int nbgpu_split_points_ok(int logq, int points)
{
    return points >= 2 && points <= logq && logq % points == 0;
}

int nbgpu_split_qam(int q, int points, float *mod)
{
    const int logq = q == 16 ? 4 : q == 64 ? 6 : q == 256 ? 8 : 0;
    if (!mod) { nbgpu_set_global_error("nbgpu_split_qam: NULL table"); return NBGPU_EINVAL; }
    if (!logq || !nbgpu_split_points_ok(logq, points) || (logq / points) % 2) {
        nbgpu_set_global_error("nbgpu_split_qam: no square QAM for GF(%d) over %d points per symbol (built in: (16, 2), (64, 3), "
                               "(256, 2), (256, 4); for other pairs bind your own table)", q, points);
        return NBGPU_EINVAL;
    }
    gray_qam(logq / points / 2, mod);
    return NBGPU_OK;
}

/* noisy[N][2]: the point mod[img] of symbol n plus Box-Muller noise, channel.c:234-263 */
int nbgpu_awgn_mapped_noise(const nbgpu_code *c, nbgpu_rng *r, const int *nbin, const float *mod, float EbN, float *noisy)
{
    if (!c || !r || !mod || !noisy) { nbgpu_set_global_error("nbgpu_awgn_mapped_noise: NULL argument"); return NBGPU_EINVAL; }
    awgn_points(c, r, nbin, NULL, c->N, 1, 2, mod, nbgpu_sigma_apsk64(EbN), noisy);
    return NBGPU_OK;
}

int nbgpu_rotate_constellation(int q, double degrees, const float *mod, float *out)
{
    if (q != 16 && q != 64 && q != 256) { nbgpu_set_global_error("nbgpu_rotate_constellation: q = %d (16, 64 or 256)", q); return NBGPU_EINVAL; }
    if (!mod || !out) { nbgpu_set_global_error("nbgpu_rotate_constellation: NULL table"); return NBGPU_EINVAL; }
    if (!isfinite(degrees)) { nbgpu_set_global_error("nbgpu_rotate_constellation: degrees = %g is not finite", degrees); return NBGPU_EINVAL; }
    const double t = degrees * (M_PI / 180.0), c = cos(t), s = sin(t);
    for (int x = 0; x < q; x++) {
        const double i = mod[2 * x], qq = mod[2 * x + 1];     /* both read before out (which may be mod) is written */
        out[2 * x] = (float)(i * c - qq * s);
        out[2 * x + 1] = (float)(i * s + qq * c);
    }
    return NBGPU_OK;
}

/* the faded channel's one symbol (include/nbldpc_b200.h, NBGPU_FADING_SYMBOL); also the host recomputation of the faded
 * symbols the device source flags (nbldpc_source.cuh) */
void nbgpu_faded_sample(float sigma, const float *m, const float *d, int fading, float *rx)
{
    const double pi = NB_PI;
    const float rho_i = (float)sqrt(-log((double)d[4]));
    const float rho_q = fading == NBGPU_FADING_COMPONENT ? (float)sqrt(-log((double)d[5])) : rho_i;
    rx[0] = (float)((double)rho_i * (double)m[0] + sigma * sqrt(-2.0 * log(d[0])) * cos(2.0 * pi * d[1]));
    rx[1] = (float)((double)rho_q * (double)m[1] + sigma * sqrt(-2.0 * log(d[2])) * cos(2.0 * pi * d[3]));
    rx[2] = rho_i;
    rx[3] = rho_q;
}

/* rx[nt][4] of one frame of the faded mapped channel, transmitted symbols as in awgn_points: per symbol u_I, v_I, u_Q, v_Q,
 * w_I (, w_Q) */
static void faded_points(const nbgpu_code *c, nbgpu_rng *r, const int *nbin, const int *tx, int nt, const float *mod, float sigma,
                         int fading, float *rx)
{
    const int S = fading == NBGPU_FADING_COMPONENT ? 6 : 5;
    int t, b;
    for (t = 0; t < nt; t++) {
        const int n = tx ? tx[t] : t;
        int som = 0;
        float d[6];
        for (b = 0; b < c->logq; b++) som += (nbin ? nbin[n * c->logq + b] : 0) << b;
        for (b = 0; b < S; b++) d[b] = draw_float(r);
        nbgpu_faded_sample(sigma, mod + 2 * som, d, fading, rx + 4 * (size_t)t);
    }
}

static int fading_ok(const char *fn, int fading)
{
    if (fading == NBGPU_FADING_SYMBOL || fading == NBGPU_FADING_COMPONENT) return 1;
    nbgpu_set_global_error("%s: fading %d (NBGPU_FADING_SYMBOL = 1, NBGPU_FADING_COMPONENT = 2)", fn, fading);
    return 0;
}

int nbgpu_awgn_faded_noise(const nbgpu_code *c, nbgpu_rng *r, const int *nbin, const float *mod, float EbN, int fading, float *rx)
{
    if (!c || !r || !mod || !rx) { nbgpu_set_global_error("nbgpu_awgn_faded_noise: NULL argument"); return NBGPU_EINVAL; }
    if (!fading_ok("nbgpu_awgn_faded_noise", fading)) return NBGPU_EINVAL;
    faded_points(c, r, nbin, NULL, c->N, mod, nbgpu_sigma_apsk64(EbN), fading, rx);
    return NBGPU_OK;
}

/* noisy[N][P][2] of one frame of the split channel: point j of symbol n is mod[sub-image j], u, v for I then u, v for Q */
int nbgpu_awgn_split_noise(const nbgpu_code *c, nbgpu_rng *r, const int *nbin, int points, const float *mod, float EbN, float *noisy)
{
    if (!c || !r || !mod || !noisy) { nbgpu_set_global_error("nbgpu_awgn_split_noise: NULL argument"); return NBGPU_EINVAL; }
    if (!nbgpu_split_points_ok(c->logq, points)) {
        nbgpu_set_global_error("nbgpu_awgn_split_noise: %d points per GF(%d) symbol (need P >= 2 dividing log2 q = %d)", points, c->q, c->logq);
        return NBGPU_EINVAL;
    }
    awgn_points(c, r, nbin, NULL, c->N, points, 2, mod, nbgpu_sigma_apsk64(EbN), noisy);
    return NBGPU_OK;
}

/* noisy[N][2] over the 64-APSK table (nbgpu_apsk64_table) */
int nbgpu_awgn_apsk64_noise(const nbgpu_code *c, nbgpu_rng *r, const int *nbin, float EbN, float *noisy)
{
    float mod[128];
    if (!c || !r || !noisy) { nbgpu_set_global_error("nbgpu_awgn_apsk64_noise: NULL argument"); return NBGPU_EINVAL; }
    if (c->q != 64) { nbgpu_set_global_error("64-APSK maps one GF(64) symbol to one constellation point (q = %d)", c->q); return NBGPU_EINVAL; }
    nbgpu_apsk64_table(mod);
    return nbgpu_awgn_mapped_noise(c, r, nbin, mod, EbN, noisy);
}

/* ---- Puncturing (include/nbldpc_b200.h, nbgpu_set_puncturing) ---- */
int nbgpu_puncture_map(int N, int p, const int *vars, int *map)
{
    int i, n, nt = 0;
    if (p < 0 || p >= N || (p > 0 && !vars)) {
        nbgpu_set_global_error("puncturing pattern: p = %d of N = %d variables (0 <= p <= N-1, and a list for p > 0)", p, N);
        return NBGPU_EINVAL;
    }
    for (n = 0; n < N; n++) map[n] = 0;
    for (i = 0; i < p; i++) {
        if (vars[i] < 0 || vars[i] >= N) { nbgpu_set_global_error("puncturing pattern: variable %d outside [0, %d)", vars[i], N); return NBGPU_EINVAL; }
        if (map[vars[i]]) { nbgpu_set_global_error("puncturing pattern: variable %d listed twice", vars[i]); return NBGPU_EINVAL; }
        map[vars[i]] = -1;
    }
    for (n = 0; n < N; n++) map[n] = map[n] ? -1 : nt++;
    return nt;
}

float nbgpu_sigma_punctured(const nbgpu_code *c, int p, float EbN)
{
    if (p < 0 || p >= c->N) { nbgpu_set_global_error("nbgpu_sigma_punctured: p = %d of N = %d variables", p, c->N); return NAN; }
    const float rate_p = (float)(c->N - c->M) / (c->N - p);                            /* init.c:167 over N - p symbols */
    return (float)sqrt(1.0 / (2.0 * rate_p * pow(10, EbN / 10.0)));                     /* channel.c:51 */
}

int nbgpu_awgn_punctured_noise(const nbgpu_code *c, nbgpu_rng *r, const int *nbin, int channel, int arg, const float *mod,
                               float EbN, int p, const int *vars, float *noisy)
{
    if (!c || !r || !noisy || (channel != NBGPU_CHANNEL_BPSK && !mod)) {
        nbgpu_set_global_error("nbgpu_awgn_punctured_noise: NULL argument");
        return NBGPU_EINVAL;
    }
    if (channel < NBGPU_CHANNEL_BPSK || channel > NBGPU_CHANNEL_SPLIT) {
        nbgpu_set_global_error("nbgpu_awgn_punctured_noise: channel %d (NBGPU_CHANNEL_BPSK .. NBGPU_CHANNEL_SPLIT = 0 .. 3)", channel);
        return NBGPU_EINVAL;
    }
    if (channel == NBGPU_CHANNEL_FADED && !fading_ok("nbgpu_awgn_punctured_noise", arg)) return NBGPU_EINVAL;
    if (channel == NBGPU_CHANNEL_SPLIT && !nbgpu_split_points_ok(c->logq, arg)) {
        nbgpu_set_global_error("nbgpu_awgn_punctured_noise: %d points per GF(%d) symbol (need P >= 2 dividing log2 q = %d)", arg, c->q, c->logq);
        return NBGPU_EINVAL;
    }
    int *map = malloc(sizeof(int) * 2 * (size_t)c->N), *tx = map + c->N;
    if (!map) { nbgpu_set_global_error("nbgpu_awgn_punctured_noise: out of memory"); return NBGPU_ENOMEM; }
    const int nt = nbgpu_puncture_map(c->N, p, vars, map);
    if (nt < 0) { free(map); return nt; }
    for (int n = 0; n < c->N; n++) if (map[n] >= 0) tx[map[n]] = n;
    const float sigma = channel == NBGPU_CHANNEL_BPSK ? nbgpu_sigma_punctured(c, p, EbN) : nbgpu_sigma_apsk64(EbN);
    if (channel == NBGPU_CHANNEL_BPSK) awgn_points(c, r, nbin, tx, nt, c->logq, 1, bpsk_points, sigma, noisy);
    else if (channel == NBGPU_CHANNEL_MAPPED) awgn_points(c, r, nbin, tx, nt, 1, 2, mod, sigma, noisy);
    else if (channel == NBGPU_CHANNEL_SPLIT) awgn_points(c, r, nbin, tx, nt, arg, 2, mod, sigma, noisy);
    else faded_points(c, r, nbin, tx, nt, mod, sigma, arg, noisy);
    free(map);
    return NBGPU_OK;
}


/* NB_LDPC.c:474-507 */
int nbgpu_accumulate_stats(const nbgpu_code *c, const int *codeword_bits, const int *decide,
                           const int *synd, const int *iters, int B, long *stats)
{
    const int N = c->N, lg = c->logq;
    int f, k, l;
    for (f = 0; f < B; f++) {
        if (stats[5]) break;
        int e = 0;
        const int *d = decide + (size_t)f * N;
        const int *cb = codeword_bits + (size_t)f * N * lg;
        for (k = 0; k < c->K; k++) {
            if (d[k] < 0 || d[k] >= c->q) { nbgpu_set_global_error("decision out of range"); return NBGPU_EINVAL; }
            for (l = 0; l < lg; l++) e += c->bingf[d[k] * lg + l] != cb[k * lg + l];
        }
        stats[0] += 1;
        stats[4] += iters[f];
        stats[3] += e;
        if (e) { stats[1] += 1; if (synd[f] == 0) stats[2] += 1; }
        if (stats[1] == 40) stats[5] = 1;
    }
    return NBGPU_OK;
}

/* the same rule fed with per-frame error counts (nbgpu_source_results) */
int nbgpu_accumulate_results(const int *bit_errors, const int *synd, const int *iters, int B, long *stats)
{
    int f;
    for (f = 0; f < B; f++) {
        if (stats[5]) break;
        stats[0] += 1;
        stats[4] += iters[f];
        stats[3] += bit_errors[f];
        if (bit_errors[f]) { stats[1] += 1; if (synd[f] == 0) stats[2] += 1; }
        if (stats[1] == 40) stats[5] = 1;
    }
    return NBGPU_OK;
}

/* ------------------------------------------------------------------------------------------------
 * Pass schedule.  The reference updates check nodes 0..M-1 in file order and rewrites APP after
 * each one (NB_LDPC.c:320, 448), so node m must see the APP rows written by every earlier node that
 * shares a variable with it -- and nothing else constrains the order.  Nodes are packed first-fit
 * into steps of at most 'cap' mutually independent nodes: step(m) > step(m') for every earlier m'
 * that shares a variable.  Any such packing reproduces the reference bit for bit.
 * ---------------------------------------------------------------------------------------------- */
int nbgpu_build_schedule(const struct nbgpu_code *c, int cap, nbgpu_schedule *out)
{
    const int M = c->M, N = c->N;
    int m, k;
    int *last_step = malloc(sizeof(int) * N);     /* step of the latest node (file order) touching a variable */
    int *step_of = malloc(sizeof(int) * M);
    int *fill = calloc((size_t)M + 1, sizeof(int));
    int *first_free = malloc(sizeof(int));
    int nsteps = 0, depth = 0;
    int *lvl_var = malloc(sizeof(int) * N);
    if (cap < 1) cap = 1;
    for (k = 0; k < N; k++) { last_step[k] = -1; lvl_var[k] = -1; }
    *first_free = 0;
    for (m = 0; m < M; m++) {
        int s = 0, lv = 0;
        for (k = c->row_ptr[m]; k < c->row_ptr[m + 1]; k++) {
            if (last_step[c->col[k]] + 1 > s) s = last_step[c->col[k]] + 1;
            if (lvl_var[c->col[k]] + 1 > lv) lv = lvl_var[c->col[k]] + 1;
        }
        if (s < *first_free) s = *first_free;
        while (fill[s] >= cap) s++;
        fill[s]++;
        while (*first_free < M && fill[*first_free] >= cap) (*first_free)++;
        step_of[m] = s;
        if (s + 1 > nsteps) nsteps = s + 1;
        if (lv + 1 > depth) depth = lv + 1;
        for (k = c->row_ptr[m]; k < c->row_ptr[m + 1]; k++) { last_step[c->col[k]] = s; lvl_var[c->col[k]] = lv; }
    }
    out->nsteps = nsteps;
    out->depth = depth;
    out->step_ptr = calloc((size_t)nsteps + 1, sizeof(int));
    out->order = malloc(sizeof(int) * M);
    for (m = 0; m < M; m++) out->step_ptr[step_of[m] + 1]++;
    for (k = 0; k < nsteps; k++) out->step_ptr[k + 1] += out->step_ptr[k];
    int *pos = malloc(sizeof(int) * (nsteps + 1));
    memcpy(pos, out->step_ptr, sizeof(int) * (nsteps + 1));
    for (m = 0; m < M; m++) out->order[pos[step_of[m]]++] = m;      /* file order inside a step */
    free(pos); free(last_step); free(step_of); free(fill); free(first_free); free(lvl_var);
    return NBGPU_OK;
}

void nbgpu_free_schedule(nbgpu_schedule *s)
{
    free(s->step_ptr); free(s->order);
    s->step_ptr = NULL; s->order = NULL; s->nsteps = 0;
}

/* ------------------------------------------------------------------------------------------------
 * Configuration table of the syndrome-based check node: what build_config_table
 * (syndrome_decoder.c:1542; generator gen_config_table2, :1661-1767) followed by sort_config_table
 * (:2285-2371) and the truncation of NB_LDPC.c:198-201 produce.  A configuration gives, per edge of
 * the check node, the index of the V->C list entry that is used (0 = most reliable).  Generated here:
 * the all-zero configuration, single deviations 1..d1, pairs with (k-1)+(l-1) < d2, triples with
 * total < d3, and the reference's hard-wired four-edge block (three of the four deviations sum to
 * less than 2, the fourth is 1 or 2).  Ordered by cost = sum over deviating edges of
 * (deviation + 3*edge), ties in generation order (the reference uses a stable insertion sort).
 * ---------------------------------------------------------------------------------------------- */
typedef struct { float cost; int id; } cfg_key;

int *nbgpu_build_config_table(int dc, int d1, int d2, int d3, int trunc, int *size_out)
{
    const int d4 = 2;
    int a, b, c, e, x, y, z, w, n = 0, cap = 64;
    int *tab = NULL;
    *size_out = 0;
    if (dc < 1 || dc > 16 || d1 < 0 || d2 < 0 || d3 < 0) return NULL;
#define CFG_PUSH() do { if (n == cap || !tab) { cap *= 2; tab = realloc(tab, sizeof(int) * (size_t)cap * dc); if (!tab) return NULL; } \
                        memset(tab + (size_t)n * dc, 0, sizeof(int) * dc); n++; } while (0)
#define CFG(i) tab[(size_t)(n - 1) * dc + (i)]
    CFG_PUSH();                                                     /* configuration 0: no deviation */
    for (a = 0; a < dc; a++) for (x = 1; x <= d1; x++) { CFG_PUSH(); CFG(a) = x; }
    for (a = 0; a < dc - 1; a++) for (b = a + 1; b < dc; b++)
        for (x = 1; x <= d2; x++) for (y = 1; y <= d2; y++)
            if (x + y - 2 < d2) { CFG_PUSH(); CFG(a) = x; CFG(b) = y; }
    for (a = 0; a < dc - 2; a++) for (b = a + 1; b < dc - 1; b++) for (c = b + 1; c < dc; c++)
        for (x = 1; x <= d3; x++) for (y = 1; y <= d3; y++) for (z = 1; z <= d3; z++)
            if (x + y + z - 3 < d3) { CFG_PUSH(); CFG(a) = x; CFG(b) = y; CFG(c) = z; }
    for (e = 0; e < dc - 3; e++) for (a = e + 1; a < dc - 2; a++) for (b = a + 1; b < dc - 1; b++) for (c = b + 1; c < dc; c++)
        for (x = 1; x <= d4; x++) for (y = 1; y <= d4; y++) for (z = 1; z <= d4; z++) for (w = 1; w <= d4; w++)
            if (x + y + z - 3 < d4) { CFG_PUSH(); CFG(a) = x; CFG(b) = y; CFG(c) = z; CFG(e) = w; }
#undef CFG
#undef CFG_PUSH
    cfg_key *k = malloc(sizeof(cfg_key) * (size_t)n);
    if (!k) { free(tab); return NULL; }
    for (a = 0; a < n; a++) {
        float cost = 0;
        for (b = 0; b < dc; b++) if (tab[(size_t)a * dc + b] > 0) cost = cost + tab[(size_t)a * dc + b] + 3.0 * b;
        k[a].cost = cost; k[a].id = a;
    }
    for (a = 1; a < n; a++) {                                       /* stable insertion sort, as sorting() :1315 */
        cfg_key t = k[a];
        for (b = a - 1; b >= 0 && k[b].cost > t.cost; b--) k[b + 1] = k[b];
        k[b + 1] = t;
    }
    const int size = (trunc > 0 && trunc < n) ? trunc : n;
    int *out = malloc(sizeof(int) * (size_t)size * dc);
    if (out) for (a = 0; a < size; a++) memcpy(out + (size_t)a * dc, tab + (size_t)k[a].id * dc, sizeof(int) * dc);
    free(k); free(tab);
    if (out) *size_out = size;
    return out;
}

/* public wrapper: copies the table into a caller buffer (NULL: only the size is returned) */
int nbgpu_config_table(int dc, int d1, int d2, int d3, int trunc, int *table, int capacity)
{
    int size = 0;
    int *t = nbgpu_build_config_table(dc, d1, d2, d3, trunc, &size);
    if (!t) { nbgpu_set_global_error("cannot build the configuration table (dc=%d d=(%d,%d,%d))", dc, d1, d2, d3); return NBGPU_EINVAL; }
    if (table) {
        if (capacity < size) { free(t); nbgpu_set_global_error("configuration table needs %d rows, buffer has %d", size, capacity); return NBGPU_EINVAL; }
        memcpy(table, t, sizeof(int) * (size_t)size * dc);
    }
    free(t);
    return size;
}
