/*
 * nbldpc_b200.h -- C ABI of the B200-native EMS NB-LDPC decoder (libnbldpc_b200.so).
 *
 * Drop-in boundary for the decode path of Lcrypto/EMS-decoder-of-NB-LDPC-codes.  The reference has no
 * FFI; its "interface" for this path is the set of C calls made by main() (NB_LDPC.c).  Every entry
 * point below names the reference call(s) it replaces.  Plain pointers and sizes only; no CUDA, torch
 * or C++ types appear here.  All functions return 0 (NBGPU_OK) or a negative NBGPU_E* code and never
 * call exit(); the message is available from nbgpu_last_error().  A context is bound to one device
 * and one CUDA stream; different contexts are independent.  There is NO CPU fallback: every compute
 * entry point fails with NBGPU_ECUDA when no sm_100 device is usable.
 *
 * Conventions kept from the reference (SURVEY.md section 3.5):
 *   - LLRs are float32 "distances": smaller = more likely; +1e5 = absent.
 *   - GF symbols are ints 0..q-1: 0 = zero element, k = alpha^(k-1); q in {16,64,256}.
 *   - edge e of check node m is the e-th entry in file order (numB in NB_LDPC.c:266-460).
 *   - "nb_iter_max" is argv[2]: at most nb_iter_max-1 decoding passes run (NB_LDPC.c:314).
 */
#ifndef NBLDPC_B200_H
#define NBLDPC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NBGPU_OK        0
#define NBGPU_EINVAL   -1   /* bad argument / unsupported parameter combination */
#define NBGPU_EIO      -2   /* matrix file missing or malformed                  */
#define NBGPU_ENOMEM   -3
#define NBGPU_ECUDA    -4   /* CUDA error or no usable GPU                        */
#define NBGPU_ESTATE   -5   /* requested frame state no longer resident           */
#define NBGPU_ERANK    -6   /* H is rank deficient (tools.c:181-185)             */

/* ------------------------------------------------------------------------------------------------
 * Host side (plain C, no GPU needed): code description = code_t + table_t of the reference.
 * ---------------------------------------------------------------------------------------------- */
typedef struct nbgpu_code nbgpu_code;

#define NBGPU_ALIST_AUTO 0
#define NBGPU_ALIST_UBS  1   /* init.c:195-207 : all columns (0-based) then all coefficients (1..q-1) */
#define NBGPU_ALIST_KN   2   /* init.c:211-227 : per row (col 1-based, exponent 0..q-2) pairs          */
#define NBGPU_ALIST_FULL 3   /* full alist (max-degree line, column lists, then row lists of (col 1-based, exponent) pairs):
                                matrices/KN/N64800_*, which the reference's LoadCode cannot read (SURVEY.md 8f.4) */

/* replaces LoadCode (init.c:143) + LoadTables (init.c:427).  The alist dialect is a runtime switch
 * instead of the compile-time '#define KN_matrix' (init.c:25). */
int nbgpu_code_load(nbgpu_code **out, const char *path, int dialect);

/* Bind an already loaded reference code_t/table_t (flattened by the caller, see INTEGRATION.md):
 * row_deg[M]; col[E], val[E] in edge order; bingf[q*logq]; addgf/mulgf/divgf[q*q] (may be NULL: the
 * tables are then generated exactly as init.c:37-130 does). */
int nbgpu_code_from_arrays(nbgpu_code **out, int N, int M, int q, const int *row_deg, const int *col,
                           const int *val, const int *bingf, const int *addgf, const int *mulgf,
                           const int *divgf);
void nbgpu_code_free(nbgpu_code *c);

/* info[10] = N, M, K, q, logq, E, dc_max, dc_min, dialect used, reserved */
void nbgpu_code_info(const nbgpu_code *c, int *info);
float nbgpu_code_rate(const nbgpu_code *c);                                  /* code_t.rate, init.c:167 */
/* copies of code_t.mat/matValue (edge order) and of the table_t tables, as ints like the reference */
void nbgpu_code_graph(const nbgpu_code *c, int *row_deg, int *col, int *val);
void nbgpu_code_tables(const nbgpu_code *c, int *bingf, int *addgf, int *mulgf, int *divgf);

/* Frame source on the host, replaces RandomBinaryGenerator + GaussianElimination + Encoding
 * (tools.c:124, 151, 232) and the noise part of ModelChannel_AWGN_BPSK (channel.c:51-62).
 * The generator is glibc's drand48 recurrence; state = 48-bit X (the reference never seeds it, so its
 * stream starts from X = 0).  All frames of a Monte-Carlo run can be generated independently with
 * nbgpu_rng_skip. */
typedef struct { uint64_t x; } nbgpu_rng;
void nbgpu_rng_reference_default(nbgpu_rng *r);
void nbgpu_rng_skip(nbgpu_rng *r, uint64_t ndraws);
double nbgpu_rng_drand48(nbgpu_rng *r);
int nbgpu_code_prepare_encoder(nbgpu_code *c);                               /* tools.c:151; NBGPU_ERANK */
int nbgpu_random_codeword(const nbgpu_code *c, nbgpu_rng *r, int *codeword /*[N]*/, int *nbin /*[N*logq]*/);
float nbgpu_sigma(const nbgpu_code *c, float EbN);                           /* channel.c:51 */
int nbgpu_awgn_bpsk_noise(const nbgpu_code *c, nbgpu_rng *r, const int *nbin, float EbN,
                          float *noisy /*[N*logq]*/);                        /* channel.c:52-62 */

/* ---- 64-APSK over AWGN: ModelChannel_AWGN_64, channel.c:112-312 (GF(64) codes only; SURVEY.md 8f row 2) ----
 * nbgpu_apsk64_table     the normalised DVB-S2X 8+16+20+20 APSK constellation, mod[64][2], indexed by the symbol's binary
 *                        image (channel.c:133-222)
 * nbgpu_sigma_apsk64     sigma = sqrt(1 / (2 * 10^(EbN/10))), channel.c:232
 * nbgpu_awgn_apsk64_noise  noisy[N][2] = constellation point + Box-Muller noise on the caller's drand48 stream, same draw
 *                        order as the reference (per symbol: u, v for I, then u, v for Q), channel.c:234-263 */
int nbgpu_apsk64_table(float *mod /*[64][2]*/);
float nbgpu_sigma_apsk64(float EbN);
int nbgpu_awgn_apsk64_noise(const nbgpu_code *c, nbgpu_rng *r, const int *nbin /*[N][6] or NULL = all-zero word*/, float EbN,
                            float *noisy /*[N][2]*/);

/* ---- Mapped channels: one GF(q) symbol = one point of a q-point 2-D constellation mod[q][2] (I, Q), indexed by the
 * symbol's binary image (LSB first), as nbgpu_apsk64_table is; two noisy reals per symbol, noisy[N][2].  q = 16, 64, 256.
 * Sigma convention of every mapped call: the one of the reference's 64-APSK channel (channel.c:232),
 * sigma = nbgpu_sigma_apsk64(EbN) = sqrt(1 / (2 * 10^(EbN/10))), with neither the code rate nor the bits per symbol.  For a
 * constellation of average power 1 the argument is therefore Es/N0 in dB; converting from Eb/N0 is the caller's job.
 *
 * nbgpu_constellation     writes mod[q][2]:
 *   NBGPU_MAP_APSK64  q = 64 only; equals nbgpu_apsk64_table.
 *   NBGPU_MAP_QAM     Gray-labelled square q-QAM, q = 16, 64 or 256, L = sqrt(q) levels per axis, m = log2(L): image bits
 *                     [0, m) give the I level and bits [m, 2m) the Q level; the level index is the inverse binary-reflected
 *                     Gray code of those bits; the coordinate is (float)((2*level - (L-1)) / sqrt(2*(q-1)/3)), evaluated in
 *                     double and rounded once (average power 1).
 *   Anything else is NBGPU_EINVAL with a message.
 * nbgpu_awgn_mapped_noise  noisy[N][2] = mod[image of symbol n] + Box-Muller noise on the caller's drand48 stream, in the
 *                     draw order of channel.c:234-263 (per symbol: u, v for I, then u, v for Q: 4N draws).
 *                     nbgpu_awgn_apsk64_noise is this call on the 64-APSK table. */
#define NBGPU_MAP_APSK64 1
#define NBGPU_MAP_QAM    2
int nbgpu_constellation(int kind, int q, float *mod /*[q][2]*/);
int nbgpu_awgn_mapped_noise(const nbgpu_code *c, nbgpu_rng *r, const int *nbin /*[N][logq] or NULL = all-zero word*/,
                            const float *mod /*[q][2]*/, float EbN, float *noisy /*[N][2]*/);

/* ---- Faded mapped channels: the mapped channel under Rayleigh fading with perfect channel state at the receiver ----
 * Symbol n is received as y_c = rho_c * mod[img(s_n)][c] + sigma * n_c, c = I, Q, with a real Rayleigh amplitude rho_c,
 * E[rho^2] = 1 (coherent detection with perfect CSI reduces complex fading to this form):
 *   NBGPU_FADING_SYMBOL     one amplitude per symbol, rho_I = rho_Q;
 *   NBGPU_FADING_COMPONENT  independent amplitudes for I and Q (signal-space diversity, for rotated constellations).
 * Sigma and EbN as for every mapped call (nbgpu_sigma_apsk64); with E[rho^2] = 1 the argument is the average Es/N0.
 * Received frame: rx[N][4] = (y_I, y_Q, rho_I, rho_Q) f32 per symbol ([B][N][4] for a batch).
 * LLR of symbol k: LLR[k] = (float)((double)(d_I*d_I)/den + (double)(d_Q*d_Q)/den), d_c = y_c - rho_c*m_c (product and
 *   difference in f32, round to nearest), den = 2*(double)(float)(sigma^2), (m_I, m_Q) = mod[img(k)].  With rho = 1 this is
 *   the mapped channel's LLR bit for bit; rho = 0 (an erased symbol) gives a constant row.  rx is not validated.
 * Stream: frame f owns the draws [f*D, (f+1)*D), D = K log2(q) + S*N, S = 5 (SYMBOL) or 6 (COMPONENT).  Symbol n reads its
 *   draws from K log2(q) + S*n on, in the order u_I, v_I, u_Q, v_Q, w_I and (COMPONENT only) w_Q, each (float)drand48();
 *   rho = (float)sqrt(-log((double)w)) (w = 1.0f gives rho = 0, a legal value);
 *   y_c = (float)((double)rho_c*(double)m_c + sigma*sqrt(-2 ln u_c)*cos(2 PI v_c)), PI = 3.1415926536.
 *
 * nbgpu_rotate_constellation  out[x] = (m_I cos t - m_Q sin t, m_I sin t + m_Q cos t), t = degrees in radians, computed in
 *                       double and rounded once; out may equal mod.  NBGPU_EINVAL for q not in {16, 64, 256}, a NULL
 *                       pointer or non-finite degrees.
 * nbgpu_awgn_faded_noise  rx[N][4] of one frame on the caller's drand48 stream (S*N draws); a bad fading value is
 *                       NBGPU_EINVAL. */
#define NBGPU_FADING_SYMBOL    1
#define NBGPU_FADING_COMPONENT 2
int nbgpu_rotate_constellation(int q, double degrees, const float *mod /*[q][2]*/, float *out /*[q][2], may equal mod*/);
int nbgpu_awgn_faded_noise(const nbgpu_code *c, nbgpu_rng *r, const int *nbin /*[N][logq] or NULL = all-zero word*/,
                           const float *mod /*[q][2]*/, float EbN, int fading, float *rx /*[N][4]*/);

/* ---- Split channel: one GF(q) symbol sent as P points of a smaller constellation (e.g. GF(256) over 16-QAM or QPSK) ----
 * P points per symbol, P >= 2 dividing log2(q): q = 16: P in {2, 4}; q = 64: {2, 3, 6}; q = 256: {2, 4, 8}.  Each point
 * carries m = log2(q)/P bits; the table is mod[M][2], M = 2^m, indexed by the point's m-bit sub-image (P*M <= 32).
 *   Point j of symbol n carries image bits [j*m, (j+1)*m) (LSB first): sub_j = (img(s_n) >> (j*m)) & (M-1), sent as
 *   mod[sub_j].  Symbol n is sent as points n*P ... n*P+P-1 (no interleaving across symbols).
 *   Frame: noisy[N][P][2] (I, Q per point), [B][N][P][2] for a batch.
 * Sigma and EbN as for every mapped call (nbgpu_sigma_apsk64); for a unit-power table the argument is Es/N0 per POINT.
 * LLR of symbol k: t_j[x] = (double)(dI*dI)/den + (double)(dQ*dQ)/den with dI = y_{j,I} - mod[x][0], dQ = y_{j,Q} - mod[x][1]
 *   (differences and squares in f32, round to nearest; divisions and the addition in f64), den = 2*(double)(float)(sigma^2);
 *   LLR[k] = (float)(((t_0[sub_0] + t_1[sub_1]) + t_2[sub_2]) + ...): summed in f64 for j = 0 ... P-1, rounded to f32 once.
 * Stream: frame f owns the draws [f*D, (f+1)*D), D = K log2(q) + 4*N*P.  Point p = n*P + j reads its draws from
 *   K log2(q) + 4p on, in the order u_I, v_I, u_Q, v_Q, each (float)drand48(); y = (float)(point + sigma*sqrt(-2 ln u)*cos(2 PI v))
 *   as for the mapped channel: the mapped stream over N*P points.
 *
 * nbgpu_split_qam     writes mod[M][2] for the pairs with an even m: Gray square M-QAM by the closed form of NBGPU_MAP_QAM with
 *                     q replaced by M: (16, 2), (64, 3) and (256, 4) give QPSK, (256, 2) gives 16-QAM (bit for bit
 *                     nbgpu_constellation(NBGPU_MAP_QAM, 16)).  Any other pair (odd m has no built-in table: bind your own) or
 *                     a NULL table is NBGPU_EINVAL with a message, and the buffer is left untouched.
 * nbgpu_awgn_split_noise  noisy[N][P][2] of one frame on the caller's drand48 stream (4*N*P draws); NBGPU_EINVAL for a bad P
 *                     or a NULL argument. */
int nbgpu_split_qam(int q, int points, float *mod /*[M][2]*/);
int nbgpu_awgn_split_noise(const nbgpu_code *c, nbgpu_rng *r, const int *nbin /*[N][logq] or NULL = all-zero word*/, int points,
                           const float *mod /*[M][2]*/, float EbN, float *noisy /*[N][P][2]*/);

/* ---- Puncturing: variables of the code that are never sent (rate matching) ----
 * Pattern: p distinct variable indices in [0, N), in any order, 0 <= p <= N-1.  Nt = N - p variables are transmitted and keep
 *   their order: compact index t is the t-th unpunctured variable.
 * Frames: while a pattern is bound to a context (nbgpu_set_puncturing), every call of it that takes or returns frames uses
 *   compact frames [B][Nt][fps] with the channel's floats per symbol fps (logq BPSK, q dense LLR, 2 64-APSK and mapped, 4
 *   faded, 2P split): upload, decode (the streamed path included), channel, frame source and nbgpu_source_download, which
 *   returns noisy [B][Nt][fps] and codewords [B][N].  The frame source's limit B*Nt*fps < 2^31 replaces B*N*fps.
 * Intake: a punctured variable's intake row is all 0.0f (no information); transmitted rows are computed exactly as without a
 *   pattern.  A punctured decode is therefore bit for bit nbgpu_decode_llr on the expanded llr[B][N][q] with zero rows there.
 *   nbgpu_channel_* return llr[B][N][q] with zero rows at punctured variables; their sorted intrinsics are all 0.0f in GF
 *   order (the stable sort).  An isolated punctured variable (no check node) decides symbol 0.
 * Stream: frame f owns the draws [f*D, (f+1)*D), D = K log2(q) + S*Nt, with the channel's draws per symbol S (2 log2(q) BPSK,
 *   4 64-APSK and mapped, 5 or 6 faded, 4P split).  The information bits are drawn as without a pattern, then each transmitted
 *   symbol in compact order takes its S draws; punctured symbols draw nothing.  This is the unpunctured stream with the
 *   punctured symbols' draws removed; p = 0 is the unpunctured stream.
 * Sigma: BPSK takes the rate of the transmitted word, rate_p = (float)(N - M) / (N - p) (init.c:167 over Nt symbols), and
 *   sigma = (float)sqrt(1 / (2 rate_p 10^(EbN/10))) as nbgpu_sigma (nbgpu_sigma_punctured; p = 0 gives nbgpu_sigma).  The
 *   constellation channels keep Es/N0 (nbgpu_sigma_apsk64) and do not depend on the rate.
 * Scoring: bit errors are counted over the first K symbols of the full decided word (NB_LDPC.c:479-485); decisions and soft
 *   output cover all N variables.
 *
 * nbgpu_sigma_punctured       sigma of the punctured BPSK channel; NaN (with a message) for p outside [0, N).
 * nbgpu_awgn_punctured_noise  the compact frame noisy[Nt][fps] of one channel on the caller's drand48 stream (S*Nt draws), with
 *                             channel = NBGPU_CHANNEL_BPSK (mod unused), _MAPPED (mod[q][2]; 64-APSK is the mapped channel on
 *                             nbgpu_apsk64_table), _FADED (arg = fading) or _SPLIT (mod[M][2], arg = points).  NBGPU_EINVAL for
 *                             a bad channel, fading or points, a NULL argument or a pattern nbgpu_set_puncturing refuses.  With
 *                             p = 0 it equals the channel's own noise call. */
#define NBGPU_CHANNEL_BPSK   0
#define NBGPU_CHANNEL_MAPPED 1
#define NBGPU_CHANNEL_FADED  2
#define NBGPU_CHANNEL_SPLIT  3
float nbgpu_sigma_punctured(const nbgpu_code *c, int p, float EbN);
int nbgpu_awgn_punctured_noise(const nbgpu_code *c, nbgpu_rng *r, const int *nbin /*[N][logq] or NULL = all-zero word*/, int channel,
                               int arg, const float *mod, float EbN, int p, const int *vars /*[p]*/, float *noisy /*[N-p][fps]*/);


/* Configuration table of the syndrome-based check node: replaces build_config_table + sort_config_table
 * (syndrome_decoder.c:1542, 2285) and the truncation NB_LDPC.c:198-201.  Returns the number of
 * configurations (rows of dc ints) or a negative error; table may be NULL to query the size. */
int nbgpu_config_table(int dc, int d1, int d2, int d3, int trunc, int *table, int capacity);

/* ------------------------------------------------------------------------------------------------
 * Device side
 * ---------------------------------------------------------------------------------------------- */
/* The sum-product check node (ecn_kind = 2).  The schedule, CtoV initialisation (all 0), Decision, Syndrom, early
 * termination, iteration counts and statistics are those of the other two kinds; only the check-node update differs.
 * Limits: q in {16, 64, 256}, check degrees 2 ... 16, irregular rows included.  For check node m with edges e = 0 ... dc-1
 * in file order, variable v_e and coefficient h_e, all arithmetic in IEEE f32 rounded to nearest, one operation at a time:
 *   1. Mvc_e[x] = APP[v_e][x] - CtoV_e[x].
 *   2. mu_e = min_x Mvc_e[x];  p_e[x] = 0 where Mvc_e[x] >= 1e5 and Mvc_e[x] > mu_e ("absent"), else E(mu_e - Mvc_e[x]).
 *      So max_x p_e[x] = 1.
 *   3. Into the check domain: u_e[img(MULGF[x][h_e])] = p_e[x]  (img = binary image).
 *   4. U_e = WHT(u_e): stage s = 0 ... log2 q - 1 pairs the indices i < j that differ in bit s only and writes
 *      (u[i] + u[j], u[i] - u[j]).  Then r_e = 1 / U_e[0] (one division) and U_e[k] = U_e[k] * r_e for every k.
 *   5. T_e[k] = fwd_e[k] * bwd_e[k] with fwd_0 = 1, fwd_{e+1} = fwd_e * U_e, bwd_{dc-1} = 1, bwd_{e-1} = bwd_e * U_e.
 *   6. t_e = WHT(T_e) with the same stages, no 1/q factor.  c_max = max_k t_e[k].
 *   7. c_e[x] = max(t_e[img(MULGF[x][h_e])], c_max * tau) with tau = 2^-20, and CtoV_e[x] = L(c_max) - L(c_e[x]),
 *      which lies in [0, 20 ln 2].  The exact t_e is q times a probability vector, so c_max >= 1; measured against a
 *      float64 brute force, the round-off of the transforms stays below 2^-24 c_max, so values under tau c_max carry
 *      round-off of 1/16 of themselves or more.
 *   8. APP[v_e][x] = Mvc_e[x] + CtoV_e[x].
 * E and L are the library's f32 exp and log (csrc/nbldpc_spa_math.h): explicit range reduction and a fixed polynomial,
 * so that every build gives the same bits.  E: d < -87 gives 0, else largest error 1.22 ulp over [-87, 0].  L: largest
 * error 1.97 ulp over [2^-24, 2^9].  Both bounds come from an exhaustive check over every float of those domains
 * (scripts/check_spa_math.c). */
/* The Min-Max check node (ecn_kind = 4; Savin, 2008).  Schedule, CtoV initialisation, Decision, Syndrom, early termination,
 * iteration counts, statistics and limits are those of the sum-product node.  For check node m with edges e = 0 ... dc-1 in
 * file order, variable v_e and coefficient h_e, all arithmetic in IEEE f32 rounded to nearest, one operation at a time:
 *   1. Mvc_e[x] = APP[v_e][x] - CtoV_e[x].
 *   2. mu_e = min_x Mvc_e[x];  w_e[x] = Mvc_e[x] - mu_e.  So w_e >= 0, and w_e = 0 at the minimum.  Values >= 1e5 get no
 *      special case: a large value loses every max/min on its own.
 *   3. Into the check domain: u_e[img(MULGF[x][h_e])] = w_e[x].
 *   4. With the min-max convolution over XOR of binary images, (A (*) B)[z] = min_a max(A[a], B[a ^ z]):
 *      t_e = (*) of u_j over j != e, i.e. t_e[z] is the least, over the configurations (y_j), j != e, with XOR y_j = z, of
 *      max_j u_j[y_j].  For dc = 2, t_0 = u_1 and t_1 = u_0.  (*) is associative and commutative and every result is one of
 *      its inputs, so any order of evaluation gives the same bits; the kernel relies on that (forward and backward partials,
 *      pruned candidates).
 *   5. Back to the variable domain: CtoV_e[x] = t_e[img(MULGF[x][h_e])].  So min_x CtoV_e[x] = 0, and CtoV_e takes only values
 *      of the w rows.
 *   6. APP[v_e][x] = Mvc_e[x] + CtoV_e[x], with Mvc the value of step 1.
 * n_m, nb_oper and offset are validated as for the other kinds and not used. */
typedef struct {
    int   n_m;          /* decoder.nbMax, argv[5]; 5 <= n_m <= min(q,32)                          */
    int   nb_oper;      /* NbOper, argv[7]: max pops per ElementaryStep                            */
    int   nb_iter_max;  /* NbIterMax, argv[2] (>= 2)                                               */
    float offset;       /* argv[6]                                                                 */
    int   ecn_kind;     /* 0 = CheckPassLogEMS (L-Bubble F/B), 1 = syndrome_ems, 2 = sum-product
                           (q-ary belief propagation, above), 4 = Min-Max (above); for 2 and 4,
                           n_m, nb_oper and offset are validated as for the other kinds but not
                           used.  3 is not assigned.                                                */
    int   early_stop;   /* 1 = stop a frame at the first zero syndrome (NB_LDPC.c:470); 0 = always
                           run nb_iter_max-1 passes (fixed-iteration throughput mode)               */
    /* syndrome_ems only (NB_LDPC.c:185-201, commented out there; see DESIGN.md "Syndrome path").
       0 = default: d1 = n_m-1, d2 = min(15, n_m-1), d3 = min(5, n_m-1), cfg_trunc = 1000, n_cv = nb_oper
       (NB_LDPC.c:185), border = 4 (syndrome_decoder.c:56; the only supported value) */
    int   d1, d2, d3, cfg_trunc, n_cv, border;
    /* tuning; 0 = automatic */
    int   frames_per_cta;  /* frames decoded together by one CTA                                  */
    int   cns_per_step;    /* upper bound on the check nodes (over all frames of a CTA) per step  */
} nbgpu_params;

typedef struct nbgpu_ctx nbgpu_ctx;

/* replaces AllocateDecoder (init.c:310): owns all device memory; code is only read during the call */
int nbgpu_create(nbgpu_ctx **out, const nbgpu_code *code, const nbgpu_params *p, int device, int max_batch);
void nbgpu_destroy(nbgpu_ctx *ctx);                                          /* FreeDecoder, init.c:395 */
const char *nbgpu_last_error(const nbgpu_ctx *ctx);   /* ctx may be NULL: error of the last failed create/load */

/* Intake (a13 minus the RNG): LLR part of ModelChannel_AWGN_BPSK (channel.c:66-91) for B frames.
 * noisy[B][N][logq] are the received BPSK samples (NoisyBin).  Outputs (host, any may be NULL):
 * llr[B][N][q] dense in GF order (what NB_LDPC.c:281-288 scatters into APP), and the sorted
 * decoder_t.intrinsic_LLR / intrinsic_GF [B][N][q]. */
int nbgpu_channel_awgn_bpsk(nbgpu_ctx *ctx, const float *noisy, float sigma, int B,
                            float *llr, float *intrinsic_llr, int *intrinsic_gf);

/* Replaces the per-frame loop body NB_LDPC.c:266-474 for B frames (B <= max_batch).
 * Inputs are HOST buffers; outputs (host): decide[B][N] hard decisions (tools.c:312), synd[B] value
 * of the last Syndrom call (tools.c:284; 0 <=> codeword), iters[B] = iter+1 as added to sum_it
 * (NB_LDPC.c:474). */
int nbgpu_decode_noisy(nbgpu_ctx *ctx, const float *noisy /*[B][N][logq]*/, float sigma, int B,
                       int *decide, int *synd, int *iters);
int nbgpu_decode_llr(nbgpu_ctx *ctx, const float *llr /*[B][N][q] GF order*/, int B,
                     int *decide, int *synd, int *iters);
/* LLR part of ModelChannel_AWGN_64 on the GPU (channel.c:266-308): dense LLR[B][N][64] and, when illr/igf are given, the sorted
 * intrinsic_LLR / intrinsic_GF; nbgpu_decode_apsk64 = the same intake fused into the decoder (replaces channel.c:266-308 +
 * NB_LDPC.c:266-474 for B frames); nbgpu_upload_apsk64 + nbgpu_run + nbgpu_download is the resident-input form. */
int nbgpu_channel_awgn_apsk64(nbgpu_ctx *ctx, const float *noisy /*[B][N][2]*/, float sigma, int B,
                              float *llr, float *illr, int *igf);
int nbgpu_decode_apsk64(nbgpu_ctx *ctx, const float *noisy /*[B][N][2]*/, float sigma, int B,
                        int *decide, int *synd, int *iters);
/* The mapped channel (see nbgpu_constellation) on any field: nbgpu_set_constellation copies a caller's mod[q][2] into the
 * context's bound table (NBGPU_EINVAL for NULL or a non-finite value, context unchanged; no table is bound after
 * nbgpu_create).  The *_mapped calls then work as their 64-APSK counterparts with that table in place of the 64-APSK one:
 * LLR[k] = (float)((double)((I - mI)^2) / (2 sigma^2) + (double)((Q - mQ)^2) / (2 sigma^2)), (mI, mQ) = mod[image of k].
 * A *_mapped call with no bound table is NBGPU_ESTATE.  Every resident batch records the table it was uploaded or generated
 * with: re-binding while a mapped batch is resident drops that batch (nbgpu_run returns NBGPU_ESTATE; its soft output and
 * source results are gone); BPSK, LLR and 64-APSK batches are unaffected, and the *_apsk64 calls always use the 64-APSK
 * table. */
int nbgpu_set_constellation(nbgpu_ctx *ctx, const float *mod /*[q][2]*/);
int nbgpu_channel_awgn_mapped(nbgpu_ctx *ctx, const float *noisy /*[B][N][2]*/, float sigma, int B,
                              float *llr, float *illr, int *igf);
int nbgpu_decode_mapped(nbgpu_ctx *ctx, const float *noisy /*[B][N][2]*/, float sigma, int B,
                        int *decide, int *synd, int *iters);
/* The faded mapped channel (see NBGPU_FADING_SYMBOL) on the bound table: as the *_mapped calls, with rx[B][N][4] =
 * (y_I, y_Q, rho_I, rho_Q) in place of noisy[B][N][2].  NBGPU_ESTATE with no bound table; re-binding drops a resident faded
 * batch as it drops a mapped one.  Soft output works on faded batches as on any other. */
int nbgpu_channel_faded(nbgpu_ctx *ctx, const float *rx /*[B][N][4]*/, float sigma, int B, float *llr, float *illr, int *igf);
int nbgpu_decode_faded(nbgpu_ctx *ctx, const float *rx /*[B][N][4]*/, float sigma, int B, int *decide, int *synd, int *iters);
/* The split channel (see nbgpu_split_qam): nbgpu_set_split_constellation copies a caller's mod[M][2], M = 2^(log2(q)/points),
 * into the context's split table, a binding of its own beside the one of nbgpu_set_constellation (NBGPU_EINVAL for a bad
 * points, NULL or a non-finite value, context unchanged; none is bound after nbgpu_create).  The *_split calls work as their
 * *_mapped counterparts with noisy[B][N][P][2] in place of noisy[B][N][2], including the streamed path of nbgpu_decode_split,
 * soft output, and nbgpu_source_download returning noisy[B][N][P][2].  NBGPU_ESTATE with no split table bound.  Re-binding the split table drops a resident split batch (nbgpu_run returns NBGPU_ESTATE; its soft output and
 * source results are gone) and leaves mapped, faded, BPSK and LLR batches alone; nbgpu_set_constellation does not drop a
 * split batch. */
int nbgpu_set_split_constellation(nbgpu_ctx *ctx, int points, const float *mod /*[M][2]*/);
int nbgpu_channel_split(nbgpu_ctx *ctx, const float *noisy /*[B][N][P][2]*/, float sigma, int B, float *llr, float *illr, int *igf);
int nbgpu_decode_split(nbgpu_ctx *ctx, const float *noisy /*[B][N][P][2]*/, float sigma, int B, int *decide, int *synd, int *iters);
/* Puncturing (semantics in "Puncturing" above): binds the pattern vars[p] to the context; p = 0 unbinds (vars may
 * then be NULL).  NBGPU_EINVAL, context unchanged, for NULL vars with p > 0, p < 0, p >= N, an index outside [0, N) or a
 * duplicate.  Binding any pattern (re-binding and unbinding included) drops the resident batch: nbgpu_run returns NBGPU_ESTATE
 * and names the reason, and the soft output, nbgpu_source_results and nbgpu_source_download return NBGPU_ESTATE until a new
 * batch is uploaded or generated.  The constellation bindings are independent of the pattern. */
int nbgpu_set_puncturing(nbgpu_ctx *ctx, int p, const int *vars /*[p]*/);

/* Same work split into stages so that a caller can keep inputs resident in HBM (bench.py "value"):
 * upload (H2D) -> run (kernel only, asynchronous on the ctx stream) -> download (D2H + sync). */
int nbgpu_upload_noisy(nbgpu_ctx *ctx, const float *noisy, float sigma, int B);
int nbgpu_upload_apsk64(nbgpu_ctx *ctx, const float *noisy /*[B][N][2]*/, float sigma, int B);   /* 64-APSK samples, see below */
int nbgpu_upload_mapped(nbgpu_ctx *ctx, const float *noisy /*[B][N][2]*/, float sigma, int B);   /* mapped samples, bound table */
int nbgpu_upload_faded(nbgpu_ctx *ctx, const float *rx /*[B][N][4]*/, float sigma, int B);       /* faded samples + CSI, bound table */
int nbgpu_upload_split(nbgpu_ctx *ctx, const float *noisy /*[B][N][P][2]*/, float sigma, int B); /* split samples, split table */
int nbgpu_upload_llr(nbgpu_ctx *ctx, const float *llr, int B);
int nbgpu_run(nbgpu_ctx *ctx);                  /* decode the resident batch; returns after launch    */
int nbgpu_sync(nbgpu_ctx *ctx);
int nbgpu_download(nbgpu_ctx *ctx, int *decide, int *synd, int *iters);
/* device time (CUDA events on the ctx stream) of the decode kernel in the last nbgpu_run, ms */
int nbgpu_last_kernel_ms(nbgpu_ctx *ctx, float *ms);
/* number of kernels launched by this ctx since creation (bench.py gpu_launches) */
long nbgpu_launch_count(const nbgpu_ctx *ctx);
/* device-side stopwatch on the ctx stream (CUDA events): begin records, end records + waits + returns ms */
int nbgpu_timer_begin(nbgpu_ctx *ctx);
int nbgpu_timer_end(nbgpu_ctx *ctx, float *ms);
/* page-lock / unlock a caller-owned host buffer so that the H2D/D2H copies of nbgpu_decode_* are DMA copies */
int nbgpu_host_register(void *ptr, size_t bytes);
int nbgpu_host_unregister(void *ptr);
/* geometry chosen by nbgpu_create: geo[8] = grid (CTAs), frames per CTA group, check nodes per step and frame,
 * steps per pass, dynamic shared memory bytes, resident frame slots, warps per CTA, check nodes per warp */
int nbgpu_geometry(const nbgpu_ctx *ctx, int *geo);
/* selection rows that needed the exact (slow) scan since creation; diagnostic */
long nbgpu_slow_selects(nbgpu_ctx *ctx);

/* Frame source on the DEVICE (SURVEY.md 8f.1): frames [frame0, frame0 + B) of the reference's Monte-Carlo stream are
 * produced where the decoder reads them, so a simulation never moves a frame across PCIe.  Replaces, per frame,
 * RandomBinaryGenerator (tools.c:124-136), Encoding (tools.c:232-270; the elimination of tools.c:151-218 is done once
 * on the host by nbgpu_code_prepare_encoder) and the noise of ModelChannel_AWGN_BPSK (channel.c:51-62).
 * `origin` is the drand48 state before frame 0 (nbgpu_rng_reference_default for the reference's stream).
 * The samples are bit-identical to nbgpu_random_codeword + nbgpu_awgn_bpsk_noise: the few samples whose f32 rounding
 * could depend on the last bits of the device's log/cos are detected and recomputed by the host's libm
 * (nbgpu_source_fixups tells how many in the last call).  Afterwards the batch is resident as after
 * nbgpu_upload_noisy: call nbgpu_run, then nbgpu_source_results (or nbgpu_download for the decisions).
 * `code` must be the code the context was created for, compared by content (sizes, graph, coefficients, BINGF, MULGF,
 * DIVGF), so another handle loaded from the same file qualifies; any other code is NBGPU_EINVAL ("the code is not the one
 * the decoder was created for") and leaves the context as it was.  The same holds for the _apsk64 and _mapped forms. */
int  nbgpu_source_frames(nbgpu_ctx *ctx, nbgpu_code *code, const nbgpu_rng *origin, uint64_t frame0, int B, float EbN);
/* The same for a GF(64) code sent as 64-APSK symbols (ModelChannel_AWGN_64, channel.c:234-263): frame f owns the draws
 * [f*D, (f+1)*D) with D = 6K + 4N, and its samples are bit-identical to nbgpu_random_codeword + nbgpu_awgn_apsk64_noise
 * (sigma = nbgpu_sigma_apsk64(EbN)).  Afterwards the batch is resident as after nbgpu_upload_apsk64; nbgpu_run,
 * nbgpu_source_results, nbgpu_download and the soft output work on it as on a BPSK batch.  One context may alternate BPSK
 * and 64-APSK batches.  NBGPU_EINVAL: q != 64 (context unchanged); B outside 1..max_batch or B*N*2 >= 2^31 (as for
 * nbgpu_source_frames, the soft output of the previous batch is dropped; the context stays usable). */
int  nbgpu_source_frames_apsk64(nbgpu_ctx *ctx, nbgpu_code *code, const nbgpu_rng *origin, uint64_t frame0, int B, float EbN);
/* The same for a code over any field sent on the bound table (nbgpu_set_constellation): D = K log2(q) + 4N draws per frame,
 * samples bit-identical to nbgpu_random_codeword + nbgpu_awgn_mapped_noise with that table; the batch is resident as after
 * nbgpu_upload_mapped.  NBGPU_ESTATE with no bound table (context unchanged); the other refusals as above. */
int  nbgpu_source_frames_mapped(nbgpu_ctx *ctx, nbgpu_code *code, const nbgpu_rng *origin, uint64_t frame0, int B, float EbN);
/* The same for the faded mapped channel (fading = NBGPU_FADING_SYMBOL or NBGPU_FADING_COMPONENT) on the bound table:
 * D = K log2(q) + S*N draws per frame, rx bit-identical to nbgpu_random_codeword + nbgpu_awgn_faded_noise (a symbol whose
 * rho or y could round differently on the device is recomputed whole by the host); the batch is resident as after
 * nbgpu_upload_faded.  NBGPU_ESTATE with no bound table, NBGPU_EINVAL for a bad fading value (context unchanged); B*N*4
 * must stay below 2^31; the other refusals as above. */
int  nbgpu_source_frames_faded(nbgpu_ctx *ctx, nbgpu_code *code, const nbgpu_rng *origin, uint64_t frame0, int B, float EbN,
                               int fading);
/* The same for the split channel on the split table (nbgpu_set_split_constellation): D = K log2(q) + 4*N*P draws per frame,
 * samples bit-identical to nbgpu_random_codeword + nbgpu_awgn_split_noise with that table; the batch is resident as after
 * nbgpu_upload_split.  NBGPU_ESTATE with no split table bound (context unchanged); B*N*2P must stay below 2^31; the other
 * refusals as above. */
int  nbgpu_source_frames_split(nbgpu_ctx *ctx, nbgpu_code *code, const nbgpu_rng *origin, uint64_t frame0, int B, float EbN);
/* what the source produced (either may be NULL): codeword symbols [B][N] (CodeWord of tools.c:258), noisy [B][N][logq]
 * after nbgpu_source_frames, noisy [B][N][2] (I, Q) after nbgpu_source_frames_apsk64 / _mapped, rx [B][N][4] after
 * nbgpu_source_frames_faded, noisy [B][N][P][2] after nbgpu_source_frames_split; NBGPU_ESTATE once an upload or a decode
 * call has replaced the batch (a batch dropped by nbgpu_set_constellation or nbgpu_set_split_constellation stays readable) */
int  nbgpu_source_download(nbgpu_ctx *ctx, int *codeword, float *noisy);
/* after nbgpu_run: information-bit errors of each frame (NB_LDPC.c:479-485), syndrome value, iteration count;
 * feed them to the frame-order statistics rule (NB_LDPC.c:474-507).  12 bytes per frame cross PCIe. */
int  nbgpu_source_results(nbgpu_ctx *ctx, int *bit_errors, int *synd, int *iters);
long nbgpu_source_fixups(const nbgpu_ctx *ctx);
/* test hook: relative width of the "ambiguous rounding" test (default 2^-46, i.e. 64 ulp of a double) */
int  nbgpu_source_set_margin(nbgpu_ctx *ctx, double margin);

/* Parity/debug: APP[N][q] and CtoV[E][q] (dense, as decoder_t.APP / decoder_t.CtoV) of one frame of
 * the last batch.  Only frames whose working set is still resident can be read (NBGPU_ESTATE). */
int nbgpu_get_state(nbgpu_ctx *ctx, int frame, float *APP, float *CtoV);

/* ---- Soft output of every frame of a batch ----
 * Computed by the decode kernel from the final APP[N][q] of each frame: the APP at the early stop (NB_LDPC.c:470) for a
 * frame that stopped early, else the APP after the last pass -- exactly the array nbgpu_get_state returns.  Isolated
 * variables report their intake row.  A context produces at most one kind per launch.
 *
 * NBGPU_SOFT_LIST, 1 <= k <= min(q, 32): per variable the k most likely symbols, by the truncation rule NB_LDPC.c:354-374
 *   with n_m = k applied to the APP row: ascending, ties -> lowest symbol; values >= 1e5 are never selected and such a
 *   slot keeps (1e5, symbol 0); then llr[i] -= llr[0], llr[0] = 0.  llr[B][N][k] f32 and sym[B][N][k] symbols in GF
 *   order (0 = zero, s = alpha^(s-1)), as nbgpu_select_nm would return for the row; sym[..][0] equals the decision.
 * NBGPU_SOFT_BITS, k = 0: per variable log2(q) bit reliabilities in the distance convention,
 *   b[l] = min{APP[s] : bingf[s][l] = 1} - min{APP[s] : bingf[s][l] = 0}, one f32 subtraction (round to nearest) of two
 *   exact minima; b[l] > 0 favours bit 0.  llr[B][N][log2 q] f32, the layout of the `noisy` input.
 * NBGPU_SOFT_NONE, k = 0: no soft output (the default). */
#define NBGPU_SOFT_NONE 0
#define NBGPU_SOFT_LIST 1
#define NBGPU_SOFT_BITS 2
/* Arms every later decode launch of ctx (nbgpu_run, nbgpu_decode_noisy / _llr / _apsk64 / _mapped / _faded / _split including
 * their streamed path, nbgpu_source_frames / _apsk64 / _mapped / _faded / _split + nbgpu_run) and allocates max_batch frames of output on the device: NBGPU_ENOMEM (with a message)
 * if that does not fit, after which ctx stays usable with soft output off.  A bad kind or k is NBGPU_EINVAL and leaves
 * the context as it was.  Invalidates the soft output of the last batch. */
int nbgpu_set_soft_output(nbgpu_ctx *ctx, int kind, int k);
/* The soft output of the B frames of the last decode launch: llr/sym [B][N][k] (LIST), llr [B][N][log2 q] (BITS).
 * NBGPU_EINVAL before any decode launch; NBGPU_ESTATE when the last launch did not produce this kind, or when the
 * soft output was invalidated since (re-armed, or another batch uploaded / generated).  Unit-boundary calls
 * (nbgpu_check_node, ...) leave it alone. */
int nbgpu_download_soft_list(nbgpu_ctx *ctx, float *llr, int *sym);
int nbgpu_download_soft_bits(nbgpu_ctx *ctx, float *llr);

/* Boundary 1 (unit parity): one check node for B independent input sets.
 * replaces CheckPassLogEMS (bubble_decoder.h:17) / syndrome_ems (syndrome_decoder.h:14):
 * vllr/vgf[B][dc][n_m] = decoder->M_VtoC_LLR/GF before the call, cllr/cgf[B][dc][q] =
 * decoder->M_CtoV_LLR/GF after it. */
int nbgpu_check_node(nbgpu_ctx *ctx, int node, const float *vllr, const int *vgf,
                     float *cllr, int *cgf, int B);
/* The dense check node of the context for check node `node` and B input sets: steps 2-7 of the sum-product node
 * (ecn_kind = 2) or steps 2-5 of the Min-Max node (ecn_kind = 4), mvc[B][dc][q] -> ctov[B][dc][q], both in symbol order,
 * through the decoder's own device functions.  NBGPU_EINVAL on a context of another ecn_kind; nbgpu_check_node is
 * NBGPU_EINVAL on an ecn_kind = 2 or 4 context. */
int nbgpu_check_node_dense(nbgpu_ctx *ctx, int node, const float *mvc, float *ctov, int B);
/* ElementaryStep (bubble_decoder.h:28) for B independent pairs of n_m-lists (symbols, -1 = absent) */
int nbgpu_elementary_step(nbgpu_ctx *ctx, const float *in1, const float *in2, const int *idx1,
                          const int *idx2, float *out, int *idxout, int B);
/* the inline truncation NB_LDPC.c:354-374: rows[B][q] -> llr/gf[B][n_m] */
int nbgpu_select_nm(nbgpu_ctx *ctx, const float *rows, float *llr, int *gf, int B);
/* Decision + Syndrom (tools.c:312, 284) on dense APP[B][N][q] */
int nbgpu_decision_syndrome(nbgpu_ctx *ctx, const float *app, int *decide, int *synd, int B);

/* Monte-Carlo statistics of NB_LDPC.c:474-507 for frames decoded in frame order.
 * codeword_bits[B][N][logq]; stats[6] accumulates: frames, erroneous frames, undetected, bit errors,
 * sum_it, stop flag (1 once the 40th erroneous frame was reached; later frames are ignored). */
int nbgpu_accumulate_stats(const nbgpu_code *c, const int *codeword_bits, const int *decide,
                           const int *synd, const int *iters, int B, long *stats);
/* the same rule fed with the per-frame error counts of nbgpu_source_results */
int nbgpu_accumulate_results(const int *bit_errors, const int *synd, const int *iters, int B, long *stats);

/* build information */
const char *nbgpu_version(void);
int nbgpu_device_count(void);

#ifdef __cplusplus
}
#endif
#endif /* NBLDPC_B200_H */
