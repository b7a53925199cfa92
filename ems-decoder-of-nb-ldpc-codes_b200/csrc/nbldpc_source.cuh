/* nbldpc_source.cuh -- the reference's Monte-Carlo frame source on the device (SURVEY.md 8f.1).
 *
 * Replaces, for a whole batch of frames and without touching the host,
 *   RandomBinaryGenerator   tools.c:124-136   information bits  floor((float)drand48() * 1.9999)
 *   Encoding                tools.c:232-270   back-substitution on the triangular matrix of GaussianElimination
 *                                             (tools.c:151-218; done once on the host, nbldpc_host.c)
 *   ModelChannel_AWGN_BPSK  channel.c:51-62   y = BPSK(b) + sigma*sqrt(-2 ln u)*cos(2 pi v), f64 -> f32
 *   ModelChannel_AWGN_64    channel.c:234-263 y[c] = mod[som][c] + sigma*sqrt(-2 ln u)*cos(2 pi v), c = I, Q, on the 64-APSK table
 *                                             or, for the mapped channel of any field, on the context's bound table
 *   the error count         NB_LDPC.c:479-485 information-bit errors of the decided word
 *
 * Frame f of the stream owns the drand48 draws [f*D, (f+1)*D), so every thread reaches its own draws by LCG jump-ahead (48
 * precomputed powers of the affine map in constant memory).  D is a property of the batch: one context may alternate the
 * channels.  The BPSK, mapped and split channels send a symbol as P points of DIMS coordinates and take two draws per
 * coordinate: D = K log2 q + 2*N*P*DIMS, with (P, DIMS) = (log2 q, 1) for BPSK, (1, 2) for a mapped channel and (P, 2) for
 * the split one (source_awgn_kernel).  A faded channel takes K log2 q + 5N or + 6N (one or two amplitude draws more per
 * symbol; source_faded_kernel).
 *
 * Exactness.  Everything except log() and cos() is IEEE arithmetic that the device reproduces bit for bit (explicit
 * __dmul_rn/__dadd_rn so that nothing is contracted into an FMA).  The device's log/cos may differ from glibc's by a
 * few ulp of a double, which changes the f32 sample only when the f64 value sits within that distance of an f32
 * rounding boundary.  Such samples (about one in 10^6) are FLAGGED by a margin test that is ~8x wider than the
 * documented error bounds, and recomputed by the host with glibc (nbgpu_mapped_sample / nbgpu_faded_sample,
 * nbldpc_host.c) before the decoder reads them.  tests/test_gpu_source.py, test_gpu_source_apsk64.py, test_gpu_mapped.py,
 * test_gpu_split.py and test_gpu_faded.py check the stream against the host source sample by sample.
 *
 * GF arithmetic of the encoder runs on binary images (addition = XOR): mulimg[h][x] = img(h * sym(x)),
 * divimg[p][x] = img(sym(x) / p), both built on the host from the code's tables.
 */
#pragma once
#include <stdint.h>

#define SRC_MASK ((1ULL << 48) - 1)
#define SRC_A 0x5DEECE66DULL
#define SRC_C 0xBULL

__constant__ uint64_t c_src_mul[48];     /* a^(2^j) mod 2^48 */
__constant__ uint64_t c_src_add[48];     /* increment of the 2^j-fold map */

struct SrcArgs {
    int N, M, K, q, logq, B;
    uint64_t x0;                 /* generator state before the first draw of this batch's first frame */
    uint64_t D;                  /* draws per frame */
    int nlevels;
    const int *level_ptr;        /* [nlevels+1] into row_order: rows of one level only need rows of earlier levels */
    const int *row_order;        /* [M] */
    const int *ut_ptr, *ut_col;  /* sparse rows of the triangular matrix (strictly right of the diagonal) */
    const uint8_t *ut_val, *piv; /* coefficients (symbols), diagonal */
    const int *perm;             /* [N] column permutation of the elimination */
    const uint8_t *mulimg, *divimg;
    const uint8_t *img;          /* [q] binary image of a symbol */
    uint8_t *cw;                 /* [B][N] codeword, binary images */
    float *noisy;                /* [B][N*logq] */
    float sigma;
    double margin;
    unsigned *flag_count, *flags;
    unsigned flag_cap;
    const int *decide;           /* [B][N] */
    int *bit_errors;             /* [B] */
    const float *mod;            /* [q][2] constellation of a mapped batch by binary image (the decoder's intake table) */
    uint8_t *flag_img;           /* [flag_cap] sub-image of the point of each flagged sample (the bit for BPSK; the symbol's
                                    image for the mapped and faded channels, q <= 256) */
    int points;                  /* source_awgn_kernel: points per symbol, P */
    int Nt;                      /* transmitted symbols per frame: N, or N - p under a puncturing pattern */
    const int *tvar;             /* [Nt] variable of each transmitted symbol, nullptr = every symbol (Nt = N) */
};

__device__ __forceinline__ uint64_t src_skip(uint64_t x, uint64_t n)
{
    for (int j = 0; n; ++j, n >>= 1)
        if (n & 1) x = (x * c_src_mul[j] + c_src_add[j]) & SRC_MASK;
    return x;
}
/* (float)drand48(), tools.c:73 */
__device__ __forceinline__ float src_draw(uint64_t &x)
{
    x = (x * SRC_A + SRC_C) & SRC_MASK;
    return __double2float_rn(__dmul_rn((double)(long long)x, 1.0 / 281474976710656.0));
}

/* One CTA per frame: information symbols, then the back-substitution level by level (a warp per row). */
__global__ void __launch_bounds__(256) source_encode_kernel(SrcArgs a)
{
    extern __shared__ uint8_t ns[];                       /* [N] symbols in elimination order, binary images */
    const int f = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const uint64_t xf = src_skip(a.x0, (uint64_t)f * a.D);
    for (int k = tid; k < a.K; k += blockDim.x) {
        uint64_t x = src_skip(xf, (uint64_t)k * a.logq);
        int bits = 0;
        for (int l = 0; l < a.logq; l++) {
            const float u = src_draw(x);
            bits |= (__dmul_rn((double)u, 1.9999) >= 1.0 ? 1 : 0) << l;       /* floor(u*1.9999), tools.c:132 */
        }
        ns[a.M + k] = (uint8_t)bits;                                          /* Bin2GF then BINGF: the image is the bits */
    }
    __syncthreads();
    for (int lv = 0; lv < a.nlevels; lv++) {
        for (int r = a.level_ptr[lv] + warp; r < a.level_ptr[lv + 1]; r += nwarps) {
            const int m = a.row_order[r];
            unsigned acc = 0;
            for (int k = a.ut_ptr[m] + lane; k < a.ut_ptr[m + 1]; k += 32)
                acc ^= a.mulimg[(int)a.ut_val[k] * a.q + ns[a.ut_col[k]]];     /* tools.c:249-250 */
            acc = __reduce_xor_sync(0xffffffffu, acc);
            if (lane == 0) ns[m] = a.divimg[(int)a.piv[m] * a.q + acc];         /* tools.c:253 */
        }
        __syncthreads();
    }
    uint8_t *cw = a.cw + (size_t)f * a.N;
    for (int n = tid; n < a.N; n += blockDim.x) cw[a.perm[n]] = ns[n];          /* tools.c:257-258 */
}

/* Box-Muller noise of one sample, sigma*sqrt(-2 ln u)*cos(2 pi v) (channel.c:59, channel.c:234-263) */
__device__ __forceinline__ double src_noise_term(double sigma, float u, float v)
{
    const double r = sqrt(-2.0 * log((double)u));
    const double cs = cos(__dmul_rn(2.0 * 3.1415926536, (double)v));             /* PI of channel.c:18 */
    return __dmul_rn(__dmul_rn(sigma, r), cs);
}
/* the f32 rounding of y = point + t could depend on the last bits of the device's log/cos (also true for inf/NaN) */
__device__ __forceinline__ bool src_ambiguous(double y, double t, double margin)
{
    const double d = margin * (fabs(t) + fabs(y));
    return !(__double2float_rn(y + d) == __double2float_rn(y - d));
}

/* BPSK, mapped and split channels: one thread per codeword symbol, sent as P = a.points points of m = log2 q / P bits each;
 * point j is the sub-image (sym >> j*m) & (2^m - 1).  DIMS = 1: BPSK (P = log2 q), the point is 1 - 2*bit and no table is
 * read.  DIMS = 2: the mapped channel (P = 1) or the split one (P >= 2), the point is (mod[sub][0], mod[sub][1]).  Every
 * coordinate takes two draws, in stream order from K log2 q + 2*P*DIMS*n on, and is written as noisy[B][N][P][DIMS].  A flag
 * records the sample index and the point's sub-image, so the host recomputes any flagged sample as the same expression. */
template <int DIMS>
__global__ void __launch_bounds__(256) source_awgn_kernel(SrcArgs a)
{
    const long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= (long long)a.B * a.Nt) return;
    const int f = (int)(id / a.Nt), t = (int)(id % a.Nt), P = a.points, m = a.logq / P, fps = P * DIMS;
    uint64_t x = src_skip(a.x0, (uint64_t)f * a.D + (uint64_t)a.K * a.logq + (uint64_t)t * 2 * fps);
    const int sym = a.cw[(size_t)f * a.N + (a.tvar ? a.tvar[t] : t)];
    const double sigma = (double)a.sigma;
    for (int k = 0; k < fps; k++) {                                             /* coordinate c of point j, in stream order */
        const int j = k / DIMS, c = k % DIMS, sub = (sym >> (j * m)) & ((1 << m) - 1);
        const float u = src_draw(x);
        const float v = src_draw(x);
        const double t = src_noise_term(sigma, u, v);
        const double y = __dadd_rn(DIMS == 1 ? (double)(1 - 2 * sub) : (double)a.mod[2 * sub + c], t);   /* channel.c:59 / :234-263 */
        const unsigned s = (unsigned)id * fps + k;                               /* sample index: B*Nt*fps < 2^31 */
        if (src_ambiguous(y, t, a.margin)) {
            const unsigned slot = atomicAdd(a.flag_count, 1u);
            if (slot < a.flag_cap) { a.flags[slot] = s; a.flag_img[slot] = (uint8_t)sub; }
        }
        a.noisy[s] = __double2float_rn(y);
    }
}

/* The faded mapped channel (include/nbldpc_b200.h): one thread per codeword symbol, FADING = NBGPU_FADING_SYMBOL / _COMPONENT,
 * 5 or 6 draws per symbol (u_I, v_I, u_Q, v_Q, w_I, w_Q), rho = (float)sqrt(-log(w)), y = rho * point + noise with the product
 * exact in f64, written as rx[B][N][4] = (y_I, y_Q, rho_I, rho_Q) in one 16-byte store.  An ambiguous rho or y flags the whole
 * symbol (its y values used that rho): the flag holds the symbol's index, and the host recomputes all four values. */
template <int FADING>
__global__ void __launch_bounds__(256) source_faded_kernel(SrcArgs a)
{
    constexpr int S = FADING == 1 ? 5 : 6;                                      /* draws per symbol */
    const long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= (long long)a.B * a.Nt) return;
    const int f = (int)(id / a.Nt), t = (int)(id % a.Nt);
    uint64_t x = src_skip(a.x0, (uint64_t)f * a.D + (uint64_t)a.K * a.logq + (uint64_t)t * S);
    const int som = a.cw[(size_t)f * a.N + (a.tvar ? a.tvar[t] : t)];
    const double sigma = (double)a.sigma;
    float d[S];
#pragma unroll
    for (int i = 0; i < S; i++) d[i] = src_draw(x);
    float rho[2], y[2];
    bool amb = false;
#pragma unroll
    for (int c = 0; c < S - 4; c++) {
        const double r = sqrt(-log((double)d[4 + c]));
        const double e = a.margin * r;
        rho[c] = __double2float_rn(r);
        amb |= !(__double2float_rn(r + e) == __double2float_rn(r - e));
    }
    if constexpr (FADING == 1) rho[1] = rho[0];
#pragma unroll
    for (int c = 0; c < 2; c++) {
        const double t = src_noise_term(sigma, d[2 * c], d[2 * c + 1]);
        const double yd = __dadd_rn(__dmul_rn((double)rho[c], (double)a.mod[2 * som + c]), t);    /* the product is exact */
        y[c] = __double2float_rn(yd);
        amb |= src_ambiguous(yd, t, a.margin);
    }
    if (amb) {
        const unsigned slot = atomicAdd(a.flag_count, 1u);
        if (slot < a.flag_cap) { a.flags[slot] = (unsigned)id; a.flag_img[slot] = (uint8_t)som; }
    }
    *reinterpret_cast<float4 *>(a.noisy + (size_t)id * 4) = make_float4(y[0], y[1], rho[0], rho[1]);
}

__global__ void source_patch_kernel(float *noisy, const unsigned *idx, const float *val, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) noisy[idx[i]] = val[i];
}

/* One CTA per frame: information-bit errors of the decided word (NB_LDPC.c:479-485: the first K symbols). */
__global__ void __launch_bounds__(256) source_errors_kernel(SrcArgs a)
{
    __shared__ int part[8];
    const int f = blockIdx.x, tid = threadIdx.x;
    const int *dec = a.decide + (size_t)f * a.N;
    const uint8_t *cw = a.cw + (size_t)f * a.N;
    int e = 0;
    for (int k = tid; k < a.K; k += blockDim.x) e += __popc((unsigned)a.img[dec[k]] ^ (unsigned)cw[k]);
    e = __reduce_add_sync(0xffffffffu, e);
    if ((tid & 31) == 0) part[tid >> 5] = e;
    __syncthreads();
    if (tid == 0) {
        int s = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) s += part[w];
        a.bit_errors[f] = s;
    }
}
