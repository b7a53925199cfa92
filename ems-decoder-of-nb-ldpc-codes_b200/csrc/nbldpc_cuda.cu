/*
 * nbldpc_cuda.cu -- CUDA layer + C ABI of the B200 EMS NB-LDPC decoder (sm_100a).
 *
 * Persistent CTAs (two per SM) each decode one GROUP of F frames at a time, start to finish (all passes,
 * early termination included), pulling groups from an atomic work queue.  A decoding pass walks the
 * host-built step schedule (nbldpc_host.c): every step holds check nodes that share no variable, so
 * ONE CTA-wide barrier per step reproduces the reference's sequential layered update
 * (NB_LDPC.c:320-466) bit for bit.  Inside a step every WARP owns a tile of up to cpw check nodes and
 * runs them through three warp-private phases (no CTA barrier in between, lists in the warp's own
 * shared memory):
 *
 *   phase 1  warp per edge, NE edges interleaved:  Mvc = APP - CtoV (NB_LDPC.c:334); top-n_m selection +
 *            normalisation (:354-374), rotation by the edge coefficient (bubble_decoder.c:133)
 *   phase 2  THREAD per ElementaryStep, 4 task slots per check node: forward/backward chains with the
 *            merges folded into the rounds where their inputs are ready (bubble_decoder.c:157-227, 316-593)
 *   phase 3  warp per edge, NE edges interleaved:  Mvc again (parked in the APP row by phase 1), saturation + offset +
 *            expansion to the dense q-vector (bubble_decoder.c:231-281), CtoV store, APP = Mcv + Mvc
 *            (NB_LDPC.c:415-450), fused Decision (tools.c:312)
 * With ecn = 1 the tile is processed one check node at a time through the syndrome-based node (nbldpc_synd.cuh), with
 * ecn = 2 through the sum-product node (nbldpc_spa.cuh), with ecn = 4 through the Min-Max node (nbldpc_minmax.cuh).
 *
 * The kernel is bound by the shared/global wavefront pipe of the SM (l1tex data stage), not by HBM or issue slots
 * (ncu, profiles/): every design choice below trades wavefronts for ALU work -- conflict-free 128-bit row moves,
 * clean scratch rows instead of fill + scatter, selection winners kept in registers, exact low bits by shuffle.
 *
 * HBM layout per resident frame (slot): APP[N][q] f32 (row = 4q bytes, one coalesced warp access);
 * CtoV as one lossless record per edge {llr[n_m] f32, sat f32, stp i32, sym[n_m] u8} -- a dense CtoV
 * row is "stp explicit (symbol, LLR) pairs + one constant" (bubble_decoder.c:262-270); decisions u8.
 * The syndrome-based, sum-product and Min-Max nodes store CtoV as dense rows instead.
 */
#include "nbldpc_device.cuh"
#include "nbldpc_synd.cuh"
#include "nbldpc_spa.cuh"
#include "nbldpc_minmax.cuh"
#include "nbldpc_source.cuh"
#include "nbldpc_internal.h"
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <vector>

#define NT_MAX 384         /* threads per CTA (upper bound; the plan may use fewer warps) */
#define NT_SYND 256        /* syndrome, sum-product and Min-Max check nodes: at most 8 warps per CTA (shared memory allows 7 at 945 configurations,
                              6 for a dc = 16 GF(256) sum-product code), 128 registers */
#define CTAS_PER_SM 2      /* resident CTAs per SM the decode kernel is compiled for (register cap 65536 / (NT_MAX * CTAS_PER_SM)) */
#define NE 2               /* edges interleaved per warp in phases 1 and 3 */

#define UNIT_NT 256       /* block size of the small unit-boundary kernels */

/* what the intake reads per variable (KArgs::input_kind): BPSK samples [logq], a dense LLR row [q], mapped (I, Q) samples [2],
 * faded (I, Q, rho_I, rho_Q) [4] or split (I, Q) samples of P points [P][2]; the mapped, faded and split intakes read KArgs::mod */
enum InputKind { INPUT_BPSK = 0, INPUT_LLR = 1, INPUT_MAPPED = 2, INPUT_FADED = 3, INPUT_SPLIT = 4 };

struct KArgs {
    int N, M, E, q, logq, dc_max, dc_min;
    int n_m, nb_oper, passes, early_stop, nb_iter_max;
    float offset;
    int F, nw, cpw, cap, nsteps, L;     /* frames per group, warps per CTA, check nodes per warp, items per step, steps, lists per node */
    int B, input_kind, frame0;          /* frames of this launch; InputKind; batch index of its first frame */
    double den;                         /* 2.0 * (double)(float)(sigma*sigma), channel.c:73 */
    const int *step_ptr, *isolated;
    int n_isolated;
    const uint32_t *cninfo;             /* [M] schedule order: first edge | degree << 24            */
    const uint32_t *einfo;              /* [E] variable | coefficient << 20 | last-visit flag << 28 */
    const int *row_ptr, *col;
    const uint8_t *hval, *rotin, *rotout, *img, *inv;
    const float *mod;                   /* [q][2] constellation of the launch's batch by binary image, INPUT_MAPPED and INPUT_FADED; [M][2] by sub-image, INPUT_SPLIT (set per launch) */
    int gf_closed;
    const float *in;
    float *app; uint8_t *ctov; uint8_t *dec;
    int rec_stride;
    int *out_decide, *out_synd, *out_iters, *frame_slot, *slot_frame;
    unsigned *queue, *slow_counter;
    const unsigned *ready;   /* streamed input (decode_host): frames copied to the device so far; nullptr = the whole batch is resident */
    unsigned *fault;         /* set when a CTA gave up waiting for its frames */
    /* shared memory map (bytes): tables | misc | per-warp scratch areas | per-warp lists */
    int off_tab, off_misc, off_wa, wa_bytes, off_wb, wb_bytes;
    int wa_mask, wa_meta, wa_einfo, wa_len;   /* offsets inside a warp's small private area: ES mask | tile meta | tile edge words | list lengths */
    int wb_scr1, wb_scr3, wb_U, wb_R;   /* offsets inside a warp's list area: phase-1 scratch (clean rows[NE] | key queues[NE] |
                                           36 unused words[NE]), phase-3 scratch (clean rows[NE]), input lists U[cpw][dc_max], other lists
                                           R[cpw][L - dc_max] directly behind them (one array of lists).
                                           Bubble path: the phase-1 scratch aliases R (unused until phase 2) and the phase-3
                                           scratch aliases U (dead after phase 2).                                         */
    int lstride;                        /* bytes per list: n_m f32 | n_m u8 | pad; an ODD number of words, so that the lists of a
                                           tile start in different banks (the ElementarySteps read one list per lane)      */
    int smem_bytes;
    /* syndrome-based check node (ecn = 1): dense CtoV rows, configuration table, per-warp sort buffers */
    int ecn, S, Spad, n_cv;
    const uint8_t *cfg;                 /* [S][dc_max] u8 */
    float *ctov_dense;                  /* [slots][E][q] f32 */
    int off_cfg, sw_key, sw_pay, sw_gf, sw_hist, sw_cand, sw_M, sw_rows, sw_perm;   /* sw_*: offsets inside a warp's list area */
    /* soft output (nbgpu_set_soft_output), read by decode_kernel<..., SOFT = true> only.  Kept at the end of the struct so
     * that the fields above keep their parameter offsets in every kernel. */
    int soft_kind, soft_k;              /* NBGPU_SOFT_LIST with k symbols per variable, or NBGPU_SOFT_BITS (k = 0)  */
    int split_p;                        /* INPUT_SPLIT: points per symbol (set per launch).  In the alignment gap in front of
                                           soft_llr: KArgs keeps its size, so the parameters behind it keep their offsets too */
    float *soft_llr;                    /* [B][N][k] (LIST) or [B][N][logq] (BITS)                                  */
    uint8_t *soft_sym;                  /* [B][N][k] symbols (LIST)                                                 */
    /* puncturing (nbgpu_set_puncturing), read by the frame initialisation and channel_kernel: pmap[n] = compact index of
     * variable n in the input frames [B][nt][..], -1 = punctured (intake row all 0.0f); nullptr with nt = N when no pattern
     * is bound.  Behind every other field, so that those keep their parameter offsets in every kernel. */
    const int *pmap;
    int nt;
};

/* Lists of a warp's tile in shared memory, by 32-bit shared-window address: one array of cpw * L lists, the input lists
 * U[c][t] first (index c * dcm + t), then the forward/backward/merge lists R[c][.].  One list = n_m f32 LLRs followed by
 * n_m u8 symbols (binary images); the lengths live in a byte array of their own. */
struct Lists {
    uint32_t base, lenb; int lstride, n_m, dcm, lr, r0;     /* lr = L - dcm lists per node in R, r0 = cpw * dcm */
    /* li < dc: input list of edge li; li >= dc: forward/backward/merge list number li - dc */
    __device__ __forceinline__ int idx(int c, int li, int dc) const { return li < dc ? c * dcm + li : r0 + c * lr + (li - dc); }
    __device__ __forceinline__ int in(int c, int t) const { return c * dcm + t; }
    __device__ __forceinline__ uint32_t addr(int i) const { return base + (uint32_t)(i * lstride); }
    __device__ __forceinline__ uint32_t sym(uint32_t list) const { return list + 4 * n_m; }
    __device__ __forceinline__ uint32_t len(int i) const { return lenb + (uint32_t)i; }
};
/* list ids of one node with degree dc: U[t] = t; F after s steps = dc+s-1 (s>=1); B after s steps =
 * dc+(dc-2)+s-1; merge k = dc+2(dc-2)+k  (bubble_decoder.c:166-227: MatriceInter rows) */
__device__ __forceinline__ int id_F(int dc, int s) { return s == 0 ? 0 : dc + s - 1; }
__device__ __forceinline__ int id_B(int dc, int s) { return s == 0 ? dc - 1 : dc + (dc - 2) + s - 1; }
__device__ __forceinline__ int id_M(int dc, int k) { return dc + 2 * (dc - 2) + k; }
/* output list of edge t: t=0 -> B after dc-2 steps, t=dc-1 -> F after dc-2 steps, else merge t-1 */
__device__ __forceinline__ int id_out(int dc, int t)
{
    if (t == 0) return id_B(dc, dc - 2);
    if (t == dc - 1) return id_F(dc, dc - 2);
    return id_M(dc, t - 1);
}

/* tile description in shared memory, per check node: {first edge | degree << 24 (0 = skip), byte offset of the frame's APP block,
 * byte offset of the node's first CtoV record (or dense row), offset of the frame's decisions}, all relative to the CTA's slot block
 * and computed once per tile by one lane per node (the phases add a variable / edge offset to them: no 64-bit multiplies per edge) */
struct TileMeta {
    int4 *p;
    __device__ __forceinline__ int4 operator[](int c) const { return p[c]; }
    __device__ __forceinline__ void set(int c, int e0, int dc, uint32_t app_off, uint32_t rec_off, uint32_t dec_off) const
    {
        p[c] = make_int4(e0 | (dc << 24), (int)app_off, (int)rec_off, (int)dec_off);
    }
    __device__ __forceinline__ static int e0(const int4 &m) { return m.x & 0xffffff; }
    __device__ __forceinline__ static int dc(const int4 &m) { return (int)((unsigned)m.x >> 24); }
};

/* a warp's private shared memory.  The scratch areas are addressed from TWO per-warp bases (s1: phase 1, s3: phase 3) with
 * compile-time offsets, so that an access is "register + immediate"; eight separately derived addresses were too many to
 * keep in registers and ptxas rebuilt them from the kernel parameters at every use (~100 instructions per check node). */
template <int Q, int ECN = 0> struct WarpMem {
    static constexpr int ROWS = ECN == 0 ? NE * Q : 0;     /* floats of clean rows in front of the queues (bubble path only) */
    uint32_t s1, s3;         /* shared-window addresses of the phase-1 scratch (clean rows | queues) and the phase-3 rows */
    unsigned char *p1, *p3;  /* the same as generic pointers (cold paths)                                    */
    uint32_t mask;           /* q = 256: ElementaryStep "seen" bits, [8][32] lane-strided (shared address)  */
    TileMeta meta;           /* [cpw] {first edge | degree << 24 (0 = skip), frame}                         */
    uint32_t *ew;            /* [cpw][dc_max] einfo words of the tile's edges (one coalesced load per tile) */
    Lists ls;
    /* phase 1, per in-flight edge: clean row for the record expansion | selection queue (sorted keys) */
    __device__ __forceinline__ uint32_t rowa(int e) const { return s1 + (uint32_t)(e * Q * 4); }
    __device__ __forceinline__ uint32_t scra(int e) const { return s1 + (uint32_t)((ROWS + e * QTraits<Q>::SCR_WORDS) * 4); }
    /* phase 3, per in-flight edge: clean row */
    __device__ __forceinline__ uint32_t row3a(int e) const { return s3 + (uint32_t)(e * Q * 4); }
    __device__ __forceinline__ float *row(int e) const { return reinterpret_cast<float *>(p1) + e * Q; }
    __device__ __forceinline__ float *row3(int e) const { return reinterpret_cast<float *>(p3) + e * Q; }
    __device__ __forceinline__ uint32_t *scr(int e) const { return reinterpret_cast<uint32_t *>(p1) + ROWS + e * QTraits<Q>::SCR_WORDS; }
    __device__ __forceinline__ WarpMem(unsigned char *smem, const KArgs &a, int warp)
    {
        unsigned char *wa = smem + a.off_wa + warp * a.wa_bytes;
        unsigned char *wb = smem + a.off_wb + warp * a.wb_bytes;
        p1 = wb + a.wb_scr1; p3 = wb + a.wb_scr3;
        s1 = smem_u32(p1); s3 = smem_u32(p3);
        asm volatile("" : "+r"(s1), "+r"(s3));              /* opaque: kept in registers, not re-derived from the parameters */
        mask = smem_u32(wa + a.wa_mask);
        meta.p = reinterpret_cast<int4 *>(wa + a.wa_meta);
        ew = reinterpret_cast<uint32_t *>(wa + a.wa_einfo);
        ls.base = smem_u32(wb + a.wb_U); ls.lenb = smem_u32(wa + a.wa_len);
        ls.lstride = a.lstride; ls.n_m = a.n_m; ls.dcm = a.dc_max; ls.lr = a.L - a.dc_max; ls.r0 = a.cpw * a.dc_max;
    }
};

/* ---- phase 2: all elementary steps of the cnt check nodes of a warp's tile ----
 * Round r = 1..dcmax-2.  Slot 0/1 of a node: forward/backward chain step r (bubble_decoder.c:166-200).
 * Slots 2/3: the merges ES(F_k, B_{dc-3-k}) (:217-227) whose later input appears in round r-1:
 * k = r-1 (if k >= dc-3-k) and k = dc-2-r (if dc-3-k = r-1 > k). */
template <int Q>
__device__ __forceinline__ void tile_elementary_steps(const Lists &ls, const TileMeta &meta, int cnt, int dcmax, uint32_t mask,
                                                      int lane, int nb_oper)
{
    for (int r = 1; r <= dcmax - 2; r++) {
        for (int cb = 0; cb < cnt; cb += 8) {
            const int c = cb + (lane >> 2), slot = lane & 3;
            if (c < cnt) {
                const int dc = TileMeta::dc(meta[c]);
                int a = 0, b = 0, o = 0;
                bool valid = false;
                if (slot == 0) { valid = r <= dc - 2; a = id_F(dc, r - 1); b = r; o = id_F(dc, r); }
                else if (slot == 1) { valid = r <= dc - 2; a = id_B(dc, r - 1); b = dc - 1 - r; o = id_B(dc, r); }
                else {
                    const int k = (slot == 2) ? r - 1 : dc - 2 - r;
                    valid = (slot == 2) ? (k <= dc - 3 && 2 * k >= dc - 3) : (k >= 0 && k <= dc - 3 && r - 1 > k);
                    a = id_F(dc, k); b = id_B(dc, dc - 3 - k); o = id_M(dc, k);
                }
                if (valid) {
                    const int ia = ls.idx(c, a, dc), ib = ls.idx(c, b, dc), io = ls.idx(c, o, dc);
                    const uint32_t la = ls.addr(ia), lb = ls.addr(ib), lo = ls.addr(io);
                    const int s = es_serial<Q>(la, ls.sym(la), (int)lds_u8(ls.len(ia)), lb, ls.sym(lb), (int)lds_u8(ls.len(ib)),
                                               lo, ls.sym(lo), mask + 4 * lane, ls.n_m, nb_oper);
                    sts_u8(ls.len(io), (uint32_t)s);
                }
            }
            __syncwarp();
        }
    }
}

/* phase 3 core: from the check node's output list of one edge (binary-image symbols) build the
 * record entry of this lane and the saturation constant (bubble_decoder.c:231-264). */
template <int Q, bool CLOSED>
__device__ __forceinline__ RecView finish_list(const Lists &ls, int li, int h, const GFTab &gf, float offset, int lane)
{
    RecView r;
    const uint32_t list = ls.addr(li);
    const int len = (int)lds_u8(ls.len(li));
    r.stp = len;                                                     /* first absent entry, :233-243 */
    r.llr = NB_SENT; r.sym = 0;
    if (lane < len) {
        r.llr = lds_f32(list + 4 * lane);
        r.sym = gf_rot_out<Q, CLOSED>(gf, (int)lds_u8(ls.sym(list) + lane), h);       /* DIVGF by the coefficient, :249-254 */
    }
    const float last = lds_f32(list + 4 * max(len - 1, 0));          /* broadcast read */
    r.sat = __fadd_rn(len > 0 ? last : NB_SENT, offset);             /* :264 (len == 0 cannot occur) */
    return r;
}
/* LLR intake for one variable (channel.c:66-76), one warp.  The reference accumulates, for every symbol g and bit b in
 * ascending order, acc = (float)((double)acc + (double)((y_b - s_b(g))^2) / (2 sigma^2)).  The value after bits 0..k only
 * depends on the low k+1 bits of the symbol's binary image, so the sums are built as a binary tree over the image bits
 * (same additions in the same order, each computed once): lane L owns the images whose low five bits are L, the remaining
 * bits fan out in registers.  t[2b + bit] are the per-bit terms; row is a q-float scratch used to go from image order to
 * symbol order. */
template <int Q>
__device__ __forceinline__ void intake_variable(const float *noisy_n, double den, const uint8_t *img, int lane,
                                                double *t, float *row, float (&v)[QTraits<Q>::VPL])
{
    constexpr int VPL = QTraits<Q>::VPL;
    constexpr int LOGQ = QTraits<Q>::LOGQ;
    constexpr int LOW = LOGQ < 5 ? LOGQ : 5;
    if (lane < 2 * LOGQ) {
        const float y = noisy_n[lane >> 1];
        const float s = (lane & 1) ? -1.0f : 1.0f;                 /* BPSK(b) = 1 - 2b */
        const float d = __fsub_rn(y, s);
        const float sq = __fmul_rn(d, d);
        t[lane] = __ddiv_rn((double)sq, den);
    }
    __syncwarp();
    float acc = 0.0f;
#pragma unroll
    for (int b = 0; b < LOW; b++) acc = __double2float_rn(__dadd_rn((double)acc, t[2 * b + ((lane >> b) & 1)]));
    float w[VPL];
    w[0] = acc;
#pragma unroll
    for (int b = LOW; b < LOGQ; b++) {                             /* fan out: w[h] for h < 2^(b-LOW) -> 2^(b-LOW+1) values */
        const int half = 1 << (b - LOW);
        const double t0 = t[2 * b], t1 = t[2 * b + 1];
#pragma unroll
        for (int h = half - 1; h >= 0; h--) {
            const float base = w[h];
            w[h + half] = __double2float_rn(__dadd_rn((double)base, t1));
            w[h] = __double2float_rn(__dadd_rn((double)base, t0));
        }
    }
#pragma unroll
    for (int h = 0; h < VPL; h++) if (Q >= 32 || lane < Q) row[lane | (h << 5)] = w[h];     /* image index = lane | h << 5 */
    __syncwarp();
#pragma unroll
    for (int j = 0; j < VPL; j++) v[j] = (Q >= 32 || lane < Q) ? row[img[QTraits<Q>::sym(lane, j)]] : 0.0f;
    __syncwarp();
}

/* LLR intake for one variable sent as one point of a q-point constellation (the mapped channel; channel.c:268-291 for
 * 64-APSK): for every symbol k, TMP[k] = (float)( (double)((I - mI)^2) / (2 sigma^2) + (double)((Q - mQ)^2) / (2 sigma^2) )
 * with (mI, mQ) = mod[binary image of k]; differences and squares in f32, divisions and the sum in f64, as the reference
 * evaluates them (a reciprocal multiply would round differently).  GF(16): lanes >= 16 hold no symbol.
 * s = (I, Q, rho_I, rho_Q): the faded channel (INPUT_FADED) scales the point by its amplitudes, I - rho_I * mI in f32
 * (include/nbldpc_b200.h, NBGPU_FADING_SYMBOL); INPUT_MAPPED passes rho = 1, and a product with 1.0f is exact. */
template <int Q>
__device__ __forceinline__ void intake_mapped(const float4 s, double den, const float *mod, const uint8_t *img, int lane,
                                              float (&v)[QTraits<Q>::VPL])
{
#pragma unroll
    for (int j = 0; j < QTraits<Q>::VPL; j++) {
        if (Q < 32 && lane >= Q) { v[j] = 0.0f; continue; }
        const int som = img[QTraits<Q>::sym(lane, j)];
        const float d0 = __fsub_rn(s.x, __fmul_rn(s.z, mod[2 * som])), d1 = __fsub_rn(s.y, __fmul_rn(s.w, mod[2 * som + 1]));
        const double a = __ddiv_rn((double)__fmul_rn(d0, d0), den), b = __ddiv_rn((double)__fmul_rn(d1, d1), den);
        v[j] = __double2float_rn(__dadd_rn(a, b));
    }
}
/* LLR intake for one variable of the split channel (include/nbldpc_b200.h, nbgpu_split_qam): P points of M = 2^m points each,
 * pts = the variable's [P][2] samples.  Lane l < P*M computes t_{l/M}[l%M] = (double)(dI^2)/den + (double)(dQ^2)/den (f32
 * differences and squares, f64 divisions and sum) into t (32 doubles of warp scratch); then every symbol adds its P entries in
 * f64, j = 0 ... P-1, and rounds once.  2*P*M <= 64 f64 divisions per variable instead of the mapped intake's 2q. */
template <int Q>
__device__ __forceinline__ void intake_split(const float *pts, int P, double den, const float *mod, const uint8_t *img, int lane,
                                             double *t, float (&v)[QTraits<Q>::VPL])
{
    /* opaque: m and mask are computed here instead of being hoisted into the callers' loops (channel_kernel<16>: 47 -> 40 registers) */
    asm volatile("" : "+r"(P));
    const int m = QTraits<Q>::LOGQ / P, mask = (1 << m) - 1;
    if (lane < P << m) {
        const int x = lane & mask, j = lane >> m;
        const float dI = __fsub_rn(pts[2 * j], mod[2 * x]), dQ = __fsub_rn(pts[2 * j + 1], mod[2 * x + 1]);
        t[lane] = __dadd_rn(__ddiv_rn((double)__fmul_rn(dI, dI), den), __ddiv_rn((double)__fmul_rn(dQ, dQ), den));
    }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < QTraits<Q>::VPL; k++) {
        if (Q < 32 && lane >= Q) { v[k] = 0.0f; continue; }
        const int im = img[QTraits<Q>::sym(lane, k)];
        double s = t[im & mask];
        for (int j = 1; j < P; j++) s = __dadd_rn(s, t[(j << m) | ((im >> (j * m)) & mask)]);
        v[k] = __double2float_rn(s);
    }
    __syncwarp();
}
/* symbol r of a mapped (INPUT_MAPPED: [..][2], rho = 1) or faded (INPUT_FADED: [..][4], one 16-byte load) input as intake_mapped
 * reads it */
__device__ __forceinline__ float4 mapped_input(const float *in, int kind, size_t r)
{
    if (kind == INPUT_FADED) return *reinterpret_cast<const float4 *>(in + r * 4);
    return make_float4(in[r * 2], in[r * 2 + 1], 1.0f, 1.0f);
}

__device__ __forceinline__ void load_gf_tables(unsigned char *smem, const KArgs &a, GFTab &gf)
{
    uint8_t *tab = smem + a.off_tab;
    for (int i = threadIdx.x; i < a.q; i += blockDim.x) { tab[i] = a.img[i]; tab[256 + i] = a.inv[i]; }
    gf.img = tab; gf.inv = tab + 256; gf.rotin = a.rotin; gf.rotout = a.rotout;
}

__device__ __forceinline__ SyndMem make_synd_mem(unsigned char *smem, const KArgs &a, int warp)
{
    SyndMem sm;
    const uint32_t wb = smem_u32(smem + a.off_wb + warp * a.wb_bytes);
    sm.lists = wb + a.wb_U;
    sm.gkey = wb + a.sw_key; sm.hsat = sm.gkey; sm.rows = sm.gkey;          /* region B */
    sm.keya = wb + a.sw_rows; sm.skey = sm.keya;                            /* region A */
    sm.gpay = wb + a.sw_pay; sm.gfa = wb + a.sw_gf; sm.hist = wb + a.sw_hist; sm.spay = sm.gfa;
    sm.cand = wb + a.sw_cand;
    sm.M = wb + a.sw_M; sm.perm = wb + a.sw_perm;
    sm.cfg = smem_u32(smem + a.off_cfg); sm.cfgmask = sm.cfg + (uint32_t)(a.S * a.dc_max);
    sm.lstride = a.lstride; sm.n_m = a.n_m; sm.dc = a.dc_max; sm.S = a.S; sm.n_cv = a.n_cv;
    return sm;
}
/* the dense nodes' rows (sum-product, Min-Max) in a warp's list area: U rows at wb_U, the permutation row at sw_rows (plan_smem) */
__device__ __forceinline__ SpaMem make_spa_mem(unsigned char *smem, const KArgs &a, int warp)
{
    const uint32_t wb = smem_u32(smem + a.off_wb + warp * a.wb_bytes);
    SpaMem sp;
    sp.urow = wb + a.wb_U; sp.prow = wb + a.sw_rows;
    return sp;
}
__device__ __forceinline__ void load_cfg_table(unsigned char *smem, const KArgs &a)
{
    if (a.ecn != 1) return;
    uint8_t *dst = smem + a.off_cfg;
    for (int i = threadIdx.x; i < a.S * (a.dc_max + 1); i += blockDim.x) dst[i] = a.cfg[i];      /* table, then one membership byte per configuration */
}
/* dense output row of one edge from the syndrome check node: Mcv[s] = M[img(MULGF[s][h])] (syndrome_decoder.c:260-266
 * followed by the scatter NB_LDPC.c:415-421) */
template <int Q, bool CLOSED>
__device__ __forceinline__ void synd_dense_row(uint32_t out, const GFTab &gf, int h, int lane, float sat, float hi, float (&mcv)[QTraits<Q>::VPL])
{
#pragma unroll
    for (int j = 0; j < QTraits<Q>::VPL; j++) {
        const int s = QTraits<Q>::sym(lane, j);
        mcv[j] = (Q >= 32 || lane < Q) ? synd_saturate(lds_f32(out + 4 * gf_rot_in<Q, CLOSED>(gf, s, h)), sat, hi) : NB_SENT;
    }
}

/* L2 prefetch of everything phase 1 reads for ONE check node of the tile: its dc APP rows (edge words already in shared memory)
 * and its dc consecutive records.  Issued one node ahead: two or three instructions per node instead of address arithmetic per
 * edge pair. */
template <int Q>
__device__ __forceinline__ void prefetch_node(const char *app, const char *ctov, const uint32_t *ew, const int4 &m, int rec_stride, int lane)
{
    constexpr int LPR = (Q * 4) / 128;                     /* 128-byte lines per row: 8 (q = 256), 2 (q = 64) */
    const int dc = TileMeta::dc(m);
    for (int i = lane; i < dc * LPR; i += 32) {
        const uint32_t ei = ew[i / LPR];
        const char *p = app + (uint32_t)m.y + (ei & 0xfffffu) * (uint32_t)(Q * 4) + (uint32_t)(i % LPR) * 128u;
        asm volatile("prefetch.global.L2 [%0];" :: "l"(p));
    }
    if (lane * 128 < dc * rec_stride) {
        const char *p = ctov + (uint32_t)m.z + (uint32_t)lane * 128u;
        asm volatile("prefetch.global.L2 [%0];" :: "l"(p));
    }
}

/* ------------------------------------------------------------------------------------------------
 * GF(16): a row is 16 values, so one warp carries TWO edges of a check node side by side -- edge t in
 * lanes 0-15, edge t+1 in lanes 16-31, lane & 15 = symbol / list entry -- instead of two half-empty
 * instruction streams.  Same arithmetic, same order of operations as the generic phases below.
 * ---------------------------------------------------------------------------------------------- */
template <bool CLOSED>
__device__ __forceinline__ void gf16_phase1(const WarpMem<16> &wm, const GFTab &gf, int c, int e0, int dc, int dcm, float *app_f,
                                            const uint8_t *ctov_f, int n_m, int rs, int lane, unsigned *slow_counter)
{
    const Lists &ls = wm.ls;
    const int h = lane >> 4, idx = lane & 15, hb = lane & 16;
    const RecLane rlh(n_m, idx, rs);
    float *scr = h ? wm.row(1) : wm.row(0);
    const int rounds = n_m + 1 < 16 ? n_m + 1 : 16;
    for (int t = 0; t < dc; t += 2) {
        const int te = min(t + h, dc - 1);                       /* t+h >= dc: duplicate of the last edge, nothing stored */
        const bool valid = t + h < dc;
        const uint32_t ei = wm.ew[c * dcm + te];
        const int hv = (ei >> 20) & 0xff;
        float *prow = app_f + (size_t)((ei & 0xfffffu) * 16u);
        float v = prow[idx];
        const RecView r = load_record(ctov_f, (uint32_t)(e0 + te), rlh);
        scr[idx] = r.sat;                                        /* dense CtoV row, bubble_decoder.c:262-270 */
        __syncwarp();
        if (idx < r.stp) scr[r.sym] = r.llr;
        __syncwarp();
        const float cv = scr[idx];
        __syncwarp();
        v = __fsub_rn(v, cv);                                    /* NB_LDPC.c:334 */
        if (valid) prow[idx] = v;                                /* parked for phase 3 */
        /* truncation, NB_LDPC.c:354-374: unique keys, 16-wide bitonic sort inside each half */
        uint32_t x = (__float_as_uint(v) & ~15u) | (uint32_t)idx;
        const bool bad = x >= 0x7f800000u;
#pragma unroll
        for (int k = 2; k <= 16; k <<= 1) {
#pragma unroll
            for (int j = k >> 1; j > 0; j >>= 1) {
                const uint32_t y = __shfl_xor_sync(NB_FULL, x, j);
                const bool up = (k == 16) || ((lane & k) == 0);
                const bool lower = (lane & j) == 0;
                x = (lower == up) ? min(x, y) : max(x, y);
            }
        }
        const uint32_t after = __shfl_down_sync(NB_FULL, x, 1);
        const bool amb = idx < n_m && idx + 1 < rounds && ((x >> 4) == (after >> 4));
        int sym = (int)(x & 15u);
        float val = __shfl_sync(NB_FULL, v, hb | sym);
        const bool over = idx < n_m && !(val < NB_SENT);
        const unsigned flags = __ballot_sync(NB_FULL, bad || amb || over);
        if (flags) {                                             /* rare: exact scan, NB_LDPC.c:356-369, one half at a time */
            for (int hh = 0; hh < 2; hh++) {
                if (!((flags >> (16 * hh)) & 0xffffu)) continue;
                if (slow_counter && lane == 0) atomicAdd(slow_counter, 1u);
                float tmp = __shfl_sync(NB_FULL, v, 16 * hh + idx);          /* both halves hold a copy of the row */
                for (int k = 0; k < n_m; k++) {
                    float bv = NB_SENT; int bg = 0x7fffffff;
                    if (tmp < bv) { bv = tmp; bg = idx; }
#pragma unroll
                    for (int o = 8; o > 0; o >>= 1) {
                        const float ov = __shfl_xor_sync(NB_FULL, bv, o);
                        const int og = __shfl_xor_sync(NB_FULL, bg, o);
                        if (ov < bv || (ov == bv && og < bg)) { bv = ov; bg = og; }
                    }
                    if (bg == 0x7fffffff) bg = 0;                              /* nothing below 1e5: (1e5, symbol 0) */
                    if (bg == idx) tmp = NB_SENT;                              /* NB_LDPC.c:368 */
                    if (h == hh && idx == k) { val = bv; sym = bg; }
                }
            }
        }
        const float v0 = __shfl_sync(NB_FULL, val, hb);
        const float llr = idx == 0 ? 0.0f : __fsub_rn(val, v0);               /* NB_LDPC.c:372-373 */
        if (valid) {
            const int li = ls.in(c, t + h);
            const uint32_t list = ls.addr(li);
            if (idx < n_m) {
                sts_f32(list + 4 * idx, llr);
                sts_u8(ls.sym(list) + idx, (uint32_t)gf_rot_in<16, CLOSED>(gf, sym, hv));   /* bubble_decoder.c:145 */
            }
            if (idx == 0) sts_u8(ls.len(li), (uint32_t)n_m);
        }
    }
}

template <bool CLOSED>
__device__ __forceinline__ void gf16_phase3(const WarpMem<16> &wm, const GFTab &gf, int c, int e0, int dc, int dcm, float *app_f,
                                            uint8_t *ctov_f, uint8_t *dec_f, int n_m, int rs, float offset, int lane)
{
    const Lists &ls = wm.ls;
    const int h = lane >> 4, idx = lane & 15, hb = lane & 16;
    const RecLane rlh(n_m, idx, rs);
    float *scr = h ? wm.row3(1) : wm.row3(0);
    for (int t = 0; t < dc; t += 2) {
        const int te = min(t + h, dc - 1);
        const bool valid = t + h < dc;
        const uint32_t ei = wm.ew[c * dcm + te];
        const uint32_t var = ei & 0xfffffu;
        float *prow = app_f + (size_t)(var * 16u);
        float v = prow[idx];                                     /* the Mvc row parked by phase 1 */
        /* record entry of this lane and saturation constant, bubble_decoder.c:231-264 */
        const int li = ls.idx(c, id_out(dc, te), dc);
        const uint32_t list = ls.addr(li);
        const int len = (int)lds_u8(ls.len(li));
        RecView nr;
        nr.stp = len; nr.llr = NB_SENT; nr.sym = 0;
        if (idx < len) {
            nr.llr = lds_f32(list + 4 * idx);
            nr.sym = gf_rot_out<16, CLOSED>(gf, (int)lds_u8(ls.sym(list) + idx), (ei >> 20) & 0xff);
        }
        const float last = __shfl_sync(NB_FULL, nr.llr, hb | max(len - 1, 0));
        nr.sat = __fadd_rn(len > 0 ? last : NB_SENT, offset);
        if (valid) {                                             /* NB_LDPC.c:438 */
            uint8_t *rec = ctov_f + (size_t)(uint32_t)(e0 + te) * rlh.stride;
            if (idx < n_m) { *reinterpret_cast<float *>(rec + rlh.llr) = nr.llr; rec[rlh.sym] = (uint8_t)nr.sym; }
            if (idx == 0) *reinterpret_cast<int2 *>(rec + rlh.tail) = make_int2(__float_as_int(nr.sat), nr.stp);
        }
        scr[idx] = nr.sat;
        __syncwarp();
        if (idx < len) scr[nr.sym] = nr.llr;
        __syncwarp();
        const float mcv = scr[idx];
        __syncwarp();
        v = __fadd_rn(mcv, v);                                   /* NB_LDPC.c:448 */
        if (valid) prow[idx] = v;
        /* Decision, tools.c:312-330: strict '<' from 1e5, ties -> lowest symbol, default 0 */
        float bv = NB_SENT; int bg = 0x7fffffff;
        if (v < bv) { bv = v; bg = idx; }
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(NB_FULL, bv, o);
            const int og = __shfl_xor_sync(NB_FULL, bg, o);
            if (ov < bv || (ov == bv && og < bg)) { bv = ov; bg = og; }
        }
        if (valid && (ei >> 28) && idx == 0) dec_f[var] = (uint8_t)(bg == 0x7fffffff ? 0 : bg);
    }
}

/* ------------------------------------------------------------------------------------------------
 * Bubble path, q >= 64: phases 1 and 3 of a warp's tile.  Two edges are in flight per warp (NE): their global loads,
 * shared-memory round trips and REDUX chains interleave.  app / ctov / dec: the CTA's slot block; the tile meta holds the
 * byte offsets of every node's frame in it.
 * ---------------------------------------------------------------------------------------------- */
template <int Q, bool CLOSED>
__device__ __forceinline__ void tile_phase1(const KArgs &a, const WarpMem<Q> &wm, const GFTab &gf, int cnt, const char *app, const char *ctov,
                                            const RecLane &rl, uint64_t pol_first, uint64_t pol_keep, bool minform, int lane)
{
    constexpr int VPL = QTraits<Q>::VPL;
    const Lists &ls = wm.ls;
    const int dcm = a.dc_max, n_m = a.n_m, rs = a.rec_stride;
#pragma unroll
    for (int e = 0; e < NE; e++) fill_row_s<Q>(wm.rowa(e), lane, NB_ROW_CLEAN);
    __syncwarp();
    for (int c = 0; c < cnt; c++) {
        const int4 mt = wm.meta[c];
        const int dc = TileMeta::dc(mt);
        /* GF(64) only: GF(256) and GF(16) hide the latency already and pay for the extra L2 traffic at the power cap */
        if constexpr (Q == 64) {
            if (c + 1 < cnt) prefetch_node<Q>(app, ctov, wm.ew + (c + 1) * dcm, wm.meta[c + 1], rs, lane);
        }
        const char *app_f = app + (uint32_t)mt.y;
        const uint8_t *rec0 = reinterpret_cast<const uint8_t *>(ctov) + (uint32_t)mt.z;      /* record of the node's edge 0 */
        for (int t = 0; t < dc; t += NE) {
            float v[NE][VPL];
            RecView r[NE];
            int hv[NE];
            float *prow[NE];
#pragma unroll
            for (int e = 0; e < NE; e++) {
                const int te = min(t + e, dc - 1);                 /* t+e >= dc: duplicate of the last edge, result ignored */
                const uint32_t ei = wm.ew[c * dcm + te];
                hv[e] = (ei >> 20) & 0xff;
                prow[e] = reinterpret_cast<float *>(const_cast<char *>(app_f) + (ei & 0xfffffu) * (uint32_t)(Q * 4));
                /* the row is not read again: phase 3 reads the parked Mvc stored over it below */
                load_row_hint<Q>(prow[e], lane, v[e], pol_first);
                r[e] = load_record(rec0, (uint32_t)te, rl);
            }
#pragma unroll
            for (int e = 0; e < NE; e++) {
                float cv[VPL];
                expand_record<Q>(r[e], lane, wm.rowa(e), cv, minform);
#pragma unroll
                for (int j = 0; j < VPL; j++) v[e][j] = __fsub_rn(v[e][j], cv[j]);      /* NB_LDPC.c:334 */
                if (t + e < dc) store_row_hint<Q>(prow[e], lane, v[e], pol_keep);     /* parked for phase 3 (NB_LDPC.c:448 adds this vector) */
            }
            float llr[NE]; int sym[NE];
            uint32_t scra[NE];
#pragma unroll
            for (int e = 0; e < NE; e++) scra[e] = wm.scra(e);
            select_edges<Q, NE>(v, lane, scra, n_m, llr, sym, a.slow_counter);
#pragma unroll
            for (int e = 0; e < NE; e++) {
                if (t + e < dc) {
                    const int li = ls.in(c, t + e);
                    const uint32_t list = ls.addr(li);
                    if (lane < n_m) {
                        sts_f32(list + 4 * lane, llr[e]);
                        sts_u8(ls.sym(list) + lane, (uint32_t)gf_rot_in<Q, CLOSED>(gf, sym[e], hv[e]));   /* bubble_decoder.c:145 */
                    }
                    if (lane == 0) sts_u8(ls.len(li), (uint32_t)n_m);
                }
            }
        }
    }
    __syncwarp();
}

template <int Q, bool CLOSED>
__device__ __forceinline__ void tile_phase3(const KArgs &a, const WarpMem<Q> &wm, const GFTab &gf, int cnt, char *app, char *ctov,
                                            uint8_t *dec, const RecLane &rl, uint64_t pol_first, bool minform, bool decide, int lane)
{
    constexpr int VPL = QTraits<Q>::VPL;
    const Lists &ls = wm.ls;
    const int dcm = a.dc_max, n_m = a.n_m;
#pragma unroll
    for (int e = 0; e < NE; e++) fill_row_s<Q>(wm.row3a(e), lane, NB_ROW_CLEAN);
    __syncwarp();
    for (int c = 0; c < cnt; c++) {
        const int4 mt = wm.meta[c];
        const int dc = TileMeta::dc(mt);
        char *app_f = app + (uint32_t)mt.y;
        uint8_t *rec0 = reinterpret_cast<uint8_t *>(ctov) + (uint32_t)mt.z;
        /* output list of edge t (id_out): t = dc-1 -> F after dc-2 steps, else B / merge number 3dc-5+t; as an index into the tile's lists */
        const int obase = dc > 2 ? ls.r0 + c * ls.lr - dc : c * dcm;
        for (int t = 0; t < dc; t += NE) {
            float v[NE][VPL];
            uint32_t ei[NE];
#pragma unroll
            for (int e = 0; e < NE; e++) {
                const int te = min(t + e, dc - 1);
                ei[e] = wm.ew[c * dcm + te];
                load_row_hint<Q>(reinterpret_cast<const float *>(app_f + (ei[e] & 0xfffffu) * (uint32_t)(Q * 4)), lane, v[e], pol_first);    /* parked Mvc */
            }
#pragma unroll
            for (int e = 0; e < NE; e++) {
                if (t + e < dc) {
                    const uint32_t var = ei[e] & 0xfffffu;
                    const int te = t + e;
                    const int li = dc > 2 ? obase + (te == dc - 1 ? 2 * dc - 3 : 3 * dc - 5 + te) : obase + (1 - te);
                    const RecView nr = finish_list<Q, CLOSED>(ls, li, (ei[e] >> 20) & 0xff, gf, a.offset, lane);
                    store_record(rec0, (uint32_t)te, rl, nr, n_m, lane);
                    float mcv[VPL];
                    expand_record<Q>(nr, lane, wm.row3a(e), mcv, minform);    /* :262-281 */
#pragma unroll
                    for (int j = 0; j < VPL; j++) v[e][j] = __fadd_rn(mcv[j], v[e][j]);      /* NB_LDPC.c:448 */
                    store_row_hint<Q>(reinterpret_cast<float *>(app_f + var * (uint32_t)(Q * 4)), lane, v[e], pol_first);
                    if (decide && (ei[e] >> 28)) {                                         /* tools.c:312 fused */
                        const int d = warp_argmin<Q>(v[e], lane);
                        if (lane == 0) dec[(uint32_t)mt.w + var] = (uint8_t)d;
                    }
                }
            }
        }
    }
}

/* Soft output of the nf frames of a finished group (include/nbldpc_b200.h), one warp per variable, from the final APP rows
 * in the group's slots (app = the CTA's slot block).  Runs after the last pass, where the phase-1 scratch of the warp is
 * free; the slots are reused by the next group, so this is the last moment the rows exist. */
template <int Q, int ECN>
__device__ __forceinline__ void soft_output(const KArgs &a, const WarpMem<Q, ECN> &wm, const GFTab &gf, const float *app, int base, int nf,
                                         int warp, int nw, int lane)
{
    constexpr int VPL = QTraits<Q>::VPL, LOGQ = QTraits<Q>::LOGQ;
    const bool active = (Q >= 32) || lane < Q;
    const int k = a.soft_k;
    for (int w = warp; w < nf * a.N; w += nw) {          /* w = f * N + n: row w of the slot block, variable base * N + w */
        const size_t var = (size_t)base * a.N + w;
        float v[1][VPL];
        load_row<Q>(app + (size_t)w * Q, lane, v[0]);
        if (a.soft_kind == NBGPU_SOFT_LIST) {
            /* the truncation NB_LDPC.c:354-374 with n_m = k; the decoder's slow-path counter is not touched */
            const uint32_t scr[1] = { wm.scra(0) };
            float llr[1]; int sym[1];
            select_edges<Q, 1>(v, lane, scr, k, llr, sym, nullptr);
            if (lane < k) { a.soft_llr[var * k + lane] = llr[0]; a.soft_sym[var * k + lane] = (uint8_t)sym[0]; }
        } else {
            /* per bit the two minima, split by the binary image; keys in the total order of the floats (the APP may be
             * negative with a negative offset), so one integer REDUX per minimum gives the exact value back */
            uint32_t m0[LOGQ], m1[LOGQ];
#pragma unroll
            for (int l = 0; l < LOGQ; l++) { m0[l] = NB_KEY_INF; m1[l] = NB_KEY_INF; }
#pragma unroll
            for (int j = 0; j < VPL; j++) {
                const uint32_t b = __float_as_uint(v[0][j]);
                const uint32_t key = active ? b ^ ((uint32_t)((int)b >> 31) | 0x80000000u) : NB_KEY_INF;
                const uint32_t im = gf.img[QTraits<Q>::sym(lane, j) & (Q - 1)];
#pragma unroll
                for (int l = 0; l < LOGQ; l++) {
                    if ((im >> l) & 1u) m1[l] = min(m1[l], key); else m0[l] = min(m0[l], key);
                }
            }
            float out = 0.0f;
#pragma unroll
            for (int l = 0; l < LOGQ; l++) {
                const uint32_t k0 = __reduce_min_sync(NB_FULL, m0[l]), k1 = __reduce_min_sync(NB_FULL, m1[l]);
                const float x0 = __uint_as_float((k0 & 0x80000000u) ? k0 ^ 0x80000000u : ~k0);
                const float x1 = __uint_as_float((k1 & 0x80000000u) ? k1 ^ 0x80000000u : ~k1);
                if (lane == l) out = __fsub_rn(x1, x0);
            }
            if (lane < LOGQ) a.soft_llr[var * LOGQ + lane] = out;
        }
    }
}

template <int Q, bool CLOSED, int ECN, bool SOFT>
__global__ void __launch_bounds__(ECN ? NT_SYND : NT_MAX, CTAS_PER_SM) decode_kernel(const KArgs a)
{
    constexpr int VPL = QTraits<Q>::VPL;
    extern __shared__ __align__(16) unsigned char smem[];
    /* read once through volatile asm: otherwise the register allocator re-reads SR_TID (S2R, ~10 per check node) instead of
     * keeping the lane number in a register */
    int tid;
    asm volatile("mov.u32 %0, %%tid.x;" : "=r"(tid));
    const int lane = tid & 31, warp = tid >> 5, nthr = blockDim.x, nw = nthr >> 5;
    WarpMem<Q, ECN> wm(smem, a, warp);
    GFTab gf;
    load_gf_tables(smem, a, gf);
    load_cfg_table(smem, a);
    int *misc = reinterpret_cast<int *>(smem + a.off_misc);
    int *s_base = misc;                 /* [1]  first frame of the group  */
    int *s_alive = misc + 1;            /* [1]  frames of the group still iterating */
    int *s_done = misc + 2;             /* [F]  0 = iterating, else iters value to report */
    int *s_badrow = misc + 2 + a.F;     /* [F]  first check row with non-zero syndrome */
    int *s_synd = misc + 2 + 2 * a.F;   /* [F]  last syndrome value */
    const int F = a.F, N = a.N, n_m = a.n_m, dcm = a.dc_max, rs = a.rec_stride;
    const size_t frame_app = (size_t)N * Q, frame_ctov = (size_t)a.E * rs;
    const RecLane rl(n_m, lane, rs);
    const uint64_t pol_keep = l2_policy_evict_last(), pol_stream = l2_policy_evict_first();
    const bool minform = a.offset >= 0.0f;
    float *app = a.app + blockIdx.x * F * frame_app;
    uint8_t *ctov = a.ctov + blockIdx.x * F * frame_ctov;
    uint8_t *dec = a.dec + (size_t)blockIdx.x * F * N;
    const size_t frame_dense = (size_t)a.E * Q;
    float *ctov_d = ECN != 0 ? a.ctov_dense + blockIdx.x * F * frame_dense : nullptr;
    const uint32_t rec_bytes = ECN != 0 ? (uint32_t)(Q * 4) : (uint32_t)rs;      /* bytes of CtoV state per edge */

    for (;;) {
        __syncthreads();
        if (tid == 0) *s_base = (int)atomicAdd(a.queue, (unsigned)F);
        __syncthreads();
        const int base = *s_base;
        if (base >= a.B) break;
        const int nf = min(F, a.B - base);
        if (a.ready) {
            /* the host is still copying the batch in (frame order, a counter after every piece): wait for this group's frames.
             * Copies run ~25x faster than the decoder consumes them, so only the first groups of a launch ever wait. */
            if (tid == 0) {
                const unsigned need = (unsigned)(base + nf);
                unsigned have, spins = 0;
                for (;;) {
                    asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(have) : "l"(a.ready) : "memory");
                    if (have >= need) break;
                    if (++spins > (1u << 23)) { atomicExch(a.fault, 1u); break; }        /* ~4 s: the copy never came */
                    __nanosleep(500);
                }
            }
            __syncthreads();
        }
        /* ---------------- frame initialisation: NB_LDPC.c:273-288 + channel.c:66-76 ---------------- */
        for (int w = warp; w < nf * N; w += nw) {
            const int f = w / N, n = w - f * N;
            const int t = a.pmap ? a.pmap[n] : n;        /* the variable's symbol in the input frame; -1: punctured */
            const size_t r = (size_t)(base + f) * a.nt + t;
            float v[VPL];
            if (t < 0) {
#pragma unroll
                for (int j = 0; j < VPL; j++) v[j] = 0.0f;
            } else if (a.input_kind == INPUT_BPSK) intake_variable<Q>(a.in + r * a.logq, a.den, gf.img, lane,
                                                                      reinterpret_cast<double *>(wm.scr(0)), reinterpret_cast<float *>(wm.scr(0)) + 32, v);
            else if (a.input_kind == INPUT_MAPPED || a.input_kind == INPUT_FADED)
                intake_mapped<Q>(mapped_input(a.in, a.input_kind, r), a.den, a.mod, gf.img, lane, v);
            else if (a.input_kind == INPUT_SPLIT)       /* scratch: 32 doubles, within the phase-1 scratch of plan_smem */
                intake_split<Q>(a.in + r * (2 * a.split_p), a.split_p, a.den, a.mod, gf.img, lane, reinterpret_cast<double *>(wm.scr(0)), v);
            else load_row<Q>(a.in + r * Q, lane, v);
            store_row<Q>(app + ((size_t)f * N + n) * Q, lane, v);
        }
        if constexpr (ECN == 0) {
            for (int i = tid; i < nf * a.E; i += nthr)       /* CtoV = 0: stp 0, constant 0.0f */
                *reinterpret_cast<int2 *>(ctov + (size_t)i * rs + rl.tail) = make_int2(0, 0);
        } else {
            float4 *z = reinterpret_cast<float4 *>(ctov_d);  /* CtoV = 0, NB_LDPC.c:273-279 */
            for (size_t i = tid; i < (size_t)nf * frame_dense / 4; i += nthr) z[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        for (int i = tid; i < F; i += nthr) { s_done[i] = (i < nf) ? 0 : -1; s_synd[i] = 0; }
        if (tid == 0) { *s_alive = nf; for (int f = 0; f < nf; f++) { a.frame_slot[base + f] = blockIdx.x * F + f; a.slot_frame[blockIdx.x * F + f] = a.frame0 + base + f; } }
        __syncthreads();
        /* variables that no check node touches keep their channel decision */
        for (int w = warp; w < nf * a.n_isolated; w += nw) {
            const int f = w / a.n_isolated, n = a.isolated[w - f * a.n_isolated];
            float v[VPL];
            load_row<Q>(app + ((size_t)f * N + n) * Q, lane, v);
            const int d = warp_argmin<Q>(v, lane);
            if (lane == 0) dec[f * N + n] = (uint8_t)d;
        }

        for (int pass = 0; pass < a.passes; pass++) {
            /* Decision + Syndrom are observable only through the early-termination test and after the last pass */
            const bool decide = a.early_stop || pass == a.passes - 1;
            for (int st = 0; st < a.nsteps; st++) {
                const int c0 = a.step_ptr[st], ncn = a.step_ptr[st + 1] - c0;
                const int items = ncn * nf;                   /* item = f * ncn + ci */
                const int per = (items + nw - 1) / nw;        /* <= cpw by construction of the schedule */
                const int first = warp * per;
                const int cnt = max(0, min(per, items - first));
                /* tile description: one lane per check node */
                if (lane < cnt) {
                    const int item = first + lane, f = item / ncn;
                    const uint32_t info = a.cninfo[c0 + item - f * ncn];
                    const uint32_t e0 = info & 0xffffff;
                    wm.meta.set(lane, (int)e0, s_done[f] ? 0 : (int)(info >> 24), (uint32_t)f * (uint32_t)(N * Q * 4),
                                ((uint32_t)f * (uint32_t)a.E + e0) * rec_bytes, (uint32_t)(f * N));
                }
                __syncwarp();
                for (int i = lane; i < cnt * dcm; i += 32) {   /* edge words of the tile: variable | coefficient | last-visit flag */
                    const int c = i / dcm, t = i - c * dcm;
                    const int4 mt = wm.meta[c];
                    if (t < TileMeta::dc(mt)) wm.ew[i] = a.einfo[TileMeta::e0(mt) + t];
                }
                __syncwarp();
                if constexpr (ECN == 0) {
                    if constexpr (Q == 16) {
                        const Lists &ls = wm.ls;
                        for (int c = 0; c < cnt; c++) {
                            const int4 mt = wm.meta[c];
                            const int e0 = TileMeta::e0(mt), dc = TileMeta::dc(mt);
                            float *app_f = reinterpret_cast<float *>(reinterpret_cast<char *>(app) + (uint32_t)mt.y);
                            const uint8_t *ctov_f = ctov + (uint32_t)mt.z - (size_t)e0 * rs;
                            gf16_phase1<CLOSED>(wm, gf, c, e0, dc, dcm, app_f, ctov_f, n_m, rs, lane, a.slow_counter);
                        }
                        __syncwarp();
                        tile_elementary_steps<Q>(ls, wm.meta, cnt, dcm, wm.mask, lane, a.nb_oper);
                        for (int c = 0; c < cnt; c++) {
                            const int4 mt = wm.meta[c];
                            const int e0 = TileMeta::e0(mt);
                            gf16_phase3<CLOSED>(wm, gf, c, e0, TileMeta::dc(mt), dcm, reinterpret_cast<float *>(reinterpret_cast<char *>(app) + (uint32_t)mt.y),
                                                ctov + (uint32_t)mt.z - (size_t)e0 * rs, dec + (uint32_t)mt.w, n_m, rs, a.offset, lane);
                        }
                    } else {
                        tile_phase1<Q, CLOSED>(a, wm, gf, cnt, reinterpret_cast<const char *>(app), reinterpret_cast<const char *>(ctov), rl, pol_stream, pol_keep, minform, lane);
                        tile_elementary_steps<Q>(wm.ls, wm.meta, cnt, dcm, wm.mask, lane, a.nb_oper);
                        tile_phase3<Q, CLOSED>(a, wm, gf, cnt, reinterpret_cast<char *>(app), reinterpret_cast<char *>(ctov), dec, rl, pol_stream, minform, decide, lane);
                    }
                } else if constexpr (ECN == 1) {
                    /* ---------------- syndrome-based check node: one node at a time per warp ---------------- */
                    const SyndMem sm = make_synd_mem(smem, a, warp);
                    for (int c = 0; c < cnt; c++) {
                        const int4 mt = wm.meta[c];
                        const int dc = TileMeta::dc(mt);
                        if (dc == 0) continue;
                        float *app_f = reinterpret_cast<float *>(reinterpret_cast<char *>(app) + (uint32_t)mt.y);
                        float *cd0 = reinterpret_cast<float *>(reinterpret_cast<char *>(ctov_d) + (uint32_t)mt.z);     /* dense CtoV row of the node's edge 0 */
                        uint8_t *dec_f = dec + (uint32_t)mt.w;
                        /* V->C messages of the node: Mvc = APP - CtoV, truncation, rotation (NB_LDPC.c:329-374, syndrome_decoder.c:41-48) */
                        for (int t = 0; t < dc; t += NE) {
                            float v[NE][VPL];
                            int hv[NE];
#pragma unroll
                            for (int e = 0; e < NE; e++) {
                                const int te = min(t + e, dc - 1);
                                const uint32_t ei = wm.ew[c * dcm + te];
                                hv[e] = (ei >> 20) & 0xff;
                                float cv[VPL];
                                load_row<Q>(app_f + (size_t)((ei & 0xfffffu) * (uint32_t)Q), lane, v[e]);
                                load_row<Q>(cd0 + (size_t)((uint32_t)te * (uint32_t)Q), lane, cv);
#pragma unroll
                                for (int j = 0; j < VPL; j++) v[e][j] = __fsub_rn(v[e][j], cv[j]);
                            }
                            float llr[NE]; int sym[NE];
                            uint32_t scra[NE];
#pragma unroll
                            for (int e = 0; e < NE; e++) scra[e] = wm.scra(e);
                            select_edges<Q, NE>(v, lane, scra, n_m, llr, sym, a.slow_counter);
#pragma unroll
                            for (int e = 0; e < NE; e++) {
                                if (t + e < dc && lane < n_m) {
                                    const uint32_t list = sm.lists + (t + e) * sm.lstride;
                                    sts_f32(list + 4 * lane, llr[e]);
                                    sts_u8(list + 4 * n_m + lane, (uint32_t)gf_rot_in<Q, CLOSED>(gf, sym[e], hv[e]));
                                }
                            }
                        }
                        __syncwarp();
                        const bool plain = synd_prepare(sm, lane);
                        for (int d = 0; d < dc; d++) {
                            if ((d & 3) == 0) { if (plain) synd_walk<false>(sm, d, min(4, dc - d), lane); else synd_walk<true>(sm, d, min(4, dc - d), lane); }
                            const uint32_t out = sm.rows + 1024 * (d & 3);
                            const int t = (int)lds_u32(sm.perm + 4 * d);                   /* un-permute, syndrome_decoder.c:234-253 */
                            const uint32_t ei = wm.ew[c * dcm + t];
                            const uint32_t var = ei & 0xfffffu;
                            float *cdrow = cd0 + (size_t)((uint32_t)t * (uint32_t)Q);
                            float mcv[VPL], v[VPL], cv[VPL];
                            const float sat = lds_f32(sm.perm + 64 + 4 * d);
                            synd_dense_row<Q, CLOSED>(out, gf, (ei >> 20) & 0xff, lane, sat, __fadd_rn(sat, a.offset), mcv);
                            load_row<Q>(app_f + (size_t)(var * (uint32_t)Q), lane, v);
                            load_row<Q>(cdrow, lane, cv);
#pragma unroll
                            for (int j = 0; j < VPL; j++) v[j] = __fadd_rn(mcv[j], __fsub_rn(v[j], cv[j]));   /* NB_LDPC.c:334, 448 */
                            store_row<Q>(cdrow, lane, mcv);                   /* NB_LDPC.c:438 */
                            store_row<Q>(app_f + (size_t)(var * (uint32_t)Q), lane, v);
                            if (decide && (ei >> 28)) {
                                const int dd = warp_argmin<Q>(v, lane);
                                if (lane == 0) dec_f[var] = (uint8_t)dd;
                            }
                            __syncwarp();
                        }
                    }
                } else {
                    /* ---------------- dense-row check nodes (sum-product, Min-Max): one node at a time per warp ---------------- */
                    const SpaMem sp = make_spa_mem(smem, a, warp);
                    for (int c = 0; c < cnt; c++) {
                        const int4 mt = wm.meta[c];
                        const int dc = TileMeta::dc(mt);
                        if (dc == 0) continue;
                        float *app_f = reinterpret_cast<float *>(reinterpret_cast<char *>(app) + (uint32_t)mt.y);
                        float *cd0 = reinterpret_cast<float *>(reinterpret_cast<char *>(ctov_d) + (uint32_t)mt.z);     /* dense CtoV row of the node's edge 0 */
                        uint8_t *dec_f = dec + (uint32_t)mt.w;
                        /* Mvc = APP - CtoV (NB_LDPC.c:334), parked in the APP row for the update below; then into the check domain */
                        for (int t = 0; t < dc; t++) {
                            const uint32_t ei = wm.ew[c * dcm + t];
                            float *arow = app_f + (size_t)((ei & 0xfffffu) * (uint32_t)Q);
                            float v[VPL], cv[VPL];
                            load_row<Q>(arow, lane, v);
                            load_row<Q>(cd0 + (size_t)((uint32_t)t * (uint32_t)Q), lane, cv);
#pragma unroll
                            for (int j = 0; j < VPL; j++) v[j] = __fsub_rn(v[j], cv[j]);
                            store_row<Q>(arow, lane, v);
                            if constexpr (ECN == 2) spa_in<Q, CLOSED>(sp, t, v, (ei >> 20) & 0xff, gf, lane);
                            else mm_in<Q, CLOSED>(sp, t, v, (ei >> 20) & 0xff, gf, lane);
                        }
                        if constexpr (ECN == 2) spa_bwd<Q>(sp, dc, cd0, lane);
                        else mm_bwd<Q>(sp, dc, cd0, lane);
                        float fwd[VPL];
#pragma unroll
                        for (int j = 0; j < VPL; j++) fwd[j] = 1.0f;
                        for (int t = 0; t < dc; t++) {
                            const uint32_t ei = wm.ew[c * dcm + t];
                            const uint32_t var = ei & 0xfffffu;
                            float *cdrow = cd0 + (size_t)((uint32_t)t * (uint32_t)Q);
                            float *arow = app_f + (size_t)(var * (uint32_t)Q);
                            float mcv[VPL], v[VPL];
                            if constexpr (ECN == 2) spa_out<Q, CLOSED>(sp, t, cdrow, fwd, (ei >> 20) & 0xff, gf, lane, mcv);
                            else mm_out<Q, CLOSED>(sp, t, dc, cdrow, fwd, (ei >> 20) & 0xff, gf, lane, mcv);
                            load_row<Q>(arow, lane, v);                       /* the parked Mvc */
#pragma unroll
                            for (int j = 0; j < VPL; j++) v[j] = __fadd_rn(mcv[j], v[j]);     /* NB_LDPC.c:448 */
                            store_row<Q>(cdrow, lane, mcv);                   /* NB_LDPC.c:438 */
                            store_row<Q>(arow, lane, v);
                            if (decide && (ei >> 28)) {
                                const int dd = warp_argmin<Q>(v, lane);
                                if (lane == 0) dec_f[var] = (uint8_t)dd;
                            }
                        }
                    }
                }
                __syncthreads();
            }
            if (!decide) continue;
            /* ---------------- Syndrom (tools.c:284-299) + early termination (NB_LDPC.c:470) ---------------- */
            for (int i = tid; i < nf; i += nthr) s_badrow[i] = a.M;
            __syncthreads();
            for (int i = tid; i < nf * a.M; i += nthr) {
                const int f = i / a.M, m = i - f * a.M;
                if (s_done[f]) continue;
                int x = 0;
                for (int e = a.row_ptr[m]; e < a.row_ptr[m + 1]; e++) x ^= gf_rot_in<Q, CLOSED>(gf, dec[f * N + a.col[e]], a.hval[e]);
                if (x) atomicMin(&s_badrow[f], m);
            }
            __syncthreads();
            if (tid < nf && !s_done[tid]) {
                const int f = tid, m = s_badrow[f];
                int x = 0;
                if (m < a.M) for (int e = a.row_ptr[m]; e < a.row_ptr[m + 1]; e++) x ^= gf_rot_in<Q, CLOSED>(gf, dec[f * N + a.col[e]], a.hval[e]);
                s_synd[f] = gf.inv[x];
                if ((x == 0 && a.early_stop)) { s_done[f] = pass + 1; atomicSub(s_alive, 1); }   /* sum_it += iter+1 */
            }
            __syncthreads();
            if (*s_alive == 0) break;
        }
        /* ---------------- results ---------------- */
        for (int i = tid; i < nf * N; i += nthr) a.out_decide[(size_t)base * N + i] = dec[i];
        if (tid < nf) {
            a.out_synd[base + tid] = s_synd[tid];
            a.out_iters[base + tid] = s_done[tid] > 0 ? s_done[tid] : a.nb_iter_max;      /* NB_LDPC.c:474 */
        }
        if constexpr (SOFT) soft_output<Q, ECN>(a, wm, gf, app, base, nf, warp, nw, lane);
    }
}

/* ------------------------------------------------------------------------------------------------
 * unit-boundary kernels (parity tests call these through the C ABI)
 * ---------------------------------------------------------------------------------------------- */
template <int Q>
__global__ void __launch_bounds__(UNIT_NT) select_kernel(const float *rows, float *llr, int *gf, int B, int n_m, unsigned *slow)
{
    constexpr int VPL = QTraits<Q>::VPL;
    constexpr int UW = UNIT_NT / 32;
    __shared__ uint32_t scr_s[UW][QTraits<Q>::SCR_WORDS + 64];     /* + slack: a lane that popped the +inf row reads one row further */
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t scr[1] = { smem_u32(scr_s[warp]) };
    for (int r = blockIdx.x * UW + warp; r < B; r += gridDim.x * UW) {
        float v[1][VPL];
        load_row<Q>(rows + (size_t)r * Q, lane, v[0]);
        float l[1]; int s[1];
        select_edges<Q, 1>(v, lane, scr, n_m, l, s, slow);
        if (lane < n_m) { llr[(size_t)r * n_m + lane] = l[0]; gf[(size_t)r * n_m + lane] = s[0]; }
        __syncwarp();
    }
}

/* ElementaryStep on B pairs; symbols already binary images (0..q-1) with lens.  One thread per step;
 * the lists are staged in shared memory because es_serial works on shared-window addresses. */
#define ES_NT 64
template <int Q>
__global__ void __launch_bounds__(ES_NT) es_kernel(const float *in1, const float *in2, const uint8_t *s1, const uint8_t *s2, const int *len1,
                                                   const int *len2, float *out, uint8_t *so, int *leno, int B, int n_m, int nb_oper)
{
    __shared__ float fl[ES_NT][3][32];
    __shared__ uint8_t sy[ES_NT][3][32];
    __shared__ uint32_t mk[8][ES_NT];
    const int t = threadIdx.x, i = blockIdx.x * ES_NT + t;
    if (i >= B) return;
    for (int k = 0; k < n_m; k++) {
        fl[t][0][k] = in1[(size_t)i * n_m + k]; fl[t][1][k] = in2[(size_t)i * n_m + k];
        sy[t][0][k] = s1[(size_t)i * n_m + k]; sy[t][1][k] = s2[(size_t)i * n_m + k];
    }
    /* mask words of one thread must be 128 bytes apart: [w][32 threads] inside this thread's half */
    const uint32_t mask = smem_u32(&mk[0][0]) + (t >> 5) * 8 * 128 + (t & 31) * 4;
    const int s = es_serial<Q>(smem_u32(fl[t][0]), smem_u32(sy[t][0]), len1[i], smem_u32(fl[t][1]), smem_u32(sy[t][1]), len2[i],
                               smem_u32(fl[t][2]), smem_u32(sy[t][2]), mask, n_m, nb_oper);
    leno[i] = s;
    for (int k = 0; k < n_m; k++) { out[(size_t)i * n_m + k] = fl[t][2][k]; so[(size_t)i * n_m + k] = k < s ? sy[t][2][k] : 0; }
}

/* one check node (bubble ECN) for B input sets: same tile code as the decoder, one warp per tile */
template <int Q, bool CLOSED>
__global__ void __launch_bounds__(NT_MAX, 1) checknode_kernel(const KArgs a, int node, const float *vllr, const int *vgf,
                                                              float *cllr, int *cgf, int B)
{
    constexpr int VPL = QTraits<Q>::VPL;
    extern __shared__ __align__(16) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
    WarpMem<Q> wm(smem, a, warp);
    const Lists &ls = wm.ls;
    GFTab gf;
    load_gf_tables(smem, a, gf);
    __syncthreads();
    const int e0 = a.row_ptr[node], dc = a.row_ptr[node + 1] - e0, n_m = a.n_m;
    for (int b0 = (blockIdx.x * nw + warp) * a.cpw; b0 < B; b0 += gridDim.x * nw * a.cpw) {
        const int cnt = min(a.cpw, B - b0);
        for (int i = lane; i < cnt * dc * n_m; i += 32) {
            const int c = i / (dc * n_m), r = i - c * dc * n_m, t = r / n_m, k = r - t * n_m;
            const size_t src = ((size_t)(b0 + c) * dc + t) * n_m + k;
            const int li = ls.in(c, t);
            const uint32_t list = ls.addr(li);
            sts_f32(list + 4 * k, vllr[src]);
            sts_u8(ls.sym(list) + k, (uint32_t)gf_rot_in<Q, CLOSED>(gf, vgf[src] & (Q - 1), a.hval[e0 + t]));
            if (k == 0) sts_u8(ls.len(li), (uint32_t)n_m);
        }
        if (lane < cnt) wm.meta.set(lane, e0, dc, 0u, 0u, 0u);
        __syncwarp();
        tile_elementary_steps<Q>(ls, wm.meta, cnt, dc, wm.mask, lane, a.nb_oper);
        fill_row_s<Q>(wm.row3a(0), lane, NB_ROW_CLEAN);       /* aliases the input lists, dead after the elementary steps (degree 2: a region of its own) */
        __syncwarp();
        for (int c = 0; c < cnt; c++)
            for (int t = 0; t < dc; t++) {
                const RecView nr = finish_list<Q, CLOSED>(ls, ls.idx(c, id_out(dc, t), dc), a.hval[e0 + t], gf, a.offset, lane);
                float mcv[VPL];
                expand_record<Q>(nr, lane, wm.row3a(0), mcv, a.offset >= 0.0f);
                float *dst = cllr + ((size_t)(b0 + c) * dc + t) * Q;
                store_row<Q>(dst, lane, mcv);
                int *gdst = cgf + ((size_t)(b0 + c) * dc + t) * Q;
#pragma unroll
                for (int j = 0; j < VPL; j++) if (Q >= 32 || lane < Q) gdst[QTraits<Q>::sym(lane, j)] = QTraits<Q>::sym(lane, j);   /* :276 */
            }
        __syncwarp();
    }
}

/* one check node (syndrome ECN) for B input sets, one warp per set: cllr[t][k] = M_CtoV_LLR[t][k] with k the rotated
 * symbol, cgf[t][k] = DIVGF[k][h_t] (syndrome_decoder.c:234-266) */
template <int Q, bool CLOSED>
__global__ void __launch_bounds__(NT_MAX, 1) checknode_synd_kernel(const KArgs a, int node, const float *vllr, const int *vgf,
                                                                   float *cllr, int *cgf, int B)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
    GFTab gf;
    load_gf_tables(smem, a, gf);
    load_cfg_table(smem, a);
    __syncthreads();
    const SyndMem sm = make_synd_mem(smem, a, warp);
    const int e0 = a.row_ptr[node], dc = a.row_ptr[node + 1] - e0, n_m = a.n_m;
    for (int b = blockIdx.x * nw + warp; b < B; b += gridDim.x * nw) {
        for (int i = lane; i < dc * n_m; i += 32) {
            const int t = i / n_m, k = i - t * n_m;
            const size_t src = ((size_t)b * dc + t) * n_m + k;
            const uint32_t list = sm.lists + t * sm.lstride;
            sts_f32(list + 4 * k, vllr[src]);
            sts_u8(list + 4 * n_m + k, (uint32_t)gf_rot_in<Q, CLOSED>(gf, vgf[src] & (Q - 1), a.hval[e0 + t]));
        }
        __syncwarp();
        const bool plain = synd_prepare(sm, lane);
        for (int d = 0; d < dc; d++) {
            if ((d & 3) == 0) { if (plain) synd_walk<false>(sm, d, min(4, dc - d), lane); else synd_walk<true>(sm, d, min(4, dc - d), lane); }
            const uint32_t out = sm.rows + 1024 * (d & 3);
            const int t = (int)lds_u32(sm.perm + 4 * d);
            float *dst = cllr + ((size_t)b * dc + t) * Q;
            int *gdst = cgf + ((size_t)b * dc + t) * Q;
            const float sat = lds_f32(sm.perm + 64 + 4 * d), hi = __fadd_rn(sat, a.offset);
            for (int k = lane; k < Q; k += 32) {
                dst[k] = synd_saturate(lds_f32(out + 4 * gf.img[k]), sat, hi);
                gdst[k] = gf_rot_out<Q, CLOSED>(gf, gf.img[k], a.hval[e0 + t]);
            }
            __syncwarp();
        }
    }
}

/* one check node (dense ECN: 2 = sum-product, 4 = Min-Max) for B input sets, one warp per set: the node's steps after Mvc
 * (include/nbldpc_b200.h) from mvc[b][t][.] (symbol order) to ctov[b][t][.], through the decoder's spa_* / mm_* functions;
 * the output rows are the backward-partial scratch, as the dense CtoV rows are in the decoder */
template <int Q, bool CLOSED, int ECN>
__global__ void __launch_bounds__(NT_SYND, 1) checknode_dense_kernel(const KArgs a, int node, const float *mvc, float *ctov, int B)
{
    constexpr int VPL = QTraits<Q>::VPL;
    extern __shared__ __align__(16) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
    GFTab gf;
    load_gf_tables(smem, a, gf);
    __syncthreads();
    const SpaMem sp = make_spa_mem(smem, a, warp);
    const int e0 = a.row_ptr[node], dc = a.row_ptr[node + 1] - e0;
    for (int b = blockIdx.x * nw + warp; b < B; b += gridDim.x * nw) {
        float *out = ctov + (size_t)b * dc * Q;
        for (int t = 0; t < dc; t++) {
            float v[VPL];
            load_row<Q>(mvc + ((size_t)b * dc + t) * Q, lane, v);
            if constexpr (ECN == 2) spa_in<Q, CLOSED>(sp, t, v, a.hval[e0 + t], gf, lane);
            else mm_in<Q, CLOSED>(sp, t, v, a.hval[e0 + t], gf, lane);
        }
        if constexpr (ECN == 2) spa_bwd<Q>(sp, dc, out, lane);
        else mm_bwd<Q>(sp, dc, out, lane);
        float fwd[VPL];
#pragma unroll
        for (int j = 0; j < VPL; j++) fwd[j] = 1.0f;
        for (int t = 0; t < dc; t++) {
            float cv[VPL];
            if constexpr (ECN == 2) spa_out<Q, CLOSED>(sp, t, out + (size_t)t * Q, fwd, a.hval[e0 + t], gf, lane, cv);
            else mm_out<Q, CLOSED>(sp, t, dc, out + (size_t)t * Q, fwd, a.hval[e0 + t], gf, lane, cv);
            store_row<Q>(out + (size_t)t * Q, lane, cv);
        }
    }
}

/* Decision + Syndrom on dense APP[B][N][q] */
template <int Q>
__global__ void __launch_bounds__(UNIT_NT) decision_kernel(const KArgs a, const float *app, int *decide, int B)
{
    constexpr int VPL = QTraits<Q>::VPL;
    constexpr int UW = UNIT_NT / 32;
    const int lane = threadIdx.x & 31;
    const long total = (long)B * a.N;
    for (long r = (long)blockIdx.x * UW + (threadIdx.x >> 5); r < total; r += (long)gridDim.x * UW) {
        float v[VPL];
        load_row<Q>(app + r * Q, lane, v);
        const int d = warp_argmin<Q>(v, lane);
        if (lane == 0) decide[r] = d;
    }
}
__global__ void syndrome_kernel(const KArgs a, const int *decide, int *synd, int B)
{
    /* one CTA per frame */
    __shared__ int badrow;
    for (int f = blockIdx.x; f < B; f += gridDim.x) {
        if (threadIdx.x == 0) badrow = a.M;
        __syncthreads();
        for (int m = threadIdx.x; m < a.M; m += blockDim.x) {
            int x = 0;
            for (int e = a.row_ptr[m]; e < a.row_ptr[m + 1]; e++) x ^= a.rotin[a.hval[e] * a.q + decide[(size_t)f * a.N + a.col[e]]];
            if (x) atomicMin(&badrow, m);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            int x = 0, m = badrow;
            if (m < a.M) for (int e = a.row_ptr[m]; e < a.row_ptr[m + 1]; e++) x ^= a.rotin[a.hval[e] * a.q + decide[(size_t)f * a.N + a.col[e]]];
            synd[f] = a.inv[x];
        }
        __syncthreads();
    }
}

/* channel intake as a standalone kernel: dense LLR and (optionally) the sorted intrinsic arrays
 * (channel.c:66-91).  The sort is only needed for interface parity with decoder_t.intrinsic_*. */
template <int Q>
__global__ void __launch_bounds__(UNIT_NT) channel_kernel(const KArgs a, const float *noisy, float *llr, float *illr, int *igf, int B, int kind)
{
    constexpr int VPL = QTraits<Q>::VPL;
    constexpr int UW = UNIT_NT / 32;
    __shared__ double ts[UW][32];
    __shared__ float rows[UW][Q];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long total = (long)B * a.N;
    for (long r = (long)blockIdx.x * UW + warp; r < total; r += (long)gridDim.x * UW) {
        float v[VPL];
        long ri = r;                                    /* output row r = f * N + n reads input symbol f * nt + pmap[n] */
        int t = 0;
        if (a.pmap) { const long f = r / a.N; t = a.pmap[r - f * a.N]; ri = f * a.nt + t; }
        if (t < 0) {
#pragma unroll
            for (int j = 0; j < VPL; j++) v[j] = 0.0f;
        } else if (kind == INPUT_MAPPED || kind == INPUT_FADED) intake_mapped<Q>(mapped_input(noisy, kind, (size_t)ri), a.den, a.mod, a.img, lane, v);
        else if (kind == INPUT_SPLIT) intake_split<Q>(noisy + ri * (2 * a.split_p), a.split_p, a.den, a.mod, a.img, lane, ts[warp], v);
        else intake_variable<Q>(noisy + ri * a.logq, a.den, a.img, lane, ts[warp], rows[warp], v);
        if (llr) store_row<Q>(llr + r * Q, lane, v);
        if (illr) {
            /* full stable sort = q rounds of the exact scan (channel.c:78-91) */
            float tmp[VPL];
#pragma unroll
            for (int j = 0; j < VPL; j++) tmp[j] = v[j];
            for (int k = 0; k < Q; k++) {
                float bv = NB_SENT; int bg = 0x7fffffff;
#pragma unroll
                for (int j = 0; j < VPL; j++) if ((Q >= 32 || lane < Q) && tmp[j] < bv) { bv = tmp[j]; bg = QTraits<Q>::sym(lane, j); }
                warp_lexmin(bv, bg);
#pragma unroll
                for (int j = 0; j < VPL; j++) if ((Q >= 32 || lane < Q) && bg == QTraits<Q>::sym(lane, j)) tmp[j] = NB_SENT;
                if (lane == 0) { illr[r * Q + k] = bv; igf[r * Q + k] = (bg == 0x7fffffff) ? -1 : bg; }
            }
        }
    }
}

template <int ECN, bool SOFT> static const void *decode_fn_e(int q, int closed)
{
    if (closed) return q == 16 ? (const void *)decode_kernel<16, true, ECN, SOFT> : q == 64 ? (const void *)decode_kernel<64, true, ECN, SOFT> : (const void *)decode_kernel<256, true, ECN, SOFT>;
    return q == 16 ? (const void *)decode_kernel<16, false, ECN, SOFT> : q == 64 ? (const void *)decode_kernel<64, false, ECN, SOFT> : (const void *)decode_kernel<256, false, ECN, SOFT>;
}
/* q is validated in nbgpu_create (16, 64 or 256); anything else never reaches a launch.  soft: a soft-output kind is armed */
static const void *decode_fn(int q, int closed, int ecn, bool soft)
{
    if (q != 16 && q != 64 && q != 256) return nullptr;
    if (ecn == 2) return soft ? decode_fn_e<2, true>(q, closed) : decode_fn_e<2, false>(q, closed);
    if (ecn == 4) return soft ? decode_fn_e<4, true>(q, closed) : decode_fn_e<4, false>(q, closed);
    if (soft) return ecn ? decode_fn_e<1, true>(q, closed) : decode_fn_e<0, true>(q, closed);
    return ecn ? decode_fn_e<1, false>(q, closed) : decode_fn_e<0, false>(q, closed);
}
template <int ECN> static const void *checknode_dense_fn(int q, int closed)
{
    if (closed) return q == 16 ? (const void *)checknode_dense_kernel<16, true, ECN> : q == 64 ? (const void *)checknode_dense_kernel<64, true, ECN> : (const void *)checknode_dense_kernel<256, true, ECN>;
    return q == 16 ? (const void *)checknode_dense_kernel<16, false, ECN> : q == 64 ? (const void *)checknode_dense_kernel<64, false, ECN> : (const void *)checknode_dense_kernel<256, false, ECN>;
}
static const void *checknode_fn(int q, int closed, int ecn)
{
    if (ecn == 2) return checknode_dense_fn<2>(q, closed);
    if (ecn == 4) return checknode_dense_fn<4>(q, closed);
    if (ecn) {
        if (closed) return q == 16 ? (const void *)checknode_synd_kernel<16, true> : q == 64 ? (const void *)checknode_synd_kernel<64, true> : (const void *)checknode_synd_kernel<256, true>;
        return q == 16 ? (const void *)checknode_synd_kernel<16, false> : q == 64 ? (const void *)checknode_synd_kernel<64, false> : (const void *)checknode_synd_kernel<256, false>;
    }
    if (closed) return q == 16 ? (const void *)checknode_kernel<16, true> : q == 64 ? (const void *)checknode_kernel<64, true> : (const void *)checknode_kernel<256, true>;
    return q == 16 ? (const void *)checknode_kernel<16, false> : q == 64 ? (const void *)checknode_kernel<64, false> : (const void *)checknode_kernel<256, false>;
}

/* ------------------------------------------------------------------------------------------------
 * context
 * ---------------------------------------------------------------------------------------------- */
/* A channel as the host code uses it, resolved once per call by channel_of(): the intake, the frame layout, how the frame
 * source draws a symbol and which constellation both read. */
enum ChannelId { CH_BPSK, CH_LLR, CH_APSK64, CH_MAPPED, CH_FADED, CH_SPLIT };
struct Channel {
    int rc;                      /* NBGPU_OK, or the refusal of channel_of (the rest is then unset) */
    int kind;                    /* InputKind */
    int fps;                     /* floats per symbol of a frame: q (LLR), 4 (faded: I, Q, rho_I, rho_Q), else points * dims */
    int draws;                   /* frame source: drand48 draws per symbol after the information bits (BPSK, mapped, split: 2 * fps) */
    bool apsk_sigma;             /* sigma = nbgpu_sigma_apsk64(EbN) (every constellation), else nbgpu_sigma(code, EbN) */
    const float *mod_d;          /* constellation [q][2] ([M][2] split) on the device; nullptr for BPSK and LLR */
    const float *mod_h;          /* its host copy ([2][1] = {+1, -1} for BPSK), indexed [sub-image][dims] by the fix-up */
    int fading;                  /* CH_FADED: NBGPU_FADING_SYMBOL or NBGPU_FADING_COMPONENT of the frame source */
    int points, dims;            /* BPSK, mapped, split: a symbol is `points` points of `dims` coordinates (source_awgn_kernel) */
};
static int split_p(const Channel &ch) { return ch.kind == INPUT_SPLIT ? ch.points : 0; }    /* KArgs::split_p */

struct nbgpu_ctx {
    int device;
    cudaStream_t stream, copy_stream;        /* kernels | host<->device copies of the chunked end-to-end path */
    cudaEvent_t ev0, ev1, ev_t0, ev_t1, ev_h2d[1];
    int per_sm;
    nbgpu_params p;
    KArgs k;
    int N, M, E, q, logq, dc_max;
    int max_batch, nslots, grid;
    uint64_t code_hash;  /* code_hash() of the code the context was created for: the frame source takes no other */
    int *row_ptr_h;  /* host copies for get_state */
    int *inv_h;
    /* device buffers */
    int *d_row_ptr, *d_col, *d_step_ptr, *d_isolated;
    uint32_t *d_cninfo, *d_einfo;
    uint8_t *d_cfg; float *d_ctov_dense;
    uint8_t *d_hval, *d_rotin, *d_rotout, *d_img, *d_inv;
    float *d_mod;                            /* the 64-APSK table (q = 64), used by every *_apsk64 call */
    float mod_h[128];                        /* host copy of the 64-APSK table, for the frame source's fix-up */
    float *d_map;                            /* the bound table of the mapped calls (nbgpu_set_constellation), NULL until bound */
    float map_h[512];                        /* host copy of the bound table, for the frame source's fix-up */
    float *d_split;                          /* the split table (nbgpu_set_split_constellation), [M][2] with M <= 16; NULL until bound */
    float split_h[32];                       /* its host copy */
    int split_p;                             /* its points per symbol */
    float *d_app; uint8_t *d_ctov; uint8_t *d_dec;
    float *d_in; size_t in_capacity;
    int *d_decide, *d_synd, *d_iters, *d_frame_slot, *d_slot_frame;
    unsigned *d_queue, *d_slow, *d_ready, *d_fault;
    unsigned *h_ready;                       /* pinned: cumulative frame counts of the input pieces of decode_host */
    int resident_B;
    Channel resident;                        /* channel of the batch in d_in (kept when nbgpu_set_constellation drops it) */
    int mapped_dropped;                      /* InputKind (mapped, faded, split) of the resident batch that re-binding its table dropped, else 0 */
    int *d_punct;                            /* puncturing pattern (nbgpu_set_puncturing): k.pmap [N], then the transmitted variables [k.nt] */
    int punct_dropped;                       /* 1: binding a pattern dropped the resident or generated batch */
    /* soft output: the armed kind and the device buffers live in k.soft_*; soft_made = the kind the last decode launch
     * produced for its soft_B frames (NBGPU_SOFT_NONE once re-armed or a new batch replaced it); decoded = a decode
     * kernel was launched at least once */
    int soft_made, soft_B, decoded;
    /* device frame source (nbldpc_source.cuh), set up by the first nbgpu_source_frames* call */
    struct {
        int ready, nlevels, B;
        int *d_level_ptr, *d_row_order, *d_ut_ptr, *d_ut_col, *d_perm, *d_bit_errors;
        uint8_t *d_ut_val, *d_piv, *d_mulimg, *d_divimg, *d_cw, *d_flag_img;
        unsigned *d_flag_count, *d_flags, *d_patch_idx;
        float *d_patch_val;
        uint64_t D;              /* draws per frame of the generated batch (depends on the channel) */
        double margin;
        long fixups;
        int state;               /* 0: nothing generated, or d_in overwritten by an upload since; 1: batch generated, not decoded;
                                    2: generated batch decoded */
    } src;
    long launches;
    float last_ms;
    char err[512];
};

static void ctx_err(nbgpu_ctx *c, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    char buf[512];
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (c) snprintf(c->err, sizeof c->err, "%s", buf);
    nbgpu_set_global_error("%s", buf);
}
#define CK(ctx, call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { ctx_err(ctx, "%s failed: %s", #call, cudaGetErrorString(e_)); return NBGPU_ECUDA; } } while (0)

extern "C" void nbgpu_destroy(nbgpu_ctx *c);
static void source_teardown(nbgpu_ctx *c);
extern "C" const char *nbgpu_last_error(const nbgpu_ctx *ctx) { return ctx ? ctx->err : nbgpu_get_global_error(); }

extern "C" int nbgpu_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

template <typename T> static int upload(nbgpu_ctx *c, T **dst, const std::vector<T> &src)
{
    CK(c, cudaMalloc((void **)dst, src.size() * sizeof(T) + 16));
    CK(c, cudaMemcpy(*dst, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice));
    return NBGPU_OK;
}

static int align_up(int x, int a) { return (x + a - 1) / a * a; }

/* FNV-1a over sizes, graph, coefficients and the GF tables (ADDGF follows from BINGF): two codes with the same hash
 * encode, decode and score frames alike, wherever they were loaded */
static uint64_t code_hash(const nbgpu_code *code)
{
    uint64_t h = 1469598103934665603ull;
    auto mix = [&h](uint64_t x) { h = (h ^ x) * 1099511628211ull; };
    mix(code->N); mix(code->M); mix(code->q); mix(code->E);
    for (int e = 0; e < code->E; e++) mix(((uint64_t)code->col[e] << 16) ^ (uint64_t)code->val[e]);
    for (int m = 0; m <= code->M; m++) mix(code->row_ptr[m]);
    for (int i = 0; i < code->q * code->logq; i++) mix((uint32_t)code->bingf[i]);
    for (int i = 0; i < code->q * code->q; i++) mix(((uint64_t)(uint32_t)code->mulgf[i] << 32) | (uint32_t)code->divgf[i]);
    return h;
}

static int scr_words(int q) { return q == 16 ? QTraits<16>::SCR_WORDS : q == 64 ? QTraits<64>::SCR_WORDS : QTraits<256>::SCR_WORDS; }

/* shared-memory plan for nw warps of cpw check nodes each (see KArgs) */
static void plan_smem(KArgs &k, int nw, int cpw)
{
    k.nw = nw; k.cpw = cpw; k.cap = nw * cpw;
    k.L = 4 * k.dc_max - 6; if (k.L < 2) k.L = 2;
    int off = 0;
    k.off_tab = off; off += 512;
    k.off_misc = off; off += align_up((2 + 3 * k.F) * 4, 16);
    /* per-warp small area: ES mask (q = 256) | meta | edge words | list lengths */
    int wa = 0;
    k.wa_mask = wa; wa += (k.q > 64 && k.ecn == 0) ? 8 * 32 * 4 : 0;
    k.wa_meta = wa; wa += cpw * 16;
    k.wa_einfo = wa; wa += cpw * k.dc_max * 4;
    k.wa_len = wa; wa += k.ecn == 0 ? align_up(cpw * k.L, 4) : 0;
    k.wa_bytes = align_up(wa, 16);
    k.off_wa = off; off += nw * k.wa_bytes;
    k.lstride = align_up(5 * k.n_m, 4);
    if (((k.lstride / 4) & 1) == 0) k.lstride += 4;       /* odd number of words: consecutive lists start in different banks */
    const int s3 = NE * k.q * 4;                                             /* clean rows */
    const int sq = NE * scr_words(k.q) * 4 + NE * 36 * 4;                     /* selection queues + 36 unused words per edge */
    if (k.ecn == 0) {
        /* per-warp lists: U[cpw][dc_max] | R[cpw][L - dc_max] as one array, each list {n_m f32 | n_m u8}.  Scratch aliases them. */
        const int ub = cpw * k.dc_max * k.lstride, rb = cpw * (k.L - k.dc_max) * k.lstride;
        k.wb_U = 0; k.wb_R = ub;
        k.wb_scr1 = align_up(ub, 16);                      /* phase-1 scratch over the R lists */
        int total = std::max(ub + rb, k.wb_scr1 + s3 + sq);
        if (s3 <= ub && k.dc_min >= 3) k.wb_scr3 = 0;      /* phase-3 rows over the input lists, dead after phase 2 ... */
        else { k.wb_scr3 = align_up(total, 16); total = k.wb_scr3 + s3; }   /* ... unless they do not fit, or degree 2: the output lists ARE input lists */
        k.wb_bytes = align_up(total, 16);
    } else if (k.ecn == 2 || k.ecn == 4) {
        /* sum-product and Min-Max check nodes, per warp: U rows [dc_max][q] (the intake and the soft output's selection use the same
         * bytes as scratch, before and after the passes) | permutation row [q] (Min-Max: also the row operand of a convolution;
         * its rows enter the check domain straight into the U rows) */
        k.wb_U = 0; k.wb_R = 0; k.wb_scr1 = 0; k.wb_scr3 = 0;
        k.sw_rows = align_up(std::max(k.dc_max * k.q * 4, sq), 16);
        k.wb_bytes = align_up(k.sw_rows + k.q * 4, 16);
    } else {
        /* syndrome check node: CTA-wide configuration table, then per warp: lists | grouped keys (aliased by the selection scratch of
         * phase 1, dead once the node's lists are written) | grouped configuration indices | histograms / output rows | group starts | perm */
        k.off_cfg = off; off += align_up(k.S * (k.dc_max + 1), 16);
        int wb2 = 0;
        k.wb_U = wb2; k.wb_R = wb2; wb2 += align_up(k.dc_max * k.lstride, 16);
        k.wb_scr1 = wb2; k.wb_scr3 = wb2;
        /* region B: selection scratch | saturation histograms | grouped keys (+16: the rank loop reads up to 3 keys past a group) | 4 output rows */
        k.sw_key = wb2; wb2 += std::max(std::max(align_up(4 * k.S + 16, 16), align_up(sq, 16)), std::max(4096, ((k.dc_max + 1) / 2) * 1024));
        k.sw_pay = wb2; wb2 += align_up(2 * k.S, 16);                                    /* payloads of the grouped keys */
        k.sw_gf = wb2; wb2 += align_up(k.S, 16);                                         /* symbols by configuration; with the next 1024 bytes: sorted payloads (2 S <= S + 1024) */
        k.sw_hist = wb2; wb2 += 1024;                                                    /* symbol histogram / cursors */
        k.sw_cand = wb2; wb2 += k.dc_max * NB_SYND_CAND * 4;
        k.sw_rows = wb2; wb2 += align_up(4 * k.S, 16);                                   /* region A: syndromes by configuration, then the sorted keys */
        k.sw_M = wb2; wb2 += align_up(257 * 2, 16);
        k.sw_perm = wb2; wb2 += NB_SYND_PERM_BYTES;
        k.wb_bytes = align_up(wb2, 16);
    }
    k.off_wb = off; off += nw * k.wb_bytes;
    k.smem_bytes = off + 256;            /* slack: select_edges may read one key row past a sentinel row */
}

extern "C" int nbgpu_create(nbgpu_ctx **out, const nbgpu_code *code, const nbgpu_params *p, int device, int max_batch)
{
    if (!out) { ctx_err(NULL, "nbgpu_create: NULL output pointer"); return NBGPU_EINVAL; }
    *out = NULL;
    if (!code || !p) { ctx_err(NULL, "nbgpu_create: NULL argument"); return NBGPU_EINVAL; }
    if (code->q != 16 && code->q != 64 && code->q != 256) { ctx_err(NULL, "GF(%d): kernels exist for GF(16), GF(64) and GF(256) only (init.c:431-435)", code->q); return NBGPU_EINVAL; }
    if (p->ecn_kind < 0 || p->ecn_kind > 4 || p->ecn_kind == 3) { ctx_err(NULL, "ecn_kind %d unknown (0 = CheckPassLogEMS, 1 = syndrome_ems, 2 = sum-product, 4 = Min-Max)", p->ecn_kind); return NBGPU_EINVAL; }
    if (p->n_m < 5 || p->n_m > 32 || p->n_m > code->q) { ctx_err(NULL, "n_m=%d unsupported: need 5 <= n_m <= min(q,32) (ElementaryStep reads row 4, bubble_decoder.c:457)", p->n_m); return NBGPU_EINVAL; }
    if (p->nb_iter_max < 2) { ctx_err(NULL, "nb_iter_max must be >= 2 (nb_iter_max-1 passes are run, NB_LDPC.c:314)"); return NBGPU_EINVAL; }
    if (p->nb_oper < 1) { ctx_err(NULL, "nb_oper must be >= 1"); return NBGPU_EINVAL; }
    if (code->dc_min < 2 || code->dc_max > 16) { ctx_err(NULL, "check degree range [%d,%d] unsupported (2..16)", code->dc_min, code->dc_max); return NBGPU_EINVAL; }
    if (max_batch < 1) { ctx_err(NULL, "max_batch must be >= 1"); return NBGPU_EINVAL; }
    for (int m = 0; m < code->M; m++)
        for (int e = code->row_ptr[m]; e < code->row_ptr[m + 1]; e++)
            for (int e2 = e + 1; e2 < code->row_ptr[m + 1]; e2++)
                if (code->col[e] == code->col[e2]) { ctx_err(NULL, "check node %d references variable %d twice", m, code->col[e]); return NBGPU_EINVAL; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); ctx_err(NULL, "no CUDA device available (this library has no CPU fallback)"); return NBGPU_ECUDA; }
    if (device < 0 || device >= ndev) { ctx_err(NULL, "device %d out of range (0..%d)", device, ndev - 1); return NBGPU_EINVAL; }
    nbgpu_ctx *c = (nbgpu_ctx *)calloc(1, sizeof *c);
    if (!c) { ctx_err(NULL, "out of memory"); return NBGPU_ENOMEM; }
    /* from here on every failure goes through nbgpu_destroy(c), which releases whatever was created so far */
#define CKF(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { ctx_err(NULL, "%s failed: %s", #call, cudaGetErrorString(e_)); cudaGetLastError(); nbgpu_destroy(c); return NBGPU_ECUDA; } } while (0)
    c->device = device; c->p = *p; c->max_batch = max_batch;
    c->N = code->N; c->M = code->M; c->E = code->E; c->q = code->q; c->logq = code->logq; c->dc_max = code->dc_max;
    c->code_hash = code_hash(code);
    CKF(cudaSetDevice(device));
    cudaDeviceProp prop;
    CKF(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) { ctx_err(c, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor); nbgpu_destroy(c); return NBGPU_ECUDA; }
    CKF(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    CKF(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    CKF(cudaEventCreateWithFlags(&c->ev_h2d[0], cudaEventDisableTiming));
    CKF(cudaEventCreate(&c->ev0)); CKF(cudaEventCreate(&c->ev1));
    CKF(cudaEventCreate(&c->ev_t0)); CKF(cudaEventCreate(&c->ev_t1));

    const int q = code->q, E = code->E, N = code->N, M = code->M;
    KArgs &k = c->k;
    memset(&k, 0, sizeof k);
    k.N = N; k.M = M; k.E = E; k.q = q; k.logq = code->logq; k.dc_max = code->dc_max; k.dc_min = code->dc_min;
    k.n_m = p->n_m; k.nb_oper = p->nb_oper; k.passes = p->nb_iter_max - 1; k.early_stop = p->early_stop;
    k.nb_iter_max = p->nb_iter_max; k.offset = p->offset;
    k.rec_stride = align_up(((4 * p->n_m + 7) & ~7) + 8 + p->n_m, 16);     /* llr[n_m] f32 | pad to 8 | sat f32, stp i32 | sym[n_m] u8 */

    /* tables */
    std::vector<uint8_t> hval(E), last(E, 0), rotin((size_t)q * q), rotout((size_t)q * q), img(q), inv(q);
    std::vector<int> lastedge(N, -1), isolated;
    for (int e = 0; e < E; e++) { hval[e] = (uint8_t)code->val[e]; lastedge[code->col[e]] = e; }
    for (int n = 0; n < N; n++) { if (lastedge[n] >= 0) last[lastedge[n]] = 1; else isolated.push_back(n); }
    for (int s = 0; s < q; s++) { img[s] = (uint8_t)code->img[s]; inv[s] = (uint8_t)code->inv[s]; }
    for (int h = 0; h < q; h++) for (int s = 0; s < q; s++) {
        rotin[(size_t)h * q + s] = (uint8_t)code->img[code->mulgf[s * q + h]];                     /* MULGF[sym][h] */
        rotout[(size_t)h * q + s] = h ? (uint8_t)code->divgf[code->inv[s] * q + h] : 0;            /* DIVGF[sym][h] */
    }
    c->row_ptr_h = (int *)malloc(sizeof(int) * (M + 1)); memcpy(c->row_ptr_h, code->row_ptr, sizeof(int) * (M + 1));
    c->inv_h = (int *)malloc(sizeof(int) * q); memcpy(c->inv_h, code->inv, sizeof(int) * q);

    /* syndrome-based check node: parameters of NB_LDPC.c:185-201 (commented out there), validated so that every index the
     * reference would use stays inside its arrays (d_1 = 40 of the commented code overruns the n_m-wide rows) */
    std::vector<uint8_t> cfg8;
    k.ecn = p->ecn_kind;
    if (p->ecn_kind == 1) {
        const int dc = code->dc_max, nm1 = p->n_m - 1;
        const int d1 = p->d1 > 0 ? p->d1 : nm1, d2 = p->d2 > 0 ? p->d2 : std::min(15, nm1), d3 = p->d3 > 0 ? p->d3 : std::min(5, nm1);
        const int trunc = p->cfg_trunc > 0 ? p->cfg_trunc : 1000, n_cv = p->n_cv > 0 ? p->n_cv : p->nb_oper;
        if (p->border != 0 && p->border != 4) { ctx_err(c, "border=%d: syndrome_ems fixes border = 4 (syndrome_decoder.c:56)", p->border); nbgpu_destroy(c); return NBGPU_EINVAL; }
        if (code->dc_min != dc || dc < 4 || dc > 8) { ctx_err(c, "syndrome_ems needs a check-regular code with 4 <= dc <= 8 (dc = %d..%d)", code->dc_min, dc); nbgpu_destroy(c); return NBGPU_EINVAL; }
        if (d1 > nm1 || d2 > nm1 || d3 > nm1 || p->n_m < 3) { ctx_err(c, "deviations (%d,%d,%d) exceed the list length n_m-1 = %d", d1, d2, d3, nm1); nbgpu_destroy(c); return NBGPU_EINVAL; }
        int size = 0;
        int *tab = nbgpu_build_config_table(dc, d1, d2, d3, trunc, &size);
        if (!tab || size < 1) { ctx_err(c, "cannot build the configuration table"); nbgpu_destroy(c); return NBGPU_ENOMEM; }
        if (size > NB_SYND_MAX) { free(tab); ctx_err(c, "%d configurations: at most %d are supported (use cfg_trunc)", size, NB_SYND_MAX); nbgpu_destroy(c); return NBGPU_EINVAL; }
        cfg8.assign((size_t)size * (dc + 1), 0);          /* table [size][dc], then per configuration the edges it does not deviate on */
        for (int d = 0; d < dc; d++) {
            int kept = 0;
            for (int i = 0; i < size; i++) {
                cfg8[(size_t)i * dc + d] = (uint8_t)tab[(size_t)i * dc + d];
                if (tab[(size_t)i * dc + d] == 0) { kept++; cfg8[(size_t)size * dc + i] |= (uint8_t)(1u << d); }
            }
            if (n_cv - 1 + 3 * d >= kept) { free(tab); ctx_err(c, "n_cv=%d: edge %d has only %d decorrelated syndromes, index %d is read (syndrome_decoder.c:195)", n_cv, d, kept, n_cv - 1 + 3 * d); nbgpu_destroy(c); return NBGPU_EINVAL; }
        }
        free(tab);
        k.S = size; k.Spad = align_up(size, 32); k.n_cv = n_cv;
    }

    /* launch geometry: shared-memory budget -> warps per CTA, check nodes per warp, frames per group, step schedule */
    if (N >= (1 << 20) || E >= (1 << 24)) { ctx_err(c, "code too large for the packed graph tables (N < 2^20, E < 2^24)"); nbgpu_destroy(c); return NBGPU_EINVAL; }
    const int budget = getenv("NBGPU_SMEM_KB") ? atoi(getenv("NBGPU_SMEM_KB")) * 1024 : (CTAS_PER_SM > 1 ? (228 * 1024) / CTAS_PER_SM - 1024 : 216 * 1024);
    k.F = 1;
    int nw = getenv("NBGPU_WARPS") ? atoi(getenv("NBGPU_WARPS")) : NT_MAX / 32, cpw = getenv("NBGPU_CPW") ? atoi(getenv("NBGPU_CPW")) : 8;
    /* the register budget is what limits residency: keep all NT_MAX/32 warps and shrink the tile before dropping warps */
    if (p->ecn_kind != 0 && !getenv("NBGPU_CPW")) cpw = 4;       /* nodes of a tile are processed one after the other: no shared-memory cost */
    nw = std::max(1, std::min(nw, (p->ecn_kind != 0 ? NT_SYND : NT_MAX) / 32)); cpw = std::max(1, std::min(cpw, 32));
    if (p->cns_per_step > 0) cpw = std::max(1, std::min(cpw, (p->cns_per_step + nw - 1) / nw));
    if (p->ecn_kind == 0 && !getenv("NBGPU_WARPS") && !getenv("NBGPU_CPW") && p->cns_per_step <= 0) {
        /* Pick (warps, nodes per warp) among the plans that fit.  Cost of one tile in instructions: phases 1/3 grow with the
         * tile (dc edges per node, heavier for larger q), the ElementarySteps do not as long as the tile's 4 task slots per
         * node fit the 32 lanes -- so high-degree codes want bigger tiles even at the price of fewer warps, whose
         * latency-hiding value is the measured `eff` (Ahmed_64800_R34_GF16: (12,4) 196, (10,5) 209, (8,6) 217, (6,8) 208 Mbit/s;
         * KN N64800_K48600_GF256: (8,4) 213, (12,3) 205). */
        static const double eff[13] = { 0, .2, .35, .5, .6, .7, .77, .84, .90, .925, .95, .975, 1.0 };
        const double w_edge = k.q == 16 ? 175.0 : k.q == 64 ? 330.0 : 660.0;
        const int dc = code->dc_max, rounds = dc - 2 + (dc > 4 ? 1 : 0);
        const double es_round = 70.0 * (k.n_m + 5) * (k.q > 64 ? 1.1 : 1.0);   /* ~n_m+5 pops of ~70 issue slots; q = 256 keeps its mask in shared memory */
        double best = -1.0; int bnw = 0, bcpw = 0;
        for (int w = NT_MAX / 32; w >= 1; w -= (w > 6 || best < 0 ? 2 : 6))          /* 12, 10, 8, 6 -- smaller only if nothing fits */
            for (int cw = 8; cw >= 1; cw--) {
                plan_smem(k, w, cw);
                if (k.smem_bytes > budget) continue;
                const double tile = cw * dc * w_edge + std::max(rounds, 1) * es_round * ((cw * 4 + 31) / 32);
                const double score = eff[w] * cw / tile;
                if (score > best * 1.0001) { best = score; bnw = w; bcpw = cw; }
            }
        if (bnw) { nw = bnw; cpw = bcpw; }
        plan_smem(k, nw, cpw);
    } else
    for (;;) {
        plan_smem(k, nw, cpw);
        if (k.smem_bytes <= budget) break;
        if (p->ecn_kind != 0) { if (nw > 1) nw--; else break; }
        else if (cpw > 4) cpw--; else if (nw > 8) nw -= 2; else if (cpw > 1) cpw--; else if (nw > 1) nw--; else break;
    }
    if (k.smem_bytes > 227 * 1024) { ctx_err(c, "decoder working set does not fit in shared memory (%d bytes for one warp)", k.smem_bytes); nbgpu_destroy(c); return NBGPU_EINVAL; }
    const int G = k.cap;
    /* choose F: smallest number of frames per group that keeps the steps reasonably full */
    int bestF = 1; double bestU = -1;
    nbgpu_schedule sched; memset(&sched, 0, sizeof sched);
    for (int F = 1; F <= G && F <= 64; F *= 2) {
        if (p->frames_per_cta > 0) F = std::min(p->frames_per_cta, G);
        nbgpu_schedule s2;
        nbgpu_build_schedule(code, G / F > 0 ? G / F : 1, &s2);
        const double util = (double)M * F / ((double)s2.nsteps * G);
        nbgpu_free_schedule(&s2);
        if (util > bestU * 1.10) { bestU = util; bestF = F; }
        if (p->frames_per_cta > 0 || util > 0.85) break;
    }
    k.F = bestF < 1 ? 1 : bestF;
    if (k.F > G) k.F = G;
    plan_smem(k, nw, cpw);
    nbgpu_build_schedule(code, G / k.F > 0 ? G / k.F : 1, &sched);
    k.nsteps = sched.nsteps;
    std::vector<int> step_ptr(sched.step_ptr, sched.step_ptr + sched.nsteps + 1);
    std::vector<uint32_t> cninfo(M), einfo(E);
    for (int i = 0; i < M; i++) {
        const int m = sched.order[i];
        cninfo[i] = (uint32_t)code->row_ptr[m] | ((uint32_t)(code->row_ptr[m + 1] - code->row_ptr[m]) << 24);
    }
    for (int e = 0; e < E; e++) einfo[e] = (uint32_t)code->col[e] | ((uint32_t)code->val[e] << 20) | ((uint32_t)last[e] << 28);
    nbgpu_free_schedule(&sched);
    std::vector<int> row_ptr(code->row_ptr, code->row_ptr + M + 1), col(code->col, code->col + E);
    if (isolated.empty()) isolated.push_back(0), k.n_isolated = 0; else k.n_isolated = (int)isolated.size();
    /* multiplication/division by the edge coefficient: closed exponent form when the tables have it */
    k.gf_closed = 1;
    for (int a2 = 0; a2 < q && k.gf_closed; a2++) for (int b2 = 1; b2 < q; b2++) {
        const int mul = a2 ? ((a2 + b2 - 2) % (q - 1)) + 1 : 0, dv = a2 ? ((a2 - b2 + (q - 1)) % (q - 1)) + 1 : 0;
        if (code->mulgf[a2 * q + b2] != mul || code->divgf[a2 * q + b2] != dv) { k.gf_closed = 0; break; }
    }
    if (getenv("NBGPU_GF_TABLES")) k.gf_closed = 0;

    int rc;
    if ((rc = upload(c, &c->d_row_ptr, row_ptr)) || (rc = upload(c, &c->d_col, col)) || (rc = upload(c, &c->d_cninfo, cninfo)) ||
        (rc = upload(c, &c->d_einfo, einfo)) ||
        (rc = upload(c, &c->d_step_ptr, step_ptr)) || (rc = upload(c, &c->d_isolated, isolated)) || (rc = upload(c, &c->d_hval, hval)) ||
        (rc = upload(c, &c->d_rotin, rotin)) || (rc = upload(c, &c->d_rotout, rotout)) ||
        (rc = upload(c, &c->d_img, img)) || (rc = upload(c, &c->d_inv, inv))) { nbgpu_destroy(c); return rc; }
    if (p->ecn_kind == 1) { if ((rc = upload(c, &c->d_cfg, cfg8))) { nbgpu_destroy(c); return rc; } k.cfg = c->d_cfg; }
    if (q == 64) {                                       /* 64-APSK intake (ModelChannel_AWGN_64): the constellation, built on the host */
        nbgpu_apsk64_table(c->mod_h);
        if ((rc = upload(c, &c->d_mod, std::vector<float>(c->mod_h, c->mod_h + 128)))) { nbgpu_destroy(c); return rc; }
    }
    k.row_ptr = c->d_row_ptr; k.col = c->d_col; k.cninfo = c->d_cninfo; k.einfo = c->d_einfo; k.step_ptr = c->d_step_ptr; k.isolated = c->d_isolated;
    k.hval = c->d_hval; k.rotin = c->d_rotin; k.rotout = c->d_rotout; k.img = c->d_img; k.inv = c->d_inv;

    /* persistent grid: one CTA per SM */
    const void *fn = decode_fn(q, k.gf_closed, k.ecn, false);
    /* opt in to the device maximum, not to this context's size: the attribute is per function and several contexts with
     * different geometries may share a kernel */
    CKF(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)prop.sharedMemPerBlockOptin));
    CKF(cudaFuncSetAttribute(decode_fn(q, k.gf_closed, k.ecn, true), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)prop.sharedMemPerBlockOptin));
    const void *fn2 = checknode_fn(q, k.gf_closed, k.ecn);
    CKF(cudaFuncSetAttribute(fn2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)prop.sharedMemPerBlockOptin));
    int per_sm = 0;
    CKF(cudaOccupancyMaxActiveBlocksPerMultiprocessorWithFlags(&per_sm, fn, k.nw * 32, k.smem_bytes, cudaOccupancyDefault));
    if (per_sm < 1) { ctx_err(c, "decode kernel does not fit on an SM (smem %d bytes)", k.smem_bytes); nbgpu_destroy(c); return NBGPU_ECUDA; }
    if (getenv("NBGPU_CTAS_PER_SM")) per_sm = std::min(per_sm, atoi(getenv("NBGPU_CTAS_PER_SM")));
    c->per_sm = per_sm;
    c->grid = prop.multiProcessorCount * per_sm;
    const int groups = (max_batch + k.F - 1) / k.F;
    if (c->grid > groups) c->grid = groups;
    c->nslots = c->grid * k.F;

    CKF(cudaMalloc((void **)&c->d_app, (size_t)c->nslots * N * q * sizeof(float)));
    CKF(cudaMalloc((void **)&c->d_ctov, (p->ecn_kind != 0 ? 0 : (size_t)c->nslots * E * k.rec_stride) + 512));
    if (p->ecn_kind != 0) CKF(cudaMalloc((void **)&c->d_ctov_dense, (size_t)c->nslots * E * q * sizeof(float)));
    CKF(cudaMalloc((void **)&c->d_dec, (size_t)c->nslots * N));
    CKF(cudaMemset(c->d_dec, 0, (size_t)c->nslots * N));
    CKF(cudaMalloc((void **)&c->d_decide, (size_t)max_batch * N * sizeof(int)));
    CKF(cudaMalloc((void **)&c->d_synd, (size_t)max_batch * sizeof(int)));
    CKF(cudaMalloc((void **)&c->d_iters, (size_t)max_batch * sizeof(int)));
    CKF(cudaMalloc((void **)&c->d_frame_slot, (size_t)max_batch * sizeof(int)));
    CKF(cudaMalloc((void **)&c->d_slot_frame, (size_t)c->nslots * sizeof(int)));
    CKF(cudaMemset(c->d_slot_frame, 0xff, (size_t)c->nslots * sizeof(int)));
    CKF(cudaMalloc((void **)&c->d_queue, 8 * sizeof(unsigned)));       /* [0] work queue, [4] slow-path counter, [5] frames copied in so far (decode_host), [6] fault flag */
    c->d_slow = c->d_queue + 4; c->d_ready = c->d_queue + 5; c->d_fault = c->d_queue + 6;
    CKF(cudaMemset(c->d_queue, 0, 8 * sizeof(unsigned)));
    CKF(cudaHostAlloc((void **)&c->h_ready, 16 * sizeof(unsigned), cudaHostAllocDefault));
    k.app = c->d_app; k.ctov = c->d_ctov; k.dec = c->d_dec; k.ctov_dense = c->d_ctov_dense;
    k.out_decide = c->d_decide; k.out_synd = c->d_synd; k.out_iters = c->d_iters;
    k.frame_slot = c->d_frame_slot; k.slot_frame = c->d_slot_frame; k.queue = c->d_queue; k.slow_counter = c->d_slow;
    k.ready = nullptr; k.fault = c->d_fault;
    k.pmap = nullptr; k.nt = N;
    /* the memsets above ran on the legacy stream, the kernels run on c->stream (non-blocking): order them once, here */
    CKF(cudaDeviceSynchronize());
#undef CKF
    *out = c;
    return NBGPU_OK;
}

extern "C" void nbgpu_destroy(nbgpu_ctx *c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    void *bufs[] = { c->d_cfg, c->d_ctov_dense, c->d_row_ptr, c->d_col, c->d_cninfo, c->d_einfo, c->d_step_ptr, c->d_isolated, c->d_hval, c->d_rotin,
                     c->d_rotout, c->d_img, c->d_inv, c->d_mod, c->d_map, c->d_split, c->d_app, c->d_ctov, c->d_dec, c->d_in, c->d_decide, c->d_synd,
                     c->d_iters, c->d_frame_slot, c->d_slot_frame, c->d_queue, c->k.soft_llr, c->k.soft_sym, c->d_punct };
    for (void *b : bufs) if (b) cudaFree(b);
    if (c->h_ready) cudaFreeHost(c->h_ready);
    source_teardown(c);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->ev_t0) cudaEventDestroy(c->ev_t0);
    if (c->ev_t1) cudaEventDestroy(c->ev_t1);
    if (c->ev_h2d[0]) cudaEventDestroy(c->ev_h2d[0]);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->stream) cudaStreamDestroy(c->stream);
    free(c->row_ptr_h); free(c->inv_h);
    free(c);
}

static int ensure_input(nbgpu_ctx *c, size_t floats)
{
    if (floats <= c->in_capacity) return NBGPU_OK;
    if (c->d_in) cudaFree(c->d_in);
    c->d_in = NULL; c->in_capacity = 0;
    CK(c, cudaMalloc((void **)&c->d_in, floats * sizeof(float)));
    c->in_capacity = floats;
    return NBGPU_OK;
}

/* Channel `id` of context c.  Refusals: the 64-APSK channel on another field than GF(64) (NBGPU_EINVAL), a mapped or faded
 * channel with no bound table or a split channel with no split table (NBGPU_ESTATE), a fading value other than NBGPU_FADING_SYMBOL / _COMPONENT (NBGPU_EINVAL).
 * fading only sets the frame source's draws: the faded intake reads the amplitudes from the frames. */
static Channel channel_of(nbgpu_ctx *c, ChannelId id, int fading = NBGPU_FADING_SYMBOL)
{
    Channel ch = {};
    if (!c) { ctx_err(NULL, "NULL context"); ch.rc = NBGPU_EINVAL; }
    else if (id == CH_APSK64 && c->q != 64) {
        ctx_err(c, "64-APSK intake (ModelChannel_AWGN_64, channel.c:112) maps one GF(64) symbol to one constellation point: q = %d", c->q);
        ch.rc = NBGPU_EINVAL;
    } else if (id == CH_FADED && fading != NBGPU_FADING_SYMBOL && fading != NBGPU_FADING_COMPONENT) {
        ctx_err(c, "faded channel: fading %d (NBGPU_FADING_SYMBOL = 1, NBGPU_FADING_COMPONENT = 2)", fading);
        ch.rc = NBGPU_EINVAL;
    } else if ((id == CH_MAPPED || id == CH_FADED) && !c->d_map) {
        ctx_err(c, "mapped channel: no constellation bound to this context (call nbgpu_set_constellation first)");
        ch.rc = NBGPU_ESTATE;
    } else if (id == CH_SPLIT && !c->d_split) {
        ctx_err(c, "split channel: no split constellation bound to this context (call nbgpu_set_split_constellation first)");
        ch.rc = NBGPU_ESTATE;
    } else if (id == CH_LLR) ch = { NBGPU_OK, INPUT_LLR, c->q };
    else if (id == CH_FADED)          /* the mapped draws, then one amplitude draw (SYMBOL) or two (COMPONENT) */
        ch = { NBGPU_OK, INPUT_FADED, 4, 4 + fading, true, c->d_map, c->map_h, fading };
    else {                            /* two draws per sample: channel.c:56-57 (BPSK, one point per bit), channel.c:234-263 */
        static const float bpsk[2] = { 1.0f, -1.0f };
        if (id == CH_BPSK) ch = { NBGPU_OK, INPUT_BPSK, 0, 0, false, nullptr, bpsk, 0, c->logq, 1 };
        else if (id == CH_SPLIT) ch = { NBGPU_OK, INPUT_SPLIT, 0, 0, true, c->d_split, c->split_h, 0, c->split_p, 2 };
        else ch = { NBGPU_OK, INPUT_MAPPED, 0, 0, true, id == CH_APSK64 ? c->d_mod : c->d_map, id == CH_APSK64 ? c->mod_h : c->map_h, 0, 1, 2 };
        ch.fps = ch.points * ch.dims;
        ch.draws = 2 * ch.fps;
    }
    return ch;
}

static double den_of(float sigma) { return 2.0 * (double)(float)(sigma * sigma); }     /* 2.0*SQR(sigma), channel.c:73 / :280 */

/* B frames of channel ch are now in d_in, uploaded by the caller or made by the frame source */
static void set_resident(nbgpu_ctx *c, const Channel &ch, int B, float sigma, bool generated)
{
    c->k.den = den_of(sigma);
    c->resident_B = B; c->resident = ch; c->mapped_dropped = 0; c->punct_dropped = 0;
    c->src.state = generated ? 1 : 0;
    if (generated) c->src.B = B;
}

static int upload_common(nbgpu_ctx *c, const Channel &ch, const float *src, float sigma, int B)
{
    if (ch.rc) return ch.rc;
    if (!src) { ctx_err(c, "NULL argument"); return NBGPU_EINVAL; }
    c->soft_made = NBGPU_SOFT_NONE;                           /* even a rejected batch: the caller moved on from the last one */
    if (B < 1 || B > c->max_batch) { ctx_err(c, "B=%d outside 1..max_batch=%d", B, c->max_batch); return NBGPU_EINVAL; }
    CK(c, cudaSetDevice(c->device));
    const size_t per_frame = (size_t)c->k.nt * ch.fps;        /* transmitted symbols only */
    int rc = ensure_input(c, per_frame * B);                  /* grows on demand: dense-LLR batches are q/log2(q) times larger */
    if (rc) return rc;
    CK(c, cudaMemcpyAsync(c->d_in, src, per_frame * B * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    set_resident(c, ch, B, sigma, false);
    return NBGPU_OK;
}

extern "C" int nbgpu_upload_noisy(nbgpu_ctx *c, const float *noisy, float sigma, int B)
{
    return upload_common(c, channel_of(c, CH_BPSK), noisy, sigma, B);
}
extern "C" int nbgpu_upload_llr(nbgpu_ctx *c, const float *llr, int B)
{
    return upload_common(c, channel_of(c, CH_LLR), llr, 0.0f, B);
}
extern "C" int nbgpu_upload_apsk64(nbgpu_ctx *c, const float *noisy, float sigma, int B)
{
    return upload_common(c, channel_of(c, CH_APSK64), noisy, sigma, B);
}
extern "C" int nbgpu_upload_mapped(nbgpu_ctx *c, const float *noisy, float sigma, int B)
{
    return upload_common(c, channel_of(c, CH_MAPPED), noisy, sigma, B);
}
extern "C" int nbgpu_upload_faded(nbgpu_ctx *c, const float *rx, float sigma, int B)
{
    return upload_common(c, channel_of(c, CH_FADED), rx, sigma, B);
}
extern "C" int nbgpu_upload_split(nbgpu_ctx *c, const float *noisy, float sigma, int B)
{
    return upload_common(c, channel_of(c, CH_SPLIT), noisy, sigma, B);
}

extern "C" int nbgpu_set_constellation(nbgpu_ctx *c, const float *mod)
{
    if (!c || !mod) { ctx_err(c, "nbgpu_set_constellation: NULL argument"); return NBGPU_EINVAL; }
    for (int i = 0; i < 2 * c->q; i++)
        if (!std::isfinite(mod[i])) { ctx_err(c, "nbgpu_set_constellation: mod[%d][%d] = %g is not finite", i / 2, i % 2, (double)mod[i]); return NBGPU_EINVAL; }
    CK(c, cudaSetDevice(c->device));
    if (!c->d_map) CK(c, cudaMalloc((void **)&c->d_map, 2 * (size_t)c->q * sizeof(float)));
    /* stream order: a launch in flight still reads the old table */
    CK(c, cudaMemcpyAsync(c->d_map, mod, 2 * (size_t)c->q * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    memcpy(c->map_h, mod, 2 * (size_t)c->q * sizeof(float));
    if (c->resident_B > 0 && c->resident.mod_d == c->d_map) {
        /* its samples were made for the old table: decoding them on the new one would be wrong (they stay downloadable) */
        c->resident_B = 0; c->mapped_dropped = c->resident.kind; c->soft_made = NBGPU_SOFT_NONE;
    }
    return NBGPU_OK;
}

extern "C" int nbgpu_set_split_constellation(nbgpu_ctx *c, int points, const float *mod)
{
    if (!c || !mod) { ctx_err(c, "nbgpu_set_split_constellation: NULL argument"); return NBGPU_EINVAL; }
    if (!nbgpu_split_points_ok(c->logq, points)) {
        ctx_err(c, "nbgpu_set_split_constellation: %d points per GF(%d) symbol (need P >= 2 dividing log2 q = %d)", points, c->q, c->logq);
        return NBGPU_EINVAL;
    }
    const int M = 1 << (c->logq / points);
    for (int i = 0; i < 2 * M; i++)
        if (!std::isfinite(mod[i])) { ctx_err(c, "nbgpu_set_split_constellation: mod[%d][%d] = %g is not finite", i / 2, i % 2, (double)mod[i]); return NBGPU_EINVAL; }
    CK(c, cudaSetDevice(c->device));
    if (!c->d_split) CK(c, cudaMalloc((void **)&c->d_split, sizeof c->split_h));
    /* stream order: a launch in flight still reads the old table */
    CK(c, cudaMemcpyAsync(c->d_split, mod, 2 * (size_t)M * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    memcpy(c->split_h, mod, 2 * (size_t)M * sizeof(float));
    c->split_p = points;
    if (c->resident_B > 0 && c->resident.mod_d == c->d_split) {
        /* made for the old table (or another P): dropped, as nbgpu_set_constellation drops a mapped batch */
        c->resident_B = 0; c->mapped_dropped = c->resident.kind; c->soft_made = NBGPU_SOFT_NONE;
    }
    return NBGPU_OK;
}

extern "C" int nbgpu_set_puncturing(nbgpu_ctx *c, int p, const int *vars)
{
    if (!c) { ctx_err(NULL, "nbgpu_set_puncturing: NULL context"); return NBGPU_EINVAL; }
    const int N = c->N;
    std::vector<int> map(2 * (size_t)N);
    const int nt = nbgpu_puncture_map(N, p, vars, map.data());
    if (nt < 0) { ctx_err(c, "nbgpu_set_puncturing: %s", nbgpu_get_global_error()); return nt; }
    for (int n = 0; n < N; n++) if (map[n] >= 0) map[N + map[n]] = n;
    CK(c, cudaSetDevice(c->device));
    if (p > 0) {
        if (!c->d_punct) CK(c, cudaMalloc((void **)&c->d_punct, 2 * (size_t)N * sizeof(int)));
        /* stream order: a launch in flight still reads the old pattern */
        CK(c, cudaMemcpyAsync(c->d_punct, map.data(), ((size_t)N + nt) * sizeof(int), cudaMemcpyHostToDevice, c->stream));
        CK(c, cudaStreamSynchronize(c->stream));
    }
    c->k.pmap = p > 0 ? c->d_punct : nullptr;
    c->k.nt = nt;
    /* frames of the old layout: neither decodable nor downloadable under the new one */
    if (c->resident_B > 0 || c->src.state || c->mapped_dropped) c->punct_dropped = 1;
    c->resident_B = 0; c->mapped_dropped = 0; c->soft_made = NBGPU_SOFT_NONE;
    return NBGPU_OK;
}

extern "C" int nbgpu_run(nbgpu_ctx *c)
{
    if (c && c->resident_B < 1 && c->punct_dropped) {
        ctx_err(c, "nbgpu_run: the batch was dropped when nbgpu_set_puncturing bound a new pattern");
        return NBGPU_ESTATE;
    }
    if (c && c->resident_B < 1 && c->mapped_dropped == INPUT_SPLIT) {
        ctx_err(c, "nbgpu_run: the split batch was dropped when nbgpu_set_split_constellation bound a new table");
        return NBGPU_ESTATE;
    }
    if (c && c->resident_B < 1 && c->mapped_dropped) {
        ctx_err(c, "nbgpu_run: the %s batch was dropped when nbgpu_set_constellation bound a new table", c->mapped_dropped == INPUT_FADED ? "faded" : "mapped");
        return NBGPU_ESTATE;
    }
    if (!c || c->resident_B < 1) { ctx_err(c, "nbgpu_run: no resident batch (call nbgpu_upload_* first)"); return NBGPU_EINVAL; }
    CK(c, cudaSetDevice(c->device));
    KArgs k = c->k;
    k.B = c->resident_B; k.input_kind = c->resident.kind; k.in = c->d_in; k.mod = c->resident.mod_d; k.split_p = split_p(c->resident);
    CK(c, cudaMemsetAsync(c->d_queue, 0, sizeof(unsigned), c->stream));
    const int groups = (k.B + k.F - 1) / k.F;
    const int grid = std::min(c->grid, groups);
    CK(c, cudaEventRecord(c->ev0, c->stream));
    {
        void *args[] = { (void *)&k };
        c->soft_made = NBGPU_SOFT_NONE;
        CK(c, cudaLaunchKernel(decode_fn(c->q, k.gf_closed, k.ecn, k.soft_kind != NBGPU_SOFT_NONE), dim3(grid), dim3(k.nw * 32), args, k.smem_bytes, c->stream));
    }
    CK(c, cudaGetLastError());
    CK(c, cudaEventRecord(c->ev1, c->stream));
    c->launches += 1;
    c->decoded = 1; c->soft_made = k.soft_kind; c->soft_B = k.B;
    if (c->src.state == 1) c->src.state = 2;
    return NBGPU_OK;
}

extern "C" int nbgpu_sync(nbgpu_ctx *c)
{
    if (!c) return NBGPU_EINVAL;
    CK(c, cudaSetDevice(c->device));
    CK(c, cudaStreamSynchronize(c->stream));
    return NBGPU_OK;
}

extern "C" int nbgpu_last_kernel_ms(nbgpu_ctx *c, float *ms)
{
    if (!c || !ms) return NBGPU_EINVAL;
    CK(c, cudaEventSynchronize(c->ev1));
    CK(c, cudaEventElapsedTime(ms, c->ev0, c->ev1));
    return NBGPU_OK;
}
extern "C" long nbgpu_launch_count(const nbgpu_ctx *c) { return c ? c->launches : 0; }

extern "C" int nbgpu_timer_begin(nbgpu_ctx *c)
{
    if (!c) return NBGPU_EINVAL;
    CK(c, cudaSetDevice(c->device));
    CK(c, cudaEventRecord(c->ev_t0, c->stream));
    return NBGPU_OK;
}
extern "C" int nbgpu_timer_end(nbgpu_ctx *c, float *ms)
{
    if (!c || !ms) return NBGPU_EINVAL;
    CK(c, cudaSetDevice(c->device));
    CK(c, cudaEventRecord(c->ev_t1, c->stream));
    CK(c, cudaEventSynchronize(c->ev_t1));
    CK(c, cudaEventElapsedTime(ms, c->ev_t0, c->ev_t1));
    return NBGPU_OK;
}
extern "C" int nbgpu_host_register(void *ptr, size_t bytes)
{
    cudaError_t e = cudaHostRegister(ptr, bytes, cudaHostRegisterDefault);
    if (e != cudaSuccess) { cudaGetLastError(); ctx_err(NULL, "cudaHostRegister failed: %s", cudaGetErrorString(e)); return NBGPU_ECUDA; }
    return NBGPU_OK;
}
extern "C" int nbgpu_host_unregister(void *ptr)
{
    cudaError_t e = cudaHostUnregister(ptr);
    if (e != cudaSuccess) { cudaGetLastError(); ctx_err(NULL, "cudaHostUnregister failed: %s", cudaGetErrorString(e)); return NBGPU_ECUDA; }
    return NBGPU_OK;
}
extern "C" int nbgpu_geometry(const nbgpu_ctx *c, int *geo)
{
    if (!c || !geo) return NBGPU_EINVAL;
    geo[0] = c->grid; geo[1] = c->k.F; geo[2] = c->k.cap / (c->k.F > 0 ? c->k.F : 1); geo[3] = c->k.nsteps;
    geo[4] = c->k.smem_bytes; geo[5] = c->nslots; geo[6] = c->k.nw; geo[7] = c->k.cpw;
    return NBGPU_OK;
}
extern "C" long nbgpu_slow_selects(nbgpu_ctx *c)
{
    if (!c) return -1;
    unsigned v = 0;
    if (cudaSetDevice(c->device) != cudaSuccess || cudaStreamSynchronize(c->stream) != cudaSuccess ||
        cudaMemcpy(&v, c->d_slow, sizeof v, cudaMemcpyDeviceToHost) != cudaSuccess) { cudaGetLastError(); return -1; }
    return (long)v;
}

extern "C" int nbgpu_download(nbgpu_ctx *c, int *decide, int *synd, int *iters)
{
    if (!c || c->resident_B < 1) { ctx_err(c, "nbgpu_download: nothing decoded"); return NBGPU_EINVAL; }
    CK(c, cudaSetDevice(c->device));
    const int B = c->resident_B;
    if (decide) CK(c, cudaMemcpyAsync(decide, c->d_decide, (size_t)B * c->N * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    if (synd) CK(c, cudaMemcpyAsync(synd, c->d_synd, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    if (iters) CK(c, cudaMemcpyAsync(iters, c->d_iters, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return NBGPU_OK;
}

/* End-to-end decode of B frames from HOST buffers.  A large batch is decoded by ONE launch that starts as soon as the first
 * wave of frames is on the device: the input goes over in up to 8 pieces on the copy stream, every piece followed by a 4-byte
 * copy of the number of frames now present (d_ready), and a CTA that takes frames [base, base+F) from the work queue first
 * waits until d_ready covers them (decode_kernel, a.ready).  Copies run ~25x faster than the decoder consumes frames, so
 * only the first groups ever wait and the H2D time disappears behind the kernel -- without cutting the batch into several
 * launches, whose starts and tails cost as much as the copies they hid (measured: 340 ms either way against 327.6 ms for the
 * kernel alone on config 5).  Small batches take the plain upload / run / download path (and keep their state readable). */
static int decode_host(nbgpu_ctx *c, const Channel &ch, const float *src, float sigma, int B, int *decide, int *synd, int *iters)
{
    if (ch.rc) return ch.rc;
    if (!src) { ctx_err(c, "NULL argument"); return NBGPU_EINVAL; }
    c->soft_made = NBGPU_SOFT_NONE;
    if (B < 1 || B > c->max_batch) { ctx_err(c, "B=%d outside 1..max_batch=%d", B, c->max_batch); return NBGPU_EINVAL; }
    const int wave = c->grid * c->k.F;
    if (B < 2 * wave || getenv("NBGPU_NO_CHUNKS")) {
        int rc = upload_common(c, ch, src, sigma, B);
        if (rc || (rc = nbgpu_run(c)) || (rc = nbgpu_download(c, decide, synd, iters))) return rc;
        return NBGPU_OK;
    }
    CK(c, cudaSetDevice(c->device));
    const size_t per_frame = (size_t)c->k.nt * ch.fps;        /* transmitted symbols only */
    int rc = ensure_input(c, per_frame * B);
    if (rc) return rc;
    set_resident(c, ch, B, sigma, false);
    /* pieces: one wave first, the rest in up to 7 equal runs of whole waves */
    int lo[9], np = 1;
    {
        const int W = B / wave, rest = W - 1, runs = rest < 7 ? rest : 7;
        lo[0] = 0; lo[1] = wave;
        for (int i = 1; i <= runs; i++) lo[1 + i] = wave + (int)((long)rest * i / runs) * wave;
        np = 1 + runs;
        lo[np] = B;
    }
    for (int i = 0; i < np; i++) c->h_ready[i] = (unsigned)lo[i + 1];
    CK(c, cudaStreamSynchronize(c->stream));                  /* earlier work on the buffers is done */
    CK(c, cudaMemsetAsync(c->d_ready, 0, 2 * sizeof(unsigned), c->copy_stream));         /* d_ready, d_fault */
    CK(c, cudaEventRecord(c->ev_h2d[0], c->copy_stream));
    for (int i = 0; i < np; i++) {
        CK(c, cudaMemcpyAsync(c->d_in + per_frame * lo[i], src + per_frame * lo[i], per_frame * (lo[i + 1] - lo[i]) * sizeof(float),
                              cudaMemcpyHostToDevice, c->copy_stream));
        CK(c, cudaMemcpyAsync(c->d_ready, c->h_ready + i, sizeof(unsigned), cudaMemcpyHostToDevice, c->copy_stream));
    }
    KArgs k = c->k;
    k.B = B; k.input_kind = ch.kind; k.in = c->d_in; k.mod = ch.mod_d; k.split_p = split_p(ch); k.ready = c->d_ready;
    CK(c, cudaMemsetAsync(c->d_queue, 0, sizeof(unsigned), c->stream));
    CK(c, cudaStreamWaitEvent(c->stream, c->ev_h2d[0], 0));   /* the counter starts at zero */
    CK(c, cudaEventRecord(c->ev0, c->stream));
    {
        void *args[] = { (void *)&k };
        CK(c, cudaLaunchKernel(decode_fn(c->q, k.gf_closed, k.ecn, k.soft_kind != NBGPU_SOFT_NONE), dim3(c->grid), dim3(k.nw * 32), args, k.smem_bytes, c->stream));
    }
    CK(c, cudaGetLastError());
    CK(c, cudaEventRecord(c->ev1, c->stream));
    c->launches += 1;
    c->decoded = 1;
    unsigned fault = 0;
    if (decide) CK(c, cudaMemcpyAsync(decide, c->d_decide, (size_t)B * c->N * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    if (synd) CK(c, cudaMemcpyAsync(synd, c->d_synd, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    if (iters) CK(c, cudaMemcpyAsync(iters, c->d_iters, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaMemcpyAsync(&fault, c->d_fault, sizeof fault, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->copy_stream));
    CK(c, cudaStreamSynchronize(c->stream));
    if (fault) { ctx_err(c, "decode: the kernel gave up waiting for its input frames (host-to-device copy did not arrive)"); return NBGPU_ECUDA; }
    c->soft_made = k.soft_kind; c->soft_B = B;                /* only a launch that saw all its frames leaves soft output */
    return NBGPU_OK;
}

extern "C" int nbgpu_decode_noisy(nbgpu_ctx *c, const float *noisy, float sigma, int B, int *decide, int *synd, int *iters)
{
    return decode_host(c, channel_of(c, CH_BPSK), noisy, sigma, B, decide, synd, iters);
}
extern "C" int nbgpu_decode_llr(nbgpu_ctx *c, const float *llr, int B, int *decide, int *synd, int *iters)
{
    return decode_host(c, channel_of(c, CH_LLR), llr, 0.0f, B, decide, synd, iters);
}
extern "C" int nbgpu_decode_apsk64(nbgpu_ctx *c, const float *noisy, float sigma, int B, int *decide, int *synd, int *iters)
{
    return decode_host(c, channel_of(c, CH_APSK64), noisy, sigma, B, decide, synd, iters);
}
extern "C" int nbgpu_decode_mapped(nbgpu_ctx *c, const float *noisy, float sigma, int B, int *decide, int *synd, int *iters)
{
    return decode_host(c, channel_of(c, CH_MAPPED), noisy, sigma, B, decide, synd, iters);
}
extern "C" int nbgpu_decode_faded(nbgpu_ctx *c, const float *rx, float sigma, int B, int *decide, int *synd, int *iters)
{
    return decode_host(c, channel_of(c, CH_FADED), rx, sigma, B, decide, synd, iters);
}
extern "C" int nbgpu_decode_split(nbgpu_ctx *c, const float *noisy, float sigma, int B, int *decide, int *synd, int *iters)
{
    return decode_host(c, channel_of(c, CH_SPLIT), noisy, sigma, B, decide, synd, iters);
}


/* ------------------------------------------------------------------------------------------------
 * Frame source on the device (SURVEY.md 8f.1; kernels in nbldpc_source.cuh)
 * ---------------------------------------------------------------------------------------------- */
#define SRC_FLAG_CAP (1u << 20)

static void source_teardown(nbgpu_ctx *c)
{
    void *sbufs[] = { c->src.d_level_ptr, c->src.d_row_order, c->src.d_ut_ptr, c->src.d_ut_col, c->src.d_perm, c->src.d_bit_errors, c->src.d_ut_val,
                      c->src.d_piv, c->src.d_mulimg, c->src.d_divimg, c->src.d_cw, c->src.d_flag_count, c->src.d_flags, c->src.d_patch_idx,
                      c->src.d_patch_val, c->src.d_flag_img };
    for (void *b : sbufs) if (b) cudaFree(b);
    const double margin = c->src.margin;
    memset(&c->src, 0, sizeof c->src);
    c->src.margin = margin;
}

static int source_setup(nbgpu_ctx *c, nbgpu_code *code)
{
    if (c->N > 48 * 1024) { ctx_err(c, "frame source: N=%d symbols do not fit the encoder's shared memory", c->N); return NBGPU_EINVAL; }
    int rc = nbgpu_code_prepare_encoder(code);
    if (rc) { ctx_err(c, "%s", nbgpu_get_global_error()); return rc; }
    const int N = c->N, M = c->M, q = c->q;
    /* level of a row = 1 + the deepest parity symbol it reads: rows of one level are independent (tools.c:244 runs m = M-1..0) */
    std::vector<int> level(M, 0), order(M), lptr;
    int depth = 0;
    for (int m = M - 1; m >= 0; m--) {
        int l = 0;
        for (int k = code->ut_ptr[m]; k < code->ut_ptr[m + 1]; k++) { const int n = code->ut_col[k]; if (n < M) l = std::max(l, level[n] + 1); }
        level[m] = l; depth = std::max(depth, l + 1);
    }
    lptr.assign(depth + 1, 0);
    for (int m = 0; m < M; m++) lptr[level[m] + 1]++;
    for (int l = 0; l < depth; l++) lptr[l + 1] += lptr[l];
    { std::vector<int> pos(lptr.begin(), lptr.end() - 1); for (int m = M - 1; m >= 0; m--) order[pos[level[m]]++] = m; }
    const int nnz = code->ut_ptr[M];
    std::vector<int> utp(code->ut_ptr, code->ut_ptr + M + 1), utc(code->ut_col, code->ut_col + nnz), perm(code->perm, code->perm + N);
    std::vector<uint8_t> utv(nnz + 1), piv(M), mulimg((size_t)q * q), divimg((size_t)q * q);
    for (int k = 0; k < nnz; k++) utv[k] = (uint8_t)code->ut_val[k];
    for (int m = 0; m < M; m++) piv[m] = (uint8_t)code->piv_col[m];
    for (int h = 0; h < q; h++)
        for (int x = 0; x < q; x++) {                       /* x = binary image of the operand symbol */
            const int sx = code->inv[x];
            mulimg[(size_t)h * q + x] = (uint8_t)code->img[code->mulgf[h * q + sx]];
            divimg[(size_t)h * q + x] = h ? (uint8_t)code->img[code->divgf[sx * q + h]] : 0;
        }
    if ((rc = upload(c, &c->src.d_level_ptr, lptr)) || (rc = upload(c, &c->src.d_row_order, order)) || (rc = upload(c, &c->src.d_ut_ptr, utp)) ||
        (rc = upload(c, &c->src.d_ut_col, utc)) || (rc = upload(c, &c->src.d_perm, perm)) || (rc = upload(c, &c->src.d_ut_val, utv)) ||
        (rc = upload(c, &c->src.d_piv, piv)) || (rc = upload(c, &c->src.d_mulimg, mulimg)) || (rc = upload(c, &c->src.d_divimg, divimg))) return rc;
    CK(c, cudaMalloc((void **)&c->src.d_cw, (size_t)c->max_batch * N));
    CK(c, cudaMalloc((void **)&c->src.d_bit_errors, (size_t)c->max_batch * sizeof(int)));
    CK(c, cudaMalloc((void **)&c->src.d_flag_count, sizeof(unsigned)));
    CK(c, cudaMalloc((void **)&c->src.d_flags, SRC_FLAG_CAP * sizeof(unsigned)));
    CK(c, cudaMalloc((void **)&c->src.d_patch_idx, SRC_FLAG_CAP * sizeof(unsigned)));
    CK(c, cudaMalloc((void **)&c->src.d_patch_val, SRC_FLAG_CAP * sizeof(float)));
    CK(c, cudaMalloc((void **)&c->src.d_flag_img, SRC_FLAG_CAP));
    uint64_t mul[48], add[48], m_ = SRC_A, a_ = SRC_C;
    for (int j = 0; j < 48; j++) { mul[j] = m_; add[j] = a_; a_ = ((m_ + 1) * a_) & SRC_MASK; m_ = (m_ * m_) & SRC_MASK; }
    CK(c, cudaMemcpyToSymbol(c_src_mul, mul, sizeof mul));
    CK(c, cudaMemcpyToSymbol(c_src_add, add, sizeof add));
    c->src.nlevels = depth;
    if (c->src.margin == 0.0) c->src.margin = 0x1p-46;
    c->src.ready = 1;
    return NBGPU_OK;
}

static SrcArgs source_args(nbgpu_ctx *c, const nbgpu_code *code, int B)
{
    SrcArgs a;
    memset(&a, 0, sizeof a);
    a.N = c->N; a.M = c->M; a.K = c->N - c->M; a.q = c->q; a.logq = c->logq; a.B = B; a.D = c->src.D; a.nlevels = c->src.nlevels;
    a.level_ptr = c->src.d_level_ptr; a.row_order = c->src.d_row_order; a.ut_ptr = c->src.d_ut_ptr; a.ut_col = c->src.d_ut_col;
    a.ut_val = c->src.d_ut_val; a.piv = c->src.d_piv; a.perm = c->src.d_perm; a.mulimg = c->src.d_mulimg; a.divimg = c->src.d_divimg;
    a.img = c->d_img; a.cw = c->src.d_cw; a.noisy = c->d_in; a.margin = c->src.margin;
    a.flag_count = c->src.d_flag_count; a.flags = c->src.d_flags; a.flag_cap = SRC_FLAG_CAP;
    a.decide = c->d_decide; a.bit_errors = c->src.d_bit_errors;
    a.flag_img = c->src.d_flag_img;
    a.Nt = c->k.nt; a.tvar = c->k.pmap ? c->d_punct + c->N : nullptr;
    (void)code;
    return a;
}

extern "C" int nbgpu_source_set_margin(nbgpu_ctx *c, double margin)
{
    if (!c || !(margin > 0.0) || margin > 0x1p-20) { ctx_err(c, "nbgpu_source_set_margin: margin must be in (0, 2^-20]"); return NBGPU_EINVAL; }
    c->src.margin = margin;
    return NBGPU_OK;
}

/* Body of every nbgpu_source_frames* call: B frames of channel `id` (fading: CH_FADED only).  The channel fixes the draws per
 * frame D, sigma, the noise kernel and the host recomputation of a flagged sample (faded: of a whole symbol); encoder, flag
 * read-back and patch are shared. */
static int source_generate(nbgpu_ctx *c, nbgpu_code *code, const nbgpu_rng *origin, uint64_t frame0, int B, float EbN, ChannelId id,
                           int fading = NBGPU_FADING_SYMBOL)
{
    if (!c || !code || !origin) { ctx_err(c, "NULL argument"); return NBGPU_EINVAL; }
    const Channel ch = channel_of(c, id, fading);
    if (ch.rc) return ch.rc;
    /* the frames are encoded with the code's tables but decoded and scored with the context's: only the context's own code
     * (by content, so that a copy loaded per thread or rank qualifies) is accepted, and the encoder tables built from it
     * stay valid for every later call */
    if (code_hash(code) != c->code_hash) { ctx_err(c, "nbgpu_source_frames: the code is not the one the decoder was created for"); return NBGPU_EINVAL; }
    c->soft_made = NBGPU_SOFT_NONE;
    if (B < 1 || B > c->max_batch) { ctx_err(c, "B=%d outside 1..max_batch=%d", B, c->max_batch); return NBGPU_EINVAL; }
    const int Nt = c->k.nt;                                   /* transmitted symbols (N without a puncturing pattern) */
    if ((double)B * Nt * ch.fps >= 2147483648.0) {
        if (Nt == c->N) ctx_err(c, "frame source: B*N*%d must stay below 2^31", ch.fps);
        else ctx_err(c, "frame source: B*Nt*%d must stay below 2^31 (Nt = %d transmitted symbols)", ch.fps, Nt);
        return NBGPU_EINVAL;
    }
    CK(c, cudaSetDevice(c->device));
    int rc;
    if (!c->src.ready && (rc = source_setup(c, code))) { source_teardown(c); return rc; }
    if ((rc = ensure_input(c, (size_t)Nt * ch.fps * B))) return rc;
    const uint64_t koff = (uint64_t)(c->N - c->M) * c->logq;   /* information-bit draws, tools.c:124-136 */
    const int S = ch.draws;
    const uint64_t D = koff + (uint64_t)Nt * S;
    const float sigma = ch.apsk_sigma ? nbgpu_sigma_apsk64(EbN) : Nt < c->N ? nbgpu_sigma_punctured(code, c->N - Nt, EbN) : nbgpu_sigma(code, EbN);
    nbgpu_rng r = *origin;
    nbgpu_rng_skip(&r, frame0 * D);
    c->src.D = D;
    SrcArgs a = source_args(c, code, B);
    a.x0 = r.x; a.sigma = sigma; a.mod = ch.mod_d; a.points = ch.points;
    if (ch.kind == INPUT_FADED) a.flag_cap = SRC_FLAG_CAP / 4;  /* a flagged symbol takes four patch entries */
    CK(c, cudaMemsetAsync(c->src.d_flag_count, 0, sizeof(unsigned), c->stream));
    source_encode_kernel<<<B, 256, c->N, c->stream>>>(a);
    const unsigned blocks = (unsigned)(((long long)B * Nt + 255) / 256);              /* one thread per transmitted symbol */
    if (ch.fading == NBGPU_FADING_COMPONENT) source_faded_kernel<NBGPU_FADING_COMPONENT><<<blocks, 256, 0, c->stream>>>(a);
    else if (ch.fading == NBGPU_FADING_SYMBOL) source_faded_kernel<NBGPU_FADING_SYMBOL><<<blocks, 256, 0, c->stream>>>(a);
    else if (ch.dims == 2) source_awgn_kernel<2><<<blocks, 256, 0, c->stream>>>(a);
    else source_awgn_kernel<1><<<blocks, 256, 0, c->stream>>>(a);
    CK(c, cudaGetLastError());
    c->launches += 2;
    unsigned nflag = 0;
    CK(c, cudaMemcpyAsync(&nflag, c->src.d_flag_count, sizeof nflag, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    if (nflag > a.flag_cap) { ctx_err(c, "frame source: %u %s flagged for host recomputation (capacity %u); margin too wide", nflag, ch.kind == INPUT_FADED ? "symbols" : "samples", a.flag_cap); return NBGPU_EINVAL; }
    c->src.fixups = nflag;
    if (nflag) {
        /* samples whose f32 rounding could depend on the last bits of log/cos: recompute with the host's libm (channel.c:59,
         * channel.c:234-263).  In the BPSK, mapped and split channels a flag is sample s of a frame, which reads the draws
         * 2s, 2s+1 after the information bits, and the sub-image of its point.  A faded flag is symbol n of the batch and its
         * image: its S draws, its four values.  Under puncturing, s and n count transmitted symbols only. */
        std::vector<unsigned> idx(nflag), pidx;
        std::vector<float> val(nflag);
        std::vector<uint8_t> img(nflag);
        CK(c, cudaMemcpy(idx.data(), c->src.d_flags, nflag * sizeof(unsigned), cudaMemcpyDeviceToHost));
        CK(c, cudaMemcpy(img.data(), c->src.d_flag_img, nflag, cudaMemcpyDeviceToHost));
        if (ch.kind == INPUT_FADED) {
            pidx.resize(4 * (size_t)nflag); val.resize(4 * (size_t)nflag);
            for (unsigned i = 0; i < nflag; i++) {
                const uint64_t f = idx[i] / Nt, t = idx[i] % Nt;
                nbgpu_rng g; g.x = a.x0;
                nbgpu_rng_skip(&g, f * D + koff + (uint64_t)S * t);
                float dr[6];
                for (int j = 0; j < S; j++) dr[j] = (float)nbgpu_rng_drand48(&g);
                nbgpu_faded_sample(sigma, ch.mod_h + 2 * img[i], dr, ch.fading, &val[4 * (size_t)i]);
                for (int j = 0; j < 4; j++) pidx[4 * (size_t)i + j] = 4 * idx[i] + j;
            }
            idx.swap(pidx);
            nflag *= 4;
        } else {
            const uint64_t per = (uint64_t)Nt * ch.fps;
            for (unsigned i = 0; i < nflag; i++) {
                const uint64_t f = idx[i] / per, s = idx[i] % per;
                nbgpu_rng g; g.x = a.x0;
                nbgpu_rng_skip(&g, f * D + koff + 2 * s);
                const float u = (float)nbgpu_rng_drand48(&g), v = (float)nbgpu_rng_drand48(&g);
                val[i] = nbgpu_mapped_sample(sigma, ch.mod_h[ch.dims * img[i] + s % ch.dims], u, v);
            }
        }
        CK(c, cudaMemcpyAsync(c->src.d_patch_idx, idx.data(), nflag * sizeof(unsigned), cudaMemcpyHostToDevice, c->stream));
        CK(c, cudaMemcpyAsync(c->src.d_patch_val, val.data(), nflag * sizeof(float), cudaMemcpyHostToDevice, c->stream));
        source_patch_kernel<<<(nflag + 255) / 256, 256, 0, c->stream>>>(c->d_in, c->src.d_patch_idx, c->src.d_patch_val, (int)nflag);
        CK(c, cudaGetLastError());
        CK(c, cudaStreamSynchronize(c->stream));                 /* idx/val are stack-scoped */
        c->launches += 1;
    }
    set_resident(c, ch, B, sigma, true);
    return NBGPU_OK;
}

extern "C" int nbgpu_source_frames(nbgpu_ctx *c, nbgpu_code *code, const nbgpu_rng *origin, uint64_t frame0, int B, float EbN)
{
    return source_generate(c, code, origin, frame0, B, EbN, CH_BPSK);
}
extern "C" int nbgpu_source_frames_apsk64(nbgpu_ctx *c, nbgpu_code *code, const nbgpu_rng *origin, uint64_t frame0, int B, float EbN)
{
    return source_generate(c, code, origin, frame0, B, EbN, CH_APSK64);
}
extern "C" int nbgpu_source_frames_mapped(nbgpu_ctx *c, nbgpu_code *code, const nbgpu_rng *origin, uint64_t frame0, int B, float EbN)
{
    return source_generate(c, code, origin, frame0, B, EbN, CH_MAPPED);
}
extern "C" int nbgpu_source_frames_faded(nbgpu_ctx *c, nbgpu_code *code, const nbgpu_rng *origin, uint64_t frame0, int B, float EbN, int fading)
{
    return source_generate(c, code, origin, frame0, B, EbN, CH_FADED, fading);
}
extern "C" int nbgpu_source_frames_split(nbgpu_ctx *c, nbgpu_code *code, const nbgpu_rng *origin, uint64_t frame0, int B, float EbN)
{
    return source_generate(c, code, origin, frame0, B, EbN, CH_SPLIT);
}

extern "C" long nbgpu_source_fixups(const nbgpu_ctx *c) { return c ? c->src.fixups : 0; }

extern "C" int nbgpu_source_download(nbgpu_ctx *c, int *codeword, float *noisy)
{
    if (!c || !c->src.ready || c->src.B < 1) { ctx_err(c, "nbgpu_source_download: no generated batch"); return NBGPU_EINVAL; }
    if (c->punct_dropped) { ctx_err(c, "nbgpu_source_download: the generated batch was dropped when nbgpu_set_puncturing bound a new pattern"); return NBGPU_ESTATE; }
    if (c->src.state == 0) { ctx_err(c, "nbgpu_source_download: the generated batch was replaced by an uploaded batch"); return NBGPU_ESTATE; }
    CK(c, cudaSetDevice(c->device));
    const int B = c->src.B;
    if (codeword) {
        std::vector<uint8_t> cw((size_t)B * c->N);
        CK(c, cudaMemcpyAsync(cw.data(), c->src.d_cw, cw.size(), cudaMemcpyDeviceToHost, c->stream));
        CK(c, cudaStreamSynchronize(c->stream));
        for (size_t i = 0; i < cw.size(); i++) codeword[i] = c->inv_h[cw[i]];
    }
    if (noisy) {
        CK(c, cudaMemcpyAsync(noisy, c->d_in, (size_t)B * c->k.nt * c->resident.fps * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
        CK(c, cudaStreamSynchronize(c->stream));
    }
    return NBGPU_OK;
}

extern "C" int nbgpu_source_results(nbgpu_ctx *c, int *bit_errors, int *synd, int *iters)
{
    if (c && c->src.B > 0 && c->punct_dropped) {
        ctx_err(c, "nbgpu_source_results: the generated batch was dropped when nbgpu_set_puncturing bound a new pattern");
        return NBGPU_ESTATE;
    }
    if (!c || !c->src.ready || c->src.B < 1 || c->resident_B != c->src.B) { ctx_err(c, "nbgpu_source_results: no generated batch"); return NBGPU_EINVAL; }
    if (c->src.state != 2) { ctx_err(c, "nbgpu_source_results: the generated batch %s", c->src.state == 1 ? "has not been decoded (call nbgpu_run)" : "was replaced by an uploaded batch"); return NBGPU_ESTATE; }
    CK(c, cudaSetDevice(c->device));
    const int B = c->src.B;
    SrcArgs a = source_args(c, NULL, B);
    source_errors_kernel<<<B, 256, 0, c->stream>>>(a);
    CK(c, cudaGetLastError());
    c->launches += 1;
    if (bit_errors) CK(c, cudaMemcpyAsync(bit_errors, c->src.d_bit_errors, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    if (synd) CK(c, cudaMemcpyAsync(synd, c->d_synd, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    if (iters) CK(c, cudaMemcpyAsync(iters, c->d_iters, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return NBGPU_OK;
}

extern "C" int nbgpu_get_state(nbgpu_ctx *c, int frame, float *APP, float *CtoV)
{
    if (!c || frame < 0 || frame >= c->resident_B) { ctx_err(c, "nbgpu_get_state: frame %d not in the last batch", frame); return NBGPU_EINVAL; }
    CK(c, cudaSetDevice(c->device));
    CK(c, cudaStreamSynchronize(c->stream));
    int slot = -1, owner = -1;
    CK(c, cudaMemcpy(&slot, c->d_frame_slot + frame, sizeof(int), cudaMemcpyDeviceToHost));
    if (slot < 0 || slot >= c->nslots) { ctx_err(c, "frame %d has no slot", frame); return NBGPU_ESTATE; }
    CK(c, cudaMemcpy(&owner, c->d_slot_frame + slot, sizeof(int), cudaMemcpyDeviceToHost));
    if (owner != frame) { ctx_err(c, "state of frame %d was overwritten by frame %d (batch larger than the resident slots)", frame, owner); return NBGPU_ESTATE; }
    const int N = c->N, q = c->q, E = c->E, n_m = c->p.n_m, rs = c->k.rec_stride;
    if (APP) CK(c, cudaMemcpy(APP, c->d_app + (size_t)slot * N * q, (size_t)N * q * sizeof(float), cudaMemcpyDeviceToHost));
    if (CtoV && c->k.ecn != 0) {
        CK(c, cudaMemcpy(CtoV, c->d_ctov_dense + (size_t)slot * E * q, (size_t)E * q * sizeof(float), cudaMemcpyDeviceToHost));
    } else if (CtoV) {
        std::vector<uint8_t> rec((size_t)E * rs);
        CK(c, cudaMemcpy(rec.data(), c->d_ctov + (size_t)slot * E * rs, rec.size(), cudaMemcpyDeviceToHost));
        for (int e = 0; e < E; e++) {
            const uint8_t *r = rec.data() + (size_t)e * rs;
            float sat; int stp;
            const int tail = (4 * n_m + 7) & ~7;
            memcpy(&sat, r + tail, 4); memcpy(&stp, r + tail + 4, 4);
            for (int g = 0; g < q; g++) CtoV[(size_t)e * q + g] = sat;
            for (int kk = 0; kk < stp; kk++) { float l; memcpy(&l, r + 4 * kk, 4); CtoV[(size_t)e * q + r[tail + 8 + kk]] = l; }
        }
    }
    return NBGPU_OK;
}

/* ---- soft output (include/nbldpc_b200.h; computed by soft_output at the end of every group of decode_kernel<..., true>) ---- */
extern "C" int nbgpu_set_soft_output(nbgpu_ctx *c, int kind, int k)
{
    if (!c) { ctx_err(NULL, "nbgpu_set_soft_output: NULL context"); return NBGPU_EINVAL; }
    const int kmax = std::min(c->q, 32);
    const bool ok = kind == NBGPU_SOFT_LIST ? (k >= 1 && k <= kmax) : (kind == NBGPU_SOFT_NONE || kind == NBGPU_SOFT_BITS) && k == 0;
    if (!ok) {
        ctx_err(c, "nbgpu_set_soft_output: kind %d with k = %d (NBGPU_SOFT_LIST: 1 <= k <= min(q, 32) = %d; NBGPU_SOFT_BITS, NBGPU_SOFT_NONE: k = 0)", kind, k, kmax);
        return NBGPU_EINVAL;
    }
    CK(c, cudaSetDevice(c->device));
    CK(c, cudaStreamSynchronize(c->stream));               /* a launch in flight may still write the old buffers */
    KArgs &ka = c->k;
    CK(c, cudaFree(ka.soft_llr)); CK(c, cudaFree(ka.soft_sym));
    ka.soft_llr = nullptr; ka.soft_sym = nullptr; ka.soft_kind = NBGPU_SOFT_NONE; ka.soft_k = 0;
    c->soft_made = NBGPU_SOFT_NONE;
    if (kind == NBGPU_SOFT_NONE) return NBGPU_OK;
    const size_t n = (size_t)c->max_batch * c->N * (kind == NBGPU_SOFT_LIST ? k : c->logq);
    float *llr = nullptr; uint8_t *sym = nullptr;
    cudaError_t e = cudaMalloc((void **)&llr, n * sizeof(float));
    if (e == cudaSuccess && kind == NBGPU_SOFT_LIST) e = cudaMalloc((void **)&sym, n);
    if (e != cudaSuccess) {
        cudaGetLastError();
        cudaFree(llr);
        ctx_err(c, "nbgpu_set_soft_output: %zu bytes of soft output for max_batch = %d frames do not fit on device %d (%s); soft output is off",
                n * (kind == NBGPU_SOFT_LIST ? 5 : 4), c->max_batch, c->device, cudaGetErrorString(e));
        return NBGPU_ENOMEM;
    }
    ka.soft_llr = llr; ka.soft_sym = sym; ka.soft_kind = kind; ka.soft_k = k;
    return NBGPU_OK;
}

static int soft_available(nbgpu_ctx *c, int kind, const char *fn)
{
    if (!c->decoded) { ctx_err(c, "%s: nothing decoded", fn); return NBGPU_EINVAL; }
    if (c->soft_made != kind) {
        ctx_err(c, "%s: the last decode launch left no %s soft output (armed kind %d; re-arming or a new batch invalidates it)", fn,
                kind == NBGPU_SOFT_LIST ? "NBGPU_SOFT_LIST" : "NBGPU_SOFT_BITS", c->k.soft_kind);
        return NBGPU_ESTATE;
    }
    return NBGPU_OK;
}

extern "C" int nbgpu_download_soft_list(nbgpu_ctx *c, float *llr, int *sym)
{
    if (!c || !llr || !sym) { ctx_err(c, "nbgpu_download_soft_list: NULL argument"); return NBGPU_EINVAL; }
    int rc = soft_available(c, NBGPU_SOFT_LIST, "nbgpu_download_soft_list");
    if (rc) return rc;
    CK(c, cudaSetDevice(c->device));
    const size_t n = (size_t)c->soft_B * c->N * c->k.soft_k;
    std::vector<uint8_t> s(n);
    CK(c, cudaMemcpyAsync(llr, c->k.soft_llr, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaMemcpyAsync(s.data(), c->k.soft_sym, n, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    for (size_t i = 0; i < n; i++) sym[i] = s[i];
    return NBGPU_OK;
}

extern "C" int nbgpu_download_soft_bits(nbgpu_ctx *c, float *llr)
{
    if (!c || !llr) { ctx_err(c, "nbgpu_download_soft_bits: NULL argument"); return NBGPU_EINVAL; }
    int rc = soft_available(c, NBGPU_SOFT_BITS, "nbgpu_download_soft_bits");
    if (rc) return rc;
    CK(c, cudaSetDevice(c->device));
    CK(c, cudaMemcpyAsync(llr, c->k.soft_llr, (size_t)c->soft_B * c->N * c->logq * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return NBGPU_OK;
}

/* ---- unit boundaries ----
 * Inputs go to the device with cudaMemcpyAsync on the context's stream (it is a non-blocking stream: work on the legacy
 * stream is not ordered against it); results come back after cudaStreamSynchronize. */
template <typename T> struct DevBuf {
    T *p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
    cudaError_t alloc(size_t n) { return cudaMalloc((void **)&p, (n ? n : 1) * sizeof(T)); }
};

extern "C" int nbgpu_select_nm(nbgpu_ctx *c, const float *rows, float *llr, int *gf, int B)
{
    if (!c || !rows || !llr || !gf || B < 1) { ctx_err(c, "nbgpu_select_nm: bad argument"); return NBGPU_EINVAL; }
    CK(c, cudaSetDevice(c->device));
    const int q = c->q, n_m = c->p.n_m;
    DevBuf<float> d_rows, d_llr; DevBuf<int> d_gf;
    CK(c, d_rows.alloc((size_t)B * q)); CK(c, d_llr.alloc((size_t)B * n_m)); CK(c, d_gf.alloc((size_t)B * n_m));
    CK(c, cudaMemcpyAsync(d_rows.p, rows, (size_t)B * q * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    const int grid = std::min((B + UNIT_NT / 32 - 1) / (UNIT_NT / 32), 148 * 8);
    if (q == 16) select_kernel<16><<<grid, UNIT_NT, 0, c->stream>>>(d_rows.p, d_llr.p, d_gf.p, B, n_m, c->d_slow);
    else if (q == 64) select_kernel<64><<<grid, UNIT_NT, 0, c->stream>>>(d_rows.p, d_llr.p, d_gf.p, B, n_m, c->d_slow);
    else select_kernel<256><<<grid, UNIT_NT, 0, c->stream>>>(d_rows.p, d_llr.p, d_gf.p, B, n_m, c->d_slow);
    CK(c, cudaGetLastError());
    c->launches++;
    CK(c, cudaMemcpyAsync(llr, d_llr.p, (size_t)B * n_m * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaMemcpyAsync(gf, d_gf.p, (size_t)B * n_m * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return NBGPU_OK;
}

extern "C" int nbgpu_elementary_step(nbgpu_ctx *c, const float *in1, const float *in2, const int *idx1, const int *idx2,
                                     float *out, int *idxout, int B)
{
    if (!c || !in1 || !in2 || !idx1 || !idx2 || !out || !idxout || B < 1) { ctx_err(c, "nbgpu_elementary_step: bad argument"); return NBGPU_EINVAL; }
    CK(c, cudaSetDevice(c->device));
    const int n_m = c->p.n_m, q = c->q;
    /* symbols -> binary images + valid lengths (first -1 ends a list, bubble_decoder.c:478) */
    std::vector<uint8_t> s1((size_t)B * n_m), s2((size_t)B * n_m);
    std::vector<int> l1(B), l2(B);
    std::vector<uint8_t> img(q);
    CK(c, cudaMemcpy(img.data(), c->d_img, q, cudaMemcpyDeviceToHost));
    for (int b = 0; b < B; b++) {
        int a = n_m, d = n_m;
        for (int k = n_m - 1; k >= 0; k--) { if (idx1[(size_t)b * n_m + k] < 0) a = k; if (idx2[(size_t)b * n_m + k] < 0) d = k; }
        /* lists with a "hole" (-1 followed by a valid symbol) do not occur in the decoder; treat as ended */
        l1[b] = a; l2[b] = d;
        for (int k = 0; k < n_m; k++) {
            const int x = idx1[(size_t)b * n_m + k], y = idx2[(size_t)b * n_m + k];
            s1[(size_t)b * n_m + k] = (x >= 0 && x < q) ? img[x] : 0;
            s2[(size_t)b * n_m + k] = (y >= 0 && y < q) ? img[y] : 0;
        }
    }
    DevBuf<float> d1, d2, dout; DevBuf<uint8_t> ds1, ds2, dso; DevBuf<int> dl1, dl2, dlo;
    CK(c, d1.alloc((size_t)B * n_m)); CK(c, d2.alloc((size_t)B * n_m)); CK(c, dout.alloc((size_t)B * n_m));
    CK(c, ds1.alloc((size_t)B * n_m)); CK(c, ds2.alloc((size_t)B * n_m)); CK(c, dso.alloc((size_t)B * n_m));
    CK(c, dl1.alloc(B)); CK(c, dl2.alloc(B)); CK(c, dlo.alloc(B));
    CK(c, cudaMemcpyAsync(d1.p, in1, (size_t)B * n_m * 4, cudaMemcpyHostToDevice, c->stream));
    CK(c, cudaMemcpyAsync(d2.p, in2, (size_t)B * n_m * 4, cudaMemcpyHostToDevice, c->stream));
    CK(c, cudaMemcpyAsync(ds1.p, s1.data(), (size_t)B * n_m, cudaMemcpyHostToDevice, c->stream));
    CK(c, cudaMemcpyAsync(ds2.p, s2.data(), (size_t)B * n_m, cudaMemcpyHostToDevice, c->stream));
    CK(c, cudaMemcpyAsync(dl1.p, l1.data(), (size_t)B * 4, cudaMemcpyHostToDevice, c->stream));
    CK(c, cudaMemcpyAsync(dl2.p, l2.data(), (size_t)B * 4, cudaMemcpyHostToDevice, c->stream));
    const int esg = (B + ES_NT - 1) / ES_NT;
    if (q == 16) es_kernel<16><<<esg, ES_NT, 0, c->stream>>>(d1.p, d2.p, ds1.p, ds2.p, dl1.p, dl2.p, dout.p, dso.p, dlo.p, B, n_m, c->p.nb_oper);
    else if (q == 64) es_kernel<64><<<esg, ES_NT, 0, c->stream>>>(d1.p, d2.p, ds1.p, ds2.p, dl1.p, dl2.p, dout.p, dso.p, dlo.p, B, n_m, c->p.nb_oper);
    else es_kernel<256><<<esg, ES_NT, 0, c->stream>>>(d1.p, d2.p, ds1.p, ds2.p, dl1.p, dl2.p, dout.p, dso.p, dlo.p, B, n_m, c->p.nb_oper);
    CK(c, cudaGetLastError());
    c->launches++;
    CK(c, cudaStreamSynchronize(c->stream));
    std::vector<uint8_t> so((size_t)B * n_m); std::vector<int> lo(B);
    CK(c, cudaMemcpy(out, dout.p, (size_t)B * n_m * 4, cudaMemcpyDeviceToHost));
    CK(c, cudaMemcpy(so.data(), dso.p, (size_t)B * n_m, cudaMemcpyDeviceToHost));
    CK(c, cudaMemcpy(lo.data(), dlo.p, (size_t)B * 4, cudaMemcpyDeviceToHost));
    for (int b = 0; b < B; b++) for (int k = 0; k < n_m; k++)
        idxout[(size_t)b * n_m + k] = (k < lo[b]) ? c->inv_h[so[(size_t)b * n_m + k]] : -1;
    return NBGPU_OK;
}

extern "C" int nbgpu_check_node(nbgpu_ctx *c, int node, const float *vllr, const int *vgf, float *cllr, int *cgf, int B)
{
    if (!c || !vllr || !vgf || !cllr || !cgf || B < 1 || node < 0 || node >= c->M) { ctx_err(c, "nbgpu_check_node: bad argument"); return NBGPU_EINVAL; }
    if (c->k.ecn == 2 || c->k.ecn == 4) { ctx_err(c, "nbgpu_check_node: the %s check node (ecn_kind = %d) takes dense rows, not n_m lists: use nbgpu_check_node_dense", c->k.ecn == 2 ? "sum-product" : "Min-Max", c->k.ecn); return NBGPU_EINVAL; }
    CK(c, cudaSetDevice(c->device));
    const int dc = c->row_ptr_h[node + 1] - c->row_ptr_h[node], n_m = c->p.n_m, q = c->q;
    DevBuf<float> dvl, dcl; DevBuf<int> dvg, dcg;
    CK(c, dvl.alloc((size_t)B * dc * n_m)); CK(c, dvg.alloc((size_t)B * dc * n_m));
    CK(c, dcl.alloc((size_t)B * dc * q)); CK(c, dcg.alloc((size_t)B * dc * q));
    CK(c, cudaMemcpyAsync(dvl.p, vllr, (size_t)B * dc * n_m * 4, cudaMemcpyHostToDevice, c->stream));
    CK(c, cudaMemcpyAsync(dvg.p, vgf, (size_t)B * dc * n_m * 4, cudaMemcpyHostToDevice, c->stream));
    const int grid = c->k.ecn == 1 ? std::min((B + c->k.nw - 1) / c->k.nw, 148) : std::min((B + c->k.cap - 1) / c->k.cap, 148);
    {
        const float *a1 = dvl.p; const int *a2 = dvg.p; float *a3 = dcl.p; int *a4 = dcg.p;
        void *args[] = { (void *)&c->k, (void *)&node, (void *)&a1, (void *)&a2, (void *)&a3, (void *)&a4, (void *)&B };
        CK(c, cudaLaunchKernel(checknode_fn(q, c->k.gf_closed, c->k.ecn), dim3(grid), dim3(c->k.nw * 32), args, c->k.smem_bytes, c->stream));
    }
    CK(c, cudaGetLastError());
    c->launches++;
    CK(c, cudaStreamSynchronize(c->stream));
    CK(c, cudaMemcpy(cllr, dcl.p, (size_t)B * dc * q * 4, cudaMemcpyDeviceToHost));
    CK(c, cudaMemcpy(cgf, dcg.p, (size_t)B * dc * q * 4, cudaMemcpyDeviceToHost));
    return NBGPU_OK;
}

extern "C" int nbgpu_check_node_dense(nbgpu_ctx *c, int node, const float *mvc, float *ctov, int B)
{
    if (!c || !mvc || !ctov || B < 1 || node < 0 || node >= c->M) { ctx_err(c, "nbgpu_check_node_dense: bad argument"); return NBGPU_EINVAL; }
    if (c->k.ecn != 2 && c->k.ecn != 4) { ctx_err(c, "nbgpu_check_node_dense: the context's check node is ecn_kind %d; dense rows are the sum-product node's (ecn_kind = 2) and the Min-Max node's (ecn_kind = 4)", c->k.ecn); return NBGPU_EINVAL; }
    CK(c, cudaSetDevice(c->device));
    const int dc = c->row_ptr_h[node + 1] - c->row_ptr_h[node], q = c->q;
    const size_t n = (size_t)B * dc * q;
    DevBuf<float> din, dout;
    CK(c, din.alloc(n)); CK(c, dout.alloc(n));
    CK(c, cudaMemcpyAsync(din.p, mvc, n * 4, cudaMemcpyHostToDevice, c->stream));
    const int grid = std::min((B + c->k.nw - 1) / c->k.nw, 148);
    {
        const float *a1 = din.p; float *a2 = dout.p;
        void *args[] = { (void *)&c->k, (void *)&node, (void *)&a1, (void *)&a2, (void *)&B };
        CK(c, cudaLaunchKernel(checknode_fn(q, c->k.gf_closed, c->k.ecn), dim3(grid), dim3(c->k.nw * 32), args, c->k.smem_bytes, c->stream));
    }
    CK(c, cudaGetLastError());
    c->launches++;
    CK(c, cudaMemcpyAsync(ctov, dout.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return NBGPU_OK;
}

extern "C" int nbgpu_decision_syndrome(nbgpu_ctx *c, const float *app, int *decide, int *synd, int B)
{
    if (!c || !app || !decide || !synd || B < 1) { ctx_err(c, "nbgpu_decision_syndrome: bad argument"); return NBGPU_EINVAL; }
    CK(c, cudaSetDevice(c->device));
    const int N = c->N, q = c->q;
    DevBuf<float> dapp; DevBuf<int> ddec, dsyn;
    CK(c, dapp.alloc((size_t)B * N * q)); CK(c, ddec.alloc((size_t)B * N)); CK(c, dsyn.alloc(B));
    CK(c, cudaMemcpyAsync(dapp.p, app, (size_t)B * N * q * 4, cudaMemcpyHostToDevice, c->stream));
    const int grid = (int)std::min<long>(((long)B * N + UNIT_NT / 32 - 1) / (UNIT_NT / 32), 148 * 8);
    if (q == 16) decision_kernel<16><<<grid, UNIT_NT, 0, c->stream>>>(c->k, dapp.p, ddec.p, B);
    else if (q == 64) decision_kernel<64><<<grid, UNIT_NT, 0, c->stream>>>(c->k, dapp.p, ddec.p, B);
    else decision_kernel<256><<<grid, UNIT_NT, 0, c->stream>>>(c->k, dapp.p, ddec.p, B);
    CK(c, cudaGetLastError());
    syndrome_kernel<<<std::min(B, 148 * 4), UNIT_NT, 0, c->stream>>>(c->k, ddec.p, dsyn.p, B);
    CK(c, cudaGetLastError());
    c->launches += 2;
    CK(c, cudaStreamSynchronize(c->stream));
    CK(c, cudaMemcpy(decide, ddec.p, (size_t)B * N * 4, cudaMemcpyDeviceToHost));
    CK(c, cudaMemcpy(synd, dsyn.p, (size_t)B * 4, cudaMemcpyDeviceToHost));
    return NBGPU_OK;
}

static int channel_common(nbgpu_ctx *c, const Channel &ch, const float *noisy, float sigma, int B, float *llr, float *illr, int *igf)
{
    if (ch.rc) return ch.rc;
    if (!noisy || B < 1 || ((illr == NULL) != (igf == NULL))) { ctx_err(c, "nbgpu_channel_awgn_*: bad argument"); return NBGPU_EINVAL; }
    CK(c, cudaSetDevice(c->device));
    const int N = c->N, q = c->q, per = ch.fps, kind = ch.kind;
    const size_t in_floats = (size_t)B * c->k.nt * per;       /* transmitted symbols only; the rows cover all N variables */
    DevBuf<float> dn, dl, dil; DevBuf<int> dig;
    CK(c, dn.alloc(in_floats)); CK(c, dl.alloc((size_t)B * N * q));
    if (illr) { CK(c, dil.alloc((size_t)B * N * q)); CK(c, dig.alloc((size_t)B * N * q)); }
    CK(c, cudaMemcpyAsync(dn.p, noisy, in_floats * 4, cudaMemcpyHostToDevice, c->stream));
    KArgs k = c->k;
    k.den = den_of(sigma);
    k.mod = ch.mod_d; k.split_p = split_p(ch);
    const int grid = (int)std::min<long>(((long)B * N + UNIT_NT / 32 - 1) / (UNIT_NT / 32), 148 * 8);
    if (q == 16) channel_kernel<16><<<grid, UNIT_NT, 0, c->stream>>>(k, dn.p, dl.p, illr ? dil.p : nullptr, illr ? dig.p : nullptr, B, kind);
    else if (q == 64) channel_kernel<64><<<grid, UNIT_NT, 0, c->stream>>>(k, dn.p, dl.p, illr ? dil.p : nullptr, illr ? dig.p : nullptr, B, kind);
    else channel_kernel<256><<<grid, UNIT_NT, 0, c->stream>>>(k, dn.p, dl.p, illr ? dil.p : nullptr, illr ? dig.p : nullptr, B, kind);
    CK(c, cudaGetLastError());
    c->launches++;
    CK(c, cudaStreamSynchronize(c->stream));
    if (llr) CK(c, cudaMemcpy(llr, dl.p, (size_t)B * N * q * 4, cudaMemcpyDeviceToHost));
    if (illr) {
        CK(c, cudaMemcpy(illr, dil.p, (size_t)B * N * q * 4, cudaMemcpyDeviceToHost));
        CK(c, cudaMemcpy(igf, dig.p, (size_t)B * N * q * 4, cudaMemcpyDeviceToHost));
    }
    return NBGPU_OK;
}
extern "C" int nbgpu_channel_awgn_bpsk(nbgpu_ctx *c, const float *noisy, float sigma, int B, float *llr, float *illr, int *igf)
{
    return channel_common(c, channel_of(c, CH_BPSK), noisy, sigma, B, llr, illr, igf);
}
extern "C" int nbgpu_channel_awgn_apsk64(nbgpu_ctx *c, const float *noisy, float sigma, int B, float *llr, float *illr, int *igf)
{
    return channel_common(c, channel_of(c, CH_APSK64), noisy, sigma, B, llr, illr, igf);
}
extern "C" int nbgpu_channel_awgn_mapped(nbgpu_ctx *c, const float *noisy, float sigma, int B, float *llr, float *illr, int *igf)
{
    return channel_common(c, channel_of(c, CH_MAPPED), noisy, sigma, B, llr, illr, igf);
}
extern "C" int nbgpu_channel_faded(nbgpu_ctx *c, const float *rx, float sigma, int B, float *llr, float *illr, int *igf)
{
    return channel_common(c, channel_of(c, CH_FADED), rx, sigma, B, llr, illr, igf);
}
extern "C" int nbgpu_channel_split(nbgpu_ctx *c, const float *noisy, float sigma, int B, float *llr, float *illr, int *igf)
{
    return channel_common(c, channel_of(c, CH_SPLIT), noisy, sigma, B, llr, illr, igf);
}
