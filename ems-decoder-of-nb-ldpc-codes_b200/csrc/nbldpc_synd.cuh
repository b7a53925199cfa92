/*
 * nbldpc_synd.cuh -- the syndrome-based check node on the GPU (sm_100a), one WARP per check node.
 *
 * Restates syndrome_ems (syndrome_decoder.c:26-284) with presorting_mvc (:289-496), sorting
 * (:1315-1334) and bayes (:2142-2211):
 *   1. presort: edges ascending by their 2nd-best LLR, then the first four by their 3rd-best LLR
 *      (selection with strict '<': ties keep the lower index first);
 *   2. one syndrome per configuration: LLR = f32 sum over the (presorted) edges of the list entry the
 *      configuration names, GF = sum (XOR of binary images) of the entries' symbols;
 *   3. the reference then sorts ALL syndromes by LLR (stable insertion sort) and, per edge d, walks the sorted
 *      syndromes whose configuration does not deviate on d ("decorrelation"): the first hit of a symbol sets its
 *      LLR, later hits go through bayes() in order; saturation at the LLR of decorrelated syndrome n_cv-1+3d, + offset.
 *
 * What the walk needs from that global order is much less than a sort of ~1000 keys:
 *   (a) hits of DIFFERENT symbols never interact, so only the order INSIDE a symbol group matters: one counting pass
 *       groups the syndromes by symbol (shared-memory histogram + cursor), and every lane orders its own eight groups
 *       (3.7 entries on average) by (LLR, configuration index) with an insertion sort -- exactly the order a stable
 *       sort by LLR leaves inside the group;
 *   (b) the saturation level of edge d is an ORDER STATISTIC: the (n_cv-1+3d)-th smallest LLR among the syndromes
 *       decorrelated on d.  A 256-bin histogram over a monotone 8-bit quantisation of the LLR (one per edge, filled in
 *       the same pass that computes the syndromes) names the bin that holds it; the few syndromes of that bin are
 *       collected and ranked exactly.  (More candidates than the collection buffer holds: a bitwise search with
 *       warp-wide counts, exact for any input.)
 * The round-1 kernel spent five 945-key LSD radix passes (MATCH-ranked scatters, 30 % of its instructions and most of its
 * latency) to obtain the same two things.  All LLRs are non-negative, so float order == bit-pattern order.
 * Symbols are binary images (GF addition == XOR) exactly as in the bubble path.
 */
#pragma once
#include "nbldpc_device.cuh"

#define NB_SYND_MAX 1024                 /* configurations per check node: 32 per lane, kept in registers */
#define NB_SYND_CAND 32                  /* candidates per edge collected for the exact saturation level (more: bitwise search) */

/* a warp's shared memory for the syndrome check node, by shared-window address */
struct SyndMem {
    uint32_t lists;      /* dc lists: n_m f32 | n_m u8 (stride lstride) in ORIGINAL edge order                          */
    uint32_t keya;       /* region A: [S] u32 syndrome LLR bits by configuration index; after the scatter the same bytes   */
    uint32_t skey;       /*   hold the keys grouped by symbol, every group ascending (written out of place by the sort)    */
    uint32_t gkey;       /* region B: [S] u32 keys grouped by symbol, any order inside a group (scatter); before that the   */
    uint32_t hsat;       /*   [ceil(dc/2)][256] u32 per-bin counts of the decorrelated syndromes, two edges per word (16+16 */
    uint32_t rows;       /*   bits); after the sort 4 output rows of 256 f32 (indexed by binary image)                      */
    uint32_t gpay;       /* [S] u16 payload of the grouped keys: decorrelation mask (cfgmask) | symbol << 8                */
    uint32_t gfa;        /* [S] u8 syndrome symbol by configuration index, directly followed by                            */
    uint32_t hist;       /* [256] u32 symbol histogram / scatter cursors; after the scatter the two hold                   */
    uint32_t spay;       /*   [S] u16 payloads in sorted order                                                             */
    uint32_t M;          /* [257] u16 first position of every symbol group                                                */
    uint32_t cand;       /* [dc][NB_SYND_CAND] u32 candidates of the saturation bins                                       */
    uint32_t perm;       /* [16] i32 original edge at presorted position i | [16] f32 saturation level | [16] i32 saturation bin |
                            [16] i32 syndromes below that bin | [16] i32 candidate counters                                */
    uint32_t cfg;        /* [S][dc] u8 configuration table (shared by the CTA)                                             */
    uint32_t cfgmask;    /* [S] u8: bit d set = the configuration does not deviate on presorted edge d (syndrome_decoder.c:96-98) */
    int lstride, n_m, dc, S, n_cv;
};
#define NB_SYND_PERM_BYTES 320

/* bayes(M1 = new LLR, M2 = current LLR), syndrome_decoder.c:2142-2211.  The reference takes double arguments, keeps float
 * locals and multiplies by double constants.  Bit-exact equivalents in f32 (conversions and f64 operations run at a quarter of
 * the f32 rate or less, and every lane of the walk evaluates this on every hit):
 *   - M1 < M2 on doubles that are floats == the float comparison;
 *   - dif = (float)((double)hi - (double)mn) == hi - mn in f32: the double difference is exact while the exponents are less
 *     than 29 apart (one rounding either way); beyond that mn < 2^-29 hi is below a quarter ulp of hi and both give hi;
 *   - (double)dif < 0.1 / 0.2 / 1 / 2  ==  dif < 0.1f / 0.2f / 1.0f / 2.0f  (0.1f and 0.2f are the first floats above 0.1, 0.2);
 *   - (float)(c * (double)min) for c = 0.5, 0.75, 0.9375: the double product of a float by a 1-4 bit constant is exact, so its
 *     rounding equals the float product;
 *   - c = 0.825 is not representable: with c1 = (float)c, c2 = (float)(c - c1),  fma(mn, c1, mn * c2)  equals
 *     (float)(c * (double)mn) for EVERY float mn >= 2^-96 and for 0 (checked exhaustively over all 2^31 non-negative floats,
 *     scripts/check_bayes_f32.c; below 2^-96 the product mn * c2 loses bits to underflow).  synd_prepare proves per check node
 *     that no operand can fall into (0, 2^-96) -- smallest non-zero syndrome LLR >= 2^-32 and no symbol group longer than 64,
 *     every bayes() step scales by at least 1/2 -- and the walk then runs without the guard; otherwise the guarded variant
 *     keeps the double multiplication behind a branch.
 * Branch-free otherwise: divergence would cost more than the few extra instructions.  An unset value is +inf: bayes(x, +inf)
 * = 1.0f * x = x, which is what the reference's "first hit sets the LLR" does. */
__device__ __noinline__ float synd_bayes_tiny(float mn) { return __double2float_rn(__dmul_rn(0.825, (double)mn)); }

/* GUARD = false: the caller has shown that no operand lies in (0, 2^-96) (synd_prepare's return value) */
template <bool GUARD>
__device__ __forceinline__ float synd_bayes_sel(float m1, float m2)
{
    const float mn = fminf(m1, m2), hi = fmaxf(m1, m2);          /* M1 < M2 ? (M1, M2) : (M2, M1); equal values give the same pair */
    const float dif = __fsub_rn(hi, mn);
    const float f = dif < 0.1f ? 0.5f : dif < 0.2f ? 0.75f : dif < 2.0f ? 0.9375f : 1.0f;
    const float a = __fmul_rn(f, mn);
    const float c1 = 0x1.a66666p-1f, c2 = 0x1.99999ap-27f;       /* 0.825 = c1 + c2 - 2^-52 */
    float b = __fmaf_rn(mn, c1, __fmul_rn(mn, c2));
    if (GUARD) { if (fabsf(mn) < 0x1p-96f && mn != 0.0f) b = synd_bayes_tiny(mn); }      /* out of line: keeps the f64 multiply off the common path */
    return (!(dif < 0.2f) && dif < 1.0f) ? b : a;
}

/* monotone 8-bit quantisation of a non-negative float: 16 bins per octave from 2^-4 upwards (bin 0: below, bin 255: beyond
 * 2^-4 * 2^(254/16)); any monotone map is correct, the resolution only decides how many candidates share the target bin */
__device__ __forceinline__ uint32_t synd_bin(uint32_t bits)
{
    const int q = (int)(bits >> 19) - ((123 << 4) - 1);
    return (uint32_t)min(max(q, 0), 255);
}

__device__ __forceinline__ uint32_t synd_M(const SyndMem &sm, uint32_t g)
{
    unsigned short v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(sm.M + 2 * g));
    return v;
}
/* first symbol group of lane L's share of the symbol-grouped order: the lanes take runs of whole groups of (almost) equal
 * length, S/32 entries each, instead of eight groups each (whose sizes vary by a factor of three) */
__device__ __forceinline__ int synd_lane_group(const SyndMem &sm, int lane)
{
    const uint32_t want = (uint32_t)(sm.S * lane) >> 5;
    int lo = 0, hi = 256;                                        /* smallest g with M[g] >= want; M[256] = S >= want */
#pragma unroll
    for (int it = 0; it < 8; it++) {
        const int mid = (lo + hi) >> 1;
        if (synd_M(sm, (uint32_t)mid) >= want) hi = mid; else lo = mid + 1;
    }
    return lo;
}

/*
 * Everything up to the walk.  On return: gkey/gmask hold the syndromes grouped by symbol, every group in the reference's
 * sorted order; M[g] the group starts; perm[0..dc) the presorting; perm+64 the dc saturation levels (:195).
 */
__device__ __forceinline__ bool synd_prepare(const SyndMem &sm, int lane)
{
    const int dc = sm.dc, n_m = sm.n_m, S = sm.S;
    uint32_t tiny = 0xffffffffu;                     /* smallest (bit pattern - 1) of the syndrome LLRs: 0.0f wraps to the top */
    /* ---- presorting_mvc ---- */
    {
        const int i = lane < dc ? lane : 0;
        const float k1 = lds_f32(sm.lists + i * sm.lstride + 4);                /* M_VtoC_LLR[i][1], :320 */
        int rank = 0;
        for (int j = 0; j < dc; j++) {
            const float kj = __shfl_sync(NB_FULL, k1, j);
            rank += (kj < k1 || (kj == k1 && j < i)) ? 1 : 0;
        }
        if (lane < dc) sts_u32(sm.perm + 4 * rank, (uint32_t)i);
        __syncwarp();
        /* first 'border' = 4 presorted edges again, by M_VtoC_LLR[.][2], :377-469 */
        const int e = (int)lds_u32(sm.perm + 4 * (lane < 4 ? lane : 0));
        const float k2 = lds_f32(sm.lists + e * sm.lstride + 8);
        int rank2 = 0;
        for (int j = 0; j < 4; j++) {
            const float kj = __shfl_sync(NB_FULL, k2, j);
            rank2 += (kj < k2 || (kj == k2 && j < lane)) ? 1 : 0;
        }
        __syncwarp();
        if (lane < 4) sts_u32(sm.perm + 4 * rank2, (uint32_t)e);
        /* histograms and counters start at zero */
        for (int w = lane; w < 256; w += 32) sts_u32(sm.hist + 4 * w, 0u);
        for (int w = lane; w < ((dc + 1) >> 1) * 256; w += 32) sts_u32(sm.hsat + 4 * w, 0u);
        if (lane < 16) sts_u32(sm.perm + 256 + 4 * lane, 0u);
        __syncwarp();
    }
    /* ---- syndromes (:64-77) + symbol histogram + saturation histograms, one pass ---- */
    if (dc == 4) {                                   /* the usual degree: list bases in registers, one table word per configuration */
        uint32_t lb[4];
#pragma unroll
        for (int j = 0; j < 4; j++) lb[j] = sm.lists + lds_u32(sm.perm + 4 * j) * sm.lstride;
#pragma unroll 2
        for (int i = lane; i < S; i += 32) {
            const uint32_t cw = lds_u32(sm.cfg + 4 * i), mem = lds_u8(sm.cfgmask + i);
            float llr = 0.0f;
            uint32_t gf = 0;
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const uint32_t c = (cw >> (8 * j)) & 255u;
                llr = __fadd_rn(llr, lds_f32(lb[j] + 4 * c));
                gf ^= lds_u8(lb[j] + 4 * n_m + c);
            }
            const uint32_t bits = __float_as_uint(llr), bin = synd_bin(bits);
            tiny = min(tiny, bits - 1u);
            sts_u32(sm.keya + 4 * i, bits);
            sts_u8(sm.gfa + i, gf);
            asm volatile("red.shared.add.u32 [%0], 1;" :: "r"(sm.hist + 4 * gf) : "memory");
            /* one word per bin and PAIR of edges, 16 bits each */
            const uint32_t inc0 = (mem & 1u) | ((mem & 2u) << 15), inc1 = ((mem >> 2) & 1u) | ((mem & 8u) << 13);
            if (inc0) asm volatile("red.shared.add.u32 [%0], %1;" :: "r"(sm.hsat + 4 * bin), "r"(inc0) : "memory");
            if (inc1) asm volatile("red.shared.add.u32 [%0], %1;" :: "r"(sm.hsat + 1024 + 4 * bin), "r"(inc1) : "memory");
        }
    } else {
        for (int i = lane; i < S; i += 32) {
            const uint32_t mem = lds_u8(sm.cfgmask + i);
            float llr = 0.0f;
            uint32_t gf = 0;
            for (int j = 0; j < dc; j++) {
                const uint32_t list = sm.lists + lds_u32(sm.perm + 4 * j) * sm.lstride;
                const uint32_t c = lds_u8(sm.cfg + i * dc + j);
                llr = __fadd_rn(llr, lds_f32(list + 4 * c));
                gf ^= lds_u8(list + 4 * n_m + c);
            }
            const uint32_t bits = __float_as_uint(llr), bin = synd_bin(bits);
            tiny = min(tiny, bits - 1u);
            sts_u32(sm.keya + 4 * i, bits);
            sts_u8(sm.gfa + i, gf);
            asm volatile("red.shared.add.u32 [%0], 1;" :: "r"(sm.hist + 4 * gf) : "memory");
            for (int p = 0; 2 * p < dc; p++) {
                const uint32_t inc = ((mem >> (2 * p)) & 1u) | (((mem >> (2 * p + 1)) & 1u) << 16);
                if (inc) asm volatile("red.shared.add.u32 [%0], %1;" :: "r"(sm.hsat + 1024 * p + 4 * bin), "r"(inc) : "memory");
            }
        }
    }
    __syncwarp();
    /* ---- group starts: exclusive prefix sum over the 256 symbol bins, lane owns bins 8*lane .. 8*lane+7 ---- */
    uint32_t gmax = 0;                               /* longest symbol group */
    {
        uint32_t h[8], tot = 0;
#pragma unroll
        for (int b = 0; b < 8; b++) { h[b] = lds_u32(sm.hist + 4 * (lane * 8 + b)); tot += h[b]; gmax = max(gmax, h[b]); }
        uint32_t inc = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(NB_FULL, inc, o); if (lane >= o) inc += t; }
        uint32_t run = inc - tot;
#pragma unroll
        for (int b = 0; b < 8; b++) {
            sts_u32(sm.hist + 4 * (lane * 8 + b), run);
            asm volatile("st.shared.u16 [%0], %1;" :: "r"(sm.M + 2 * (lane * 8 + b)), "h"((unsigned short)run) : "memory");
            run += h[b];
        }
        if (lane == 31) asm volatile("st.shared.u16 [%0], %1;" :: "r"(sm.M + 2 * 256), "h"((unsigned short)run) : "memory");
    }
    /* ---- saturation bins: the bin of edge d that holds its decorrelated syndrome number n_cv-1+3d, and how many lie below ---- */
    for (int p = 0; 2 * p < dc; p++) {
        uint32_t h[8], tot = 0;                                                  /* packed: edge 2p in the low half, 2p+1 in the high half */
#pragma unroll
        for (int b = 0; b < 8; b++) { h[b] = lds_u32(sm.hsat + 1024 * p + 4 * (lane * 8 + b)); tot += h[b]; }
        uint32_t inc = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(NB_FULL, inc, o); if (lane >= o) inc += t; }
        uint32_t run = inc - tot;
#pragma unroll
        for (int b = 0; b < 8; b++) {
#pragma unroll
            for (int s = 0; s < 2; s++) {
                const int d = 2 * p + s, target = sm.n_cv - 1 + 3 * d;
                const int below = (int)((run >> (16 * s)) & 0xffffu), here = (int)((h[b] >> (16 * s)) & 0xffffu);
                if (d < dc && below <= target && target < below + here) {
                    sts_u32(sm.perm + 128 + 4 * d, (uint32_t)(lane * 8 + b));
                    sts_u32(sm.perm + 192 + 4 * d, (uint32_t)below);
                }
            }
            run += h[b];
        }
    }
    __syncwarp();
    /* ---- scatter into the symbol groups (any order inside a group) + candidates of the saturation bins ---- */
    {
        /* the four (eight) saturation bins packed into one (two) words: a candidate test is a byte compare */
        uint32_t sb0 = 0, sb1 = 0;
        for (int d = 0; d < dc; d++) {
            const uint32_t b = lds_u32(sm.perm + 128 + 4 * d) & 255u;
            if (d < 4) sb0 |= b << (8 * d); else sb1 |= b << (8 * (d - 4));
        }
        __syncwarp();                                    /* the saturation histograms are about to be overwritten by the grouped keys */
#pragma unroll 2
        for (int i = lane; i < S; i += 32) {
            const uint32_t key = lds_u32(sm.keya + 4 * i), gf = lds_u8(sm.gfa + i), mem = lds_u8(sm.cfgmask + i);
            uint32_t pos;
            asm volatile("atom.shared.add.u32 %0, [%1], 1;" : "=r"(pos) : "r"(sm.hist + 4 * gf) : "memory");
            sts_u32(sm.gkey + 4 * pos, key);
            asm volatile("st.shared.u16 [%0], %1;" :: "r"(sm.gpay + 2 * pos), "h"((unsigned short)(mem | (gf << 8))) : "memory");
            const uint32_t bin4 = synd_bin(key) * 0x01010101u;
            /* byte d of eq is 0xff where the syndrome's bin is edge d's saturation bin */
            uint32_t hit = (__vcmpeq4(bin4, sb0) & 0x08040201u);
            hit = (hit | (hit >> 8) | (hit >> 16) | (hit >> 24)) & 15u;
            if (dc > 4) { uint32_t h2 = __vcmpeq4(bin4, sb1) & 0x08040201u; h2 = (h2 | (h2 >> 8) | (h2 >> 16) | (h2 >> 24)) & 15u; hit |= h2 << 4; }
            hit &= mem;
            while (hit) {                                /* rare: a few syndromes per edge share the bin */
                const int d = __ffs(hit) - 1;
                hit &= hit - 1u;
                uint32_t cpos;
                asm volatile("atom.shared.add.u32 %0, [%1], 1;" : "=r"(cpos) : "r"(sm.perm + 256 + 4 * d) : "memory");
                if (cpos < NB_SYND_CAND) sts_u32(sm.cand + 4 * (d * NB_SYND_CAND + cpos), key);
            }
        }
    }
    __syncwarp();
    /* ---- saturation levels (:195): exact order statistic among the candidates of the bin ---- */
    for (int d = 0; d < dc; d++) {
        const int m = (int)lds_u32(sm.perm + 256 + 4 * d);
        const int want = sm.n_cv - 1 + 3 * d - (int)lds_u32(sm.perm + 192 + 4 * d);      /* rank inside the bin */
        if (m <= NB_SYND_CAND) {
            for (int u = 0; 32 * u < m; u++) {
                const int ci = lane + 32 * u;
                const uint32_t c = ci < m ? lds_u32(sm.cand + 4 * (d * NB_SYND_CAND + ci)) : 0xffffffffu;
                int lt = 0, le = 0;
                for (int j = 0; j < m; j++) {
                    const uint32_t x = lds_u32(sm.cand + 4 * (d * NB_SYND_CAND + j));
                    lt += x < c; le += x <= c;
                }
                if (ci < m && lt <= want && want < le) sts_u32(sm.perm + 64 + 4 * d, c);   /* equal candidates write the same value */
            }
        } else {
            /* more syndromes in one bin than the buffer holds (e.g. many equal LLRs): the k-th smallest bit pattern among the
             * edge's decorrelated syndromes by a bitwise search, counts over the warp */
            const int target = sm.n_cv - 1 + 3 * d;
            uint32_t prefix = 0;
            for (int bit = 31; bit >= 0; bit--) {
                const uint32_t cand = prefix | (1u << bit), himask = ~((1u << bit) - 1u);
                int cnt = 0;                                                              /* syndromes whose bits above 'bit' are below cand's */
                for (int i = lane; i < S; i += 32)
                    cnt += ((lds_u8(sm.cfgmask + i) >> d) & 1u) && ((lds_u32(sm.keya + 4 * i) & himask) < cand);
                cnt = __reduce_add_sync(NB_FULL, cnt);
                if (cnt <= target) prefix = cand;                                         /* the k-th value has this bit set */
            }
            if (lane == 0) sts_u32(sm.perm + 64 + 4 * d, prefix);
        }
    }
    __syncwarp();
    /* ---- order every symbol group by LLR, out of place (gkey/gpay -> skey/spay; region A is free since the scatter, gfa and
     * the cursors too): the rank of an entry inside its group is the number of members before it in (LLR, position) order.
     * Every entry is independent of every other -- lane L takes entries L, L+32, ...; the loads of a group's members do
     * not depend on each other, unlike the steps of an insertion sort ---- */
    {
#pragma unroll 1
        for (int i = lane; i < S; i += 32) {
            const uint32_t k = lds_u32(sm.gkey + 4 * i);
            unsigned short pay;
            asm volatile("ld.shared.u16 %0, [%1];" : "=h"(pay) : "r"(sm.gpay + 2 * i));
            const uint32_t g = (uint32_t)pay >> 8;
            const int gs = (int)synd_M(sm, g), ge = (int)synd_M(sm, g + 1u);
            const unsigned long long me = ((unsigned long long)k << 32) | (uint32_t)i;
            int rank = gs;
#pragma unroll 1
            for (int j0 = gs; j0 < ge; j0 += 4) {
#pragma unroll
                for (int u = 0; u < 4; u++) {                    /* region B extends 16 bytes past its S keys */
                    const int j = j0 + u;
                    const unsigned long long other = ((unsigned long long)lds_u32(sm.gkey + 4 * j) << 32) | (uint32_t)j;
                    rank += (j < ge && other < me) ? 1 : 0;
                }
            }
            sts_u32(sm.skey + 4 * rank, k);
            asm volatile("st.shared.u16 [%0], %1;" :: "r"(sm.spay + 2 * rank), "h"(pay) : "memory");
        }
    }
    __syncwarp();
    /* bayes() may run without its small-operand guard (see synd_bayes_sel) */
    tiny = __reduce_min_sync(NB_FULL, tiny);
    gmax = __reduce_max_sync(NB_FULL, gmax);
    return tiny >= 0x2f800000u - 1u && gmax <= 64u;            /* 0x2f800000 = 2^-32 */
}

/* step 4 for the presorted positions d0 .. d0+nd-1 (nd <= 4) in ONE walk: on return out_k[256] = sm.rows + 1024 k
 * (f32, indexed by the binary image of the rotated symbol) holds M_CtoV_LLR[d0+k][.] BEFORE the saturation of
 * syndrome_decoder.c:198-209, which the reader of the row applies (synd_saturate: 8 values per lane and edge instead of one
 * per lane and walk step).  The reference walks the sorted syndromes and, per symbol, lets the first hit set the LLR
 * and every later hit go through bayes(); hits of different symbols do not interact, so every lane replays the syndromes of
 * a run of whole symbol groups (contiguous in the symbol-grouped order, ascending inside a group, about S/32 entries) for
 * all nd edges at once and scatters the results to the symbols (group ^ best symbol of the edge).
 * GUARD: see synd_bayes_sel; synd_prepare's return value says whether it can be dropped. */
/* saturation of one output value (syndrome_decoder.c:198-209): above the level of edge d -> level + offset; symbols no syndrome
 * reached still hold the initial 1500.0 and take the same test */
__device__ __forceinline__ float synd_saturate(float v, float sat, float hi) { return v > sat ? hi : v; }

template <bool GUARD>
__device__ __forceinline__ void synd_walk(const SyndMem &sm, int d0, int nd, int lane)
{
    uint32_t xs[4]; float m[4];
    const float unset_m = __int_as_float(0x7f800000);
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int d = d0 + (k < nd ? k : 0);
        xs[k] = lds_u8(sm.lists + lds_u32(sm.perm + 4 * d) * sm.lstride + 4 * sm.n_m) << 2;  /* M_VtoC_GF[d][0], :103 */
        m[k] = unset_m;
    }
    const int gfirst = synd_lane_group(sm, lane);
    int glast = __shfl_down_sync(NB_FULL, gfirst, 1);
    if (lane == 31) glast = 256;
    const int lo = (int)synd_M(sm, (uint32_t)gfirst), hi_i = (int)synd_M(sm, (uint32_t)glast);
#pragma unroll
    for (int k = 0; k < 4; k++)                                  /* symbols without a hit keep the initial 1500.0 (:131) */
        if (k < nd) {
            const uint32_t a = sm.rows + 1024 * k + lane * 16;
            const float unset = 1500.0f;
            asm volatile("st.shared.v4.f32 [%0], {%1, %1, %1, %1};\n\tst.shared.v4.f32 [%0+512], {%1, %1, %1, %1};" :: "r"(a), "f"(unset) : "memory");
        }
    __syncwarp();
    const uint32_t ndmask = (1u << nd) - 1u;
    /* one entry ahead: the next entry's symbol also tells whether this one closes its group */
    float llr = __uint_as_float(lds_u32(sm.skey + 4 * min(lo, sm.S - 1)));
    uint32_t pay = lds_u16(sm.spay + 2 * min(lo, sm.S - 1));
#pragma unroll 1
    for (int i = lo; i < hi_i; i++) {
        const int nx = min(i + 1, sm.S - 1);
        const float llr_n = __uint_as_float(lds_u32(sm.skey + 4 * nx));
        const uint32_t pay_n = lds_u16(sm.spay + 2 * nx);
        const uint32_t mem = (pay >> d0) & ndmask;               /* decorrelation, :96-98 */
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const float nb = synd_bayes_sel<GUARD>(llr, m[k]);
            m[k] = ((mem >> k) & 1u) ? nb : m[k];
        }
        if (i + 1 == hi_i || ((pay ^ pay_n) >> 8) != 0u) {       /* last syndrome of the symbol: store */
            const uint32_t g4 = (pay >> 8) << 2;
#pragma unroll
            for (int k = 0; k < 4; k++) {
                if (m[k] < unset_m) sts_f32(sm.rows + 1024 * k + (g4 ^ xs[k]), m[k]);
                m[k] = unset_m;
            }
        }
        llr = llr_n; pay = pay_n;
    }
    __syncwarp();
}
