/*
 * nbldpc_device.cuh -- device functions of the EMS decoder (sm_100a).
 *
 * Building blocks (reference lines they replace):
 *   expand_record    bubble_decoder.c:262-270   dense q-vector of one stored C->V message
 *   select_edges     NB_LDPC.c:354-374          stable top-n_m of q values + normalisation, one warp
 *                                               per edge, NEDG edges interleaved for latency hiding
 *   es_serial        bubble_decoder.c:316-593   ElementaryStep, one THREAD per step (32 per warp)
 *   warp_argmin      tools.c:312-330            Decision
 * GF symbols travel through the check node as BINARY IMAGES so that GF addition is XOR
 * (ADDGF[a][b] == inv[img[a]^img[b]] is verified on the host); the multiplication by the edge
 * coefficient on the way in (bubble_decoder.c:133-152) and the division on the way out (:249-254) use
 * the exponent form of the reference tables (MULGF[a][b] = ((a+b-2) mod (q-1))+1, verified on the
 * host; a table fallback exists for caller-supplied tables of another shape).
 *
 * All LLR arithmetic uses the explicit round-to-nearest intrinsics (__fadd_rn/__fsub_rn): one IEEE
 * f32 operation where the reference has one, never contracted or re-associated.
 */
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define NB_SENT 1e5f
#define NB_FULL 0xffffffffu
#define NB_KEY_INF 0xffffffffu

/* A warp holds one q-vector ("row"); lane L owns VPL slots.  The slot -> symbol map is chosen so that every row move is
 * one or two 128-bit accesses per lane over CONTIGUOUS 512-byte spans (bank-conflict free in shared memory, four 128-byte
 * lines per instruction in global memory): for q = 256 slots 0-3 are symbols 4L..4L+3 and slots 4-7 symbols
 * 128+4L..128+4L+3.  (A lane-major map, symbols 8L..8L+7, costs twice the wavefronts: the round-1 kernel was bound by
 * exactly that pipe, l1tex data-stage 81 % busy.) */
template <int Q> struct QTraits {
    static constexpr int VPL = (Q >= 32) ? Q / 32 : 1;      /* values per lane when a warp holds one row */
    static constexpr int LOGQ = (Q == 16) ? 4 : (Q == 64) ? 6 : 8;
    static constexpr int KEY_WORDS = (VPL + 1) * 32;        /* selection queue: sorted keys [rank][lane] + one row of +inf */
    static constexpr int SCR_WORDS = KEY_WORDS > Q ? KEY_WORDS : Q;   /* per-edge scratch that can hold either the queue or a dense row */
    __device__ __forceinline__ static int sym(int lane, int j)
    {
        if constexpr (Q == 256) return ((j & 4) << 5) | (lane << 2) | (j & 3);
        else if constexpr (Q == 64) return lane * 2 + j;
        else return lane;
    }
};

/* GF(q) helpers shared by every kernel: byte tables in shared memory (+ global fallback tables) */
struct GFTab {
    const uint8_t *img;      /* [q] symbol -> binary image (shared)            */
    const uint8_t *inv;      /* [q] binary image -> symbol (shared)            */
    const uint8_t *rotin;    /* [q*q] global fallback: img[MULGF[sym][h]]       */
    const uint8_t *rotout;   /* [q*q] global fallback: DIVGF[inv[s]][h]         */
};

/* img[MULGF[sym][h]], bubble_decoder.c:145.  CLOSED: MULGF[a][b] = ((a+b-2) mod (q-1))+1 (checked on the host) */
template <int Q, bool CLOSED> __device__ __forceinline__ int gf_rot_in(const GFTab &g, int sym, int h)
{
    if constexpr (CLOSED) {
        int e = sym + h - 2;
        e = (e >= Q - 1) ? e - (Q - 1) : e;
        return g.img[sym ? e + 1 : 0];
    } else {
        return g.rotin[h * Q + sym];
    }
}
/* DIVGF[inv[s]][h], bubble_decoder.c:251 */
template <int Q, bool CLOSED> __device__ __forceinline__ int gf_rot_out(const GFTab &g, int s, int h)
{
    if constexpr (CLOSED) {
        const int sym = g.inv[s];
        int e = sym - h;
        e = (e < 0) ? e + (Q - 1) : e;
        return sym ? e + 1 : 0;
    } else {
        return g.rotout[h * Q + s];
    }
}

/* ---- explicit shared-window accesses (32-bit addresses: no generic-pointer arithmetic in hot loops) ---- */
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ float lds_f32(uint32_t a) { float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint32_t lds_u16(uint32_t a) { unsigned short v; asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint32_t lds_u8(uint32_t a) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ void sts_f32(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" :: "r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ void sts_u32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts_u8(uint32_t a, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }

/* ---- row I/O: a warp moves one q-float row; lane holds symbols lane*VPL .. lane*VPL+VPL-1 ---- */
template <int Q> __device__ __forceinline__ void load_row(const float *row, int lane, float (&v)[QTraits<Q>::VPL])
{
    if constexpr (Q == 256) {
        const float4 a = reinterpret_cast<const float4 *>(row)[lane];
        const float4 b = reinterpret_cast<const float4 *>(row)[lane + 32];
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    } else if constexpr (Q == 64) {
        const float2 a = reinterpret_cast<const float2 *>(row)[lane];
        v[0] = a.x; v[1] = a.y;
    } else {
        v[0] = (lane < Q) ? row[lane] : NB_SENT;
    }
}
template <int Q> __device__ __forceinline__ void store_row(float *row, int lane, const float (&v)[QTraits<Q>::VPL])
{
    if constexpr (Q == 256) {
        reinterpret_cast<float4 *>(row)[lane] = make_float4(v[0], v[1], v[2], v[3]);
        reinterpret_cast<float4 *>(row)[lane + 32] = make_float4(v[4], v[5], v[6], v[7]);
    } else if constexpr (Q == 64) {
        reinterpret_cast<float2 *>(row)[lane] = make_float2(v[0], v[1]);
    } else {
        if (lane < Q) row[lane] = v[0];
    }
}
/* ---- the same row moves with an L2 eviction policy (createpolicy): a parked row is wanted again a few microseconds
 * later (evict_last); APP rows and records are touched once per pass and are streamed (evict_first) ---- */
__device__ __forceinline__ uint64_t l2_policy_evict_last()
{
    uint64_t p; asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p)); return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_first()
{
    uint64_t p; asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p)); return p;
}
__device__ __forceinline__ float4 ldg_f4_hint(const float4 *p, uint64_t pol)
{
    float4 v;
    asm volatile("ld.global.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ void stg_f4_hint(float4 *p, const float4 &v, uint64_t pol)
{
    asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;" :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(pol) : "memory");
}
template <int Q> __device__ __forceinline__ void load_row_hint(const float *row, int lane, float (&v)[QTraits<Q>::VPL], uint64_t pol)
{
    if constexpr (Q == 256) {
        const float4 a = ldg_f4_hint(reinterpret_cast<const float4 *>(row) + lane, pol);
        const float4 b = ldg_f4_hint(reinterpret_cast<const float4 *>(row) + lane + 32, pol);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    } else {
        load_row<Q>(row, lane, v);
    }
}
template <int Q> __device__ __forceinline__ void store_row_hint(float *row, int lane, const float (&v)[QTraits<Q>::VPL], uint64_t pol)
{
    if constexpr (Q == 256) {
        stg_f4_hint(reinterpret_cast<float4 *>(row) + lane, make_float4(v[0], v[1], v[2], v[3]), pol);
        stg_f4_hint(reinterpret_cast<float4 *>(row) + lane + 32, make_float4(v[4], v[5], v[6], v[7]), pol);
    } else {
        store_row<Q>(row, lane, v);
    }
}
template <int Q> __device__ __forceinline__ void fill_row(float *row, int lane, float x)
{
    if constexpr (Q == 256) {                        /* one register, stored as a quad twice: no broadcast moves */
        const uint32_t a = smem_u32(row) + lane * 16;
        asm volatile("st.shared.v4.f32 [%0], {%1, %1, %1, %1};\n\tst.shared.v4.f32 [%0+512], {%1, %1, %1, %1};" :: "r"(a), "f"(x) : "memory");
    } else if constexpr (Q == 64) {
        reinterpret_cast<float2 *>(row)[lane] = make_float2(x, x);
    } else {
        if (lane < Q) row[lane] = x;
    }
}

/* the same row moves on a shared-window address (no generic-pointer arithmetic in the hot loops) */
template <int Q> __device__ __forceinline__ void lds_row(uint32_t row, int lane, float (&v)[QTraits<Q>::VPL])
{
    if constexpr (Q == 256) {
        const uint32_t a = row + lane * 16;
        asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(a));
        asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4+512];" : "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]) : "r"(a));
    } else if constexpr (Q == 64) {
        asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v[0]), "=f"(v[1]) : "r"(row + lane * 8));
    } else {
        v[0] = (lane < Q) ? lds_f32(row + 4 * lane) : NB_SENT;
    }
}
template <int Q> __device__ __forceinline__ void fill_row_s(uint32_t row, int lane, float x)
{
    if constexpr (Q == 256) {
        const uint32_t a = row + lane * 16;
        asm volatile("st.shared.v4.f32 [%0], {%1, %1, %1, %1};\n\tst.shared.v4.f32 [%0+512], {%1, %1, %1, %1};" :: "r"(a), "f"(x) : "memory");
    } else if constexpr (Q == 64) {
        asm volatile("st.shared.v2.f32 [%0], {%1, %1};" :: "r"(row + lane * 8), "f"(x) : "memory");
    } else {
        if (lane < Q) sts_f32(row + 4 * lane, x);
    }
}

/* ---- stored C->V message of one edge ("record"): llr[n_m] f32 | pad to 8 | sat f32 | stp i32 | sym[n_m] u8 ----
 * A dense CtoV row is "stp explicit (symbol, LLR) pairs + the constant sat everywhere else"
 * (bubble_decoder.c:262-270), so the record is lossless. */
struct RecView {
    float llr; int sym; float sat; int stp;     /* llr/sym: entry 'lane' (garbage for lane >= stp) */
};
/* Per-lane byte offsets into a record, computed once per kernel: the record of edge 'ed' of a frame is
 * at ctov_f + ed * stride, so a field address is one 32x32->64 multiply-add away. */
struct RecLane {
    uint32_t llr, sym, tail, stride;    /* byte offsets of llr[lane'], sym[lane'], {sat,stp}; lane' = lane < n_m ? lane : 0 */
    __device__ __forceinline__ RecLane(int n_m, int lane, int rec_stride)
    {
        const int k = lane < n_m ? lane : 0;
        tail = (4 * n_m + 7) & ~7;              /* {sat, stp} is accessed as one 8-byte word: keep it aligned for odd n_m */
        llr = 4 * k; sym = tail + 8 + k; stride = (uint32_t)rec_stride;
    }
};
__device__ __forceinline__ RecView load_record(const uint8_t *ctov_f, uint32_t ed, const RecLane &rl)
{
    RecView r;
    const uint8_t *rec = ctov_f + (size_t)ed * rl.stride;
    r.llr = *reinterpret_cast<const float *>(rec + rl.llr);
    const int2 tail = *reinterpret_cast<const int2 *>(rec + rl.tail);
    r.sat = __int_as_float(tail.x);
    r.stp = tail.y;
    r.sym = rec[rl.sym];
    return r;
}
__device__ __forceinline__ void store_record(uint8_t *ctov_f, uint32_t ed, const RecLane &rl, const RecView &r, int n_m, int lane)
{
    uint8_t *rec = ctov_f + (size_t)ed * rl.stride;
    if (lane < n_m) { *reinterpret_cast<float *>(rec + rl.llr) = r.llr; rec[rl.sym] = (uint8_t)r.sym; }
    if (lane == 0) *reinterpret_cast<int2 *>(rec + rl.tail) = make_int2(__float_as_int(r.sat), r.stp);
}
/* Dense values of this lane's symbols from a record, through a CLEAN scratch row (every word +inf on entry and again on
 * return): the explicit pairs are scattered, the row is read back, the touched words are reset.  A word that still holds
 * +inf is a symbol without explicit pair and takes the constant.  minform: llr <= sat for every explicit pair (offset >= 0,
 * bubble_decoder.c:264), so the merge is one FMNMX per value; otherwise a compare + select. */
#define NB_ROW_CLEAN __int_as_float(0x7f800000)
template <int Q>
__device__ __forceinline__ void expand_record(const RecView &r, int lane, uint32_t scr, float (&c)[QTraits<Q>::VPL], bool minform)
{
    constexpr int VPL = QTraits<Q>::VPL;
    const bool mine = lane < r.stp;
    const uint32_t slot = scr + 4 * (uint32_t)r.sym;
    if (mine) sts_f32(slot, r.llr);
    __syncwarp();
    float x[VPL];
    lds_row<Q>(scr, lane, x);
    __syncwarp();
    if (mine) sts_f32(slot, NB_ROW_CLEAN);
    if (minform) {
#pragma unroll
        for (int j = 0; j < VPL; j++) c[j] = fminf(x[j], r.sat);
    } else {
#pragma unroll
        for (int j = 0; j < VPL; j++) c[j] = (x[j] < NB_ROW_CLEAN) ? x[j] : r.sat;
    }
    __syncwarp();
}

/* ---- in-lane sorting networks on u32 keys ---- */
__device__ __forceinline__ void cswap(uint32_t &a, uint32_t &b)
{
    const uint32_t lo = min(a, b), hi = max(a, b);
    a = lo; b = hi;
}
template <int VPL> __device__ __forceinline__ void sort_keys(uint32_t (&k)[VPL])
{
    if constexpr (VPL == 8) {
        cswap(k[0], k[1]); cswap(k[2], k[3]); cswap(k[4], k[5]); cswap(k[6], k[7]);
        cswap(k[0], k[2]); cswap(k[1], k[3]); cswap(k[4], k[6]); cswap(k[5], k[7]);
        cswap(k[1], k[2]); cswap(k[5], k[6]); cswap(k[0], k[4]); cswap(k[3], k[7]);
        cswap(k[1], k[5]); cswap(k[2], k[6]);
        cswap(k[1], k[4]); cswap(k[3], k[6]);
        cswap(k[2], k[4]); cswap(k[3], k[5]);
        cswap(k[3], k[4]);
    } else if constexpr (VPL == 2) {
        cswap(k[0], k[1]);
    }
}

/* lexicographic (value, symbol) minimum across the warp with the reference's scan semantics:
 * strict '<' from the +1e5 sentinel, ties -> lowest symbol; "nothing below 1e5" -> (1e5, BIG). */
__device__ __forceinline__ void warp_lexmin(float &bv, int &bg)
{
#pragma unroll
    for (int off = 16; off; off >>= 1) {
        const float ov = __shfl_xor_sync(NB_FULL, bv, off);
        const int og = __shfl_xor_sync(NB_FULL, bg, off);
        if (ov < bv || (ov == bv && og < bg)) { bv = ov; bg = og; }
    }
}

/* Decision for one row held by a warp (tools.c:317-329): argmin with strict '<' from 1e5, ties ->
 * lowest symbol, default 0.  For non-negative finite rows (the normal case) the float bit pattern is
 * monotone: one integer REDUX finds the minimum value, a second one the lowest symbol that holds it. */
template <int Q> __device__ __forceinline__ int warp_argmin(const float (&v)[QTraits<Q>::VPL], int lane)
{
    constexpr int VPL = QTraits<Q>::VPL;
    const bool active = (Q >= 32) || lane < Q;
    uint32_t mb = NB_KEY_INF, ob = 0;
#pragma unroll
    for (int j = 0; j < VPL; j++) { const uint32_t b = __float_as_uint(v[j]); mb = min(mb, b); ob |= b; }
    if (!active) { mb = NB_KEY_INF; ob = 0; }
    if (!__any_sync(NB_FULL, ob >= 0x7f800000u)) {
        const uint32_t m = __reduce_min_sync(NB_FULL, mb);
        if (!(__uint_as_float(m) < NB_SENT)) return 0;
        uint32_t best = 0xffffu;
#pragma unroll
        for (int j = VPL - 1; j >= 0; j--) if (__float_as_uint(v[j]) == m) best = (uint32_t)QTraits<Q>::sym(lane, j);   /* slots ascend in symbol */
        if (!active) best = 0xffffu;
        return (int)__reduce_min_sync(NB_FULL, best);
    }
    float bv = NB_SENT; int bg = 0x7fffffff;
#pragma unroll
    for (int j = 0; j < VPL; j++) if (active && v[j] < bv) { bv = v[j]; bg = QTraits<Q>::sym(lane, j); }   /* strict '<' + ascending slots: lowest symbol of the lane */
    warp_lexmin(bv, bg);
    return (bg == 0x7fffffff) ? 0 : bg;
}

/*
 * Truncation of V->C messages (NB_LDPC.c:354-374) for NEDG edges at once: the n_m smallest of the q
 * values mvc[e][], ascending, ties -> lowest symbol, values >= 1e5 never selected (slot keeps
 * (1e5, symbol 0) and symbol 0 is masked), then LLR[k] -= LLR[0], LLR[0] = 0.
 *
 * Fast path: every value becomes a UNIQUE 32-bit key (f32 bits & ~(q-1)) | symbol.  For non-negative
 * finite floats the bit pattern is monotone in the value, so key order == (value, symbol) order except
 * when two values differ only in the log2(q) dropped mantissa bits.  Each lane sorts its VPL keys with
 * a register network and parks them in shared memory ([rank][lane], row VPL = +inf); n_m+1 rounds of
 * one REDUX.MIN over the lane heads pop the global minimum, the owning lane stepping to its next row;
 * every lane then re-reads its head row, so the load needs no predicate and no copy.  The minimum comes
 * back warp-uniform, so lane r simply keeps the result of round r: one compare + select, no shared-memory
 * traffic.  n_m = 20 and n_m = 16 run their rounds straight-line, other n_m a rolled loop.  The NEDG independent
 * REDUX chains are interleaved so that their latencies overlap.  The dropped low bits of the winners come
 * from the owning lane by two shuffles (each lane keeps the low bytes of its VPL values packed in one or two
 * registers), so no dense row is written for the read-back.  A result is accepted only if (a) no value was
 * negative/NaN/Inf, (b) adjacent winners (including the (n_m+1)-th) differ in their kept bits, (c) the
 * n_m winners are < 1e5.  If only (b) fails and not at the n_m boundary, the winners are re-ordered in
 * place with full comparisons; otherwise that edge re-runs the exact scan (same semantics as the
 * reference loop).
 *
 * scr[e]: SCR_WORDS u32 of warp-private scratch as a shared-window address (free on entry, free on return).
 * Result: lane k < n_m holds (out_llr[e], out_sym[e]) = k-th entry of edge e.
 */
template <int Q, int NEDG>
__device__ __forceinline__ void select_edges(const float (&mvc)[NEDG][QTraits<Q>::VPL], int lane, const uint32_t (&scr)[NEDG],
                                             int n_m, float (&out_llr)[NEDG], int (&out_sym)[NEDG], unsigned *slow_counter)
{
    constexpr int VPL = QTraits<Q>::VPL;
    constexpr int LOGQ = QTraits<Q>::LOGQ;
    const bool active = (Q >= 32) || lane < Q;
    const int rounds = (n_m + 1 < Q) ? n_m + 1 : Q;
    uint32_t head[NEDG], nxt[NEDG], mine[NEDG], lo[NEDG][2];
    bool bad[NEDG];
#pragma unroll
    for (int e = 0; e < NEDG; e++) {
        uint32_t key[VPL];
        if constexpr (Q == 256) {
            /* key = value bits with the low byte replaced by the symbol: one PRMT per value */
            const uint32_t symA = 0x03020100u + 0x04040404u * (uint32_t)lane, symB = symA | 0x80808080u;
            uint32_t b[VPL];
#pragma unroll
            for (int j = 0; j < VPL; j++) b[j] = __float_as_uint(mvc[e][j]);
#pragma unroll
            for (int j = 0; j < VPL; j++) key[j] = __byte_perm(b[j], j < 4 ? symA : symB, 0x3214 + (j & 3));
            lo[e][0] = __byte_perm(__byte_perm(b[0], b[1], 0x0040), __byte_perm(b[2], b[3], 0x0040), 0x5410);
            lo[e][1] = __byte_perm(__byte_perm(b[4], b[5], 0x0040), __byte_perm(b[6], b[7], 0x0040), 0x5410);
        } else {
#pragma unroll
            for (int j = 0; j < VPL; j++) {
                const uint32_t b = __float_as_uint(mvc[e][j]);
                key[j] = active ? ((b & ~uint32_t(Q - 1)) | uint32_t(QTraits<Q>::sym(lane, j))) : NB_KEY_INF;
            }
            if constexpr (Q == 64) lo[e][0] = (__float_as_uint(mvc[e][0]) & 63u) | ((__float_as_uint(mvc[e][1]) & 63u) << 8);
            else lo[e][0] = 0;
            lo[e][1] = 0;
        }
        sort_keys<VPL>(key);
        bad[e] = active && key[VPL - 1] >= 0x7f800000u;
        const uint32_t col = scr[e] + 4 * lane;            /* the lane's column of the queue [rank][lane] */
#pragma unroll
        for (int j = 0; j < VPL; j++) sts_u32(col + 128 * j, key[j]);
        sts_u32(col + 128 * VPL, NB_KEY_INF);
        head[e] = key[0];
        nxt[e] = col;                                   /* row of the lane's current head */
        mine[e] = NB_KEY_INF;
    }
    if constexpr (Q == 16 && NEDG == 2) {
        /* GF(16): a row is one key per lane of a half warp.  Both edges are sorted at once, edge 0 in lanes 0-15 and edge 1 in
         * lanes 16-31, by a 16-wide bitonic network (10 exchanges) instead of 2 x 16 reduction rounds. */
        const uint32_t other = __shfl_sync(NB_FULL, head[1], lane & 15);
        uint32_t x = lane < 16 ? head[0] : other;
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
        mine[0] = __shfl_sync(NB_FULL, x, lane & 15);
        mine[1] = __shfl_sync(NB_FULL, x, 16 | (lane & 15));
    } else {
    /* no __syncwarp needed: every lane only reads back what it wrote itself */
#define NB_SEL_ROUND(E, OFF)                                                                                   \
    asm volatile("{\n\t"                                                                                        \
                 ".reg .pred p, c;\n\t"                                                                         \
                 ".reg .u32 m;\n\t"                                                                             \
                 "redux.sync.min.u32 m, %0, 0xffffffff;\n\t"                                                    \
                 "setp.eq.u32 p, %0, m;\n\t"                                                                    \
                 "@p add.u32 %1, %1, 128;\n\t"                                                                  \
                 "ld.shared.u32 %0, [%1];\n\t"                                                                  \
                 "setp.eq.u32 c, %3, " #OFF ";\n\t"                                                             \
                 "selp.u32 %2, m, %2, c;\n\t"                                                                   \
                 "}"                                                                                             \
                 : "+r"(head[E]), "+r"(nxt[E]), "+r"(mine[E]) : "r"(lr) : "memory")
/* the last round only has to name the (n_m+1)-th key for the boundary test: nothing is popped */
#define NB_SEL_PEEK(E)                                                                                          \
    asm volatile("{\n\t"                                                                                        \
                 ".reg .pred c;\n\t"                                                                            \
                 ".reg .u32 m;\n\t"                                                                             \
                 "redux.sync.min.u32 m, %1, 0xffffffff;\n\t"                                                    \
                 "setp.eq.u32 c, %2, 0;\n\t"                                                                    \
                 "selp.u32 %0, m, %0, c;\n\t"                                                                   \
                 "}"                                                                                             \
                 : "+r"(mine[E]) : "r"(head[E]), "r"(lr))
    const int full = rounds - 1;
    int r = 0;
    int lr = lane;                                    /* lane - r: lane r keeps the minimum of round r */
    /* the usual list lengths straight-line: the rolled loop below spends 13 of its 61 instructions per four rounds on
     * loop-carried register moves, the convergence check in front of the first REDUX and the counter */
#define NB_SEL_ROUNDS4(A, B, C, D)                                      \
    _Pragma("unroll") for (int e = 0; e < NEDG; e++) NB_SEL_ROUND(e, A); \
    _Pragma("unroll") for (int e = 0; e < NEDG; e++) NB_SEL_ROUND(e, B); \
    _Pragma("unroll") for (int e = 0; e < NEDG; e++) NB_SEL_ROUND(e, C); \
    _Pragma("unroll") for (int e = 0; e < NEDG; e++) NB_SEL_ROUND(e, D);
    if (full == 20 || full == 16) {
        NB_SEL_ROUNDS4(0, 1, 2, 3) NB_SEL_ROUNDS4(4, 5, 6, 7) NB_SEL_ROUNDS4(8, 9, 10, 11) NB_SEL_ROUNDS4(12, 13, 14, 15)
        if (full == 20) { NB_SEL_ROUNDS4(16, 17, 18, 19) }
        r = full; lr = lane - full;
    }
#pragma unroll 1
    for (; r + 4 <= full; r += 4) {
#pragma unroll
        for (int e = 0; e < NEDG; e++) NB_SEL_ROUND(e, 0);
#pragma unroll
        for (int e = 0; e < NEDG; e++) NB_SEL_ROUND(e, 1);
#pragma unroll
        for (int e = 0; e < NEDG; e++) NB_SEL_ROUND(e, 2);
#pragma unroll
        for (int e = 0; e < NEDG; e++) NB_SEL_ROUND(e, 3);
        lr -= 4;
    }
#pragma unroll 1
    for (; r < full; r++) {
#pragma unroll
        for (int e = 0; e < NEDG; e++) NB_SEL_ROUND(e, 0);
        lr -= 1;
    }
#pragma unroll
    for (int e = 0; e < NEDG; e++) NB_SEL_PEEK(e);
    }
    __syncwarp();
#pragma unroll
    for (int e = 0; e < NEDG; e++) {
        /* lane k: k-th winner; lanes >= rounds hold a copy of the last one (or +inf), which no test below looks at */
        const uint32_t after = __shfl_down_sync(NB_FULL, mine[e], 1);
        const bool amb = lane < n_m && lane + 1 < rounds && ((mine[e] >> LOGQ) == (after >> LOGQ));
        int sym = int(mine[e] & uint32_t(Q - 1));
        /* the exact value: kept bits from the key, dropped bits from the lane that owns the symbol */
        uint32_t vb;
        if constexpr (Q == 256) {
            const int owner = (sym >> 2) & 31;
            const uint32_t wa = __shfl_sync(NB_FULL, lo[e][0], owner), wb = __shfl_sync(NB_FULL, lo[e][1], owner);
            vb = __byte_perm(mine[e], __byte_perm(wa, wb, (uint32_t)((sym & 3) | ((sym >> 5) & 4))), 0x3214);
        } else if constexpr (Q == 64) {
            const uint32_t w = __shfl_sync(NB_FULL, lo[e][0], sym >> 1);
            vb = (mine[e] & ~63u) | ((w >> (8 * (sym & 1))) & 63u);
        } else {
            vb = __float_as_uint(__shfl_sync(NB_FULL, mvc[e][0], sym));
        }
        float val = __uint_as_float(vb);
        const bool over = lane < n_m && !(val < NB_SENT);
        if (__any_sync(NB_FULL, bad[e] || amb || over)) {                      /* rare: one vote on the common path */
        const unsigned ambs = __ballot_sync(NB_FULL, amb);
        if (ambs && !(ambs >> (n_m - 1)) && !__any_sync(NB_FULL, bad[e] || over)) {
            /* winners whose kept bits coincide, none of them at the n_m boundary: the SET is right (equal kept bits are
             * contiguous in key order), only the order inside such runs needs the full (value, symbol) comparison --
             * odd-even transposition over the n_m lanes until nothing moves */
            bool moved;
            do {
                moved = false;
#pragma unroll
                for (int par = 0; par < 2; par++) {
                    const bool left = (lane & 1) == par;
                    const int partner = left ? lane + 1 : lane - 1;
                    const float pv = __shfl_sync(NB_FULL, val, partner & 31);
                    const int ps = __shfl_sync(NB_FULL, sym, partner & 31);
                    const bool less = pv < val || (pv == val && ps < sym);
                    const bool sw = lane < n_m && partner >= 0 && partner < n_m && (left ? less : !less);
                    if (sw) { val = pv; sym = ps; }
                    moved |= sw;
                }
            } while (__any_sync(NB_FULL, moved));
        } else {
            /* exact scan, NB_LDPC.c:356-369.  Inside a lane the slots ascend in symbol, so strict '<' keeps the lowest */
            if (slow_counter && lane == 0) atomicAdd(slow_counter, 1u);
            float tmp[VPL];
#pragma unroll
            for (int j = 0; j < VPL; j++) tmp[j] = mvc[e][j];
            for (int k = 0; k < n_m; k++) {
                float bv = NB_SENT; int bg = 0x7fffffff;
#pragma unroll
                for (int j = 0; j < VPL; j++) if (active && tmp[j] < bv) { bv = tmp[j]; bg = QTraits<Q>::sym(lane, j); }
                warp_lexmin(bv, bg);
                if (bg == 0x7fffffff) bg = 0;                      /* nothing below 1e5: (1e5, symbol 0) */
#pragma unroll
                for (int j = 0; j < VPL; j++) if (active && bg == QTraits<Q>::sym(lane, j)) tmp[j] = NB_SENT;   /* NB_LDPC.c:368 */
                if (lane == k) { val = bv; sym = bg; }
            }
        }
        }
        const float v0 = __shfl_sync(NB_FULL, val, 0);
        out_llr[e] = (lane == 0) ? 0.0f : __fsub_rn(val, v0);                               /* NB_LDPC.c:372-373 */
        out_sym[e] = sym;
    }
    __syncwarp();
}

/*
 * ElementaryStep (bubble_decoder.c:316-593), one thread per step; all lists live in shared memory and
 * are addressed by 32-bit shared-window addresses.
 * A list is n_m f32 LLRs at 'l', n_m u8 symbols at 's', and a length: entries >= len are "absent"
 * (reference: LLR 1e5, symbol -1); their LLR slot holds 1e5 so that sums with them are >= 1e5 exactly
 * as in tab_aux.  Symbols are binary images: ADDGF == XOR.  The "already output" set is a q-bit mask:
 * registers for q <= 64, q/32 words 128 bytes apart in shared memory for q = 256.
 * Eight bubbles (nb_bubble = 8, :327): p < 4 walks row p to the right, p >= 4 walks column p-4 down
 * from row 4 (:445-460, :548-555).  Pop = first strictly smallest candidate below 1e5, else bubble 0
 * (minimum(), :38-56).
 */
#define NB_BV_UPDATE(P) asm("{\n\t.reg .pred q;\n\tsetp.eq.s32 q, %2, " #P ";\n\tselp.f32 %0, %1, %0, q;\n\t}" : "+f"(bv[P]) : "f"(nv), "r"(bp))
template <int Q>
__device__ __forceinline__ int es_serial(uint32_t l1, uint32_t s1, int len1, uint32_t l2, uint32_t s2, int len2,
                                         uint32_t lo, uint32_t so, uint32_t mask, int n_m, int nb_oper)
{
    float bv[8];
    unsigned long long seen = 0ull;
    uint32_t seen32 = 0u;                                  /* q <= 32: one word */
    if constexpr (Q > 64) {
#pragma unroll
        for (int w = 0; w < Q / 32; w++) sts_u32(mask + w * 128, 0u);
    }
    {
        const float a4 = lds_f32(l1 + 16), b0 = lds_f32(l2);
        bv[0] = __fadd_rn(lds_f32(l1), b0); bv[1] = __fadd_rn(lds_f32(l1 + 4), b0);
        bv[2] = __fadd_rn(lds_f32(l1 + 8), b0); bv[3] = __fadd_rn(lds_f32(l1 + 12), b0);
        bv[4] = __fadd_rn(a4, b0); bv[5] = __fadd_rn(a4, lds_f32(l2 + 4));
        bv[6] = __fadd_rn(a4, lds_f32(l2 + 8)); bv[7] = __fadd_rn(a4, lds_f32(l2 + 12));
    }
    /* walk coordinate of each bubble, 8 bits each: column j for p<4 (starts 0), row i for p>=4 (starts 4) */
    uint32_t posr = 0u, posc = 0x04040404u;
    int s = 0;
    for (int ss = 0; ss < nb_oper; ss++) {
        /* 8-way strict minimum, ties -> lowest bubble (tree of "right < left") */
        const bool c01 = bv[1] < bv[0], c23 = bv[3] < bv[2], c45 = bv[5] < bv[4], c67 = bv[7] < bv[6];
        const float m01 = c01 ? bv[1] : bv[0], m23 = c23 ? bv[3] : bv[2], m45 = c45 ? bv[5] : bv[4], m67 = c67 ? bv[7] : bv[6];
        const int i01 = c01 ? 1 : 0, i23 = c23 ? 3 : 2, i45 = c45 ? 5 : 4, i67 = c67 ? 7 : 6;
        const bool c03 = m23 < m01, c47 = m67 < m45;
        const float m03 = c03 ? m23 : m01, m47 = c47 ? m67 : m45;
        const int i03 = c03 ? i23 : i01, i47 = c47 ? i67 : i45;
        const bool c07 = m47 < m03;
        float val = c07 ? m47 : m03;
        int bp = c07 ? i47 : i03;
        if (!(val < NB_SENT)) { bp = 0; val = bv[0]; }
        const bool isrow = bp < 4;
        const uint32_t sh = 8u * (bp & 3);
        const int c = int(((isrow ? posr : posc) >> sh) & 0xffu);
        const int i = isrow ? bp : c;
        const int j = isrow ? c : bp - 4;
        if (i >= len1 || j >= len2) break;                                  /* :478-484 */
        const uint32_t g = lds_u8(s1 + i) ^ lds_u8(s2 + j);                 /* :486 */
        bool fresh;
        if constexpr (Q > 64) {
            const uint32_t wa = mask + (g >> 5) * 128;
            const uint32_t w = lds_u32(wa), bit = 1u << (g & 31);
            fresh = !(w & bit);
            if (fresh) sts_u32(wa, w | bit);
        } else if constexpr (Q > 32) {
            fresh = !((seen >> g) & 1ull);
            seen |= 1ull << g;
        } else {
            const uint32_t bit = 1u << g;
            fresh = !(seen32 & bit);
            seen32 |= bit;
        }
        if (fresh) { sts_f32(lo + 4 * s, val); sts_u8(so + s, g); s++; }     /* :490-496 */
        if (s == n_m) break;                                                /* :502 */
        if (i >= n_m - 1 || j >= n_m - 1) break;                            /* :506-544 */
        const uint32_t inc = 1u << sh;                                      /* :548-555 */
        posr += isrow ? inc : 0u;
        posc += isrow ? 0u : inc;
        const int ni = isrow ? i : i + 1;
        const int nj = isrow ? j + 1 : j;
        const float nv = __fadd_rn(lds_f32(l1 + 4 * ni), lds_f32(l2 + 4 * nj));   /* :557 */
        NB_BV_UPDATE(0); NB_BV_UPDATE(1); NB_BV_UPDATE(2); NB_BV_UPDATE(3);
        NB_BV_UPDATE(4); NB_BV_UPDATE(5); NB_BV_UPDATE(6); NB_BV_UPDATE(7);
    }
    for (int k = s; k < n_m; k++) sts_f32(lo + 4 * k, NB_SENT);             /* :370-374 */
    return s;
}
