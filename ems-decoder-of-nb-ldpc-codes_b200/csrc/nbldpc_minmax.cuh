/*
 * nbldpc_minmax.cuh -- the Min-Max check node (ecn_kind = 4) on the GPU (sm_100a), one WARP per check node.
 *
 * include/nbldpc_b200.h states the node exactly.  For the node's edges e = 0 .. dc-1 with coefficient h_e:
 *   mm_in   w_e = Mvc_e - mu_e, rotated into the check domain (u_e[img(h_e x)] = w_e[x]) straight into the warp's U row e;
 *   mm_bwd  the backward partials bwd_e = u_{e+1} (*) ... (*) u_{dc-1} into dc-1 scratch rows (the node's dense CtoV rows:
 *           their old values are dead once every Mvc has been formed);
 *   mm_out  t_e = fwd_e (*) bwd_e with fwd_e = u_0 (*) ... (*) u_{e-1} kept in registers, back to the variable domain
 *           (CtoV_e[x] = t_e[img(h_e x)]) through the warp's permutation row.
 * (*) is the min-max convolution over XOR, (A (*) B)[z] = min_a max(A[a], B[a ^ z]).  It is associative and commutative and
 * every result is one of its inputs, so the order of evaluation does not change a bit: the convolutions with the identity
 * (fwd_0, bwd_{dc-1}) are skipped, and a node costs 3 (dc - 2) convolutions.
 *
 * mm_conv holds A in registers in the row layout of QTraits<Q>::sym and B in a shared-memory row, which is in symbol order
 * (lds_row / sts_row).  For a candidate a held by lane l in slot J, lane L needs B[a ^ z] for its own z: for q = 256 that is
 * the 16-byte chunks at words 4 (L ^ l) and 128 + 4 (L ^ l) with the slots permuted by J (bit 2 of J swaps the chunks, bits
 * 0-1 permute inside them), so two conflict-free LDS.128 and a permutation fixed at compile time; for q = 64 one LDS.64
 * at word 2 (L ^ l), for q = 16 one word (lanes 16-31 idle).  A[a] is one shuffle from lane l.
 *
 * Pruning, exact: every running value C[z] is the max of some candidate pair, so it bounds the final C[z] from above, and
 * so does T = max_z C[z].  A candidate with A[a] >= T gives max(A[a], .) >= T for every z and cannot lower any C[z]: it is
 * skipped.  Candidates are taken slot by slot from a ballot of A[.] < T, and T is refreshed every MM_REFRESH candidates.
 * All values are >= +0 (w = Mvc - mu, and every result is one of them), so the warp maxima of T are integer REDUX on the
 * bit patterns.  Pruning changes the cost, never the bits.
 */
#pragma once
#include "nbldpc_device.cuh"
#include "nbldpc_spa.cuh"         /* SpaMem (the dense nodes' warp rows), sts_row */

#define MM_REFRESH 4              /* candidates between two refreshes of the pruning bound T */

/* C[z] = min(C[z], max(av, B[a ^ z])) for the candidate a = sym(l, J), B the shared row brow in symbol order */
template <int Q, int J>
__device__ __forceinline__ void mm_cand(float av, int l, uint32_t brow, int lane, float (&c)[QTraits<Q>::VPL])
{
    if constexpr (Q == 256) {
        float b[8];
        const uint32_t p = brow + 16u * (uint32_t)(l ^ lane);
        asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(b[0]), "=f"(b[1]), "=f"(b[2]), "=f"(b[3]) : "r"(p));
        asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4+512];" : "=f"(b[4]), "=f"(b[5]), "=f"(b[6]), "=f"(b[7]) : "r"(p));
#pragma unroll
        for (int i = 0; i < 8; i++) c[i] = fminf(c[i], fmaxf(av, b[i ^ J]));
    } else if constexpr (Q == 64) {
        float b[2];
        asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(b[0]), "=f"(b[1]) : "r"(brow + 8u * (uint32_t)(l ^ lane)));
#pragma unroll
        for (int i = 0; i < 2; i++) c[i] = fminf(c[i], fmaxf(av, b[i ^ J]));
    } else {
        c[0] = fminf(c[0], fmaxf(av, lds_f32(brow + 4u * (uint32_t)((l ^ lane) & 15))));
    }
}

/* the pruning bound: warp max of the running C over the active lanes (all values >= +0: integer order is float order) */
template <int Q>
__device__ __forceinline__ float mm_bound(const float (&c)[QTraits<Q>::VPL], int lane)
{
    uint32_t m = 0;
#pragma unroll
    for (int i = 0; i < QTraits<Q>::VPL; i++) m = max(m, __float_as_uint(c[i]));
    return __uint_as_float(__reduce_max_sync(NB_FULL, (Q >= 32 || lane < Q) ? m : 0u));
}

template <int Q, int J>
__device__ __forceinline__ void mm_slot(const float (&A)[QTraits<Q>::VPL], uint32_t brow, int lane, float (&c)[QTraits<Q>::VPL])
{
    const bool active = (Q >= 32) || lane < Q;
    float T = mm_bound<Q>(c, lane);
    uint32_t m = __ballot_sync(NB_FULL, active && A[J] < T);
    for (int n = 1; m; n++) {
        const int l = __ffs(m) - 1;
        m &= m - 1;
        mm_cand<Q, J>(__shfl_sync(NB_FULL, A[J], l), l, brow, lane, c);
        if (n % MM_REFRESH == 0 && m) { T = mm_bound<Q>(c, lane); m &= __ballot_sync(NB_FULL, active && A[J] < T); }
    }
}

/* c = A (*) B: A in registers (row layout), B the shared row brow (symbol order) */
template <int Q>
__device__ __forceinline__ void mm_conv(const float (&A)[QTraits<Q>::VPL], uint32_t brow, int lane, float (&c)[QTraits<Q>::VPL])
{
#pragma unroll
    for (int i = 0; i < QTraits<Q>::VPL; i++) c[i] = __int_as_float(0x7f800000);
    mm_slot<Q, 0>(A, brow, lane, c);
    if constexpr (Q >= 64) mm_slot<Q, 1>(A, brow, lane, c);
    if constexpr (Q == 256) {
        mm_slot<Q, 2>(A, brow, lane, c); mm_slot<Q, 3>(A, brow, lane, c); mm_slot<Q, 4>(A, brow, lane, c);
        mm_slot<Q, 5>(A, brow, lane, c); mm_slot<Q, 6>(A, brow, lane, c); mm_slot<Q, 7>(A, brow, lane, c);
    }
}

/* steps 2-3 for edge e: Mvc row (symbol order, row layout) -> U row e (check domain) */
template <int Q, bool CLOSED>
__device__ __forceinline__ void mm_in(const SpaMem &sp, int e, const float (&mvc)[QTraits<Q>::VPL], int h, const GFTab &gf, int lane)
{
    constexpr int VPL = QTraits<Q>::VPL;
    const bool active = (Q >= 32) || lane < Q;
    float mu = __int_as_float(0x7f800000);
#pragma unroll
    for (int j = 0; j < VPL; j++) if (active) mu = fminf(mu, mvc[j]);
#pragma unroll
    for (int o = 16; o; o >>= 1) mu = fminf(mu, __shfl_xor_sync(NB_FULL, mu, o));
    const uint32_t u = sp.urow + (uint32_t)(e * Q * 4);
#pragma unroll
    for (int j = 0; j < VPL; j++)
        if (active) sts_f32(u + 4 * gf_rot_in<Q, CLOSED>(gf, QTraits<Q>::sym(lane, j), h), __fsub_rn(mvc[j], mu));
    __syncwarp();
}

/* step 4, backward half: scr + e * Q (global, row layout) = u_{e+1} (*) ... (*) u_{dc-1} for e = 0 .. dc-2 */
template <int Q>
__device__ __forceinline__ void mm_bwd(const SpaMem &sp, int dc, float *scr, int lane)
{
    constexpr int VPL = QTraits<Q>::VPL;
    float b[VPL];
    lds_row<Q>(sp.urow + (uint32_t)((dc - 1) * Q * 4), lane, b);
    for (int e = dc - 2;; e--) {
        store_row<Q>(scr + (size_t)e * Q, lane, b);
        if (e == 0) break;
        float c[VPL];
        mm_conv<Q>(b, sp.urow + (uint32_t)(e * Q * 4), lane, c);
#pragma unroll
        for (int j = 0; j < VPL; j++) b[j] = c[j];
    }
}

/* steps 4-5 for edge e, in edge order: fwd = u_0 (*) ... (*) u_{e-1} on entry (set here for e = 0), u_0 (*) ... (*) u_e on
 * return for e < dc - 1; bwd = the row mm_bwd left for e (not read for e = dc - 1); cv = CtoV_e in symbol order (row layout) */
template <int Q, bool CLOSED>
__device__ __forceinline__ void mm_out(const SpaMem &sp, int e, int dc, const float *bwd, float (&fwd)[QTraits<Q>::VPL], int h,
                                       const GFTab &gf, int lane, float (&cv)[QTraits<Q>::VPL])
{
    constexpr int VPL = QTraits<Q>::VPL;
    const bool active = (Q >= 32) || lane < Q;
    float t[VPL];
    if (e == 0) {
        load_row<Q>(bwd, lane, t);
        lds_row<Q>(sp.urow, lane, fwd);
    } else if (e == dc - 1) {
#pragma unroll
        for (int j = 0; j < VPL; j++) t[j] = fwd[j];
    } else {
        float b[VPL];
        load_row<Q>(bwd, lane, b);
        sts_row<Q>(sp.prow, lane, b);
        __syncwarp();
        mm_conv<Q>(fwd, sp.prow, lane, t);
        mm_conv<Q>(fwd, sp.urow + (uint32_t)(e * Q * 4), lane, b);
#pragma unroll
        for (int j = 0; j < VPL; j++) fwd[j] = b[j];
        __syncwarp();
    }
    sts_row<Q>(sp.prow, lane, t);
    __syncwarp();
#pragma unroll
    for (int j = 0; j < VPL; j++)
        cv[j] = active ? lds_f32(sp.prow + 4 * gf_rot_in<Q, CLOSED>(gf, QTraits<Q>::sym(lane, j), h)) : 0.0f;
    __syncwarp();
}
