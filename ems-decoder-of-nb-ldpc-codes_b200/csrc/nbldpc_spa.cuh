/*
 * nbldpc_spa.cuh -- the sum-product check node (ecn_kind = 2) on the GPU (sm_100a), one WARP per check node.
 *
 * The q-ary sum-product (belief-propagation) update in the Walsh-Hadamard domain; include/nbldpc_b200.h states it exactly.
 * For the node's edges e = 0 .. dc-1 with coefficient h_e:
 *   spa_in   p_e[x] = E(mu_e - Mvc_e[x]), rotated into the check domain (u_e[img(h_e x)] = p_e[x]) through the warp's
 *            permutation row, U_e = WHT(u_e) * (1 / U_e[0]), parked in the warp's U row e (shared memory);
 *   spa_bwd  the backward products bwd_e = U_{dc-1} ... U_{e+1} into dc scratch rows (the node's dense CtoV rows: their
 *            old values are dead once every Mvc has been formed);
 *   spa_out  T_e = fwd_e * bwd_e with fwd_e = U_0 ... U_{e-1} kept in registers, t_e = WHT(T_e), back to the variable
 *            domain (c_e[x] = t_e[img(h_e x)]) through the permutation row, capped at tau c_max,
 *            CtoV_e[x] = L(c_max) - L(c_e[x]).
 * A row lives in the row layout of QTraits<Q>::sym: for q = 256 index bits 0, 1 and 7 are inside a lane and bits 2-6
 * across lanes, for q = 64 bit 0 inside and bits 1-5 across, for q = 16 bits 0-3 across (lanes 16-31 idle).  The WHT
 * stages across lanes are shfl_xor.  Every lane reads and writes only its own slots of the U rows and the scratch rows;
 * only the permutations cross lanes.
 */
#pragma once
#include "nbldpc_device.cuh"
#include "nbldpc_spa_math.h"

#define NB_SPA_TAU 0x1p-20f       /* c_e[x] >= tau * c_max: smaller values are f32 round-off of the transform */

/* a warp's shared memory for the sum-product node: U rows [dc_max][q] f32 and one permutation row [q] f32 */
struct SpaMem {
    uint32_t urow, prow;
};

/* the row store that mirrors lds_row (conflict-free 128-bit moves) */
template <int Q> __device__ __forceinline__ void sts_row(uint32_t row, int lane, const float (&v)[QTraits<Q>::VPL])
{
    if constexpr (Q == 256) {
        const uint32_t a = row + lane * 16;
        asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" :: "r"(a), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]) : "memory");
        asm volatile("st.shared.v4.f32 [%0+512], {%1,%2,%3,%4};" :: "r"(a), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]) : "memory");
    } else if constexpr (Q == 64) {
        asm volatile("st.shared.v2.f32 [%0], {%1,%2};" :: "r"(row + lane * 8), "f"(v[0]), "f"(v[1]) : "memory");
    } else {
        if (lane < Q) sts_f32(row + 4 * lane, v[0]);
    }
}

/* one butterfly stage inside a lane: slots j and j | JM hold indices that differ in one bit, (a + b, a - b) */
template <int VPL, int JM> __device__ __forceinline__ void spa_stage_lane(float (&v)[VPL])
{
#pragma unroll
    for (int j = 0; j < VPL; j++)
        if (!(j & JM)) { const float a = v[j], b = v[j | JM]; v[j] = __fadd_rn(a, b); v[j | JM] = __fsub_rn(a, b); }
}
/* one butterfly stage across lanes lane and lane ^ LM: the lower lane keeps a + b, the upper a - b */
template <int VPL> __device__ __forceinline__ void spa_stage_shfl(float (&v)[VPL], int lane, int lm)
{
    const bool hi = (lane & lm) != 0;
#pragma unroll
    for (int j = 0; j < VPL; j++) {
        const float o = __shfl_xor_sync(NB_FULL, v[j], lm);
        v[j] = hi ? __fsub_rn(o, v[j]) : __fadd_rn(v[j], o);
    }
}
/* WHT without scaling, stage s = 0 .. log2 q - 1 pairing the indices that differ in bit s */
template <int Q> __device__ __forceinline__ void spa_wht(float (&v)[QTraits<Q>::VPL], int lane)
{
    constexpr int VPL = QTraits<Q>::VPL;
    if constexpr (Q == 256) {
        spa_stage_lane<VPL, 1>(v); spa_stage_lane<VPL, 2>(v);
#pragma unroll
        for (int lm = 1; lm < 32; lm <<= 1) spa_stage_shfl<VPL>(v, lane, lm);
        spa_stage_lane<VPL, 4>(v);
    } else if constexpr (Q == 64) {
        spa_stage_lane<VPL, 1>(v);
#pragma unroll
        for (int lm = 1; lm < 32; lm <<= 1) spa_stage_shfl<VPL>(v, lane, lm);
    } else {
#pragma unroll
        for (int lm = 1; lm < 16; lm <<= 1) spa_stage_shfl<VPL>(v, lane, lm);
    }
}

/* steps 2-4 for edge e: Mvc row (symbol order, row layout) -> U row e */
template <int Q, bool CLOSED>
__device__ __forceinline__ void spa_in(const SpaMem &sp, int e, const float (&mvc)[QTraits<Q>::VPL], int h, const GFTab &gf, int lane)
{
    constexpr int VPL = QTraits<Q>::VPL;
    const bool active = (Q >= 32) || lane < Q;
    float mu = __int_as_float(0x7f800000);
#pragma unroll
    for (int j = 0; j < VPL; j++) if (active) mu = fminf(mu, mvc[j]);
#pragma unroll
    for (int o = 16; o; o >>= 1) mu = fminf(mu, __shfl_xor_sync(NB_FULL, mu, o));
#pragma unroll
    for (int j = 0; j < VPL; j++) {
        const float m = mvc[j];
        const float p = (m >= NB_SENT && m > mu) ? 0.0f : nb_spa_exp(__fsub_rn(mu, m));     /* absent values other than the minimum */
        if (active) sts_f32(sp.prow + 4 * gf_rot_in<Q, CLOSED>(gf, QTraits<Q>::sym(lane, j), h), p);
    }
    __syncwarp();
    float u[VPL];
    lds_row<Q>(sp.prow, lane, u);
    __syncwarp();
    spa_wht<Q>(u, lane);
    const float r = __fdiv_rn(1.0f, __shfl_sync(NB_FULL, u[0], 0));        /* index 0 is slot 0 of lane 0 in every layout */
#pragma unroll
    for (int j = 0; j < VPL; j++) u[j] = __fmul_rn(u[j], r);
    sts_row<Q>(sp.urow + (uint32_t)(e * Q * 4), lane, u);
}

/* step 5, backward half: scr + e * Q (global, row layout) = U_{dc-1} * ... * U_{e+1} (1 for e = dc-1) */
template <int Q>
__device__ __forceinline__ void spa_bwd(const SpaMem &sp, int dc, float *scr, int lane)
{
    constexpr int VPL = QTraits<Q>::VPL;
    float b[VPL];
#pragma unroll
    for (int j = 0; j < VPL; j++) b[j] = 1.0f;
    for (int e = dc - 1; e >= 0; e--) {
        store_row<Q>(scr + (size_t)e * Q, lane, b);
        if (e == 0) break;
        float u[VPL];
        lds_row<Q>(sp.urow + (uint32_t)(e * Q * 4), lane, u);
#pragma unroll
        for (int j = 0; j < VPL; j++) b[j] = __fmul_rn(b[j], u[j]);
    }
}

/* steps 5-7 for edge e, in edge order: fwd = U_0 * ... * U_{e-1} on entry (all 1 for e = 0), U_0 * ... * U_e on return;
 * bwd = the row spa_bwd left for e; cv = CtoV_e in symbol order (row layout) */
template <int Q, bool CLOSED>
__device__ __forceinline__ void spa_out(const SpaMem &sp, int e, const float *bwd, float (&fwd)[QTraits<Q>::VPL], int h, const GFTab &gf,
                                        int lane, float (&cv)[QTraits<Q>::VPL])
{
    constexpr int VPL = QTraits<Q>::VPL;
    const bool active = (Q >= 32) || lane < Q;
    float t[VPL], u[VPL];
    load_row<Q>(bwd, lane, t);
    lds_row<Q>(sp.urow + (uint32_t)(e * Q * 4), lane, u);
#pragma unroll
    for (int j = 0; j < VPL; j++) { t[j] = __fmul_rn(fwd[j], t[j]); fwd[j] = __fmul_rn(fwd[j], u[j]); }
    spa_wht<Q>(t, lane);
    float cmax = -__int_as_float(0x7f800000);
#pragma unroll
    for (int j = 0; j < VPL; j++) if (active) cmax = fmaxf(cmax, t[j]);
#pragma unroll
    for (int o = 16; o; o >>= 1) cmax = fmaxf(cmax, __shfl_xor_sync(NB_FULL, cmax, o));
    sts_row<Q>(sp.prow, lane, t);
    __syncwarp();
    const float floor_c = __fmul_rn(cmax, NB_SPA_TAU), lmax = nb_spa_log(cmax);
#pragma unroll
    for (int j = 0; j < VPL; j++) {
        const float c = active ? lds_f32(sp.prow + 4 * gf_rot_in<Q, CLOSED>(gf, QTraits<Q>::sym(lane, j), h)) : cmax;
        cv[j] = __fsub_rn(lmax, nb_spa_log(fmaxf(c, floor_c)));
    }
    __syncwarp();
}
