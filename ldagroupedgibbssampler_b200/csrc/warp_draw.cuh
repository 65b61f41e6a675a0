// warp_draw.cuh -- the categorical draw of the register path (K <= 1024) shared by the z-step (kernels_z.cu) and
// the held-out estimator (kernels_heldout.cu): scores, the lane-local fma prefix, the Kogge-Stone warp scan of the
// lane totals and the lane -> tile -> element search (contract: DESIGN.md 4.2).
#pragma once
#include "common.cuh"

namespace ldagpu {

constexpr unsigned FULL = 0xffffffffu;
template <int NT> __device__ __forceinline__ int pos_of(int k) { return tpos_lg(lg_of_tiles(NT), k); }

template <int NT> struct RowScan {
    float p[NT][4];   // lane-local inclusive prefix over the lane's 4*NT consecutive topics (p[NT-1][3] = lane total)
    float inc, prev;  // inclusive scan of the lane totals at this lane, and at the lane before (0 for lane 0)
    float S;          // total
};

// Scores, lane-local prefix, warp scan of the lane totals (contract: DESIGN.md 4.2).
// The first NREG tiles of the per-document vector come from registers, the others from the lane's float4 in shared
// memory (a_sm[(j - NREG) * 32 + lane]): at 8 tiles theta (32 registers) and the prefixes (32) do not fit 80
// registers together, and two LDS.128 per run are cheaper than the eight local-memory reloads the compiler spills to.
template <int NT, int NREG>
__device__ __forceinline__ void scan_scores(const float4 (&a)[NREG], const float4 *a_sm, const float4 (&ph)[NT],
                                            RowScan<NT> &rs, int lane)
{
    float run = 0.0f;
#pragma unroll
    for (int j = 0; j < NT; ++j) {
        float4 aj;
        if (j < NREG) aj = a[j < NREG ? j : 0];
        else aj = a_sm[(j - NREG) * 32 + lane];
        // one product starts the lane's chain, every other topic is one fused multiply-add
        const float p0 = j == 0 ? __fmul_rn(aj.x, ph[j].x) : __fmaf_rn(aj.x, ph[j].x, run);
        const float p1 = __fmaf_rn(aj.y, ph[j].y, p0);
        const float p2 = __fmaf_rn(aj.z, ph[j].z, p1);
        const float p3 = __fmaf_rn(aj.w, ph[j].w, p2);
        rs.p[j][0] = p0; rs.p[j][1] = p1; rs.p[j][2] = p2; rs.p[j][3] = p3;
        run = p3;
    }
    float inc = run;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const float y = __shfl_up_sync(FULL, inc, off);
        if (lane >= off) inc = __fadd_rn(inc, y);
    }
    float prev = __shfl_up_sync(FULL, inc, 1);
    if (lane == 0) prev = 0.0f;
    rs.inc = inc;
    rs.prev = prev;
    rs.S = __shfl_sync(FULL, inc, 31);
}

// first k with cumsum_k >= U * sum, searched lane -> tile -> element; returns the topic (natural order)
template <int NT>
__device__ __forceinline__ int draw_topic(const RowScan<NT> &rs, float U, int lane, int K)
{
    const float u = __fmul_rn(U, rs.S);
    const unsigned m = __ballot_sync(FULL, rs.inc >= u);
    const int ls = m ? __ffs(m) - 1 : 31;
    const float r = __fsub_rn(u, rs.prev);   // the value lane ls needs; the other lanes' results are discarded
    int jsel = 0;
    float q0 = rs.p[0][0], q1 = rs.p[0][1], q2 = rs.p[0][2];
    if (NT > 1) {
        // the prefixes never decrease (scores >= 0): the tiles whose last prefix is < r come first, so their number
        // is a binary search over the NT - 1 tile ends (three dependent compares at 8 tiles instead of seven)
        int jc = 0;
        if (NT == 8) {
            jc = rs.p[3][3] < r ? 4 : 0;
            jc += (jc ? rs.p[5][3] : rs.p[1][3]) < r ? 2 : 0;
            const float lo = (jc & 2) ? rs.p[2][3] : rs.p[0][3], hi = (jc & 2) ? rs.p[6][3] : rs.p[4][3];
            jc += ((jc & 4) ? hi : lo) < r ? 1 : 0;
        } else {
#pragma unroll
            for (int j = 0; j + 1 < NT; ++j) jc += (rs.p[j][3] >= r) ? 0 : 1;
        }
        jsel = __shfl_sync(FULL, jc, ls);   // warp-uniform: a real branch picks the tile's registers
#define LDAGPU_PICK(J)                                                                              \
    case J:                                                                                         \
        if (J < NT) { q0 = rs.p[J < NT ? J : 0][0]; q1 = rs.p[J < NT ? J : 0][1]; q2 = rs.p[J < NT ? J : 0][2]; } \
        break;
        switch (jsel) {
            LDAGPU_PICK(1) LDAGPU_PICK(2) LDAGPU_PICK(3) LDAGPU_PICK(4) LDAGPU_PICK(5) LDAGPU_PICK(6) LDAGPU_PICK(7)
            default: break;
        }
#undef LDAGPU_PICK
    }
    int i = 3;
    if (q2 >= r) i = 2;
    if (q1 >= r) i = 1;
    if (q0 >= r) i = 0;
    const int k = __shfl_sync(FULL, lane * (4 * NT) + 4 * jsel + i, ls);
    return k < K ? k : K - 1;
}

}  // namespace ldagpu
