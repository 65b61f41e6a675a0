// kernels_z_big.cu -- the dense z-step and theta draw for K > 1024 (more than 8 tiles per row).
//
// Same arithmetic contract as kernels_z.cu (DESIGN.md 4.2-4.3) -- the tile totals are formed 8 tiles at
// a time with a carry between groups -- but a Phi^T row no longer fits in registers: the row, and the
// per-document vector it is multiplied with (theta for GGS, n_dk + alpha for PCGS), stay in shared
// memory; a run first computes the cumulative tile totals of all groups, then each token of the run
// locates its group, tile and lane and recomputes the 4 prefix values of that one tile.
// Correct for any K the shared memory can hold (K <= ~28 000 GGS, ~18 000 PCGS); it is the reference's
// dense O(K) per token loop, so for K = 10 000 it is 40 KB of Phi per token -- the sparse z-step
// (SURVEY 8f row 1) is the intended path there.
//
// Replaces: topics/LDAGroupedGibbsSampler.java:47-132, topics/UncollapsedParallelLDA.java:1466-1545.
#include "common.cuh"
#include "contract_math.cuh"

namespace ldagpu {

constexpr unsigned FULL = 0xffffffffu;

// cumulative totals of 8 tiles (DESIGN.md 4.2): distributed butterfly, then Kogge-Stone over tiles.
// On return lane l holds the cumulative total through tile (l >> 2) & 7 of the group.
__device__ __forceinline__ float group_totals(const float (&t)[8], int lane)
{
    const bool h16 = (lane & 16) != 0, h8 = (lane & 8) != 0, h4 = (lane & 4) != 0;
    float u[4], v[2];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float keep = h16 ? t[4 + i] : t[i], send = h16 ? t[i] : t[4 + i];
        u[i] = __fadd_rn(keep, __shfl_xor_sync(FULL, send, 16));
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        float keep = h8 ? u[2 + i] : u[i], send = h8 ? u[i] : u[2 + i];
        v[i] = __fadd_rn(keep, __shfl_xor_sync(FULL, send, 8));
    }
    float keep = h4 ? v[1] : v[0], send = h4 ? v[0] : v[1];
    float w = __fadd_rn(keep, __shfl_xor_sync(FULL, send, 4));
    w = __fadd_rn(w, __shfl_xor_sync(FULL, w, 2));
    w = __fadd_rn(w, __shfl_xor_sync(FULL, w, 1));
#pragma unroll
    for (int off = 4; off < 32; off <<= 1) {
        float y = __shfl_up_sync(FULL, w, off);
        if (lane >= off) w = __fadd_rn(w, y);
    }
    return w;
}

struct BigLayout {
    size_t row, vec, cnt, bf, bar, per_warp;
};
__host__ __device__ inline BigLayout big_layout(int NT, bool pcgs)
{
    BigLayout L;
    const size_t rowf = (size_t)NT * TILE, ng = (size_t)(NT + 7) / 8;
    L.row = 0;
    L.vec = L.row + rowf * 4;
    L.cnt = L.vec + rowf * 4;
    L.bf = L.cnt + (pcgs ? rowf * 4 : 0);
    L.bar = L.bf + ng * 32 * 4;
    L.per_warp = (L.bar + 8 + 127) / 128 * 128;
    return L;
}

template <bool PCGS>
__global__ void __launch_bounds__(256) z_kernel_big(ZArgs a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int NT = a.dm.NT, NG = (NT + 7) / 8, K = a.dm.K, Ks = a.dm.Ks;
    const int ROWF = NT * TILE;
    const BigLayout L = big_layout(NT, PCGS);
    unsigned char *wb = smem_raw + (size_t)warp * L.per_warp;
    float *row = reinterpret_cast<float *>(wb + L.row);
    float *vec = reinterpret_cast<float *>(wb + L.vec);
    int *cnt = reinterpret_cast<int *>(wb + L.cnt);
    float *Bf = reinterpret_cast<float *>(wb + L.bf);
    uint64_t *bar = reinterpret_cast<uint64_t *>(wb + L.bar);
    const uint32_t row_bytes = (uint32_t)Ks * 4u;

    for (int i = lane; i < ROWF; i += 32) { row[i] = 0.0f; vec[i] = 0.0f; if (PCGS) cnt[i] = 0; }
    if (lane == 0) { mbar_init(bar, 1); mbar_fence_init(); }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    uint32_t fills = 0;

    for (;;) {
        unsigned long long item = 0;
        if (lane == 0) item = atomicAdd(a.work_counter, 1ull);
        item = __shfl_sync(FULL, item, 0);
        if ((int64_t)item >= a.n_items) break;
        int64_t d = a.item_doc[item], t0, t1;
        if (PCGS) {
            t0 = a.doc_off[d]; t1 = a.doc_off[d + 1];
            if (t0 == t1) continue;
            for (int64_t t = t0 + lane; t < t1; t += 32) atomicAdd(&cnt[a.z[t]], 1);
            __syncwarp();
            for (int k = lane; k < ROWF; k += 32)
                vec[k] = k < K ? __fadd_rn(__int2float_rn(cnt[k]), a.alpha[k]) : 0.0f;
        } else {
            t0 = a.item_begin[item];
            const int64_t de = a.doc_off[d + 1];
            t1 = t0 + a.chunk < de ? t0 + a.chunk : de;
            const float *trow = a.theta + (size_t)d * Ks;
            for (int k = lane; k < ROWF; k += 32) vec[k] = k < Ks ? trow[k] : 0.0f;
        }
        __syncwarp();

        for (int64_t tb = t0; tb < t1; tb += 32) {
            const int64_t t = tb + lane;
            const bool valid = t < t1;
            const int nvalid = (int)((t1 - tb) < 32 ? (t1 - tb) : 32);
            const int w = valid ? a.tokens[t] : -1;
            const int zold = (PCGS && valid) ? a.z[t] : 0;
            const int wprev = __shfl_up_sync(FULL, w, 1);
            unsigned rem = __ballot_sync(FULL, valid && (lane == 0 || w != wprev));
            float U = 0.0f;
            if (valid) {
                unsigned long long gt = (unsigned long long)(a.dm.token_base + t);
                uint4 r = philox4x32_10((uint32_t)gt, (uint32_t)(gt >> 32), a.sweep, STREAM_Z << 24, a.seed_lo, a.seed_hi);
                U = uniform23(r.x);
            }
            int znew = 0;
            while (rem) {
                const int b = __ffs(rem) - 1;
                rem &= rem - 1;
                const int e = rem ? __ffs(rem) - 1 : nvalid;
                const int wrow = __shfl_sync(FULL, w, b);
                __syncwarp();
                if (lane == 0) {
                    mbar_expect_tx(bar, row_bytes);
                    bulk_g2s(row, a.phiT + (size_t)wrow * Ks, row_bytes, bar);
                }
                mbar_wait(bar, fills & 1u);
                ++fills;

                float S = 0.0f;
                bool have_totals = false;
                for (int tt = b; tt < e; ++tt) {
                    if (PCGS) {
                        const int old = __shfl_sync(FULL, zold, tt);
                        if (lane == 0) {
                            const int c = cnt[old] - 1;
                            cnt[old] = c;
                            vec[old] = __fadd_rn(__int2float_rn(c), a.alpha[old]);
                        }
                        __syncwarp();
                    }
                    if (PCGS || !have_totals) {
                        // cumulative tile totals of every group of 8 tiles, with the carry between groups
                        float carry = 0.0f;
                        for (int g = 0; g < NG; ++g) {
                            float tl[8];
#pragma unroll
                            for (int tau = 0; tau < 8; ++tau) {
                                const int j = 8 * g + tau;
                                float p3 = 0.0f;
                                if (j < NT) {
                                    const float4 v = reinterpret_cast<const float4 *>(vec)[j * 32 + lane];
                                    const float4 ph = reinterpret_cast<const float4 *>(row)[j * 32 + lane];
                                    p3 = __fmul_rn(v.x, ph.x);
                                    p3 = __fmaf_rn(v.y, ph.y, p3);
                                    p3 = __fmaf_rn(v.z, ph.z, p3);
                                    p3 = __fmaf_rn(v.w, ph.w, p3);
                                }
                                tl[tau] = p3;
                            }
                            float wv = group_totals(tl, lane);
                            if (g > 0) wv = __fadd_rn(carry, wv);
                            Bf[g * 32 + lane] = wv;
                            carry = __shfl_sync(FULL, wv, 31);
                        }
                        S = carry;
                        have_totals = true;
                        __syncwarp();
                    }
                    // locate group, tile, lane, element
                    const float Ut = __shfl_sync(FULL, U, tt);
                    const float u = __fmul_rn(Ut, S);
                    int g = NG - 1;
                    unsigned mt = 0;
                    for (int gg = 0; gg < NG; ++gg) {
                        mt = __ballot_sync(FULL, Bf[gg * 32 + lane] >= u);
                        if (mt) { g = gg; break; }
                    }
                    int tau = (mt ? __ffs(mt) - 1 : 31) >> 2;
                    int js = 8 * g + tau;
                    if (js > NT - 1) { js = NT - 1; g = js >> 3; tau = js & 7; }
                    const float base = tau > 0 ? Bf[g * 32 + 4 * tau - 1] : (g > 0 ? Bf[(g - 1) * 32 + 31] : 0.0f);
                    const float r = __fsub_rn(u, base);
                    const float4 v = reinterpret_cast<const float4 *>(vec)[js * 32 + lane];
                    const float4 ph = reinterpret_cast<const float4 *>(row)[js * 32 + lane];
                    const float q0 = __fmul_rn(v.x, ph.x);
                    const float q1 = __fmaf_rn(v.y, ph.y, q0);
                    const float q2 = __fmaf_rn(v.z, ph.z, q1);
                    float inc = __fmaf_rn(v.w, ph.w, q2);
#pragma unroll
                    for (int off = 1; off < 32; off <<= 1) {
                        float y = __shfl_up_sync(FULL, inc, off);
                        if (lane >= off) inc = __fadd_rn(inc, y);
                    }
                    const unsigned m = __ballot_sync(FULL, inc >= r);
                    const int ls = m ? __ffs(m) - 1 : 31;
                    float prev = __shfl_up_sync(FULL, inc, 1);
                    if (lane == 0) prev = 0.0f;
                    const float r2 = __fsub_rn(r, prev);
                    int i = 3;
                    if (q2 >= r2) i = 2;
                    if (q1 >= r2) i = 1;
                    if (q0 >= r2) i = 0;
                    int k = __shfl_sync(FULL, TILE * js + 4 * lane + i, ls);
                    if (k > K - 1) k = K - 1;
                    if (lane == tt) znew = k;
                    if (PCGS) {
                        if (lane == 0) {
                            const int c = cnt[k] + 1;
                            cnt[k] = c;
                            vec[k] = __fadd_rn(__int2float_rn(c), a.alpha[k]);
                        }
                        __syncwarp();
                    }
                }
            }
            if (valid) {
                a.z[t] = znew;
                if (a.n_wk_out) atomicAdd(&a.n_wk_out[(size_t)w * Ks + znew], 1);
            }
        }
        if (PCGS) {
            for (int i = lane; i < ROWF; i += 32) cnt[i] = 0;
            __syncwarp();
        }
    }
}

template <bool PCGS> static cudaError_t launch_big(const ZArgs &a, int sm_count, cudaStream_t st)
{
    if (a.n_items == 0) return cudaSuccess;
    const BigLayout L = big_layout(a.dm.NT, PCGS);
    int warps = (int)((size_t)(226 * 1024) / L.per_warp);
    if (warps < 1) return cudaErrorInvalidValue;   // K too large for one row + vector in shared memory
    if (warps > 8) warps = 8;
    const size_t smem = (size_t)warps * L.per_warp;
    cudaError_t e = cudaFuncSetAttribute(z_kernel_big<PCGS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int per_sm = 1;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, z_kernel_big<PCGS>, warps * 32, smem);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    int64_t grid = (int64_t)sm_count * per_sm;
    const int64_t need = (a.n_items + warps - 1) / warps;
    if (need < grid) grid = need;
    z_kernel_big<PCGS><<<(unsigned)grid, warps * 32, smem, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_z_ggs_big(const ZArgs &a, int sm_count, cudaStream_t st) { return launch_big<false>(a, sm_count, st); }
cudaError_t launch_z_pcgs_big(const ZArgs &a, int sm_count, cudaStream_t st) { return launch_big<true>(a, sm_count, st); }

// ---------------------------------------------------------------------------------------
// theta for K > 1024: one warp per document, cells drawn with the plain per-cell loop
// (c_gamma); the normalising sum follows the contract (lane-sequential over the lane's cells in
// (tile, element) order, then xor butterfly).  Values in shared memory: 4*ROWF bytes per warp.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) theta_kernel_big(ThetaArgs a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int NT = a.dm.NT, K = a.dm.K, Ks = a.dm.Ks, ROWF = NT * TILE;
    int *cg = reinterpret_cast<int *>(smem_raw) + (size_t)warp * ROWF;
    for (int i = lane; i < ROWF; i += 32) cg[i] = 0;
    __syncwarp();
    for (;;) {
        unsigned long long dd = 0;
        if (lane == 0) dd = atomicAdd(a.work_counter, 1ull);
        dd = __shfl_sync(FULL, dd, 0);
        if ((int64_t)dd >= a.dm.D) break;
        const int64_t d = (int64_t)dd, t0 = a.doc_off[d], t1 = a.doc_off[d + 1];
        float *trow = a.theta + (size_t)d * Ks;
        if (t0 == t1) {
            for (int i = lane; i < Ks; i += 32) trow[i] = 0.0f;
            continue;
        }
        for (int64_t t = t0 + lane; t < t1; t += 32) atomicAdd(&cg[a.z[t]], 1);
        __syncwarp();
        const unsigned long long cell0 = (unsigned long long)(a.dm.doc_base + d) * (unsigned long long)K;
        float acc = 0.0f;
        for (int q = 0; q < NT * 4; ++q) {
            const int k = (q >> 2) * TILE + lane * 4 + (q & 3);
            float gv = 0.0f;
            if (k < K) {
                gv = c_gamma<float>(__fadd_rn(__int2float_rn(cg[k]), a.alpha[k]), a.seed_lo, a.seed_hi,
                                    cell0 + (unsigned long long)k, a.sweep, STREAM_THETA);
                if (K > MAX_REG_TILES * TILE) acc = __fadd_rn(acc, gv);
            }
            cg[k] = __float_as_int(gv);
        }
        __syncwarp();
        if (K <= MAX_REG_TILES * TILE) {
            // the sparse scheme's rows at K <= 1024: the contract sums over the lane's L consecutive topics, L = 4 x the
            // register path's tile count (DESIGN.md 4.3), whatever the row layout
            const int L = 4 * reg_tiles(K);
            for (int m = 0; m < L; ++m) {
                const int k = lane * L + m;
                if (k < K) acc = __fadd_rn(acc, __int_as_float(cg[k]));
            }
        }
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) acc = __fadd_rn(acc, __shfl_xor_sync(FULL, acc, off));
        const float sum = acc;
        const float inv = sum != 0.0f ? __fdiv_rn(1.0f, sum) : 0.0f;   // contract 4.3: theta = g * (1 / sum)
        for (int j = 0; j < NT; ++j) {
            const int k0 = j * TILE + lane * 4;
            float4 v = reinterpret_cast<const float4 *>(cg)[j * 32 + lane];
            float *c = &v.x;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if (sum != 0.0f) {
                    c[i] = __fmul_rn(c[i], inv);
                    if (c[i] <= 0.0f) c[i] = 0x1p-149f;
                }
                if (k0 + i >= K) c[i] = 0.0f;
            }
            if (k0 < Ks) reinterpret_cast<float4 *>(trow)[k0 >> 2] = v;
            reinterpret_cast<int4 *>(cg)[j * 32 + lane] = make_int4(0, 0, 0, 0);
        }
        __syncwarp();
    }
}

cudaError_t launch_theta_big(const ThetaArgs &a, int sm_count, cudaStream_t st)
{
    if (a.dm.D == 0) return cudaSuccess;
    const size_t per_warp = (size_t)a.dm.NT * TILE * 4;
    int warps = (int)((size_t)(226 * 1024) / per_warp);
    if (warps < 1) return cudaErrorInvalidValue;
    if (warps > 8) warps = 8;
    const size_t smem = warps * per_warp;
    cudaError_t e = cudaFuncSetAttribute(theta_kernel_big, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int per_sm = 1;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, theta_kernel_big, warps * 32, smem);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    int64_t grid = (int64_t)sm_count * per_sm;
    const int64_t need = (a.dm.D + warps - 1) / warps;
    if (need < grid) grid = need;
    theta_kernel_big<<<(unsigned)grid, warps * 32, smem, st>>>(a);
    return cudaGetLastError();
}

}  // namespace ldagpu
