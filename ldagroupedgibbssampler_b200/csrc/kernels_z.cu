// kernels_z.cu -- K1: the z-step of one Gibbs sweep for K <= 1024, with the GGS theta draw fused into it.
//
// Replaces (reference, src/main/java/cc/mallet/topics/):
//   LDAGroupedGibbsSampler.java:47-132      GGS  z-step (theta draw :60-72, token loop :79-130)
//   UncollapsedParallelLDA.java:1466-1545   PCGS z-step
//   UncollapsedParallelLDA.java:1354-1437   RecursiveDocumentSampler / loopOverBatches (scheduling)
//
// Design (DESIGN.md section 5): one warp owns one work item (GGS: a chunk of 32..256 tokens of one
// document; PCGS: one whole document, because n_dk changes token by token).  Lane l owns the L = 4 * NT
// consecutive topics [l*L, (l+1)*L); rows of Phi^T / n_wk / theta are stored so that those topics are the
// lane's float4 of every 128-column tile (common.cuh: tpos / ttopic), i.e. one row is NT coalesced float4
// loads per lane.  Rows are fetched by the TMA engine (cp.async.bulk, 1-D) into a per-warp shared-memory
// slot; the row is copied to registers as soon as it lands and the slot is refilled with the next run's
// row -- across 32-token blocks too -- while the warp computes.  A run of equal word types shares one
// row fetch and (GGS) one prefix scan.  The categorical draw is a two-level fp32 prefix tree (contract
// 4.2): the lane's sequential fma prefix over its L topics, ONE Kogge-Stone warp scan of the 32 lane
// totals; a token then costs a ballot, NT-1 compares and two shuffles.  Uniforms are Philox4x32-10 keyed
// by the global token index, so the CPU oracle reproduces every sampled topic bit for bit.
//
// GGS fuses the theta draw (LDAGroupedGibbsSampler.java:60-72): a warp whose work item is a whole document
// draws theta_d ~ Dir(n_d + alpha) into its own shared memory and registers and samples the document's
// tokens at once -- the reference does the same per document (GGS:66-72 then :79-130).  The Gamma math is
// issue bound, the token loop is bound by Phi^T traffic, so the two overlap across the warps of an SM.
// Chunks of longer documents read the theta row that theta_kernel wrote before the z-step.
#include "common.cuh"
#include "contract_math.cuh"
#include "warp_draw.cuh"

namespace ldagpu {

// warps per CTA / CTAs per SM.  GGS at 1024 topics keeps theta (32 registers) and the prefixes (32) live;
// 24 warps per SM leave 80 registers per thread (profiles/README.md, round 2)
constexpr int Z_WARPS = 8;
template <int NT, bool PCGS> __host__ __device__ constexpr int z_minb() { return NT == 8 ? (PCGS ? 2 : 3) : 4; }

// ---------------------------------------------------------------------------------------
// GGS theta draw for one document by one warp: theta_d ~ Dir(n_d + alpha) from the counts before the
// document is resampled (LDAGroupedGibbsSampler.java:60-72; ParallelDirichlet.java:46-70 = K Gammas,
// normalise, floor).  Everything is indexed by COLUMN (the row layout of common.cuh); lane l works on
// columns 128*j + 4*l + i = its topics l*L + 4*j + i.
//   phase 1  branch-free lock step over the lane's 4*NT cells: attempt 0 of every ZERO-COUNT cell
//            (shape = alpha_k, the vast majority; Marsaglia-Tsang constants from a per-CTA table,
//            cf. the reference's MarsagliaSparseDirichlet.java:9-29) is settled when the squeeze
//            accepts it (~92 %); all other cells are appended to a per-warp list in shared memory
//            in the same step (ballot + popc)
//   phase 2  the list is drained by all 32 lanes with a flattened attempt loop: a lane whose cell
//            is accepted takes the next list entry, so rejections do not idle the warp
//   phase 3  normalising sum in the contract's order (lane-sequential over its topics, then xor butterfly),
//            one reciprocal, products, floor
// Cells are independent and keyed by (document, topic, attempt): the order of evaluation does not
// change any value.  cg[] (one word per column, zero on entry) holds the count until the cell is drawn,
// the Gamma value afterwards and the normalised theta on return.
// ---------------------------------------------------------------------------------------
constexpr int TH_WARPS = 8;
constexpr int TH_PLIST = 512;   // pending-list capacity per warp (drained early when nearly full)

struct ThetaTables {
    const float *d0, *c0, *i0;   // [ROWF] by column: Marsaglia-Tsang constants of shape alpha_k
};

template <int NT>
__device__ __forceinline__ void theta_tables_fill(float *d0, float *c0, float *i0, const float *__restrict__ alpha, int K)
{
    for (int p = threadIdx.x; p < NT * TILE; p += blockDim.x) {
        const int k = ttopic_lg(lg_of_tiles(NT), p);
        bool b; float dd, cc, ii;
        gamma_setup<float>(k < K ? alpha[k] : 1.0f, b, dd, cc, ii);
        d0[p] = dd; c0[p] = cc; i0[p] = ii;
    }
}

template <int NT>
__device__ __forceinline__ void theta_draw_doc(int *cg, unsigned short *plist, const ThetaTables &tb,
                                               const float *__restrict__ alpha, const int32_t *__restrict__ z,
                                               int64_t t0, int64_t t1, int K, unsigned long long cell0,
                                               uint32_t sweep, const PhiloxKeys &rk, int lane)
{
    constexpr int LG = lg_of_tiles(NT);
    const unsigned lt_mask = (1u << lane) - 1u;
    for (int64_t t = t0 + lane; t < t1; t += 32) atomicAdd(&cg[pos_of<NT>(z[t])], 1);
    __syncwarp();
    int npend = 0;

    // phase 2 body: drain plist[0, npend) with a flattened attempt loop
    auto drain = [&]() {
        __syncwarp();
        int next = 32, idx = lane, p = 0, k = 0;
        bool have = idx < npend, boost = false;
        float dd_ = 0.f, cc_ = 0.f, ii_ = 0.f;
        uint32_t attempt = 0;
        if (have) {
            p = plist[idx];
            k = ttopic_lg(LG, p);
            gamma_setup<float>(__fadd_rn(__int2float_rn(cg[p]), alpha[k]), boost, dd_, cc_, ii_);
        }
        while (__any_sync(FULL, have)) {
            bool finished = false;
            if (have) {
                const unsigned long long cell = cell0 + (unsigned long long)k;
                uint4 w = philox4x32_10((uint32_t)cell, (uint32_t)(cell >> 32), sweep, (STREAM_THETA << 24) | attempt, rk);
                float gv;
                if (gamma_attempt<float>(boost, dd_, cc_, ii_, w, gv)) {
                    cg[p] = __float_as_int(gv);
                    finished = true;
                } else {
                    ++attempt;
                }
            }
            const unsigned fm = __ballot_sync(FULL, finished);
            if (finished) {
                idx = next + __popc(fm & lt_mask);
                have = idx < npend;
                attempt = 0;
                if (have) {
                    p = plist[idx];
                    k = ttopic_lg(LG, p);
                    gamma_setup<float>(__fadd_rn(__int2float_rn(cg[p]), alpha[k]), boost, dd_, cc_, ii_);
                }
            }
            next += __popc(fm);
        }
        npend = 0;
        __syncwarp();
    };

    // ---- phase 1; the cells it leaves open are appended to the pending list as they are found
    //      (ballot + popc, all lanes) and the list is drained whenever another 32 might not fit
    //      two cells of the lane (q, q + 1: adjacent columns) go through the attempt side by side in packed FP32
    //      (gamma_attempt_squeeze2; the values are those of the scalar attempt)
#pragma unroll 1
    for (int q = 0; q < NT * 4; q += 2) {
        int p[2];
        bool valid[2], zero[2], done[2];
        uint4 rnd[2];
#pragma unroll
        for (int w = 0; w < 2; ++w) {
            p[w] = ((q + w) >> 2) * TILE + lane * 4 + ((q + w) & 3);
            const int k = lane * (4 * NT) + q + w;
            valid[w] = k < K;
            zero[w] = valid[w] && cg[p[w]] == 0;
            const unsigned long long cell = cell0 + (unsigned long long)k;
            rnd[w] = philox4x32_10((uint32_t)cell, (uint32_t)(cell >> 32), sweep, STREAM_THETA << 24, rk);
        }
        // q is even, so the two cells are one aligned float2 of each table
        const float2 dd = *reinterpret_cast<const float2 *>(tb.d0 + p[0]);
        const float2 cc = *reinterpret_cast<const float2 *>(tb.c0 + p[0]);
        const float2 ii = *reinterpret_cast<const float2 *>(tb.i0 + p[0]);
        float2 gv;
        gamma_attempt_squeeze2(dd, cc, ii, rnd[0], rnd[1], done[0], done[1], gv);
        const float g2[2] = {gv.x, gv.y};
#pragma unroll
        for (int w = 0; w < 2; ++w) {
            const bool settled = zero[w] && done[w];
            if (settled) cg[p[w]] = __float_as_int(g2[w]);
            const bool open = valid[w] && !settled;
            const unsigned open_mask = __ballot_sync(FULL, open);
            if (open) plist[npend + __popc(open_mask & lt_mask)] = (unsigned short)p[w];
            npend += __popc(open_mask);
        }
        if (npend > TH_PLIST - 64) drain();
    }
    // ---- phase 2
    if (npend > 0) drain();
    __syncwarp();
    // ---- phase 3: sum in contract order, normalise in place
    float4 *g4 = reinterpret_cast<float4 *>(cg);
    float acc = 0.0f;
#pragma unroll
    for (int j = 0; j < NT; ++j) {
        const float4 v = g4[j * 32 + lane];
        acc = __fadd_rn(acc, v.x); acc = __fadd_rn(acc, v.y);
        acc = __fadd_rn(acc, v.z); acc = __fadd_rn(acc, v.w);
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) acc = __fadd_rn(acc, __shfl_xor_sync(FULL, acc, off));
    const float sum = acc;
    // contract 4.3: theta = g * (1 / sum) -- one division per document; the products handle the
    // many denormal g (alpha << 1) at full speed, where a division would take its slow path
    const float inv = sum != 0.0f ? __fdiv_rn(1.0f, sum) : 0.0f;
#pragma unroll
    for (int j = 0; j < NT; ++j) {
        const int k0 = lane * (4 * NT) + 4 * j;
        float4 v = g4[j * 32 + lane];
        if (sum != 0.0f) {
            v.x = __fmul_rn(v.x, inv); v.y = __fmul_rn(v.y, inv);
            v.z = __fmul_rn(v.z, inv); v.w = __fmul_rn(v.w, inv);
            if (v.x <= 0.0f) v.x = 0x1p-149f;
            if (v.y <= 0.0f) v.y = 0x1p-149f;
            if (v.z <= 0.0f) v.z = 0x1p-149f;
            if (v.w <= 0.0f) v.w = 0x1p-149f;
        }
        // padding topics (k >= K) carry no probability
        if (k0 + 0 >= K) v.x = 0.0f;
        if (k0 + 1 >= K) v.y = 0.0f;
        if (k0 + 2 >= K) v.z = 0.0f;
        if (k0 + 3 >= K) v.w = 0.0f;
        g4[j * 32 + lane] = v;
    }
    __syncwarp();
}

// theta tiles kept in registers: 3 in the 8-tile GGS kernel (the rest in shared memory; measured 1..8, profiles/README.md)
template <int NT, bool PCGS> __host__ __device__ constexpr int z_th_reg() { return (NT == 8 && !PCGS) ? 3 : NT; }
// shared-memory footprint, in bytes
template <int NT, bool PCGS> __host__ __device__ constexpr size_t z_warp_smem()
{
    // GGS: row slot + one auxiliary area that is the pending list during the theta draw and the home of the theta tiles
    // that do not stay in registers afterwards
    constexpr size_t aux = (size_t)(NT - z_th_reg<NT, PCGS>()) * 32 * 16 > (size_t)TH_PLIST * 2
                               ? (size_t)(NT - z_th_reg<NT, PCGS>()) * 32 * 16 : (size_t)TH_PLIST * 2;
    return (size_t)NT * TILE * 4 + (PCGS ? (size_t)NT * TILE * 8 : aux);
}
template <int NT, bool PCGS> __host__ __device__ constexpr size_t z_cta_smem()
{
    return Z_WARPS * z_warp_smem<NT, PCGS>() + (PCGS ? 1 : 3) * (size_t)NT * TILE * 4 +
           (size_t)Z_WARPS * 8;
}

template <int NT, bool PCGS>
__global__ void __launch_bounds__(Z_WARPS * 32, z_minb<NT, PCGS>()) z_kernel(ZArgs a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int ROWF = NT * TILE;
    unsigned char *wbase = smem_raw + (size_t)warp * z_warp_smem<NT, PCGS>();
    float *const slot = reinterpret_cast<float *>(wbase);           // the warp's Phi^T row slot (GGS: also the theta scratch)
    int *cnt = reinterpret_cast<int *>(wbase + (size_t)ROWF * 4);   // PCGS: n_dk by column
    float *av = reinterpret_cast<float *>(wbase + (size_t)ROWF * 8);   // PCGS: n_dk + alpha by column
    unsigned short *plist = reinterpret_cast<unsigned short *>(wbase + (size_t)ROWF * 4);   // GGS: pending theta cells
    // GGS at 8 tiles: the theta tiles beyond TH_REG stay in shared memory -- the area of the pending list, idle once theta is drawn
    constexpr int TH_REG = z_th_reg<NT, PCGS>();
    float4 *th_sm = reinterpret_cast<float4 *>(plist);
    float *cta_f = reinterpret_cast<float *>(smem_raw + Z_WARPS * z_warp_smem<NT, PCGS>());
    float *alpha_s = cta_f;                                         // PCGS: alpha by column
    uint64_t *const bar = reinterpret_cast<uint64_t *>(smem_raw + Z_WARPS * z_warp_smem<NT, PCGS>() +
                                                       (PCGS ? 1 : 3) * (size_t)ROWF * 4) + warp;
    const int K = a.dm.K, Ks = a.dm.Ks;   // Ks == ROWF on this path: a bulk copy fills the whole slot
    const uint32_t row_bytes = (uint32_t)Ks * 4u;
    ThetaTables tb{cta_f, cta_f + ROWF, cta_f + 2 * ROWF};

    if (PCGS) {
        for (int i = lane; i < ROWF / 4; i += 32) reinterpret_cast<int4 *>(cnt)[i] = make_int4(0, 0, 0, 0);
        for (int p = threadIdx.x; p < ROWF; p += blockDim.x) {
            const int k = ttopic_lg(lg_of_tiles(NT), p);
            alpha_s[p] = k < K ? a.alpha[k] : 0.0f;
        }
    } else if (a.fuse_theta) {
        theta_tables_fill<NT>(cta_f, cta_f + ROWF, cta_f + 2 * ROWF, a.alpha, K);
    }
    if (lane == 0) {
        mbar_init(bar, 1);
        mbar_fence_init();
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();

    uint32_t phase = 0;            // parity of the slot's mbarrier (one completed fetch flips it)
    // lane 0 drives the TMA: row of word type `wrow` into the slot
    auto request = [&](int wrow) {
        if (lane == 0) {
            mbar_expect_tx(bar, row_bytes);
            bulk_g2s(slot, a.phiT + (size_t)wrow * Ks, row_bytes, bar);
        }
    };

    // the next work item is claimed one item ahead, so the atomic's round trip hides under the work
    unsigned long long claimed = 0;
    if (lane == 0) claimed = atomicAdd(a.work_counter, 1ull);
    for (;;) {
        const unsigned long long item = __shfl_sync(FULL, claimed, 0);
        if ((int64_t)item >= a.n_items) break;
        if (lane == 0) claimed = atomicAdd(a.work_counter, 1ull);

        int64_t d, t0, t1;
        float4 th[TH_REG];
        if (PCGS) {
            d = a.item_doc[item];
            t0 = a.doc_off[d];
            t1 = a.doc_off[d + 1];
            if (t0 == t1) continue;   // UncollapsedParallelLDA.java:1474
            for (int64_t t = t0 + lane; t < t1; t += 32) atomicAdd(&cnt[pos_of<NT>(a.z[t])], 1);
            __syncwarp();
#pragma unroll
            for (int j = 0; j < NT; ++j) {
                int4 c = reinterpret_cast<const int4 *>(cnt)[j * 32 + lane];
                float4 al = reinterpret_cast<const float4 *>(alpha_s)[j * 32 + lane];
                float4 v;
                v.x = __fadd_rn(__int2float_rn(c.x), al.x);
                v.y = __fadd_rn(__int2float_rn(c.y), al.y);
                v.z = __fadd_rn(__int2float_rn(c.z), al.z);
                v.w = __fadd_rn(__int2float_rn(c.w), al.w);
                reinterpret_cast<float4 *>(av)[j * 32 + lane] = v;
            }
            __syncwarp();
        } else {
            d = a.item_doc[item];
            t0 = a.item_begin[item];
            const int64_t ds = a.doc_off[d], de = a.doc_off[d + 1];
            t1 = t0 + a.chunk < de ? t0 + a.chunk : de;
            float *trow = a.theta + (size_t)d * Ks;
            if (a.fuse_theta && t0 == ds && t1 == de) {
                // the item is a whole document: draw its theta here (GGS:60-72), keep it in registers and
                // leave a copy in the theta matrix (GGS:72 thetaMatrix[docId]; log-posterior, getTheta)
                int *cg = reinterpret_cast<int *>(slot);
#pragma unroll
                for (int j = 0; j < NT; ++j) reinterpret_cast<int4 *>(cg)[j * 32 + lane] = make_int4(0, 0, 0, 0);
                __syncwarp();
                theta_draw_doc<NT>(cg, plist, tb, a.alpha, a.z, t0, t1, K,
                                   (unsigned long long)(a.dm.doc_base + d) * (unsigned long long)K, a.sweep, a.rk, lane);
#pragma unroll
                for (int j = 0; j < NT; ++j) {
                    const float4 v = reinterpret_cast<const float4 *>(slot)[j * 32 + lane];
                    if (j < TH_REG) th[j < TH_REG ? j : 0] = v;
                    else th_sm[(j - TH_REG) * 32 + lane] = v;   // the pending list is idle from here on
                    __stcs(reinterpret_cast<float4 *>(trow) + j * 32 + lane, v);
                }
                // the slot goes back to the TMA engine: order the generic-proxy accesses above before its writes
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
            } else {
#pragma unroll
                for (int j = 0; j < NT; ++j) {
                    const float4 v = __ldg(reinterpret_cast<const float4 *>(trow) + j * 32 + lane);
                    if (j < TH_REG) th[j < TH_REG ? j : 0] = v;
                    else th_sm[(j - TH_REG) * 32 + lane] = v;
                }
                if (TH_REG < NT) __syncwarp();
            }
        }

        bool row_in_flight = false;    // the row of this block's first token was requested by the previous block
        // 32-bit offsets inside the item (an item is at most one document: < 2^31 tokens) keep the loop state small
        const int ntok = (int)(t1 - t0);
        const int32_t *const tok = a.tokens + t0;
        int32_t *const zz = a.z + t0;
        int w = lane < ntok ? tok[lane] : -1;
        for (int o = 0; o < ntok; o += 32) {
            const int idx = o + lane;
            const bool valid = idx < ntok;
            const int nvalid = ntok - o < 32 ? ntok - o : 32;
            const bool more = o + 32 < ntok;
            const int w_next = (idx + 32 < ntok) ? tok[idx + 32] : -1;     // next block's word types, loaded early
            const int zold = (PCGS && valid) ? zz[idx] : 0;
            const int wprev = __shfl_up_sync(FULL, w, 1);
            const unsigned heads = __ballot_sync(FULL, valid && (lane == 0 || w != wprev));
            float U = 0.0f;
            if (valid) {
                unsigned long long gt = (unsigned long long)(a.dm.token_base + t0 + idx);
                uint4 r = philox4x32_10((uint32_t)gt, (uint32_t)(gt >> 32), a.sweep, STREAM_Z << 24, a.rk);
                U = uniform23(r.x);
            }
            int znew = 0;
            // One row slot per warp: the row of a run is copied to registers as soon as it lands, and the
            // slot is refilled with the next run's row while the warp computes.
            unsigned rem = heads;          // lane 0 of a non-empty block is always a head
            int b = 0;
            if (!row_in_flight) request(__shfl_sync(FULL, w, 0));
            for (;;) {
                rem &= rem - 1;
                const int e = rem ? __ffs(rem) - 1 : nvalid;   // run = tokens [b, e) of this block
                mbar_wait(bar, phase);
                phase ^= 1u;
                float4 ph[NT];
#pragma unroll
                for (int j = 0; j < NT; ++j) ph[j] = reinterpret_cast<const float4 *>(slot)[j * 32 + lane];
                __syncwarp();
                if (rem) request(__shfl_sync(FULL, w, e));
                else if (more) request(__shfl_sync(FULL, w_next, 0));

                RowScan<NT> rs;
                if (!PCGS) scan_scores<NT, TH_REG>(th, th_sm, ph, rs, lane);
                // not unrolled: runs average 1.4 tokens here; the compiler's 4x unrolled loop with its remainder
                // handling cost 3.7 % of the z-step (11.29 -> 10.88 ms on the 400 000-document slice)
#pragma unroll 1
                for (int tt = b; tt < e; ++tt) {
                    if (PCGS) {
                        // remove the token from the document counts (UncollapsedParallelLDA.java:1494);
                        // every lane computes the new entry (broadcast reads), lane 0 stores it
                        const int old = pos_of<NT>(__shfl_sync(FULL, zold, tt));
                        const int c = cnt[old] - 1;
                        const float v = __fadd_rn(__int2float_rn(c), alpha_s[old]);
                        __syncwarp();
                        if (lane == 0) { cnt[old] = c; av[old] = v; }
                        __syncwarp();
                        float4 aa[NT];
#pragma unroll
                        for (int j = 0; j < NT; ++j) aa[j] = reinterpret_cast<const float4 *>(av)[j * 32 + lane];
                        scan_scores<NT, NT>(aa, nullptr, ph, rs, lane);
                    }
                    const float Ut = __shfl_sync(FULL, U, tt);
                    const int k = draw_topic<NT>(rs, Ut, lane, K);
                    if (lane == tt) znew = k;
                    if (PCGS) {
                        // add it back under its new topic (UncollapsedParallelLDA.java:1535)
                        const int pk = pos_of<NT>(k);
                        const int c = cnt[pk] + 1;
                        const float v = __fadd_rn(__int2float_rn(c), alpha_s[pk]);
                        __syncwarp();
                        if (lane == 0) { cnt[pk] = c; av[pk] = v; }
                        __syncwarp();
                    }
                }
                if (!rem) break;
                b = e;
            }
            row_in_flight = more;
            if (valid) {
                zz[idx] = znew;
                // fused count rebuild (the reference adds its +-1 deltas inside the token loop too,
                // UncollapsedParallelLDA.java:1505,1542): fire-and-forget reductions
                if (a.n_wk_out) atomicAdd(&a.n_wk_out[(size_t)w * Ks + pos_of<NT>(znew)], 1);
            }
            w = w_next;
        }
        if (PCGS) {
            // leave the histogram clean for the next document
            for (int i = lane; i < ROWF / 4; i += 32) reinterpret_cast<int4 *>(cnt)[i] = make_int4(0, 0, 0, 0);
            __syncwarp();
        }
    }
}

template <int NT, bool PCGS>
static cudaError_t launch_z_t(const ZArgs &a, int sm_count, cudaStream_t st)
{
    constexpr size_t smem = z_cta_smem<NT, PCGS>();
    int ctas_per_sm = 1;
    cudaError_t e = kernel_config(reinterpret_cast<const void *>(z_kernel<NT, PCGS>), Z_WARPS * 32, smem, &ctas_per_sm);
    if (e != cudaSuccess) return e;
    int64_t grid = (int64_t)sm_count * ctas_per_sm;   // persistent: every resident warp pulls items
    int64_t need = (a.n_items + Z_WARPS - 1) / Z_WARPS;
    if (need < grid) grid = need;
    if (grid < 1) grid = 1;
    z_kernel<NT, PCGS><<<(unsigned)grid, Z_WARPS * 32, smem, st>>>(a);
    return cudaGetLastError();
}

template <bool PCGS> static cudaError_t launch_z_any(const ZArgs &a, int sm_count, cudaStream_t st)
{
    if (a.n_items == 0) return cudaSuccess;
    if (a.dm.K <= MAX_REG_TILES * TILE) {
        switch (a.dm.NT) {   // reg_tiles(K) (row layout, common.cuh)
        case 1: return launch_z_t<1, PCGS>(a, sm_count, st);
        case 2: return launch_z_t<2, PCGS>(a, sm_count, st);
        case 4: return launch_z_t<4, PCGS>(a, sm_count, st);
        case 8: return launch_z_t<8, PCGS>(a, sm_count, st);
        default: break;
        }
    }
    return PCGS ? launch_z_pcgs_big(a, sm_count, st) : launch_z_ggs_big(a, sm_count, st);
}

cudaError_t launch_z_ggs(const ZArgs &a, int sm_count, cudaStream_t st) { return launch_z_any<false>(a, sm_count, st); }
cudaError_t launch_z_pcgs(const ZArgs &a, int sm_count, cudaStream_t st) { return launch_z_any<true>(a, sm_count, st); }

// ---------------------------------------------------------------------------------------
// stand-alone theta draw: documents split into chunks (longer than one GGS work item), the step-wise
// API (ldagpu_sample_theta) and the PCGS diagnostic theta (UncollapsedParallelLDA.java:710-714).
// One warp per document from a dynamic queue over doc_list (or all documents).
// ---------------------------------------------------------------------------------------
template <int NT>
__global__ void __launch_bounds__(TH_WARPS * 32) theta_kernel(ThetaArgs a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int ROWF = NT * TILE;
    const int K = a.dm.K, Ks = a.dm.Ks;
    float *tabs = reinterpret_cast<float *>(smem_raw);
    unsigned char *wb = smem_raw + (size_t)3 * ROWF * 4 + (size_t)warp * ((size_t)ROWF * 4 + TH_PLIST * 2);
    int *cg = reinterpret_cast<int *>(wb);                     // count, then Gamma value bits
    unsigned short *plist = reinterpret_cast<unsigned short *>(wb + (size_t)ROWF * 4);
    theta_tables_fill<NT>(tabs, tabs + ROWF, tabs + 2 * ROWF, a.alpha, K);
    ThetaTables tb{tabs, tabs + ROWF, tabs + 2 * ROWF};
    for (int i = lane; i < ROWF; i += 32) cg[i] = 0;
    __syncthreads();

    for (;;) {
        unsigned long long dd = 0;
        if (lane == 0) dd = atomicAdd(a.work_counter, 1ull);
        dd = __shfl_sync(FULL, dd, 0);
        if ((int64_t)dd >= a.n_docs) break;
        const int64_t d = a.doc_list ? (int64_t)a.doc_list[dd] : (int64_t)dd;
        const int64_t t0 = a.doc_off[d], t1 = a.doc_off[d + 1];
        float *trow = a.theta + (size_t)d * Ks;
        if (t0 == t1) {   // empty document: the reference skips it, its theta row stays zero
            for (int i = lane; i < Ks; i += 32) trow[i] = 0.0f;
            continue;
        }
        theta_draw_doc<NT>(cg, plist, tb, a.alpha, a.z, t0, t1, K,
                           (unsigned long long)(a.dm.doc_base + d) * (unsigned long long)K, a.sweep, a.rk, lane);
#pragma unroll
        for (int j = 0; j < NT; ++j) {
            reinterpret_cast<float4 *>(trow)[j * 32 + lane] = reinterpret_cast<const float4 *>(cg)[j * 32 + lane];
            reinterpret_cast<int4 *>(cg)[j * 32 + lane] = make_int4(0, 0, 0, 0);
        }
        __syncwarp();
    }
}

template <int NT> static cudaError_t launch_theta_t(const ThetaArgs &a, int sm_count, cudaStream_t st)
{
    constexpr size_t rowf = (size_t)NT * TILE;
    constexpr size_t smem = 3 * rowf * 4 + TH_WARPS * (rowf * 4 + TH_PLIST * 2);
    int per_sm = 1;
    cudaError_t e = kernel_config(reinterpret_cast<const void *>(theta_kernel<NT>), TH_WARPS * 32, smem, &per_sm);
    if (e != cudaSuccess) return e;
    int64_t grid = (int64_t)sm_count * per_sm;
    int64_t need = (a.n_docs + TH_WARPS - 1) / TH_WARPS;
    if (need < grid) grid = need;
    theta_kernel<NT><<<(unsigned)grid, TH_WARPS * 32, smem, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_theta(const ThetaArgs &a, int sm_count, cudaStream_t st)
{
    if (a.n_docs <= 0) return cudaSuccess;
    // theta_kernel<NT> writes rows in the register path's layout (Ks = 128 * NT, permuted columns); the sparse scheme
    // keeps its rows in natural topic order with Ks = round_up(K, 32) and takes the general kernel at every K
    const int NT = a.dm.NT;
    if (a.dm.K <= MAX_REG_TILES * TILE && a.dm.Ks == NT * TILE && a.dm.lg == lg_of_tiles(NT)) {
        switch (NT) {
        case 1: return launch_theta_t<1>(a, sm_count, st);
        case 2: return launch_theta_t<2>(a, sm_count, st);
        case 4: return launch_theta_t<4>(a, sm_count, st);
        case 8: return launch_theta_t<8>(a, sm_count, st);
        default: break;
        }
    }
    return launch_theta_big(a, sm_count, st);
}

}  // namespace ldagpu
