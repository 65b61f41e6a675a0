// kernels_heldout.cu -- held-out log-likelihood of a test set by the left-to-right estimator, for K <= 1024.
//
// Serves (reference, src/main/java/cc/mallet/topics/):
//   UncollapsedParallelLDA.java:604-611,840-844   the held-out evaluation during sample() (MarginalProbEstimatorPlain)
// and MALLET's MarginalProbEstimator.evaluateLeftToRight (Wallach et al. 2009) without resampling, which the
// reference's Plain variant restates over plain count arrays.
//
// Contract (DESIGN.md 4.8):
//   phihat_kw = (float)(((double)n_wk + beta) / ((double)n_k + V*beta))           heldout_phihat_kernel
//   for every test document d and particle r, from n_dk = 0, position i = 0 .. N_d-1, word w:
//     S_i^r = sum_k (float(n_dk) + alpha_k) * phihat_kw   (the lane-contiguous tree of 4.2, warp_draw.cuh)
//     z_i drawn from the same tree with the uniform of Philox stream 5, n_{d,z_i} += 1   heldout_l2r_kernel
//   m_i = (sum_r (double)S_i^r) / (R * (i + alpha_sum)),  l_d = sum_i ln(m_i)     heldout_reduce_kernel
//
// heldout_l2r_kernel is the PCGS z-step of a fresh document: one warp per (document, particle) work item from an
// atomic queue; n_dk + alpha lives in shared memory by column; phihat rows come through the TMA row slot, the row of
// the next token's type is requested as soon as the current one is in registers, and a run of equal types shares one
// fetch.  S_i^r goes to a [R][batch tokens] fp32 scratch buffer; the engine cuts the test set into document batches
// whose scratch fits its bound.
#include "common.cuh"
#include "contract_math.cuh"
#include "warp_draw.cuh"

namespace ldagpu {

constexpr int HO_WARPS = 8;
template <int NT> __host__ __device__ constexpr int ho_minb() { return NT == 8 ? 2 : NT == 4 ? 3 : 4; }   // no spills (-Xptxas -v)
// per warp: row slot, n_dk and n_dk + alpha by column; per CTA: alpha by column and one mbarrier per warp
template <int NT> __host__ __device__ constexpr size_t ho_cta_smem()
{
    return (size_t)HO_WARPS * 3 * NT * TILE * 4 + (size_t)NT * TILE * 4 + (size_t)HO_WARPS * 8;
}

__global__ void heldout_phihat_kernel(Dims src, Dims dst, const int32_t *__restrict__ n_wk, const int32_t *__restrict__ n_k,
                                      double beta, double vbeta, float *__restrict__ phihat)
{
    const int64_t cells = (int64_t)dst.Vp * dst.Ks;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < cells; i += (int64_t)gridDim.x * blockDim.x) {
        const int w = (int)(i / dst.Ks), p = (int)(i % dst.Ks);
        const int k = ttopic(dst, p);
        float v = 0.0f;
        if (w < dst.V && k < dst.K) {
            const double n = (double)n_wk[(size_t)w * src.Ks + tpos(src, k)];
            v = __double2float_rn(__ddiv_rn(__dadd_rn(n, beta), __dadd_rn((double)n_k[k], vbeta)));
        }
        phihat[i] = v;
    }
}

template <int NT>
__global__ void __launch_bounds__(HO_WARPS * 32, ho_minb<NT>()) heldout_l2r_kernel(HeldoutArgs a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int ROWF = NT * TILE;
    float *const slot = reinterpret_cast<float *>(smem_raw + (size_t)warp * 3 * ROWF * 4);
    int *const cnt = reinterpret_cast<int *>(slot + ROWF);
    float *const av = slot + 2 * ROWF;
    float *const alpha_s = reinterpret_cast<float *>(smem_raw + (size_t)HO_WARPS * 3 * ROWF * 4);
    uint64_t *const bar = reinterpret_cast<uint64_t *>(alpha_s + ROWF) + warp;
    const int K = a.dm.K;
    const uint32_t row_bytes = (uint32_t)ROWF * 4u;

    for (int p = threadIdx.x; p < ROWF; p += blockDim.x) {
        const int k = ttopic_lg(lg_of_tiles(NT), p);
        alpha_s[p] = k < K ? a.alpha[k] : 0.0f;
    }
    if (lane == 0) {
        mbar_init(bar, 1);
        mbar_fence_init();
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();

    uint32_t phase = 0;
    auto request = [&](int wrow) {
        if (lane == 0) {
            mbar_expect_tx(bar, row_bytes);
            bulk_g2s(slot, a.phihat + (size_t)wrow * ROWF, row_bytes, bar);
        }
    };

    const int64_t n_items = (a.doc1 - a.doc0) * (int64_t)a.R;
    unsigned long long claimed = 0;
    if (lane == 0) claimed = atomicAdd(a.work_counter, 1ull);
    for (;;) {
        const unsigned long long item = __shfl_sync(FULL, claimed, 0);
        if ((int64_t)item >= n_items) break;
        if (lane == 0) claimed = atomicAdd(a.work_counter, 1ull);
        const int64_t d = a.doc0 + (int64_t)item / a.R;
        const uint32_t r = (uint32_t)((int64_t)item % a.R);
        const int64_t t0 = a.doc_off[d], t1 = a.doc_off[d + 1];
        if (t0 == t1) continue;   // an empty document contributes 0

        // n_dk = 0: the vector is alpha
#pragma unroll
        for (int j = 0; j < NT; ++j) {
            reinterpret_cast<int4 *>(cnt)[j * 32 + lane] = make_int4(0, 0, 0, 0);
            reinterpret_cast<float4 *>(av)[j * 32 + lane] = reinterpret_cast<const float4 *>(alpha_s)[j * 32 + lane];
        }
        __syncwarp();

        const int ntok = (int)(t1 - t0);
        const int32_t *const tok = a.tokens + t0;
        float *const sout = a.S + (size_t)r * (size_t)a.batch_tokens + (size_t)(t0 - a.tok0);
        int w = lane < ntok ? tok[lane] : -1;
        int cur = -1;              // type of the row in ph
        float4 ph[NT];
        request(__shfl_sync(FULL, w, 0));
        for (int o = 0; o < ntok; o += 32) {
            const int idx = o + lane;
            const bool valid = idx < ntok;
            const int nvalid = ntok - o < 32 ? ntok - o : 32;
            const int w_next = (idx + 32 < ntok) ? tok[idx + 32] : -1;
            float U = 0.0f, s_mine = 0.0f;
            if (valid) {
                const unsigned long long gt = (unsigned long long)(a.token_base + t0 + idx);
                const uint4 q = philox4x32_10((uint32_t)gt, (uint32_t)(gt >> 32), a.iteration, (STREAM_HELDOUT << 24) | r, a.rk);
                U = uniform23(q.x);
            }
#pragma unroll 1
            for (int tt = 0; tt < nvalid; ++tt) {
                const int wt = __shfl_sync(FULL, w, tt);
                const int wn = tt + 1 < 32 ? __shfl_sync(FULL, w, (tt + 1) & 31) : __shfl_sync(FULL, w_next, 0);
                if (wt != cur) {
                    // the slot holds (or is receiving) this token's row: it was requested by the previous token
                    mbar_wait(bar, phase);
                    phase ^= 1u;
#pragma unroll
                    for (int j = 0; j < NT; ++j) ph[j] = reinterpret_cast<const float4 *>(slot)[j * 32 + lane];
                    __syncwarp();
                    cur = wt;
                }
                if (wn >= 0 && wn != wt) request(wn);   // the slot is free: its row is in registers
                float4 aa[NT];
#pragma unroll
                for (int j = 0; j < NT; ++j) aa[j] = reinterpret_cast<const float4 *>(av)[j * 32 + lane];
                RowScan<NT> rs;
                scan_scores<NT, NT>(aa, nullptr, ph, rs, lane);
                if (lane == tt) s_mine = rs.S;
                if (o + tt + 1 < ntok) {   // the last draw of a document changes nothing that is read
                    const float Ut = __shfl_sync(FULL, U, tt);
                    const int k = draw_topic<NT>(rs, Ut, lane, K);
                    const int pk = pos_of<NT>(k);
                    const int c = cnt[pk] + 1;
                    const float v = __fadd_rn(__int2float_rn(c), alpha_s[pk]);
                    __syncwarp();
                    if (lane == 0) { cnt[pk] = c; av[pk] = v; }
                    __syncwarp();
                }
            }
            if (valid) sout[idx] = s_mine;
            w = w_next;
        }
    }
}

// one warp per document of the batch: m_i from the particles' S in particle order, l_d = sum_i ln(m_i) in token order
__global__ void heldout_reduce_kernel(HeldoutArgs a, double alpha_sum, double *__restrict__ doc_ll)
{
    const int lane = threadIdx.x & 31;
    const int64_t nd = a.doc1 - a.doc0;
    const double R = (double)a.R;
    for (int64_t q = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; q < nd; q += ((int64_t)gridDim.x * blockDim.x) >> 5) {
        const int64_t d = a.doc0 + q;
        const int64_t t0 = a.doc_off[d], t1 = a.doc_off[d + 1];
        const float *const s = a.S + (size_t)(t0 - a.tok0);
        double acc = 0.0;
        for (int64_t o = 0; o < t1 - t0; o += 32) {
            const int64_t i = o + lane;
            double l = 0.0;
            if (i < t1 - t0) {
                double sum = 0.0;
                for (int r = 0; r < a.R; ++r) sum = __dadd_rn(sum, (double)s[(size_t)r * (size_t)a.batch_tokens + (size_t)i]);
                l = c_ln<double>(__ddiv_rn(sum, __dmul_rn(R, __dadd_rn((double)i, alpha_sum))));
            }
            const int n = t1 - t0 - o < 32 ? (int)(t1 - t0 - o) : 32;
            for (int j = 0; j < n; ++j) acc = __dadd_rn(acc, __shfl_sync(FULL, l, j));
        }
        if (lane == 0) doc_ll[q] = acc;
    }
}

cudaError_t launch_heldout_phihat(const Dims &src, const Dims &dst, const int32_t *n_wk, const int32_t *n_k, double beta,
                                  float *phihat, int sm_count, cudaStream_t st)
{
    const double vbeta = (double)dst.V * beta;
    heldout_phihat_kernel<<<(unsigned)(sm_count * 8), 256, 0, st>>>(src, dst, n_wk, n_k, beta, vbeta, phihat);
    return cudaGetLastError();
}

template <int NT> static cudaError_t launch_l2r_t(const HeldoutArgs &a, int sm_count, cudaStream_t st)
{
    constexpr size_t smem = ho_cta_smem<NT>();
    int per_sm = 1;
    cudaError_t e = kernel_config(reinterpret_cast<const void *>(heldout_l2r_kernel<NT>), HO_WARPS * 32, smem, &per_sm);
    if (e != cudaSuccess) return e;
    int64_t grid = (int64_t)sm_count * per_sm;
    const int64_t need = ((a.doc1 - a.doc0) * (int64_t)a.R + HO_WARPS - 1) / HO_WARPS;
    if (need < grid) grid = need;
    if (grid < 1) grid = 1;
    heldout_l2r_kernel<NT><<<(unsigned)grid, HO_WARPS * 32, smem, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_heldout_l2r(const HeldoutArgs &a, int sm_count, cudaStream_t st)
{
    if (a.doc1 <= a.doc0) return cudaSuccess;
    switch (a.dm.NT) {   // reg_tiles(K): phihat is in the register path's row layout
    case 1: return launch_l2r_t<1>(a, sm_count, st);
    case 2: return launch_l2r_t<2>(a, sm_count, st);
    case 4: return launch_l2r_t<4>(a, sm_count, st);
    case 8: return launch_l2r_t<8>(a, sm_count, st);
    default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_heldout_reduce(const HeldoutArgs &a, double alpha_sum, double *doc_ll, int sm_count, cudaStream_t st)
{
    const int64_t nd = a.doc1 - a.doc0;
    if (nd <= 0) return cudaSuccess;
    int64_t grid = (nd + 7) / 8;
    if (grid > (int64_t)sm_count * 16) grid = (int64_t)sm_count * 16;
    heldout_reduce_kernel<<<(unsigned)grid, 256, 0, st>>>(a, alpha_sum, doc_ll);
    return cudaGetLastError();
}

}  // namespace ldagpu
