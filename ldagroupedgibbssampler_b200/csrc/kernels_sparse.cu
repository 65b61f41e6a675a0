// kernels_sparse.cu -- the sparse PCGS z-step ("spalias") for large K, and its alias tables.
//
// Replaces (reference, src/main/java/cc/mallet/):
//   topics/SpaliasUncollapsedParallelLDA.java:39-60    per-type alias table over alpha_k * phi[k][w]
//   topics/SpaliasUncollapsedParallelLDA.java:124-245  token loop: p(k) = alpha_k phi_kw (alias draw)
//                                                      + n_dk phi_kw (sparse cumulative sum over n_dk > 0)
//   topics/SpaliasUncollapsedParallelLDA.java:262-312  sampleNewTopic, insert / remove of the non-zero list
//   util/OptimizedGentleAliasMethod.java:52-79,100-107 table construction and generateSample(u)
//
// Cost per token is O(nnz_d) gathered Phi entries instead of the dense step's K: 12 + ~32 nnz_d bytes
// (a 4-byte gather costs a 32-byte sector) against 4 K.  Arithmetic contract: DESIGN.md 4.6; the CPU
// oracle (oracle/lda_oracle_sparse.c) reproduces tables and z bit for bit.
#include <cstdlib>

#include "common.cuh"
#include "contract_math.cuh"

namespace ldagpu {

constexpr unsigned FULL = 0xffffffffu;

// ---------------------------------------------------------------------------------------
// Alias tables.  The reference's stack algorithm is order dependent, so the pairing loop stays
// sequential per word type; types are independent.  Two kernels per round of T types (T = scratch slots):
//   alias_classify_kernel (one WARP per type, coalesced): the lanes stream the Phi^T row, form the
//            normaliser (lane-strided fp64 partial sums + xor butterfly), classify every topic as "low"
//            (b < 0) or "high" and compact (topic, b) pairs, in topic order, into the type's two stacks
//            (ballot + popc prefix) -- the same stacks the sequential classification would build;
//   alias_pair_kernel (one LANE per type): the sequential pairing loop on the type's private scratch
//            (si[K] topics + sb[K] fp64 values in STACK order: "low" from the front, "high" from the back).
//            Both stacks are consumed top first and nothing is ever pushed back on them (a high that turns low is
//            the next one popped: it stays in registers), so each is a sequential stream: a lane keeps the next
//            ALIAS_Q entries of either stack in registers and the warp tops all of them up together whenever one
//            lane runs dry -- one memory round trip per ALIAS_Q steps instead of two dependent ones per step.
//            (Two other structures were measured and lost: per-lane rings in shared memory filled by cp.async removed
//            the remaining load stalls but cost as many extra instructions as they saved cycles, 9.9 ms against 9.05
//            for the whole build; all lanes walking their low stacks in step, four entries per round from aligned
//            vector loads one round ahead, left the rare per-lane events -- a new high, a high turned low -- running
//            with one or two active lanes: 15 active threads per instruction on average, 14.4 ms.)
// Round 1 ran both phases in one kernel, a warp classifying its 32 types one after the other: with ~45 000 active
// types that is 9.5 warps per SM in long latency-bound loops (ncu: 12 long-scoreboard stalls per issue, 14 % issue
// utilisation, 20.4 ms at K = 10 000).
// Only the types that occur in this rank's tokens get a table (no token ever reads the others).
// ---------------------------------------------------------------------------------------
constexpr int ALIAS_Q = 4;      // stack entries a lane of the pairing kernel holds ahead in registers (measured 2, 4, 8: 9.5, 9.05, 9.3 ms)
constexpr int ALIAS_TPS = 1024; // scratch slots per SM: one round covers 151 552 types
constexpr int ALIAS_CW = 8;     // warps per CTA of the classify kernel

__global__ void __launch_bounds__(ALIAS_CW * 32)
alias_classify_kernel(Dims dm, const float *__restrict__ alpha, const float *__restrict__ phiT,
                      AliasSlot *__restrict__ table, float *__restrict__ type_norm,
                      double *__restrict__ sb_all, int32_t *__restrict__ si_all, int2 *__restrict__ counts,
                      const int32_t *__restrict__ active, int32_t n)
{
    const int lane = threadIdx.x & 31;
    const int K = dm.K;
    const double k1 = 1.0 / (double)K;
    const unsigned lt_mask = (1u << lane) - 1u;
    const int nwarps = gridDim.x * ALIAS_CW;
    for (int slot = blockIdx.x * ALIAS_CW + (threadIdx.x >> 5); slot < n; slot += nwarps) {
        const int64_t w = active[slot];
        const float *ph = phiT + (size_t)w * dm.Ks;
        AliasSlot *tw = table + (size_t)w * dm.Ks;
        double *sb = sb_all + (size_t)slot * K;
        int32_t *si = si_all + (size_t)slot * K;
        // normaliser: the lane's terms are added in topic order; four loads are in flight per step
        double acc = 0.0;
        int k = lane;
        for (; k + 96 < K; k += 128) {
            const float a0 = alpha[k], a1 = alpha[k + 32], a2 = alpha[k + 64], a3 = alpha[k + 96];
            const float p0 = ph[k], p1 = ph[k + 32], p2 = ph[k + 64], p3 = ph[k + 96];
            acc = __dadd_rn(acc, (double)__fmul_rn(a0, p0));
            acc = __dadd_rn(acc, (double)__fmul_rn(a1, p1));
            acc = __dadd_rn(acc, (double)__fmul_rn(a2, p2));
            acc = __dadd_rn(acc, (double)__fmul_rn(a3, p3));
        }
        for (; k < K; k += 32) acc = __dadd_rn(acc, (double)__fmul_rn(alpha[k], ph[k]));
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) acc = __dadd_rn(acc, __shfl_xor_sync(FULL, acc, off));
        const double norm = acc;
        if (lane == 0) type_norm[w] = __double2float_rn(norm);
        int low = 0, high = 0;
        for (int c0 = 0; c0 < K; c0 += 128) {
            float av[4], pv[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int i = c0 + 32 * r + lane;
                av[r] = i < K ? alpha[i] : 0.0f;
                pv[r] = i < K ? ph[i] : 0.0f;
            }
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int i = c0 + 32 * r + lane;
                const bool valid = i < K;
                // a type whose Phi column is all zero (possible with the Polya-urn Phi draw) has no prior part:
                // its table is never consulted (tn = 0), keep the arithmetic finite
                const double b = (valid && norm > 0.0)
                                     ? __dsub_rn(__ddiv_rn((double)__fmul_rn(av[r], pv[r]), norm), k1) : 0.0;
                if (valid) tw[i] = AliasSlot{0.0f, i};
                const bool is_low = valid && b < 0.0;
                const unsigned lm = __ballot_sync(FULL, is_low), hm = __ballot_sync(FULL, valid && !is_low);
                const int pos = is_low ? low + __popc(lm & lt_mask) : K - 1 - (high + __popc(hm & lt_mask));
                if (valid) { si[pos] = i; sb[pos] = b; }
                low += __popc(lm);
                high += __popc(hm);
            }
        }
        if (lane == 0) counts[slot] = make_int2(low, high);
    }
}

__global__ void __launch_bounds__(128)
alias_pair_kernel(Dims dm, AliasSlot *__restrict__ table, const double *__restrict__ sb_all,
                  const int32_t *__restrict__ si_all, const int2 *__restrict__ counts,
                  const int32_t *__restrict__ active, int32_t n)
{
    const int slot = blockIdx.x * blockDim.x + threadIdx.x;
    const int K = dm.K;
    const bool mine = slot < n;
    AliasSlot *tw = table + (size_t)(mine ? active[slot] : 0) * dm.Ks;
    const double *sb = sb_all + (size_t)(mine ? slot : 0) * K;
    const int32_t *si = si_all + (size_t)(mine ? slot : 0) * K;
    const int2 cn = mine ? counts[slot] : make_int2(0, 0);
    // low stack: positions [0, low), top = low - 1; high stack: [K - high, K), top = K - high.  The reference loop
    //   while (low>0 && high>0) { l = pop low; h = top high; b[h] += b[l]; b[l] = 0;
    //                             if (b[h] <= 0) pop high; if (b[h] < 0) push h on low; a[l] = h; ps[l] = 1 + K c }
    // with the two values it keeps re-reading held in registers: the residual of the current top
    // high, and a high that just turned low (it is pushed on top of the low stack, so it is the
    // next one popped).  Every stack entry is then read once, in stack order.
    int low = cn.x, high = cn.y, h = 0, pl = 0;
    int lnext = low - 1, hnext = K - high;      // next positions to fetch (top first); -1 / K: stack exhausted
    int lq_n = 0, hq_n = 0, lq_i[ALIAS_Q], hq_i[ALIAS_Q];
    double lq_b[ALIAS_Q], hq_b[ALIAS_Q];
#pragma unroll
    for (int r = 0; r < ALIAS_Q; ++r) { lq_i[r] = hq_i[r] = 0; lq_b[r] = hq_b[r] = 0.0; }
    double d = 0.0, pc = 0.0;
    bool have_h = false, pending = false;
    bool act = low > 0 && high > 0;
    while (__any_sync(FULL, act)) {
        // every lane tops its queues up whenever one lane runs dry: the loads of a top-up are independent, so the warp
        // pays one memory round trip per ALIAS_Q steps
        const bool dry = act && ((!pending && lq_n == 0) || (!have_h && hq_n == 0));
        if (__any_sync(FULL, dry)) {
#pragma unroll
            for (int r = 0; r < ALIAS_Q; ++r) {
                if (r == lq_n && lnext >= 0) { lq_i[r] = si[lnext]; lq_b[r] = sb[lnext]; --lnext; ++lq_n; }
                if (r == hq_n && hnext < K) { hq_i[r] = si[hnext]; hq_b[r] = sb[hnext]; ++hnext; ++hq_n; }
            }
        }
        if (act) {
            int l;
            double c;
            if (pending) { l = pl; c = pc; pending = false; }
            else {
                l = lq_i[0]; c = lq_b[0];
#pragma unroll
                for (int r = 0; r + 1 < ALIAS_Q; ++r) { lq_i[r] = lq_i[r + 1]; lq_b[r] = lq_b[r + 1]; }
                --lq_n; --low;
            }
            if (!have_h) {
                h = hq_i[0]; d = hq_b[0];
#pragma unroll
                for (int r = 0; r + 1 < ALIAS_Q; ++r) { hq_i[r] = hq_i[r + 1]; hq_b[r] = hq_b[r + 1]; }
                --hq_n; have_h = true;
            }
            const double nb = __dadd_rn(c, d);
            d = nb;
            if (nb <= 0.0) { high--; have_h = false; }
            if (nb < 0.0) { pending = true; pl = h; pc = nb; }
            tw[l] = AliasSlot{__double2float_rn(__dadd_rn(1.0, __dmul_rn((double)K, c))), h};
            act = (pending || low > 0) && high > 0;
        }
    }
}

// scratch slots (types per round of the two kernels): all of the vocabulary when it fits sm_count * ALIAS_TPS slots.
// LDAGPU_ALIAS_SLOTS caps it -- 12 K bytes of scratch per slot (1.2 GB per 10 000 slots at K = 10 000); the tables do
// not depend on it, only the number of rounds.
int64_t alias_scratch_threads(const Dims &dm, int sm_count)
{
    int64_t t = (int64_t)sm_count * ALIAS_TPS;
    if (const char *e = getenv("LDAGPU_ALIAS_SLOTS")) {
        const long long v = atoll(e);
        if (v > 0 && v < t) t = (v + 127) / 128 * 128;
    }
    int64_t need = ((int64_t)dm.V + 127) / 128 * 128;
    return need < t ? need : t;
}

// scratch: sb[T][K] doubles; si[T][K] ints followed by the T (low, high) count pairs
size_t alias_value_doubles(const Dims &dm, int64_t T) { return (size_t)T * (size_t)dm.K; }
size_t alias_stack_ints(const Dims &dm, int64_t T) { return alias_value_doubles(dm, T) + 2 * (size_t)T; }

cudaError_t launch_alias_build(const Dims &dm, const float *alpha, const float *phiT, AliasSlot *table,
                               float *type_norm, double *bs_scratch, int32_t *stack_scratch,
                               const int32_t *active, int32_t n_active, int64_t T, int sm_count, cudaStream_t st)
{
    if (n_active == 0) return cudaSuccess;
    int2 *counts = reinterpret_cast<int2 *>(stack_scratch + (size_t)T * dm.K);   // 8-byte aligned: T is a multiple of 128
    int per_sm = 1;
    cudaError_t e = kernel_config(reinterpret_cast<const void *>(alias_classify_kernel), ALIAS_CW * 32, 0, &per_sm);
    if (e != cudaSuccess) return e;
    // rounds of up to T types; when they do not fit one round, split them evenly
    const int64_t rounds = ((int64_t)n_active + T - 1) / T;
    const int64_t per_round = ((int64_t)n_active + rounds - 1) / rounds;
    for (int64_t first = 0; first < n_active; first += per_round) {
        const int32_t n = (int32_t)(n_active - first < per_round ? n_active - first : per_round);
        int64_t cgrid = ((int64_t)n + ALIAS_CW - 1) / ALIAS_CW;
        if (cgrid > (int64_t)sm_count * per_sm) cgrid = (int64_t)sm_count * per_sm;
        alias_classify_kernel<<<(unsigned)cgrid, ALIAS_CW * 32, 0, st>>>(dm, alpha, phiT, table, type_norm, bs_scratch,
                                                                        stack_scratch, counts, active + first, n);
        alias_pair_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(dm, table, bs_scratch, stack_scratch, counts,
                                                                      active + first, n);
    }
    return cudaGetLastError();
}


// ---------------------------------------------------------------------------------------
// Sparse z-step.  One warp per document (PCGS is sequential inside a document).  The document's
// non-zero topics and their counts form a list in the reference's order (append on first use,
// swap-remove when a count reaches 0).  The list is cut into blocks of 256 entries and lane l owns
// entries 8l..8l+7 of a block (two 16-byte loads per array): finding a topic, gathering Phi at the
// listed topics, the cumulative sum (lane-local prefix + one warp scan per block) and the search all
// work on those eight registers.
//   fast path  lists of up to 256 topics live in shared memory (2 KB per warp, 64 warps per SM);
//   slow path  a document whose list outgrows that continues on per-warp lists in global memory with
//              the same arithmetic block by block (early sweeps from a random start, very long documents).
// ---------------------------------------------------------------------------------------
constexpr int SP_BLOCK = 256;   // list entries per block (8 per lane)
constexpr int SP_WARPS = 8;     // warps per CTA

struct SparseArgs {
    ZArgs z;
    const AliasSlot *table;
    const float *type_norm;
    int *lists;   // per resident warp: nz[cap], cnt[cap], cum[cap] in global memory (slow path)
    int cap;      // list capacity per warp (multiple of SP_BLOCK)
};

__device__ __forceinline__ void load8(const int *a, int (&v)[8])
{
    const int4 x = reinterpret_cast<const int4 *>(a)[0], y = reinterpret_cast<const int4 *>(a)[1];
    v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w; v[4] = y.x; v[5] = y.y; v[6] = y.z; v[7] = y.w;
}

// position of topic k in the list, -1 if absent
template <bool MULTI>
__device__ __forceinline__ int list_find(const int *nz, int nnz, int k, int lane)
{
    for (int b0 = 0; b0 < (MULTI ? nnz : 1); b0 += SP_BLOCK) {
        int v[8];
        load8(nz + b0 + 8 * lane, v);
        const int nvalid = nnz - (b0 + 8 * lane);
        int pe = -1;
#pragma unroll
        for (int e = 7; e >= 0; --e)
            if (e < nvalid && v[e] == k) pe = e;
        const unsigned m = __ballot_sync(FULL, pe >= 0);
        if (m) {
            const int l = __ffs(m) - 1;
            return b0 + 8 * l + __shfl_sync(FULL, pe, l);
        }
    }
    return -1;
}

// add one token of topic k (SpaliasUncollapsedParallelLDA.java:223-230,306-312); pos = its list position when known
__device__ __forceinline__ void list_add_at(int *nz, int *cnt, int &nnz, int k, int pos, int lane)
{
    const int c = pos >= 0 ? cnt[pos] : 0;
    __syncwarp();
    if (lane == 0) {
        if (pos < 0) { nz[nnz] = k; cnt[nnz] = 1; }
        else cnt[pos] = c + 1;
    }
    if (pos < 0) ++nnz;
    __syncwarp();
}

// remove one token of topic `old` (:159-166, :295-304)
template <bool MULTI>
__device__ __forceinline__ void list_remove(int *nz, int *cnt, int &nnz, int old, int lane)
{
    const int pos = list_find<MULTI>(nz, nnz, old, lane);
    const int c = cnt[pos] - 1;
    const int lk = nz[nnz - 1], lc = cnt[nnz - 1];
    __syncwarp();
    if (lane == 0) {
        if (c == 0) { nz[pos] = lk; cnt[pos] = lc; }
        else cnt[pos] = c;
    }
    if (c == 0) --nnz;
    __syncwarp();
}

// One token: scores over the list, cumulative sum, prior/likelihood branch.  Returns the new topic and, in
// `slot`, its list position when the likelihood branch found it (-1 otherwise).
template <bool MULTI>
__device__ __forceinline__ int sparse_draw(const SparseArgs &sa, const int *nz, const int *cnt, float *cum, int nnz,
                                           int wt, float u, int lane, int &slot)
{
    const int K = sa.z.dm.K, Ks = sa.z.dm.Ks;
    const float *ph = sa.z.phiT + (size_t)wt * Ks;
    const float tn = __ldg(sa.type_norm + wt);
    float carry = 0.0f, E = 0.0f;
    float q[8];
    int nvalid0 = 0;
    for (int b0 = 0; b0 < (MULTI ? nnz : 1); b0 += SP_BLOCK) {
        int kk[8], cc[8];
        load8(nz + b0 + 8 * lane, kk);
        load8(cnt + b0 + 8 * lane, cc);
        const int nvalid = nnz - (b0 + 8 * lane);
        float s[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) s[e] = e < nvalid ? __ldg(ph + kk[e]) : 0.0f;
#pragma unroll
        for (int e = 0; e < 8; ++e) s[e] = e < nvalid ? __fmul_rn(__int2float_rn(cc[e]), s[e]) : 0.0f;
        q[0] = s[0];
#pragma unroll
        for (int e = 1; e < 8; ++e) q[e] = __fadd_rn(q[e - 1], s[e]);
        float inc = q[7];
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const float y = __shfl_up_sync(FULL, inc, off);
            if (lane >= off) inc = __fadd_rn(inc, y);
        }
        E = __shfl_up_sync(FULL, inc, 1);
        if (lane == 0) E = 0.0f;
        if (MULTI) {
#pragma unroll
            for (int e = 0; e < 8; ++e)
                if (e < nvalid) cum[b0 + 8 * lane + e] = __fadd_rn(carry, __fadd_rn(E, q[e]));
        }
        carry = __fadd_rn(carry, __shfl_sync(FULL, inc, 31));
        nvalid0 = nvalid;
    }
    if (MULTI) __syncwarp();
    const float sum = carry;
    const float tot = __fadd_rn(tn, sum);
    slot = -1;
    if (!(tot > 0.0f)) {
        // neither the prior nor the document gives this type any mass (its Phi column is all zero over the topics
        // that matter): the reference draws the topic uniformly (topics/PolyaUrnSpaliasLDA.java:275-277)
        int i = __float2int_rz(__fmul_rn(u, __int2float_rn(K)));
        return i > K - 1 ? K - 1 : i;
    }
    if (u < __fdiv_rn(tn, tot) || nnz == 0) {
        // prior part: alias draw (:265-267, OptimizedGentleAliasMethod.java:100-107)
        const float up = __fadd_rn(u, __fdiv_rn(__fmul_rn(sum, u), tn));
        const float ups = __fmul_rn(up, __int2float_rn(K));
        int i = __float2int_rz(ups);
        if (i > K - 1) i = K - 1;
        const int2 entry = __ldg(reinterpret_cast<const int2 *>(sa.table + (size_t)wt * Ks + i));   // {ps, alias}
        if (__fsub_rn(ups, __int2float_rn(i)) > __int_as_float(entry.x)) i = entry.y;
        return i;
    }
    // likelihood part: first slot with u*tot - tn <= cum (:269-275, findIdx :347-375)
    const float ul = __fsub_rn(__fmul_rn(u, tot), tn);
    slot = nnz - 1;
    if (!MULTI) {
        int pe = -1;
#pragma unroll
        for (int e = 7; e >= 0; --e)
            if (e < nvalid0 && ul <= __fadd_rn(E, q[e])) pe = e;
        const unsigned m = __ballot_sync(FULL, pe >= 0);
        if (m) {
            const int l = __ffs(m) - 1;
            slot = 8 * l + __shfl_sync(FULL, pe, l);
        }
    } else {
        for (int b0 = 0; b0 < nnz; b0 += SP_BLOCK) {
            const int nvalid = nnz - (b0 + 8 * lane);
            int pe = -1;
#pragma unroll
            for (int e = 7; e >= 0; --e)
                if (e < nvalid && ul <= cum[b0 + 8 * lane + e]) pe = e;
            const unsigned m = __ballot_sync(FULL, pe >= 0);
            if (m) {
                const int l = __ffs(m) - 1;
                slot = b0 + 8 * l + __shfl_sync(FULL, pe, l);
                break;
            }
        }
    }
    return nz[slot];
}

// tokens [ta, t1) of one document on the given lists; MULTI = lists of any length (global memory)
template <bool MULTI>
__device__ __forceinline__ int64_t sparse_tokens(const SparseArgs &sa, int *nz, int *cnt, float *cum, int &nnz,
                                                 int64_t ta, int64_t t1, int lane)
{
    const ZArgs &a = sa.z;
    const int Ks = a.dm.Ks;
    for (int64_t tb = ta; tb < t1; tb += 32) {
        const int64_t t = tb + lane;
        const bool valid = t < t1;
        const int nv = (int)((t1 - tb) < 32 ? (t1 - tb) : 32);
        const int w = valid ? a.tokens[t] : 0;
        const int zold = valid ? a.z[t] : 0;
        float U = 0.0f;
        if (valid) {
            const unsigned long long gt = (unsigned long long)(a.dm.token_base + t);
            const uint4 r = philox4x32_10((uint32_t)gt, (uint32_t)(gt >> 32), a.sweep, STREAM_Z << 24, a.seed_lo, a.seed_hi);
            U = uniform23(r.x);
        }
        int znew = 0, done = nv;
        for (int tt = 0; tt < nv; ++tt) {
            if (!MULTI && nnz >= SP_BLOCK) { done = tt; break; }   // the list may outgrow shared memory: hand over
            const int wt = __shfl_sync(FULL, w, tt);
            const int old = __shfl_sync(FULL, zold, tt);
            const float u = __shfl_sync(FULL, U, tt);
            list_remove<MULTI>(nz, cnt, nnz, old, lane);
            int slot;
            const int nw = sparse_draw<MULTI>(sa, nz, cnt, cum, nnz, wt, u, lane, slot);
            if (lane == tt) znew = nw;
            if (slot < 0) slot = list_find<MULTI>(nz, nnz, nw, lane);
            list_add_at(nz, cnt, nnz, nw, slot, lane);
        }
        if (lane < done) {
            a.z[t] = znew;
            if (a.n_wk_out) atomicAdd(&a.n_wk_out[(size_t)w * Ks + znew], 1);
        }
        if (done < nv) return tb + done;   // first token not processed
    }
    return t1;
}

// 4 CTAs (32 warps, 64 registers) per SM: 5, 6 and 8 CTAs were measured slower on B200 (spills; the kernel is
// bound by the DRAM sectors of the Phi gathers, not by latency)
__global__ void __launch_bounds__(SP_WARPS * 32, 4) z_spalias_kernel(SparseArgs sa)
{
    __shared__ __align__(16) int s_nz[SP_WARPS][SP_BLOCK];
    __shared__ __align__(16) int s_cnt[SP_WARPS][SP_BLOCK];
    const ZArgs &a = sa.z;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int cap = sa.cap;
    int *gnz = sa.lists + ((size_t)blockIdx.x * SP_WARPS + warp) * (size_t)cap * 3;
    int *gcnt = gnz + cap;
    float *gcum = reinterpret_cast<float *>(gcnt + cap);
    int *nz = s_nz[warp], *cnt = s_cnt[warp];

    for (;;) {
        unsigned long long item = 0;
        if (lane == 0) item = atomicAdd(a.work_counter, 1ull);
        item = __shfl_sync(FULL, item, 0);
        if ((int64_t)item >= a.n_items) break;
        const int64_t d = a.item_doc[item], t0 = a.doc_off[d], t1 = a.doc_off[d + 1];
        if (t0 == t1) continue;
        // non-zero topic list in first-occurrence order (SpaliasUncollapsedParallelLDA.java:147-153)
        int nnz = 0;
        bool in_smem = true;
        for (int64_t tb = t0; tb < t1 && in_smem; tb += 32) {
            const int zz = (tb + lane < t1) ? a.z[tb + lane] : -1;
            const int nv = (int)((t1 - tb) < 32 ? (t1 - tb) : 32);
            for (int tt = 0; tt < nv; ++tt) {
                const int k = __shfl_sync(FULL, zz, tt);
                const int pos = list_find<false>(nz, nnz, k, lane);
                if (pos < 0 && nnz >= SP_BLOCK) { in_smem = false; break; }
                list_add_at(nz, cnt, nnz, k, pos, lane);
            }
        }
        int64_t next = t0;
        if (in_smem) next = sparse_tokens<false>(sa, nz, cnt, nullptr, nnz, t0, t1, lane);
        if (next < t1) {
            // slow path: continue (or, when the initial list did not fit, start over) on the global lists
            if (in_smem) {
                for (int i = lane; i < nnz; i += 32) { gnz[i] = nz[i]; gcnt[i] = cnt[i]; }
                __syncwarp();
            } else {
                nnz = 0;
                for (int64_t tb = t0; tb < t1; tb += 32) {
                    const int zz = (tb + lane < t1) ? a.z[tb + lane] : -1;
                    const int nv = (int)((t1 - tb) < 32 ? (t1 - tb) : 32);
                    for (int tt = 0; tt < nv; ++tt) {
                        const int k = __shfl_sync(FULL, zz, tt);
                        const int pos = list_find<true>(gnz, nnz, k, lane);
                        list_add_at(gnz, gcnt, nnz, k, pos, lane);
                    }
                }
            }
            sparse_tokens<true>(sa, gnz, gcnt, gcum, nnz, next, t1, lane);
        }
    }
}

size_t spalias_list_bytes(const Dims &dm, int max_doc_len, int sm_count)
{
    int cap = max_doc_len < dm.K ? max_doc_len : dm.K;
    cap = (cap + 1 + SP_BLOCK - 1) / SP_BLOCK * SP_BLOCK + SP_BLOCK;   // whole blocks are loaded
    return (size_t)sm_count * 8 * SP_WARPS * (size_t)cap * 12;   // up to 8 CTAs of 8 warps per SM
}

cudaError_t launch_z_spalias(const ZArgs &z, const AliasSlot *table, const float *type_norm,
                             int *lists, int max_doc_len, int sm_count, cudaStream_t st)
{
    if (z.n_items == 0) return cudaSuccess;
    SparseArgs sa;
    sa.z = z; sa.table = table; sa.type_norm = type_norm; sa.lists = lists;
    int cap = max_doc_len < z.dm.K ? max_doc_len : z.dm.K;
    sa.cap = (cap + 1 + SP_BLOCK - 1) / SP_BLOCK * SP_BLOCK + SP_BLOCK;
    int per_sm = 1;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, z_spalias_kernel, SP_WARPS * 32, 0);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 8) per_sm = 8;
    int64_t grid = (int64_t)sm_count * per_sm;
    const int64_t need = (z.n_items + SP_WARPS - 1) / SP_WARPS;
    if (need < grid) grid = need;
    z_spalias_kernel<<<(unsigned)grid, SP_WARPS * 32, 0, st>>>(sa);
    return cudaGetLastError();
}

}  // namespace ldagpu
