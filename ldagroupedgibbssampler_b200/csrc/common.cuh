// common.cuh -- shared declarations of the libldagpu kernels and their launchers.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "contract_math.cuh"

#include <map>
#include <mutex>
#include <tuple>

namespace ldagpu {

constexpr int TILE = 128;            // topics per warp tile: lane l owns topics 4l..4l+3 of the tile
constexpr int MAX_REG_TILES = 8;     // K <= 1024 keeps a whole Phi^T row in registers
constexpr int GGS_CHUNK_MAX = 256;   // most tokens per GGS work item (x4 for corpora beyond ~10^8 tokens per GPU) (documents are split freely; the engine
                                     // picks a multiple of 32 so that every resident warp gets several items)
constexpr int PHI_ROW_BLOCK = 8;     // words per sequential partial sum of the Phi normaliser
constexpr int PHI_SEGMENTS = 8;      // vocabulary segments (= max ranks) of the Phi normaliser tree

inline int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

struct Dims {
    int32_t K;        // topics
    int32_t Ks;       // row stride of Phi^T / n_wk / theta in elements: 128 * NT on the register path, else round_up(K, 32)
    int32_t NT;       // tiles of a row: 1, 2, 4 or 8 for K <= 1024 (register path), ceil(K / 128) above
    int32_t lg;       // log2 of the topics one lane owns on the register path (2 = rows in natural topic order)
    int32_t V;        // vocabulary
    int32_t Vp;       // padded vocabulary rows: round_up(V, 64)
    int64_t D;        // local documents
    int64_t N;        // local tokens
    int64_t doc_base;    // global index of local document 0
    int64_t token_base;  // global index of local token 0
};

// Row layout (DESIGN.md section 2).  On the register path (K <= 1024) lane l of a warp owns the L = 4 * NT
// CONSECUTIVE topics [l * L, (l + 1) * L) (contract 4.2), but reads them as one coalesced float4 per tile: a
// row of Phi^T / n_wk / theta stores topic k = l * L + 4 * j + i at column 128 * j + 4 * l + i -- a
// permutation of the bits of k.  Topic indicators (z), alpha and n_k stay in natural topic order; every
// kernel that indexes a row by topic goes through these two functions.  lg == 2 is the identity
// (K <= 128, the K > 1024 path and the sparse scheme).
// NT of the register path for K <= MAX_REG_TILES * TILE, and lg of NT tiles (L = 4 * NT = 1 << lg)
__host__ __device__ constexpr int reg_tiles(int K) { return K <= 128 ? 1 : K <= 256 ? 2 : K <= 512 ? 4 : 8; }
__host__ __device__ constexpr int lg_of_tiles(int NT) { return NT == 1 ? 2 : NT == 2 ? 3 : NT == 4 ? 4 : 5; }
// a row layout turned into the register path's (host code): NT, Ks = 128 * NT and lg from K
inline Dims reg_path_dims(Dims dm)
{
    dm.NT = reg_tiles(dm.K);
    dm.Ks = dm.NT * TILE;
    dm.lg = lg_of_tiles(dm.NT);
    return dm;
}
__host__ __device__ __forceinline__ int tpos_lg(int lg, int k)
{
    return (((k & ((1 << lg) - 1)) >> 2) << 7) | ((k >> lg) << 2) | (k & 3);
}
__host__ __device__ __forceinline__ int ttopic_lg(int lg, int p)
{
    return lg == 2 ? p : ((((p >> 2) & 31) << lg) | ((p >> 7) << 2) | (p & 3));
}
__host__ __device__ __forceinline__ int tpos(const Dims &dm, int k) { return tpos_lg(dm.lg, k); }      // topic -> column
__host__ __device__ __forceinline__ int ttopic(const Dims &dm, int p) { return ttopic_lg(dm.lg, p); }  // column -> topic

struct ZArgs {
    Dims dm;
    const int64_t *doc_off;   // [D+1] local CSR
    const int32_t *tokens;    // [N]
    int32_t *z;               // [N] in/out
    const float *phiT;        // [Vp][Ks]
    float *theta;             // [D][Ks] (GGS): read for chunks of long documents, written when the warp draws it
    const float *alpha;       // [Ks], natural topic order
    const int32_t *item_doc;  // GGS: [n_items] document of each chunk; PCGS: [D] LPT order
    const int64_t *item_begin;// GGS: [n_items] first token of each chunk
    int64_t n_items;
    int32_t chunk;            // GGS: tokens per work item
    int32_t fuse_theta;       // GGS: a work item that covers a whole document draws its theta itself
    unsigned long long *work_counter;
    int32_t *n_wk_out;        // when set (zeroed by the caller), the z-step also adds the new (w, z) counts
    uint32_t seed_lo, seed_hi, sweep;
    PhiloxKeys rk;            // round keys of (seed_lo, seed_hi)
};

struct ThetaArgs {
    Dims dm;
    const int64_t *doc_off;
    const int32_t *z;
    const float *alpha;   // [Ks]
    float *theta;         // [D][Ks]
    const int32_t *doc_list;  // documents to draw (n_docs entries), or null = all D documents
    int64_t n_docs;
    unsigned long long *work_counter;
    uint32_t seed_lo, seed_hi, sweep;
    PhiloxKeys rk;
};

// held-out left-to-right estimator (kernels_heldout.cu), one batch of documents [doc0, doc1) of the local test set
struct HeldoutArgs {
    Dims dm;                  // of phihat: K <= 1024, the register path's NT / Ks / lg, V, Vp
    const int64_t *doc_off;   // [D_test + 1] local test CSR
    const int32_t *tokens;    // [N_test]
    const float *phihat;      // [Vp][Ks]
    const float *alpha;       // [>= K], natural topic order
    int64_t doc0, doc1;       // the batch
    int64_t tok0;             // doc_off[doc0]: token t of the batch is column t - tok0 of S
    int64_t batch_tokens;     // doc_off[doc1] - tok0
    int32_t R;                // particles
    float *S;                 // [R][batch_tokens] score totals S_i^r
    int64_t token_base;       // global index of local test token 0 (Philox counter)
    uint32_t iteration;
    PhiloxKeys rk;
    unsigned long long *work_counter;
};

// ---------------------------------------------------------------------------------------
// Peer-memory exchange (kernels_p2p.cu, kernels_phi.cu): one process per GPU; every rank maps the
// other ranks' buffers with CUDA IPC, and the count exchange / Phi broadcast of a sweep are loads
// and stores over NVLink inside the Phi kernels instead of collectives around them.
// ---------------------------------------------------------------------------------------
constexpr int P2P_MAX = 8;           // ranks of one NVSwitch box (= PHI_SEGMENTS)
enum : int { P2P_FLAG_COUNTS = 0, P2P_FLAG_SEG = 1, P2P_FLAG_PHI = 2, P2P_FLAG_BAR = 3, P2P_FLAG_KINDS = 4 };

struct PeerTable {
    int32_t *n_wk[P2P_MAX];      // [Vp][Ks] partial counts of every rank (own entry = local buffer)
    float *phiT[P2P_MAX];        // [Vp][Ks] replicated Phi^T of every rank
    double *seg[P2P_MAX];        // [PHI_SEGMENTS][Ks] segment sums of every rank
    int32_t *nk_parts[P2P_MAX];  // [P2P_MAX][Ks] per-source topic totals landing on every rank
    uint32_t *flags[P2P_MAX];    // [P2P_FLAG_KINDS][P2P_MAX] epoch written by source rank, on every rank
    uint32_t *done_ctr;          // local: [P2P_FLAG_KINDS] CTA completion counters ("last block signals")
    int *error;                  // local: set when a wait timed out
    unsigned long long timeout_ns;
    int rank, world;
};

// n_k parts to every rank + "my partial counts are complete" (epoch) to every rank
cudaError_t launch_p2p_push_topic_totals(const PeerTable &pt, const int32_t *n_k_local, int32_t Ks, uint32_t epoch,
                                         cudaStream_t st);
// stand-alone reduce of the rank's vocabulary rows over all ranks' partial counts (+ n_k from the parts)
cudaError_t launch_p2p_reduce_counts(const PeerTable &pt, const Dims &dm, int32_t *n_k, int32_t row0, int32_t row1,
                                     uint32_t epoch, int sm_count, cudaStream_t st);
// signal `kind` with `epoch` to every rank / wait until every rank has signalled it
cudaError_t launch_p2p_signal(const PeerTable &pt, int kind, uint32_t epoch, cudaStream_t st);
cudaError_t launch_p2p_wait(const PeerTable &pt, int kind, uint32_t epoch, cudaStream_t st);
// fused variants of the three Phi kernels (kernels_phi.cu)
cudaError_t launch_phi_draw_p2p(const PeerTable &pt, bool reduce_counts, uint32_t epoch_counts, const Dims &dm,
                                int32_t *n_wk, int32_t *n_k, double beta, float *phiT, double *partial, int32_t row0,
                                int32_t row1, uint32_t seed_lo, uint32_t seed_hi, uint32_t sweep, int32_t poisson_L,
                                cudaStream_t st);
cudaError_t launch_phi_segment_sums_p2p(const PeerTable &pt, uint32_t epoch_seg, const Dims &dm, const double *partial,
                                        int seg0, int seg1, cudaStream_t st);
cudaError_t launch_phi_normalise_p2p(const PeerTable &pt, uint32_t epoch_seg, uint32_t epoch_phi, const Dims &dm,
                                     double *topic_sum, double *phi_mean_sum, int32_t row0, int32_t row1, int keep_zeros,
                                     cudaStream_t st);

// Opt a kernel into `smem` bytes of dynamic shared memory and report how many CTAs of `threads` threads fit
// one SM.  Both are properties of the CURRENT DEVICE, so the cache is keyed by the device ordinal (a second
// handle on another GPU of the same process gets its own opt-in) and guarded by a mutex.
inline cudaError_t kernel_config(const void *func, int threads, size_t smem, int *ctas_per_sm)
{
    static std::mutex mu;
    static std::map<std::tuple<const void *, int, int, size_t>, int> cache;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lock(mu);
    const auto key = std::make_tuple(func, dev, threads, smem);
    auto it = cache.find(key);
    if (it == cache.end()) {
        if (smem > 48 * 1024) {   // below that no opt-in is needed
            e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
        }
        int n = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, func, threads, smem);
        if (e != cudaSuccess) return e;
        it = cache.emplace(key, n < 1 ? 1 : n).first;
    }
    if (ctas_per_sm) *ctas_per_sm = it->second;
    return cudaSuccess;
}

// launchers (each returns the cudaError of the launch)
cudaError_t launch_theta(const ThetaArgs &a, int sm_count, cudaStream_t st);
cudaError_t launch_z_ggs(const ZArgs &a, int sm_count, cudaStream_t st);
cudaError_t launch_z_pcgs(const ZArgs &a, int sm_count, cudaStream_t st);
// K > 1024 (kernels_z_big.cu): row and per-document vector in shared memory
cudaError_t launch_theta_big(const ThetaArgs &a, int sm_count, cudaStream_t st);
cudaError_t launch_z_ggs_big(const ZArgs &a, int sm_count, cudaStream_t st);
cudaError_t launch_z_pcgs_big(const ZArgs &a, int sm_count, cudaStream_t st);
// sparse PCGS z-step and its alias tables (kernels_sparse.cu)
// one slot of a type's alias table (util/OptimizedGentleAliasMethod.java:52-79: ps[i], a[i]) -- kept side by
// side so that building a slot is one 8-byte store and a draw one 8-byte load
struct __align__(8) AliasSlot {
    float ps;
    int32_t alias;
};
int64_t alias_scratch_threads(const Dims &dm, int sm_count);
size_t alias_stack_ints(const Dims &dm, int64_t T);     // ints of the stack scratch for T slots (topics + the count pairs)
size_t alias_value_doubles(const Dims &dm, int64_t T);  // doubles of the value scratch for T slots
cudaError_t launch_alias_build(const Dims &dm, const float *alpha, const float *phiT, AliasSlot *table,
                               float *type_norm, double *bs_scratch, int32_t *stack_scratch,
                               const int32_t *active, int32_t n_active, int64_t slots, int sm_count, cudaStream_t st);
size_t spalias_list_bytes(const Dims &dm, int max_doc_len, int sm_count);
cudaError_t launch_z_spalias(const ZArgs &z, const AliasSlot *table, const float *type_norm,
                             int *lists, int max_doc_len, int sm_count, cudaStream_t st);
// largest K the dense z-step can hold in shared memory (row + vector [+ counts] per warp)
inline int max_dense_topics(bool pcgs) { return pcgs ? 18000 : 27000; }
cudaError_t launch_counts(const Dims &dm, const int32_t *tokens, const int32_t *z, int32_t *n_wk,
                          int32_t *n_k, int sm_count, cudaStream_t st);
cudaError_t launch_counts_chunk(const Dims &dm, const int32_t *tokens, const int32_t *z, int64_t n, int32_t *n_wk,
                                int *bad, int sm_count, cudaStream_t st);
cudaError_t launch_unpack16(const uint16_t *in, int32_t *out, int64_t n, int sm_count, cudaStream_t st);
cudaError_t launch_pack16(const int32_t *in, uint16_t *out, int64_t n, int sm_count, cudaStream_t st);
cudaError_t launch_topic_totals(const Dims &dm, const int32_t *n_wk, int32_t *n_k, cudaStream_t st);
cudaError_t launch_doc_topic_counts(const Dims &dm, const int64_t *doc_off, const int32_t *z,
                                    int32_t *n_dk /*[D][K] dense*/, cudaStream_t st);
// Phi draw over rows [row0, row1) (multiples of 64); partial[(row/8)][Ks] fp64
cudaError_t launch_phi_draw(const Dims &dm, const int32_t *n_wk, double beta, float *phiT,
                            double *partial, int32_t row0, int32_t row1, uint32_t seed_lo,
                            uint32_t seed_hi, uint32_t sweep, int32_t poisson_L /* > 0: Polya-urn Poisson draw */, cudaStream_t st);
// segment sums seg[s][Ks] for segments [seg0, seg1)
cudaError_t launch_phi_segment_sums(const Dims &dm, const double *partial, double *seg, int seg0,
                                    int seg1, cudaStream_t st);
// S_k from the 8 segment sums, then normalise rows [row0,row1) and optionally add into phi_sum
cudaError_t launch_phi_normalise(const Dims &dm, const double *seg, double *topic_sum, float *phiT,
                                 double *phi_mean_sum, int32_t row0, int32_t row1, int keep_zeros, cudaStream_t st);
// log-likelihood pieces: per-block partial sums (ll_type: pairs {sum, nnz})
cudaError_t launch_lgs_table(int K, const double *alpha, double *out /*[K] lgS(alpha_k)*/, cudaStream_t st);
cudaError_t launch_ll_doc(const Dims &dm, const int64_t *doc_off, const int32_t *z,
                          const double *alpha, const double *lgs_alpha, double alpha_sum, double *partials,
                          int n_partials, int sm_count, cudaStream_t st);
cudaError_t launch_ll_type(const Dims &dm, const int32_t *n_wk, double beta, int32_t row0,
                           int32_t row1, double *partials, int n_partials, cudaStream_t st);
// histograms of the count values for the hyper-parameter optimisation (ModifiedSimpleLDA.java:812-905)
cudaError_t launch_count_histograms(const Dims &dm, const int64_t *doc_off, const int32_t *z, const int32_t *n_wk,
                                    int32_t row0, int32_t row1, unsigned long long *doc_hist, int n_doc_bins,
                                    unsigned long long *type_hist, int n_type_bins, cudaStream_t st);
// log-posterior pieces (UncollapsedParallelLDA.java:1573-1634)
cudaError_t launch_lp_tokens(const Dims &dm, const int32_t *tokens, const int32_t *z,
                             const float *phiT, double *partials, int n_partials, cudaStream_t st);
cudaError_t launch_lp_theta(const Dims &dm, const int64_t *doc_off, const int32_t *z,
                            const float *theta, const double *alpha, double *partials,
                            int n_partials, int sm_count, cudaStream_t st);
cudaError_t launch_lp_phi(const Dims &dm, const float *phiT, double beta, int32_t row0, int32_t row1,
                          double *partials, int n_partials, cudaStream_t st);
// held-out log-likelihood (kernels_heldout.cu): phihat in dst's layout from n_wk in src's layout and n_k; the
// particles' score totals of one batch; the per-document values of that batch into doc_ll[0, doc1 - doc0)
cudaError_t launch_heldout_phihat(const Dims &src, const Dims &dst, const int32_t *n_wk, const int32_t *n_k, double beta,
                                  float *phihat, int sm_count, cudaStream_t st);
cudaError_t launch_heldout_l2r(const HeldoutArgs &a, int sm_count, cudaStream_t st);
cudaError_t launch_heldout_reduce(const HeldoutArgs &a, double alpha_sum, double *doc_ll, int sm_count, cudaStream_t st);
// out[j] = sum_i partials[i*stride + j], sequential in i
cudaError_t launch_sum_partials(const double *partials, int n, int stride, double *out, cudaStream_t st);

// transposes / conversions for the accessors
cudaError_t launch_export_phi(const Dims &dm, const float *phiT, double *phi_kv /*[K][V]*/, cudaStream_t st);
cudaError_t launch_import_phi(const Dims &dm, const double *phi_kv, float *phiT, cudaStream_t st);
cudaError_t launch_export_mean(const Dims &dm, const double *sum_vk, double scale, double *out_kv, cudaStream_t st);
cudaError_t launch_export_counts(const Dims &dm, const int32_t *n_wk, int32_t *out_vk /*[V][K] dense*/, cudaStream_t st);
cudaError_t launch_export_theta(const Dims &dm, const float *theta, double *out /*[D][K]*/, cudaStream_t st);
cudaError_t launch_import_theta(const Dims &dm, const double *in, float *theta, cudaStream_t st);
cudaError_t launch_validate(const Dims &dm, const int32_t *tokens, const int32_t *z, int *bad, cudaStream_t st);

// ---------------------------------------------------------------------------------------
// device helpers: mbarrier + 1-D bulk async copy (TMA engine, cp.async.bulk)
// ---------------------------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// global -> shared bulk copy, completion signalled on the mbarrier (bytes % 16 == 0, 16 B aligned)
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// ---- cross-GPU flags: release/acquire at system scope over peer-mapped memory ----------------
__device__ __forceinline__ void st_release_sys(uint32_t *p, uint32_t v)
{
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t *p)
{
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long globaltimer_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
// One thread: spin until every rank's flag of `kind` (in THIS rank's flag array) has reached epoch.
// A rank that never arrives (dead peer process) must not hang the GPU: after timeout_ns the wait
// gives up and raises the error word, which the host checks after every synchronise.
__device__ __forceinline__ void p2p_wait_all(const PeerTable &pt, int kind, uint32_t epoch)
{
    const uint32_t *f = pt.flags[pt.rank] + kind * P2P_MAX;
    const unsigned long long t0 = globaltimer_ns();
    for (int r = 0; r < pt.world; ++r) {
        // epochs only grow; the signed difference keeps the comparison valid across a wrap
        while ((int32_t)(ld_acquire_sys(f + r) - epoch) < 0) {
            if (globaltimer_ns() - t0 > pt.timeout_ns) { atomicExch(pt.error, 1 + kind); return; }
            __nanosleep(200);
        }
    }
}
// One thread per destination rank (tid < world): publish epoch in every rank's flag array.
__device__ __forceinline__ void p2p_signal_one(const PeerTable &pt, int kind, uint32_t epoch, int dst)
{
    st_release_sys(pt.flags[dst] + kind * P2P_MAX + pt.rank, epoch);
}
// "last block signals": every thread has finished its peer stores; the CTA that arrives last at the
// local counter publishes the epoch to all ranks.
__device__ __forceinline__ void p2p_cta_done_signal(const PeerTable &pt, int kind, uint32_t epoch, unsigned total_ctas)
{
    __threadfence_system();
    __syncthreads();
    __shared__ bool s_last;
    if (threadIdx.x == 0) {
        const unsigned prev = atomicAdd(pt.done_ctr + kind, 1u);
        s_last = prev == total_ctas - 1;
        if (s_last) pt.done_ctr[kind] = 0;   // ready for the next launch (stream order separates launches)
    }
    __syncthreads();
    if (s_last) {
        __threadfence_system();
        if ((int)threadIdx.x < pt.world) p2p_signal_one(pt, kind, epoch, (int)threadIdx.x);
    }
}
#endif

}  // namespace ldagpu
