// engine.cu -- host side of libldagpu.so: the handle, the sweep driver, the NCCL exchange step and
// the C ABI declared in include/ldagpu.h.
//
// One sweep (reference order: topics/UncollapsedParallelLDA.java:645-693):
//   [GGS] theta_kernel        theta_d ~ Dir(n_d + alpha) for the documents the z-step does not draw itself:
//                             those longer than one work item (all of them above the register path's K)  (GGS:60-72)
//   z_kernel                  [GGS] theta_d of a whole-document work item, then z_i | theta/n_d, Phi; n_wk
//                             accumulated from the new z                  (GGS:79-130, UPL:1491-1543, 1107-1221)
//   topic_totals_kernel       n_k from n_wk
//   [G>1] reduce-scatter n_wk by vocabulary slice, all-reduce n_k         (stand-in for the shared
//                                                                         AtomicInteger[K][V], UPL:102)
//   phi_draw / segments       Gamma(beta + n_wk) for the rank's slice     (GGS:182-192, PCGS:91-101)
//   [G>1] all-gather the 8 segment sums
//   phi_normalise             rows of the slice
//   [G>1] all-gather Phi^T
// With peer access between the GPUs (the default on an NVSwitch box) the three [G>1] steps are not
// collectives: the Phi kernels load the peers' partial counts and store the segment sums and the
// normalised rows into every rank's buffers themselves (kernels_p2p.cu, kernels_phi.cu); NCCL only
// bootstraps (IPC handle exchange) and serves the accessors.  LDAGPU_EXCHANGE=nccl keeps the
// collective path.
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

#include "../../include/ldagpu.h"
#include "common.cuh"

using namespace ldagpu;

namespace {

thread_local std::string g_create_error;

// ---- NCCL through dlopen: single-GPU users need no NCCL at all -----------------------------
struct NcclApi {
    void *lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*ReduceScatter)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    std::string err;
    bool load()
    {
        if (lib) return true;
        // resolves to the copy already mapped into the process (torch's bundled NCCL) when there is one
        lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) { err = std::string("dlopen libnccl.so.2: ") + dlerror(); return false; }
#define LD(field, sym)                                                          \
    field = reinterpret_cast<decltype(field)>(dlsym(lib, sym));                 \
    if (!field) { err = std::string("dlsym ") + sym + " failed"; lib = nullptr; return false; }
        LD(GetUniqueId, "ncclGetUniqueId")
        LD(CommInitRank, "ncclCommInitRank")
        LD(CommDestroy, "ncclCommDestroy")
        LD(ReduceScatter, "ncclReduceScatter")
        LD(AllGather, "ncclAllGather")
        LD(AllReduce, "ncclAllReduce")
        LD(GetErrorString, "ncclGetErrorString")
#undef LD
        return true;
    }
};
NcclApi g_nccl;

// Device memory owned by one object, freed when it is destroyed or overwritten.  That must happen with its own device
// current: the engine never relies on a cudaFree issued from another device.
template <typename T> struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    DevBuf(DevBuf &&o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
    DevBuf &operator=(DevBuf &&o) noexcept
    {
        if (this != &o) {
            release();
            p = o.p; n = o.n;
            o.p = nullptr; o.n = 0;
        }
        return *this;
    }
    ~DevBuf() { release(); }
    cudaError_t alloc(size_t count)
    {
        release();
        n = count;
        if (count == 0) return cudaSuccess;
        return cudaMalloc(reinterpret_cast<void **>(&p), sizeof(T) * count);
    }
    void release()
    {
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
    }
};

// java.util.Random, JDK 8 specification (the reference's initial z: UPL:398-406,458-460)
struct JavaRandom {
    uint64_t s;
    explicit JavaRandom(int64_t seed) : s(((uint64_t)seed ^ 0x5DEECE66Dull) & ((1ull << 48) - 1)) {}
    int32_t next(int bits)
    {
        s = (s * 0x5DEECE66Dull + 0xBull) & ((1ull << 48) - 1);
        return (int32_t)(uint32_t)(s >> (48 - bits));
    }
    int32_t nextInt(int32_t bound)
    {
        int32_t r = next(31);
        int32_t m = bound - 1;
        if ((bound & m) == 0) return (int32_t)(((int64_t)bound * (int64_t)r) >> 31);
        for (int32_t u = r;; u = next(31)) {
            r = u % bound;
            if ((int32_t)((uint32_t)u - (uint32_t)r + (uint32_t)m) >= 0) break;
        }
        return r;
    }
};

constexpr int N_PARTIALS = 592;   // 4 CTAs per SM on a 148-SM part; fixed so sums are reproducible
constexpr int EV_PER_SWEEP = 9;
// bound of the held-out score buffer S[R][batch tokens]: a test set whose R * N_test floats do not fit is evaluated in
// document batches (a single document longer than the bound gets a batch, and a buffer, of its own)
constexpr int64_t HELDOUT_SCRATCH_BYTES = 1ll << 30;

}  // namespace

struct ldagpu_handle_s {
    Dims dm{};
    int scheme = 0, device = 0, sm_count = 148;
    double beta = 0.0, alpha_sum = 0.0;
    std::vector<double> alpha;
    uint64_t seed = 0;
    int32_t iteration = 0;
    int64_t D_global = 0;

    DevBuf<int64_t> doc_off, item_begin;
    DevBuf<int32_t> tokens, z, z_stage, n_wk, n_k, item_doc, long_docs, scratch_i32;
    DevBuf<uint16_t> z16;   // 16-bit transport buffer of the topic indicators (ldagpu_set_z16 / ldagpu_sweep_get_z16)
    struct ZPart { int64_t item0, item1, tok0, tok1; };
    std::vector<ZPart> z_parts;   // GGS, >= 8 Mi tokens: document-aligned parts of the work items for the streamed read-back of z
    int64_t n_long_docs = 0;   // GGS: documents longer than one work item (their theta is drawn before the z-step)
    DevBuf<float> phiT, theta, alpha_f;
    // sparse scheme: per-type alias tables over alpha_k * phi_kw and the build scratch
    DevBuf<float> type_norm;
    DevBuf<AliasSlot> alias_table;
    DevBuf<int32_t> alias_stack, active_types, sparse_lists;
    int32_t n_active_types = 0;
    DevBuf<double> alias_bs;
    int64_t alias_slots = 0;   // types per round of the alias-table kernels (scratch slots)
    int max_doc_len = 0;
    DevBuf<double> alpha_d, lgs_alpha, partial, seg, topic_sum, phi_mean, red, red_out, scratch_f64;
    DevBuf<unsigned long long> counter;
    DevBuf<int> bad;
    int64_t n_items = 0;
    int32_t ggs_chunk = GGS_CHUNK_MAX;
    std::vector<int64_t> h_doc_off;

    // held-out test set (ldagpu_set_test_documents): local CSR on the device and on the host, and the global index of
    // its first document / token.  A group keeps the shard bounds of its test set in test_doc0 / test_tok0.
    DevBuf<int64_t> test_doc_off;
    DevBuf<int32_t> test_tokens;
    std::vector<int64_t> h_test_doc_off{0}, test_doc0{0, 0}, test_tok0{0, 0};
    int64_t test_doc_base = 0, test_token_base = 0;
    DevBuf<float> phihat, ho_scores;   // during an evaluation: phihat [Vp][Ks of the register path], S [R][batch tokens]
    DevBuf<double> ho_ll;               // during an evaluation: [D_test] per-document values

    int32_t mean_burn_in = 0, mean_thin = 1, n_sampled_phi = 0;
    int32_t poisson_L = 0;   // > 0: Phi rows are drawn by the Poisson Polya urn (ldagpu_set_phi_sampler)

    cudaStream_t stream = nullptr;
    std::vector<cudaEvent_t> events;
    // host <-> device copies of z overlap the kernels next to them: a second stream and a few ordering events
    cudaStream_t copy_stream = nullptr;
    std::vector<cudaEvent_t> copy_events;

    int rank = 0, world = 1;
    ncclComm_t comm = nullptr;
    int32_t row0 = 0, row1 = 0, seg0 = 0, seg1 = PHI_SEGMENTS;
    // peer-memory exchange
    bool p2p = false;
    PeerTable pt{};
    DevBuf<int32_t> nk_parts;
    DevBuf<uint32_t> p2p_flags, p2p_local;   // shared epoch flags; local {done counters[4], error}
    std::vector<void *> ipc_opened;
    uint32_t ep[P2P_FLAG_KINDS] = {0, 0, 0, 0};
    uint32_t counts_epoch = 0;   // epoch of the last "counts complete" signal (consumed by the reduce)
    uint32_t bar_epoch = 0, seg_epoch = 0, phi_epoch = 0;   // epochs in flight between the stages of an exchange
    std::string p2p_note;

    // single-process multi-GPU (ldagpu_create_multi): this handle only coordinates; the shards hold the state
    std::vector<ldagpu_handle> shards;
    std::vector<int64_t> shard_doc0, shard_tok0;   // [parts + 1] first document / token of every part, in this handle's order
    bool multi() const { return !shards.empty(); }
    // what an entry point fans out to, in shard order: the shards of a group, else the handle itself (a group of one)
    std::vector<ldagpu_handle> parts() { return multi() ? shards : std::vector<ldagpu_handle>{this}; }

    std::atomic<int> abort_flag{0};
    std::string err;
    double t_z = 0, t_counts = 0, t_phi = 0, t_comm = 0;
    double last_zk_ms = 0, last_call_ms = 0;
    int64_t last_zk_launches = 0, last_launches = 0;

    int fail(const char *fmt, ...)
    {
        char buf[512];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof buf, fmt, ap);
        va_end(ap);
        err = buf;
        return 1;
    }
};

#define CK(h, call)                                                                              \
    do {                                                                                         \
        cudaError_t e__ = (call);                                                                \
        if (e__ != cudaSuccess)                                                                  \
            return (h)->fail("%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
    } while (0)
#define NK(h, call)                                                                                       \
    do {                                                                                                  \
        ncclResult_t r__ = (call);                                                                        \
        if (r__ != ncclSuccess)                                                                           \
            return (h)->fail("%s:%d %s: %s", __FILE__, __LINE__, #call, g_nccl.GetErrorString(r__));      \
    } while (0)
#define NEED(h)                                  \
    if (!(h)) return 1;                          \
    CK(h, cudaSetDevice((h)->device))
// one part's share of a call: on the part's device; a failure is reported on the caller's handle
#define MC(P, c, call)                               \
    do {                                             \
        cudaSetDevice((c)->device);                  \
        if (call) return part_fail(P, c);            \
    } while (0)

namespace {

using Parts = std::vector<ldagpu_handle>;

int part_fail(ldagpu_handle P, ldagpu_handle c)
{
    P->err = c->err;
    return 1;
}

int ensure_events(ldagpu_handle h, size_t n)
{
    while (h->events.size() < n) {
        cudaEvent_t e;
        CK(h, cudaEventCreate(&e));
        h->events.push_back(e);
    }
    return 0;
}

int ensure_theta(ldagpu_handle h)
{
    if (h->theta.p) return 0;
    CK(h, h->theta.alloc((size_t)std::max<int64_t>(h->dm.D, 1) * h->dm.Ks));
    CK(h, cudaMemsetAsync(h->theta.p, 0, sizeof(float) * h->theta.n, h->stream));
    return 0;
}

// theta_d ~ Dir(n_d + alpha) for every document, or (only_long, inside a sweep) for the documents that the
// z-step splits into several work items -- the others draw their theta inside the z kernel
int step_theta(ldagpu_handle h, bool only_long = false)
{
    if (ensure_theta(h)) return 1;
    const bool fused_path = h->dm.K <= MAX_REG_TILES * TILE;
    if (only_long && fused_path && h->n_long_docs == 0) return 0;
    CK(h, cudaMemsetAsync(h->counter.p, 0, sizeof(unsigned long long), h->stream));
    ThetaArgs a{};
    a.dm = h->dm; a.doc_off = h->doc_off.p; a.z = h->z.p; a.alpha = h->alpha_f.p; a.theta = h->theta.p;
    a.doc_list = nullptr; a.n_docs = h->dm.D;
    if (only_long && fused_path) { a.doc_list = h->long_docs.p; a.n_docs = h->n_long_docs; }
    a.work_counter = h->counter.p;
    a.seed_lo = (uint32_t)h->seed; a.seed_hi = (uint32_t)(h->seed >> 32); a.sweep = (uint32_t)h->iteration;
    a.rk = philox_keys(a.seed_lo, a.seed_hi);
    CK(h, launch_theta(a, h->sm_count, h->stream));
    h->last_launches += 1;
    return 0;
}

// fused: the z kernel also accumulates n_wk (which the caller has zeroed)
// part >= 0 (GGS): only the work items of part `part` of h->z_parts -- the last sweep of a call that returns z runs the
// z-step in parts, so that the read-back of one part overlaps the z-step of the next (sweep_enqueue)
int step_z(ldagpu_handle h, bool fused = false, bool fuse_theta = false, int part = -1)
{
    unsigned long long *counter = h->counter.p + (part >= 0 ? 1 + part : 0);
    CK(h, cudaMemsetAsync(counter, 0, sizeof(unsigned long long), h->stream));
    ZArgs a{};
    a.dm = h->dm; a.doc_off = h->doc_off.p; a.tokens = h->tokens.p; a.z = h->z.p; a.phiT = h->phiT.p;
    a.theta = h->theta.p; a.alpha = h->alpha_f.p; a.item_doc = h->item_doc.p; a.item_begin = h->item_begin.p;
    a.n_items = h->n_items; a.chunk = h->ggs_chunk; a.work_counter = counter;
    if (part >= 0) {
        const auto &zp = h->z_parts[(size_t)part];
        a.item_doc += zp.item0; a.item_begin += zp.item0; a.n_items = zp.item1 - zp.item0;
    }
    a.n_wk_out = fused ? h->n_wk.p : nullptr;
    a.fuse_theta = fuse_theta ? 1 : 0;
    a.seed_lo = (uint32_t)h->seed; a.seed_hi = (uint32_t)(h->seed >> 32); a.sweep = (uint32_t)h->iteration;
    a.rk = philox_keys(a.seed_lo, a.seed_hi);
    if (h->scheme == LDAGPU_SCHEME_GGS) {
        if (!h->theta.p) return h->fail("GGS z-step needs theta: call ldagpu_sample_theta or ldagpu_set_theta first");
        CK(h, launch_z_ggs(a, h->sm_count, h->stream));
    } else if (h->scheme == LDAGPU_SCHEME_SPALIAS) {
        CK(h, launch_z_spalias(a, h->alias_table.p, h->type_norm.p, h->sparse_lists.p, h->max_doc_len,
                               h->sm_count, h->stream));
    } else {
        CK(h, launch_z_pcgs(a, h->sm_count, h->stream));
    }
    if (a.n_items) { h->last_launches += 1; h->last_zk_launches += part > 0 ? 0 : 1; }
    return 0;
}

// sparse scheme: the alias tables follow every change of Phi (SpaliasUncollapsedParallelLDA.java:39-60)
int step_alias(ldagpu_handle h)
{
    if (h->scheme != LDAGPU_SCHEME_SPALIAS) return 0;
    CK(h, launch_alias_build(h->dm, h->alpha_f.p, h->phiT.p, h->alias_table.p, h->type_norm.p,
                             h->alias_bs.p, h->alias_stack.p, h->active_types.p, h->n_active_types, h->alias_slots,
                             h->sm_count, h->stream));
    // classify + pair per round (one round unless the active vocabulary exceeds the scratch slots)
    h->last_launches += 2 * (int)((h->n_active_types + h->alias_slots - 1) / std::max<int64_t>(h->alias_slots, 1));
    return 0;
}

int step_counts_local(ldagpu_handle h)
{
    CK(h, launch_counts(h->dm, h->tokens.p, h->z.p, h->n_wk.p, h->n_k.p, h->sm_count, h->stream));
    h->last_launches += h->dm.N > 0 ? 2 : 1;   // counts_kernel + topic_totals_kernel
    return 0;
}

// Peer-memory mode: the in-kernel waits are bounded (a dead rank must not hang the GPU), so host-side skew
// between the ranks -- one rank still generating its shard, replaying java.util.Random for a later shard --
// must not reach them.  Every API call that exchanges starts with one tiny NCCL all-reduce, which waits as
// long as it takes; after it the ranks are microseconds apart and the flag waits only absorb compute skew.
int rendezvous(ldagpu_handle h, int *abort_any = nullptr)
{
    if (abort_any) *abort_any = h->abort_flag.load(std::memory_order_relaxed);
    if (h->world == 1 || !h->comm) return 0;   // single GPU, or shards driven by one caller thread (no skew to absorb)
    if (!h->p2p && !abort_any) return 0;       // the NCCL collectives wait as long as it takes anyway
    uint32_t *word = h->p2p_local.p + P2P_FLAG_KINDS + 1;
    uint32_t mine = abort_any ? (uint32_t)(*abort_any != 0) : 0u;
    CK(h, cudaMemcpyAsync(word, &mine, sizeof mine, cudaMemcpyHostToDevice, h->stream));
    NK(h, g_nccl.AllReduce(word, word, 1, ncclUint32, ncclMax, h->comm, h->stream));
    if (abort_any) {
        CK(h, cudaMemcpyAsync(&mine, word, sizeof mine, cudaMemcpyDeviceToHost, h->stream));
        CK(h, cudaStreamSynchronize(h->stream));
        *abort_any = (int)mine;
    }
    return 0;
}

// Stages.  With several shards driven by ONE caller thread (ldagpu_create_multi) a kernel that waits, on the device,
// for another shard's signal must only be enqueued after the kernel that gives the signal: a launch can block the
// host until the device drains (first use of a kernel under lazy module loading, a larger local-memory pool), and a
// device that waits for work the blocked host has not enqueued yet would never drain.  So the exchange and the Phi
// draw are cut into stages -- every waiter in a later stage than the signals it waits for -- and every operation that
// exchanges runs stage by stage over all parts (run_stages); a single GPU is a group of one.  The NCCL collectives and a
// single GPU have nothing to order: they do all their work in the first stage of the exchange and of the Phi draw.
enum Stage {
    ST_LOCAL,       // [theta +] z-step, topic totals, push n_k parts + "my partial counts are complete"
    ST_REDUCE,      // reduce the rank's vocabulary rows over all ranks' counts (waits for ST_LOCAL of all), signal the barrier
    ST_BARRIER,     // wait for the barrier: nobody touches its partial counts again before every rank has read them
    ST_DRAW,        // Phi draw (+ the peers' counts when fused) + segment sums stored to every rank + "segments in place"
    ST_NORMALISE,   // normalise (waits for every rank's segments) + rows stored to every rank + "rows in place"
    ST_LAND,        // wait until every rank's rows have landed here; [sparse scheme] rebuild the alias tables
    N_STAGES
};

// every stage on every part before the next stage on any part
template <typename F> int run_stages(ldagpu_handle h, const Parts &parts, F &&stage_of_part)
{
    for (int st = 0; st < N_STAGES; ++st)
        for (size_t g = 0; g < parts.size(); ++g) MC(h, parts[g], stage_of_part(g, (Stage)st));
    return 0;
}

// defer_reduce (peer-memory mode): only announce the partial counts; the Phi draw that follows sums them.
int step_counts_exchange(ldagpu_handle h, bool defer_reduce, Stage stage)
{
    if (h->world == 1) return 0;
    if (h->p2p) {
        if (stage == ST_LOCAL) {
            h->counts_epoch = ++h->ep[P2P_FLAG_COUNTS];
            CK(h, launch_p2p_push_topic_totals(h->pt, h->n_k.p, h->dm.Ks, h->counts_epoch, h->stream));
            h->last_launches += 1;
        }
        if (defer_reduce) return 0;
        if (stage == ST_REDUCE) {
            CK(h, launch_p2p_reduce_counts(h->pt, h->dm, h->n_k.p, h->row0, h->row1, h->counts_epoch, h->sm_count, h->stream));
            h->bar_epoch = ++h->ep[P2P_FLAG_BAR];
            CK(h, launch_p2p_signal(h->pt, P2P_FLAG_BAR, h->bar_epoch, h->stream));
            h->last_launches += 2;
        }
        if (stage == ST_BARRIER) {
            CK(h, launch_p2p_wait(h->pt, P2P_FLAG_BAR, h->bar_epoch, h->stream));
            h->last_launches += 1;
        }
        return 0;
    }
    if (stage != ST_LOCAL) return 0;
    const size_t slice = (size_t)(h->dm.Vp / h->world) * h->dm.Ks;
    NK(h, g_nccl.ReduceScatter(h->n_wk.p, h->n_wk.p + (size_t)h->rank * slice, slice, ncclInt32, ncclSum, h->comm, h->stream));
    NK(h, g_nccl.AllReduce(h->n_k.p, h->n_k.p, (size_t)h->dm.Ks, ncclInt32, ncclSum, h->comm, h->stream));
    return 0;
}

int phi_mean_buffer(ldagpu_handle h, bool accumulate_mean, double **mean)
{
    *mean = nullptr;
    if (!accumulate_mean) return 0;
    if (!h->phi_mean.p) {
        CK(h, h->phi_mean.alloc((size_t)h->dm.Vp * h->dm.Ks));
        CK(h, cudaMemsetAsync(h->phi_mean.p, 0, sizeof(double) * h->phi_mean.n, h->stream));
    }
    *mean = h->phi_mean.p;
    return 0;
}

// peer-memory mode: the fused draw (fused_reduce) sums the peers' partial counts, waiting for their "counts complete"
int step_phi_p2p(ldagpu_handle h, bool accumulate_mean, cudaEvent_t *ev, bool fused_reduce, Stage stage)
{
    const uint32_t lo = (uint32_t)h->seed, hi = (uint32_t)(h->seed >> 32);
    if (stage == ST_DRAW) {
        CK(h, launch_phi_draw_p2p(h->pt, fused_reduce, h->counts_epoch, h->dm, h->n_wk.p, h->n_k.p, h->beta, h->phiT.p,
                                  h->partial.p, h->row0, h->row1, lo, hi, (uint32_t)h->iteration, h->poisson_L, h->stream));
        h->seg_epoch = ++h->ep[P2P_FLAG_SEG];
        CK(h, launch_phi_segment_sums_p2p(h->pt, h->seg_epoch, h->dm, h->partial.p, h->seg0, h->seg1, h->stream));
        h->last_launches += 2;
        if (ev) { CK(h, cudaEventRecord(ev[0], h->stream)); CK(h, cudaEventRecord(ev[1], h->stream)); }
    }
    if (stage == ST_NORMALISE) {
        double *mean = nullptr;
        if (phi_mean_buffer(h, accumulate_mean, &mean)) return 1;
        h->phi_epoch = ++h->ep[P2P_FLAG_PHI];
        CK(h, launch_phi_normalise_p2p(h->pt, h->seg_epoch, h->phi_epoch, h->dm, h->topic_sum.p, mean, h->row0, h->row1,
                                       h->poisson_L > 0, h->stream));
        h->last_launches += 1;
        if (ev) CK(h, cudaEventRecord(ev[2], h->stream));
    }
    if (stage == ST_LAND) {
        CK(h, launch_p2p_wait(h->pt, P2P_FLAG_PHI, h->phi_epoch, h->stream));
        h->last_launches += 1;
        if (step_alias(h)) return 1;
        if (ev) CK(h, cudaEventRecord(ev[3], h->stream));
    }
    return 0;
}

// ev != nullptr: record events after draw+segments, segment all-gather, normalise, Phi all-gather
int step_phi(ldagpu_handle h, bool accumulate_mean, cudaEvent_t *ev, bool fused_reduce, Stage stage)
{
    if (h->p2p) return step_phi_p2p(h, accumulate_mean, ev, fused_reduce, stage);
    if (stage != ST_DRAW) return 0;
    const uint32_t lo = (uint32_t)h->seed, hi = (uint32_t)(h->seed >> 32);
    CK(h, launch_phi_draw(h->dm, h->n_wk.p, h->beta, h->phiT.p, h->partial.p, h->row0, h->row1, lo, hi,
                          (uint32_t)h->iteration, h->poisson_L, h->stream));
    CK(h, launch_phi_segment_sums(h->dm, h->partial.p, h->seg.p, h->seg0, h->seg1, h->stream));
    h->last_launches += 2;
    if (ev) CK(h, cudaEventRecord(ev[0], h->stream));
    if (h->world > 1) {
        const size_t per = (size_t)(PHI_SEGMENTS / h->world) * h->dm.Ks;
        NK(h, g_nccl.AllGather(h->seg.p + (size_t)h->rank * per, h->seg.p, per, ncclDouble, h->comm, h->stream));
    }
    if (ev) CK(h, cudaEventRecord(ev[1], h->stream));
    double *mean = nullptr;
    if (phi_mean_buffer(h, accumulate_mean, &mean)) return 1;
    CK(h, launch_phi_normalise(h->dm, h->seg.p, h->topic_sum.p, h->phiT.p, mean, h->row0, h->row1, h->poisson_L > 0, h->stream));
    h->last_launches += 1;
    if (ev) CK(h, cudaEventRecord(ev[2], h->stream));
    if (h->world > 1) {
        const size_t slice = (size_t)(h->dm.Vp / h->world) * h->dm.Ks;
        NK(h, g_nccl.AllGather(h->phiT.p + (size_t)h->rank * slice, h->phiT.p, slice, ncclFloat, h->comm, h->stream));
    }
    if (step_alias(h)) return 1;
    if (ev) CK(h, cudaEventRecord(ev[3], h->stream));
    return 0;
}

bool mean_this_iteration(ldagpu_handle h)
{
    // UPL:1350-1352 samplePhiThisIteration()
    return h->mean_burn_in > 0 && h->iteration > h->mean_burn_in && h->mean_thin > 0 &&
           h->iteration % h->mean_thin == 0;
}

int sync_check(ldagpu_handle h)
{
    CK(h, cudaStreamSynchronize(h->stream));
    CK(h, cudaGetLastError());
    if (h->p2p) {
        int err = 0;
        CK(h, cudaMemcpy(&err, h->p2p_local.p + P2P_FLAG_KINDS, sizeof err, cudaMemcpyDeviceToHost));
        if (err) {
            static const char *what[] = {"partial counts", "segment sums", "Phi rows", "barrier"};
            return h->fail("peer-memory exchange: waiting for the %s of another rank timed out (is a rank dead?)",
                           what[(err - 1) & 3]);
        }
    }
    return 0;
}

int sync_all(ldagpu_handle h, const Parts &parts)
{
    for (ldagpu_handle c : parts) MC(h, c, sync_check(c));
    return 0;
}

int ensure_z16(ldagpu_handle h)
{
    if (!h->z16.p) CK(h, h->z16.alloc((size_t)std::max<int64_t>(h->dm.N, 1) + 8));
    return 0;
}

// z[o, o + cnt) to z_out[o, ...) on `stream`, or narrowed on the device to z16_out[o, ...) when that is given
int copy_z_out(ldagpu_handle h, int32_t *z_out, uint16_t *z16_out, int64_t o, int64_t cnt, cudaStream_t stream)
{
    if (z16_out) {
        CK(h, launch_pack16(h->z.p + o, h->z16.p + o, cnt, h->sm_count, stream));
        CK(h, cudaMemcpyAsync(z16_out + o, h->z16.p + o, sizeof(uint16_t) * (size_t)cnt, cudaMemcpyDeviceToHost, stream));
    } else {
        CK(h, cudaMemcpyAsync(z_out + o, h->z.p + o, sizeof(int32_t) * (size_t)cnt, cudaMemcpyDeviceToHost, stream));
    }
    return 0;
}

// ---- a call of n sweeps in three pieces, so that one caller thread can drive several shards (ldagpu_create_multi):
// sweeps_prepare, then sweep_enqueue once per sweep and stage (asynchronous), then sweeps_finish (synchronise, timers).
// z_out / z16_out != nullptr: the topic indicators of the last sweep are copied to the host on the copy stream as
// soon as its z-step has finished, under the count exchange and the Phi draw (the Java shim copies z back into
// the documents' LabelSequences after every sample() call, INTEGRATION.md section 2)
struct SweepCall {
    int32_t n = 0, ran = 0;
    bool with_phi = true, z_copied = false;
    int32_t *z_out = nullptr;
    uint16_t *z16_out = nullptr;
};

int sweeps_prepare(ldagpu_handle h, SweepCall &c)
{
    h->last_zk_ms = 0; h->last_call_ms = 0; h->last_zk_launches = 0; h->last_launches = 0;
    c.ran = 0; c.z_copied = false;
    if (c.z16_out && ensure_z16(h)) return 1;
    if (c.n <= 0) return 0;
    return ensure_events(h, (size_t)c.n * EV_PER_SWEEP);
}

// one stage of the next sweep (see "Stages" above); ST_REDUCE and ST_BARRIER only run in z-only sweeps, where no fused
// Phi draw sums the counts
int sweep_enqueue(ldagpu_handle h, SweepCall &c, Stage stage)
{
    const int32_t s = c.ran;
    cudaEvent_t *ev = h->events.data() + (size_t)s * EV_PER_SWEEP;
    if (stage == ST_LOCAL) {
        h->iteration += 1;
        CK(h, cudaEventRecord(ev[0], h->stream));
        // the count rebuild is fused into the z kernel: zero n_wk first (Phi, not n_wk, feeds the z-step)
        CK(h, cudaMemsetAsync(h->n_wk.p, 0, sizeof(int32_t) * h->n_wk.n, h->stream));
        // GGS draws theta inside the z kernel for the documents that are one work item, and in the stand-alone
        // kernel beforehand for the documents split into several
        const bool fuse_theta = h->scheme == LDAGPU_SCHEME_GGS;
        if (fuse_theta && step_theta(h, /*only_long=*/true)) return 1;
        CK(h, cudaEventRecord(ev[1], h->stream));
        const bool stream_out = (c.z_out || c.z16_out) && s == c.n - 1 && h->scheme == LDAGPU_SCHEME_GGS && h->z_parts.size() > 1;
        if (stream_out) {
            // the z-step in document-aligned parts: as soon as a part's indicators are final they are narrowed (16-bit
            // transport) and copied to the host on the copy stream, under the z-step of the following parts
            for (size_t p = 0; p < h->z_parts.size(); ++p) {
                const auto &zp = h->z_parts[p];
                if (step_z(h, true, fuse_theta, (int)p)) return 1;
                CK(h, cudaEventRecord(h->copy_events[1 + p], h->stream));
                CK(h, cudaStreamWaitEvent(h->copy_stream, h->copy_events[1 + p], 0));
                if (copy_z_out(h, c.z_out, c.z16_out, zp.tok0, zp.tok1 - zp.tok0, h->copy_stream)) return 1;
                h->last_launches += c.z16_out ? 1 : 0;
            }
            c.z_copied = true;
        } else if (step_z(h, true, fuse_theta)) return 1;
        CK(h, cudaEventRecord(ev[2], h->stream));
        if (!stream_out && (c.z_out || c.z16_out) && s == c.n - 1 && h->dm.N) {
            CK(h, cudaEventRecord(h->copy_events[0], h->stream));
            CK(h, cudaStreamWaitEvent(h->copy_stream, h->copy_events[0], 0));
            // 16-bit transport: narrowed on the device (copy stream, under the Phi draw), half the PCIe bytes
            if (copy_z_out(h, c.z_out, c.z16_out, 0, h->dm.N, h->copy_stream)) return 1;
            h->last_launches += c.z16_out ? 1 : 0;
            c.z_copied = true;
        }
        CK(h, launch_topic_totals(h->dm, h->n_wk.p, h->n_k.p, h->stream));
        h->last_launches += 1;
        CK(h, cudaEventRecord(ev[3], h->stream));
    }
    if (step_counts_exchange(h, c.with_phi, stage)) return 1;
    if (stage == ST_BARRIER) CK(h, cudaEventRecord(ev[4], h->stream));
    if (c.with_phi) {
        const bool acc = mean_this_iteration(h);
        if (step_phi(h, acc, ev + 5, true, stage)) return 1;
        if (stage == ST_LAND && acc) h->n_sampled_phi += 1;   // GGS:168-170
    } else if (stage == ST_LAND) {
        for (int i = 5; i < EV_PER_SWEEP; ++i) CK(h, cudaEventRecord(ev[i], h->stream));
    }
    if (stage == ST_LAND) c.ran += 1;
    return 0;
}

int sweeps_finish(ldagpu_handle h, SweepCall &c)
{
    const int32_t ran = c.ran;
    // aborted before the last sweep: plain copy of the current z
    if (!c.z_copied && h->dm.N && (c.z_out || c.z16_out) && copy_z_out(h, c.z_out, c.z16_out, 0, h->dm.N, h->stream)) return 1;
    if (sync_check(h)) return 1;
    if (c.z_copied) CK(h, cudaStreamSynchronize(h->copy_stream));
    for (int32_t s = 0; s < ran; ++s) {
        cudaEvent_t *ev = h->events.data() + (size_t)s * EV_PER_SWEEP;
        float ms[EV_PER_SWEEP - 1];
        for (int i = 0; i + 1 < EV_PER_SWEEP; ++i) CK(h, cudaEventElapsedTime(&ms[i], ev[i], ev[i + 1]));
        if (getenv("LDAGPU_TRACE"))
            fprintf(stderr, "[ldagpu rank %d sweep %d] theta %.3f z %.3f totals %.3f exchange %.3f draw+seg %.3f seg-gather %.3f "
                            "normalise %.3f phi-gather/wait+alias %.3f ms\n", h->rank, h->iteration - ran + s + 1, ms[0], ms[1], ms[2],
                    ms[3], ms[4], ms[5], ms[6], ms[7]);
        h->t_z += ms[0] + ms[1];
        h->last_zk_ms += ms[1];
        h->t_counts += ms[2];
        // ms[7] = Phi all-gather + (sparse scheme) alias-table build: on one GPU it is all table build
        h->t_comm += ms[3] + ms[5] + (h->world > 1 ? ms[7] : 0.0f);
        if (h->world == 1) h->t_phi += ms[7];
        h->t_phi += ms[4] + ms[6];
    }
    if (ran > 0) {
        float total = 0.f;
        CK(h, cudaEventElapsedTime(&total, h->events[0], h->events[(size_t)(ran - 1) * EV_PER_SWEEP + EV_PER_SWEEP - 1]));
        h->last_call_ms = total;
    }
    return 0;
}

// n sweeps on every part: sweep s is enqueued on every part before sweep s + 1 on any (a shard's kernels wait, on the
// device, for the other shards' kernels of the same sweep).  z_out / z16_out are in corpus order.
int run_sweeps(ldagpu_handle h, int32_t n, bool with_phi, int32_t *done, int32_t *z_out, uint16_t *z16_out)
{
    if (done) *done = 0;
    const Parts parts = h->parts();
    std::vector<SweepCall> calls(parts.size());
    for (size_t g = 0; g < parts.size(); ++g) {
        SweepCall &c = calls[g];
        c.n = n; c.with_phi = with_phi;
        c.z_out = z_out ? z_out + h->shard_tok0[g] : nullptr;
        c.z16_out = z16_out ? z16_out + h->shard_tok0[g] : nullptr;
        MC(h, parts[g], sweeps_prepare(parts[g], c));
    }
    if (n > 0) {
        // one process per GPU: every rank must run the same number of sweeps, or the others would wait for this one in
        // the exchange -- the ranks agree on the abort flag in the rendezvous, once per call, and a call is short (the
        // host side caps the sweeps per call); otherwise the flag is looked at before every sweep and stops all shards
        // at the same one (UPL:645)
        int stop = 0;
        for (ldagpu_handle c : parts) {
            int s = 0;
            MC(h, c, rendezvous(c, &s));
            stop |= s;
        }
        // fault injection for the tests of the bounded waits: LDAGPU_FAULT_STALL_SHARD=g leaves the Phi stages of shard g
        // of a group out, as if its process had died -- the other shards must report a timeout instead of hanging
        static const int stall_env = getenv("LDAGPU_FAULT_STALL_SHARD") ? atoi(getenv("LDAGPU_FAULT_STALL_SHARD")) : -1;
        const int stall = h->multi() ? stall_env : -1;
        for (int32_t s = 0; s < n && !stop; ++s) {
            if (!h->comm && parts[0]->abort_flag.load(std::memory_order_relaxed)) break;
            if (run_stages(h, parts, [&](size_t g, Stage st) {
                    if ((int)g != stall || st < ST_DRAW) return sweep_enqueue(parts[g], calls[g], st);
                    if (st == ST_LAND) calls[g].ran += 1;
                    return 0;
                }))
                return 1;
        }
        for (size_t g = 0; g < parts.size(); ++g) MC(h, parts[g], sweeps_finish(parts[g], calls[g]));
    }
    // the call's statistics: the slowest part sets the time, launches add up
    double call_ms = 0, zk_ms = 0;
    int64_t zk_launches = 0, launches = 0;
    for (ldagpu_handle c : parts) {
        call_ms = std::max(call_ms, c->last_call_ms);
        zk_ms = std::max(zk_ms, c->last_zk_ms);
        zk_launches = std::max(zk_launches, c->last_zk_launches);
        launches += c->last_launches;
    }
    h->last_call_ms = call_ms; h->last_zk_ms = zk_ms; h->last_zk_launches = zk_launches; h->last_launches = launches;
    if (done) *done = calls[0].ran;
    return 0;
}

int build_items(ldagpu_handle h)
{
    const std::vector<int64_t> &off = h->h_doc_off;
    const int64_t D = h->dm.D;
    std::vector<int32_t> item_doc;
    std::vector<int64_t> item_begin;
    if (h->scheme == LDAGPU_SCHEME_GGS) {
        // documents split freely into chunks: tokens are independent given theta (GGS:97-101).  Few long
        // documents (NIPS shape: 1 500 documents of ~1 300 tokens) would leave most resident warps with one
        // item and some with two; smaller chunks give every warp of the persistent grid ~8 items.
        const int64_t resident_warps = (int64_t)h->sm_count * 40;
        int64_t chunk = (h->dm.N / (8 * resident_warps) + 31) / 32 * 32;
        // a work item that is a whole document draws its theta inside the z kernel; documents longer than the cap
        // need the stand-alone theta pass first.  The cap grows with the corpus (the tail a long item can leave at
        // the end of the launch stays below ~1 % of it): 256 tokens up to ~10^8 tokens per GPU, 1024 beyond
        const int64_t cap = std::min<int64_t>(4 * GGS_CHUNK_MAX,
                                              std::max<int64_t>(GGS_CHUNK_MAX, h->dm.N / (64 * resident_warps) / 32 * 32));
        chunk = std::min<int64_t>(std::max<int64_t>(chunk, 32), cap);
        h->ggs_chunk = (int32_t)chunk;
        std::vector<int32_t> long_docs;
        for (int64_t d = 0; d < D; ++d) {
            if (off[d + 1] - off[d] > chunk) long_docs.push_back((int32_t)d);
            for (int64_t t = off[d]; t < off[d + 1]; t += chunk) {
                item_doc.push_back((int32_t)d);
                item_begin.push_back(t);
            }
        }
        // parts for the streamed read-back: 8 document-aligned ranges of about equal token counts
        h->z_parts.clear();
        if (h->dm.N >= (8 << 20)) {
            const int nparts = 8;
            size_t i0 = 0;
            for (int p = 0; p < nparts && i0 < item_doc.size(); ++p) {
                const int64_t target = h->dm.N / nparts * (p + 1);
                size_t i1 = i0;
                if (p == nparts - 1) i1 = item_doc.size();
                else {
                    while (i1 < item_doc.size() && item_begin[i1] < target) ++i1;
                    while (i1 < item_doc.size() && i1 > 0 && item_doc[i1] == item_doc[i1 - 1]) ++i1;   // never split a document
                }
                if (i1 > i0)
                    h->z_parts.push_back({(int64_t)i0, (int64_t)i1, item_begin[i0],
                                          i1 < item_doc.size() ? item_begin[i1] : h->dm.N});
                i0 = i1;
            }
        }
        h->n_long_docs = (int64_t)long_docs.size();
        CK(h, h->long_docs.alloc(std::max<size_t>(long_docs.size(), 1)));
        if (!long_docs.empty())
            CK(h, cudaMemcpy(h->long_docs.p, long_docs.data(), sizeof(int32_t) * long_docs.size(), cudaMemcpyHostToDevice));
    } else {
        // PCGS is sequential inside a document: one item per document, longest first
        item_doc.resize((size_t)D);
        std::iota(item_doc.begin(), item_doc.end(), 0);
        std::stable_sort(item_doc.begin(), item_doc.end(), [&](int32_t a, int32_t b) {
            return off[a + 1] - off[a] > off[b + 1] - off[b];
        });
        item_begin.assign(1, 0);
    }
    h->n_items = (int64_t)item_doc.size();
    CK(h, h->item_doc.alloc(std::max<size_t>(item_doc.size(), 1)));
    CK(h, h->item_begin.alloc(std::max<size_t>(item_begin.size(), 1)));
    if (!item_doc.empty())
        CK(h, cudaMemcpy(h->item_doc.p, item_doc.data(), sizeof(int32_t) * item_doc.size(), cudaMemcpyHostToDevice));
    if (!item_begin.empty())
        CK(h, cudaMemcpy(h->item_begin.p, item_begin.data(), sizeof(int64_t) * item_begin.size(), cudaMemcpyHostToDevice));
    return 0;
}

// Peer-memory exchange: map every other rank's n_wk / Phi^T / segment sums / n_k parts / flags with
// CUDA IPC (handles travel through one NCCL all-gather).  All ranks agree on the outcome; when a mapping
// fails (no peer access, IPC disabled) or LDAGPU_EXCHANGE=nccl, the NCCL collectives stay in charge.
struct IpcBlob {
    cudaIpcMemHandle_t n_wk, phiT, seg, nk_parts, flags;
};

void close_peer_exchange(ldagpu_handle h)
{
    for (void *p : h->ipc_opened) cudaIpcCloseMemHandle(p);
    h->ipc_opened.clear();
    h->p2p = false;
}

// rank `rank` of `world` owns the vocabulary rows [row0, row1) and the Phi segments [seg0, seg1)
void set_rank(ldagpu_handle h, int rank, int world)
{
    h->rank = rank;
    h->world = world;
    const int32_t rows = h->dm.Vp / world;
    h->row0 = rank * rows;
    h->row1 = h->row0 + rows;
    h->seg0 = rank * (PHI_SEGMENTS / world);
    h->seg1 = h->seg0 + PHI_SEGMENTS / world;
}

// what the peer-memory exchange needs besides the peers' pointers: the zeroed n_k parts and flag buffers and the
// PeerTable's own fields
int init_peer_table(ldagpu_handle h)
{
    CK(h, h->nk_parts.alloc((size_t)P2P_MAX * h->dm.Ks));
    CK(h, h->p2p_flags.alloc((size_t)P2P_FLAG_KINDS * P2P_MAX));
    CK(h, h->p2p_local.alloc((size_t)P2P_FLAG_KINDS + 4));
    CK(h, cudaMemset(h->nk_parts.p, 0, sizeof(int32_t) * h->nk_parts.n));
    CK(h, cudaMemset(h->p2p_flags.p, 0, sizeof(uint32_t) * h->p2p_flags.n));
    CK(h, cudaMemset(h->p2p_local.p, 0, sizeof(uint32_t) * h->p2p_local.n));
    PeerTable &pt = h->pt;
    pt = PeerTable{};
    pt.rank = h->rank; pt.world = h->world;
    pt.done_ctr = h->p2p_local.p;
    pt.error = reinterpret_cast<int *>(h->p2p_local.p + P2P_FLAG_KINDS);
    const char *to = getenv("LDAGPU_P2P_TIMEOUT_MS");
    pt.timeout_ns = (unsigned long long)(to ? std::max(1L, atol(to)) : 60000L) * 1000000ull;
    return 0;
}

int setup_peer_exchange(ldagpu_handle h)
{
    const char *mode = getenv("LDAGPU_EXCHANGE");
    const bool want = !(mode && std::strcmp(mode, "nccl") == 0);
    const int G = h->world;
    if (init_peer_table(h)) return 1;

    int ok = want && G <= P2P_MAX ? 1 : 0;
    if (!want) h->p2p_note = "LDAGPU_EXCHANGE=nccl";
    IpcBlob mine{};
    if (ok) {
        cudaError_t e = cudaIpcGetMemHandle(&mine.n_wk, h->n_wk.p);
        if (e == cudaSuccess) e = cudaIpcGetMemHandle(&mine.phiT, h->phiT.p);
        if (e == cudaSuccess) e = cudaIpcGetMemHandle(&mine.seg, h->seg.p);
        if (e == cudaSuccess) e = cudaIpcGetMemHandle(&mine.nk_parts, h->nk_parts.p);
        if (e == cudaSuccess) e = cudaIpcGetMemHandle(&mine.flags, h->p2p_flags.p);
        if (e != cudaSuccess) { ok = 0; h->p2p_note = std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e); cudaGetLastError(); }
    }
    // all-gather the handles (as bytes) and every rank's device ordinal
    DevBuf<unsigned char> blobs;
    CK(h, blobs.alloc(sizeof(IpcBlob) * (size_t)G));
    CK(h, cudaMemcpyAsync(blobs.p + sizeof(IpcBlob) * (size_t)h->rank, &mine, sizeof mine, cudaMemcpyHostToDevice, h->stream));
    NK(h, g_nccl.AllGather(blobs.p + sizeof(IpcBlob) * (size_t)h->rank, blobs.p, sizeof(IpcBlob), ncclChar, h->comm, h->stream));
    std::vector<IpcBlob> all((size_t)G);
    CK(h, cudaMemcpyAsync(all.data(), blobs.p, sizeof(IpcBlob) * (size_t)G, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));

    PeerTable &pt = h->pt;
    if (ok) {
        for (int r = 0; r < G && ok; ++r) {
            if (r == h->rank) {
                pt.n_wk[r] = h->n_wk.p; pt.phiT[r] = h->phiT.p; pt.seg[r] = h->seg.p;
                pt.nk_parts[r] = h->nk_parts.p; pt.flags[r] = h->p2p_flags.p;
                continue;
            }
            auto open = [&](const cudaIpcMemHandle_t &mh, void **out) {
                cudaError_t e = cudaIpcOpenMemHandle(out, mh, cudaIpcMemLazyEnablePeerAccess);
                if (e != cudaSuccess) {
                    ok = 0;
                    h->p2p_note = std::string("cudaIpcOpenMemHandle (rank ") + std::to_string(r) + "): " + cudaGetErrorString(e);
                    cudaGetLastError();
                    return;
                }
                h->ipc_opened.push_back(*out);
            };
            open(all[(size_t)r].n_wk, reinterpret_cast<void **>(&pt.n_wk[r]));
            if (ok) open(all[(size_t)r].phiT, reinterpret_cast<void **>(&pt.phiT[r]));
            if (ok) open(all[(size_t)r].seg, reinterpret_cast<void **>(&pt.seg[r]));
            if (ok) open(all[(size_t)r].nk_parts, reinterpret_cast<void **>(&pt.nk_parts[r]));
            if (ok) open(all[(size_t)r].flags, reinterpret_cast<void **>(&pt.flags[r]));
        }
    }
    // every rank must take the same path
    DevBuf<int> agree;
    CK(h, agree.alloc(1));
    CK(h, cudaMemcpyAsync(agree.p, &ok, sizeof ok, cudaMemcpyHostToDevice, h->stream));
    NK(h, g_nccl.AllReduce(agree.p, agree.p, 1, ncclInt32, ncclMin, h->comm, h->stream));
    int all_ok = 0;
    CK(h, cudaMemcpyAsync(&all_ok, agree.p, sizeof all_ok, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    if (!all_ok) {
        if (ok) h->p2p_note = "another rank could not map peer memory";
        close_peer_exchange(h);
        if (want && getenv("LDAGPU_EXCHANGE") && std::strcmp(getenv("LDAGPU_EXCHANGE"), "p2p") == 0)
            return h->fail("LDAGPU_EXCHANGE=p2p but peer memory is unavailable: %s", h->p2p_note.c_str());
        return 0;
    }
    h->p2p = true;
    return 0;
}

double lgamma_stirling_host(double z)
{
    int shift = 0;
    while (z < 2) { z++; shift++; }
    double r = 0.5 * std::log(2 * M_PI) + (z - 0.5) * std::log(z) - z + 1 / (12 * z) - 1 / (360 * z * z * z) +
               1 / (1260 * z * z * z * z * z);
    while (shift > 0) { shift--; z--; r -= std::log(z); }
    return r;
}

// alpha (validated by the caller) into the handle: the host copy and its sum (sequential, as MSL:139-143), the float and
// double device copies and the lgS(alpha_k) table
int upload_alpha(ldagpu_handle h, const double *alpha)
{
    const int K = h->dm.K;
    h->alpha.assign(alpha, alpha + K);
    h->alpha_sum = 0.0;
    for (int k = 0; k < K; ++k) h->alpha_sum += alpha[k];
    std::vector<float> af((size_t)h->dm.Ks, 0.0f);
    std::vector<double> ad((size_t)h->dm.Ks, 0.0);
    for (int k = 0; k < K; ++k) { af[(size_t)k] = (float)alpha[k]; ad[(size_t)k] = alpha[k]; }
    CK(h, cudaMemcpyAsync(h->alpha_f.p, af.data(), sizeof(float) * af.size(), cudaMemcpyHostToDevice, h->stream));
    CK(h, cudaMemcpyAsync(h->alpha_d.p, ad.data(), sizeof(double) * ad.size(), cudaMemcpyHostToDevice, h->stream));
    CK(h, launch_lgs_table(K, h->alpha_d.p, h->lgs_alpha.p, h->stream));
    return 0;
}

// An accessor that converts between the device layout and the host's [K][V] / [D][K] layout: the conversion kernel
// (`launch`, given the scratch buffer) writes or reads `cells` values in host layout in a scratch buffer, which is
// copied to `out` after it or from `in` before it.
template <typename T, typename F>
int via_scratch(ldagpu_handle h, DevBuf<T> &scratch, size_t cells, std::common_type_t<T> *out, const std::common_type_t<T> *in,
                F &&launch)
{
    CK(h, scratch.alloc(cells));
    if (in) CK(h, cudaMemcpyAsync(scratch.p, in, sizeof(T) * cells, cudaMemcpyHostToDevice, h->stream));
    if (launch(scratch.p)) return 1;
    if (out) CK(h, cudaMemcpyAsync(out, scratch.p, sizeof(T) * cells, cudaMemcpyDeviceToHost, h->stream));
    int rc = sync_check(h);
    scratch.release();
    return rc;
}

// Every rank, and every shard of a group, holds the global values of its own vocabulary rows only (n_wk after the
// exchange, the Phi-mean sums): collect all rows on parts[0], which exports them.  Ranks all-gather them with NCCL,
// the shards of a group copy theirs to shard 0 over peer access.
template <typename T>
int gather_rows(ldagpu_handle h, const Parts &parts, DevBuf<T> ldagpu_handle_s::*buf, ncclDataType_t type)
{
    if (h->world > 1 && h->comm) {
        const size_t slice = (size_t)(h->dm.Vp / h->world) * h->dm.Ks;
        T *p = (h->*buf).p;
        NK(h, g_nccl.AllGather(p + (size_t)h->rank * slice, p, slice, type, h->comm, h->stream));
        return 0;
    }
    ldagpu_handle c0 = parts[0];
    for (size_t g = 1; g < parts.size(); ++g) {
        ldagpu_handle c = parts[g];
        if (!(c->*buf).p || !(c0->*buf).p) continue;
        const size_t o = (size_t)c->row0 * c->dm.Ks, cnt = (size_t)(c->row1 - c->row0) * c->dm.Ks;
        cudaSetDevice(c->device);
        CK(h, cudaMemcpyPeerAsync((c0->*buf).p + o, c0->device, (c->*buf).p + o, c->device, sizeof(T) * cnt, c->stream));
        CK(h, cudaStreamSynchronize(c->stream));
    }
    return 0;
}

// counts from the resident z on every part, exchanged; redraw_phi: then Phi from them (UPL:450, 1842)
int refresh_counts_and_phi(ldagpu_handle h, bool redraw_phi)
{
    const Parts parts = h->parts();
    if (run_stages(h, parts, [&](size_t g, Stage st) {
            ldagpu_handle c = parts[g];
            if (st == ST_LOCAL && (rendezvous(c) || step_counts_local(c))) return 1;
            return step_counts_exchange(c, redraw_phi, st) || (redraw_phi && step_phi(c, false, nullptr, true, st)) ? 1 : 0;
        }))
        return 1;
    return sync_all(h, parts);
}

// what is wrong with the CSR offsets of D documents (appended to the array's name), or nullptr
const char *csr_offsets_error(const int64_t *off, int64_t D)
{
    if (off[0] != 0) return "[0] must be 0";
    for (int64_t d = 0; d < D; ++d)
        if (off[d + 1] < off[d]) return " must be non-decreasing";
    return nullptr;
}

// The shard rule of a group, for its training set and its test set: documents [0, D) with offsets `off` split by token
// count into `parts` contiguous ranges; part g holds documents [d0[g], d0[g + 1]) and tokens [t0[g], t0[g + 1])
void shard_bounds_by_tokens(const int64_t *off, int64_t D, int parts, std::vector<int64_t> &d0, std::vector<int64_t> &t0)
{
    d0.assign((size_t)parts + 1, D);
    d0[0] = 0;
    const int64_t N = off[D];
    for (int g = 1; g < parts; ++g) {
        const int64_t target = N / parts * g;
        int64_t d = std::lower_bound(off, off + D + 1, target) - off;
        d0[(size_t)g] = std::min<int64_t>(std::max<int64_t>(d, d0[(size_t)g - 1]), D);
    }
    t0.resize(d0.size());
    for (size_t g = 0; g < d0.size(); ++g) t0[g] = off[d0[g]];
}

// documents [d0, d1) of `off` as a part's own offsets: off[d0..d1] - off[d0]
std::vector<int64_t> local_offsets(const int64_t *off, int64_t d0, int64_t d1)
{
    std::vector<int64_t> loc((size_t)(d1 - d0) + 1);
    for (int64_t d = d0; d <= d1; ++d) loc[(size_t)(d - d0)] = off[d] - off[d0];
    return loc;
}

// held-out evaluation runs the register path's draw only
int heldout_refuses_k(ldagpu_handle h)
{
    if (h->dm.K <= MAX_REG_TILES * TILE) return 0;
    return h->fail("held-out evaluation is limited to K <= %d topics (the dense left-to-right estimator); K = %d",
                   MAX_REG_TILES * TILE, h->dm.K);
}

}  // namespace

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

const char *ldagpu_version(void) { return "libldagpu 0.4 (sm_100a; GGS with fused theta, PCGS, sparse PCGS; peer-memory exchange; single-process multi-GPU)"; }

const char *ldagpu_last_error(ldagpu_handle h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int ldagpu_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int ldagpu_create(int32_t K, int32_t V, int64_t D, const int64_t *doc_offsets, const int32_t *tokens,
                  const double *alpha, double beta, uint64_t seed, int32_t scheme, int32_t device,
                  int64_t doc_base, int64_t token_base, ldagpu_handle *out)
{
    if (out) *out = nullptr;
    auto bail = [&](const std::string &m) { g_create_error = m; return 1; };
    if (!out || !doc_offsets || (!tokens && D > 0 && doc_offsets[D] > 0) || !alpha) return bail("null argument");
    if (K < 1 || V < 1 || D < 0) return bail("K, V must be >= 1 and D >= 0");
    if (scheme != LDAGPU_SCHEME_GGS && scheme != LDAGPU_SCHEME_PCGS && scheme != LDAGPU_SCHEME_SPALIAS)
        return bail("unknown scheme");
    if (scheme != LDAGPU_SCHEME_SPALIAS && K > max_dense_topics(scheme == LDAGPU_SCHEME_PCGS))
        return bail("K is too large for the dense z-step (one Phi row + one document vector per warp in shared memory)");
    if (scheme == LDAGPU_SCHEME_SPALIAS && K > (1 << 20)) return bail("K is too large");
    if (!(beta > 0.0)) return bail("beta must be > 0");   // ParallelRandoms.java:61-63
    for (int k = 0; k < K; ++k)
        if (!(alpha[k] > 0.0)) return bail("alpha must be > 0");
    if (const char *e = csr_offsets_error(doc_offsets, D)) return bail(std::string("doc_offsets") + e);
    int ndev = ldagpu_device_count();
    if (ndev == 0) return bail("no CUDA device: libldagpu has no CPU fallback");
    if (device < 0 || device >= ndev) return bail("device ordinal out of range");

    ldagpu_handle h = new ldagpu_handle_s();
    auto fail_out = [&]() { g_create_error = h->err; ldagpu_destroy(h); return 1; };
    h->device = device;
    h->scheme = scheme;
    h->beta = beta;
    h->seed = seed;
    Dims &dm = h->dm;
    dm.K = K; dm.Ks = (int32_t)round_up(K, 32); dm.NT = (K + TILE - 1) / TILE; dm.lg = 2;
    if (scheme != LDAGPU_SCHEME_SPALIAS && K <= MAX_REG_TILES * TILE) {
        // register path of the dense z-step: 1, 2, 4 or 8 tiles, lane l owns 4 * NT consecutive topics and the
        // rows of Phi^T / n_wk / theta are stored in the matching column order (common.cuh: tpos / ttopic)
        dm = reg_path_dims(dm);
    }
    dm.V = V; dm.Vp = (int32_t)round_up(V, PHI_ROW_BLOCK * PHI_SEGMENTS);
    dm.D = D; dm.N = doc_offsets[D]; dm.doc_base = doc_base; dm.token_base = token_base;
    h->D_global = D;
    set_rank(h, 0, 1);
    h->shard_doc0 = {0, D};
    h->shard_tok0 = {0, dm.N};
    h->h_doc_off.assign(doc_offsets, doc_offsets + D + 1);

    auto body = [&]() -> int {
        CK(h, cudaSetDevice(device));
        cudaDeviceProp prop;
        CK(h, cudaGetDeviceProperties(&prop, device));
        h->sm_count = prop.multiProcessorCount;
        CK(h, cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
        CK(h, cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
        for (int i = 0; i < 10; ++i) {
            cudaEvent_t e;
            CK(h, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            h->copy_events.push_back(e);
        }
        const size_t N1 = (size_t)std::max<int64_t>(dm.N, 1);
        CK(h, h->doc_off.alloc((size_t)D + 1));
        CK(h, h->tokens.alloc(N1 + 4));
        CK(h, h->z.alloc(N1 + 4));
        CK(h, h->phiT.alloc((size_t)dm.Vp * dm.Ks));
        CK(h, h->n_wk.alloc((size_t)dm.Vp * dm.Ks));
        CK(h, h->n_k.alloc((size_t)dm.Ks));
        CK(h, h->alpha_f.alloc((size_t)dm.Ks));
        CK(h, h->alpha_d.alloc((size_t)dm.Ks));
        CK(h, h->lgs_alpha.alloc((size_t)dm.Ks));
        CK(h, h->partial.alloc((size_t)(dm.Vp / PHI_ROW_BLOCK) * dm.Ks));
        CK(h, h->seg.alloc((size_t)PHI_SEGMENTS * dm.Ks));
        CK(h, h->topic_sum.alloc((size_t)dm.Ks));
        CK(h, h->red.alloc((size_t)N_PARTIALS * 2));
        CK(h, h->red_out.alloc(8));
        CK(h, h->counter.alloc(16));
        CK(h, h->bad.alloc(1));
        for (int64_t d = 0; d < D; ++d)
            h->max_doc_len = (int)std::max<int64_t>(h->max_doc_len, doc_offsets[d + 1] - doc_offsets[d]);
        if (scheme == LDAGPU_SCHEME_SPALIAS) {
            CK(h, h->alias_table.alloc((size_t)dm.Vp * dm.Ks));
            CK(h, h->type_norm.alloc((size_t)dm.Vp));
            h->alias_slots = alias_scratch_threads(dm, h->sm_count);
            CK(h, h->alias_bs.alloc(alias_value_doubles(dm, h->alias_slots)));
            CK(h, h->alias_stack.alloc(alias_stack_ints(dm, h->alias_slots)));
            CK(h, h->sparse_lists.alloc(spalias_list_bytes(dm, h->max_doc_len, h->sm_count) / sizeof(int32_t)));
            // only the types that occur in this rank's tokens are ever looked up
            std::vector<char> seen((size_t)V, 0);
            for (int64_t i = 0; i < dm.N; ++i)
                if (tokens[i] >= 0 && tokens[i] < V) seen[(size_t)tokens[i]] = 1;
            std::vector<int32_t> act;
            for (int32_t w = 0; w < V; ++w)
                if (seen[(size_t)w]) act.push_back(w);
            h->n_active_types = (int32_t)act.size();
            CK(h, h->active_types.alloc(std::max<size_t>(act.size(), 1)));
            if (!act.empty())
                CK(h, cudaMemcpy(h->active_types.p, act.data(), sizeof(int32_t) * act.size(), cudaMemcpyHostToDevice));
            CK(h, cudaMemset(h->alias_table.p, 0, sizeof(AliasSlot) * h->alias_table.n));
            CK(h, cudaMemset(h->type_norm.p, 0, sizeof(float) * h->type_norm.n));
        }
        CK(h, cudaMemcpy(h->doc_off.p, doc_offsets, sizeof(int64_t) * ((size_t)D + 1), cudaMemcpyHostToDevice));
        CK(h, cudaMemset(h->tokens.p, 0, sizeof(int32_t) * h->tokens.n));
        CK(h, cudaMemset(h->z.p, 0, sizeof(int32_t) * h->z.n));
        if (dm.N) CK(h, cudaMemcpy(h->tokens.p, tokens, sizeof(int32_t) * (size_t)dm.N, cudaMemcpyHostToDevice));
        CK(h, cudaMemset(h->phiT.p, 0, sizeof(float) * h->phiT.n));
        CK(h, cudaMemset(h->n_wk.p, 0, sizeof(int32_t) * h->n_wk.n));
        CK(h, cudaMemset(h->n_k.p, 0, sizeof(int32_t) * h->n_k.n));
        CK(h, cudaMemset(h->partial.p, 0, sizeof(double) * h->partial.n));
        CK(h, cudaMemset(h->seg.p, 0, sizeof(double) * h->seg.n));
        if (upload_alpha(h, alpha)) return 1;
        // type ids must be inside the alphabet (UPL:360 numTypes = alphabet.size())
        CK(h, launch_validate(dm, h->tokens.p, nullptr, h->bad.p, h->stream));
        int bad = 0;
        CK(h, cudaMemcpyAsync(&bad, h->bad.p, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CK(h, cudaStreamSynchronize(h->stream));
        if (bad) return h->fail("token type id out of range [0, %d)", V);
        if (build_items(h)) return 1;
        if (scheme == LDAGPU_SCHEME_GGS && ensure_theta(h)) return 1;
        return sync_check(h);
    };
    if (body()) return fail_out();
    *out = h;
    return 0;
}

int ldagpu_destroy(ldagpu_handle h)
{
    if (!h) return 0;
    for (ldagpu_handle c : h->shards) ldagpu_destroy(c);   // a group's own buffers are all empty
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    for (void *p : h->ipc_opened) cudaIpcCloseMemHandle(p);
    h->ipc_opened.clear();
    if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
    for (cudaEvent_t e : h->events) cudaEventDestroy(e);
    for (cudaEvent_t e : h->copy_events) cudaEventDestroy(e);
    if (h->copy_stream) { cudaStreamSynchronize(h->copy_stream); cudaStreamDestroy(h->copy_stream); }
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;   // its device buffers, with its device current
    return 0;
}

int ldagpu_comm_unique_id(void *id128)
{
    if (!id128) return 1;
    if (!g_nccl.load()) { g_create_error = g_nccl.err; return 1; }
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    ncclUniqueId id;
    if (g_nccl.GetUniqueId(&id) != ncclSuccess) { g_create_error = "ncclGetUniqueId failed"; return 1; }
    std::memcpy(id128, &id, sizeof id);
    return 0;
}

int ldagpu_comm_init(ldagpu_handle h, int32_t rank, int32_t world, const void *id128)
{
    NEED(h);
    if (world < 1 || rank < 0 || rank >= world) return h->fail("bad rank/world");
    if (world == 1) return 0;
    if (PHI_SEGMENTS % world != 0) return h->fail("world size must divide %d", PHI_SEGMENTS);
    if (!g_nccl.load()) return h->fail("%s", g_nccl.err.c_str());
    ncclUniqueId id;
    std::memcpy(&id, id128, sizeof id);
    NK(h, g_nccl.CommInitRank(&h->comm, world, id, rank));
    set_rank(h, rank, world);
    // global document count for the D * lgS(alphaSum) term of the log-likelihood
    DevBuf<long long> tmp;
    CK(h, tmp.alloc(1));
    long long d = h->dm.D;
    CK(h, cudaMemcpyAsync(tmp.p, &d, sizeof d, cudaMemcpyHostToDevice, h->stream));
    NK(h, g_nccl.AllReduce(tmp.p, tmp.p, 1, ncclInt64, ncclSum, h->comm, h->stream));
    CK(h, cudaMemcpyAsync(&d, tmp.p, sizeof d, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    h->D_global = d;
    return setup_peer_exchange(h);
}

int ldagpu_get_exchange_mode(ldagpu_handle h, int32_t *mode)
{
    if (!h || !mode) return 1;
    if (h->multi()) { *mode = 2; return 0; }
    *mode = h->world == 1 ? 0 : (h->p2p ? 2 : 1);
    return 0;
}

int ldagpu_init_z_java_random(ldagpu_handle h, int32_t seed)
{
    NEED(h);
    // java.util.Random(seed).nextInt(K) is one stream over the whole corpus in document order (UPL:398-406,458-460):
    // skip the draws of the ranks before this one, then every part takes its slice
    const Parts parts = h->parts();
    JavaRandom r((int64_t)seed);
    for (int64_t i = 0; i < parts[0]->dm.token_base; ++i) (void)r.nextInt(h->dm.K);
    std::vector<int32_t> z;
    for (ldagpu_handle c : parts) {
        z.resize((size_t)c->dm.N);
        for (int64_t i = 0; i < c->dm.N; ++i) z[(size_t)i] = r.nextInt(c->dm.K);
        CK(h, cudaSetDevice(c->device));
        if (c->dm.N) CK(h, cudaMemcpyAsync(c->z.p, z.data(), sizeof(int32_t) * z.size(), cudaMemcpyHostToDevice, c->stream));
        CK(h, cudaStreamSynchronize(c->stream));
    }
    return refresh_counts_and_phi(h, true);   // initialSamplePhi, UPL:450
}

// setZIndicators: the upload and the count rebuild are pipelined chunk by chunk -- the copy stream brings z in,
// the main stream checks the range and accumulates n_wk for the chunk that has landed (UPL:1797-1830 rebuilds
// while it copies too).  The new indicators land in a STAGING buffer and only replace the resident z once every
// one of them is inside [0, K): on an out-of-range indicator the reference throws and keeps its state
// (UPL:475-481), so do we -- the counts are rebuilt from the untouched z and the call fails.
// is16: the host buffer holds uint16 (half the PCIe bytes); it is widened on the device.
// Two pieces, so that one caller thread can drive several shards: set_z_upload enqueues the upload and the counts,
// set_z_commit (once the range flags of ALL shards are known) commits or restores and enqueues the exchange.
static int set_z_upload(ldagpu_handle h, const void *z, bool is16)
{
    const int64_t N = h->dm.N;
    if (!h->z_stage.p) {
        CK(h, h->z_stage.alloc((size_t)std::max<int64_t>(N, 1) + 4));
        CK(h, cudaMemsetAsync(h->z_stage.p, 0, sizeof(int32_t) * h->z_stage.n, h->stream));
    }
    if (is16 && ensure_z16(h)) return 1;
    CK(h, cudaMemsetAsync(h->n_wk.p, 0, sizeof(int32_t) * h->n_wk.n, h->stream));
    CK(h, cudaMemsetAsync(h->bad.p, 0, sizeof(int), h->stream));
    CK(h, cudaEventRecord(h->copy_events[0], h->stream));
    CK(h, cudaStreamWaitEvent(h->copy_stream, h->copy_events[0], 0));   // earlier users of the staging buffers are done
    const int nchunk = N >= (8 << 20) ? 8 : 1;
    const int64_t per = ((N + nchunk - 1) / nchunk + 7) / 8 * 8;        // vector loads: chunks start on 16-byte boundaries
    const size_t esz = is16 ? sizeof(uint16_t) : sizeof(int32_t);
    for (int c = 0; c < nchunk; ++c) {
        const int64_t o = (int64_t)c * per, cnt = std::min<int64_t>(per, N - o);
        if (cnt <= 0) break;
        void *dst = is16 ? static_cast<void *>(h->z16.p + o) : static_cast<void *>(h->z_stage.p + o);
        CK(h, cudaMemcpyAsync(dst, static_cast<const char *>(z) + (size_t)o * esz, esz * (size_t)cnt, cudaMemcpyHostToDevice,
                              h->copy_stream));
        CK(h, cudaEventRecord(h->copy_events[1 + c], h->copy_stream));
        CK(h, cudaStreamWaitEvent(h->stream, h->copy_events[1 + c], 0));
        if (is16) {
            CK(h, launch_unpack16(h->z16.p + o, h->z_stage.p + o, cnt, h->sm_count, h->stream));
            h->last_launches += 1;
        }
        CK(h, launch_counts_chunk(h->dm, h->tokens.p + o, h->z_stage.p + o, cnt, h->n_wk.p, h->bad.p, h->sm_count, h->stream));
    }
    h->last_launches += nchunk;
    return 0;
}

// the range flag of this shard (synchronises the shard's stream)
static int set_z_read_flag(ldagpu_handle h, int *bad)
{
    // one process per GPU: every rank must take the same exit, or the others would wait for this one in the exchange
    if (h->world > 1 && h->comm) NK(h, g_nccl.AllReduce(h->bad.p, h->bad.p, 1, ncclInt32, ncclMax, h->comm, h->stream));
    CK(h, cudaMemcpyAsync(bad, h->bad.p, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    return 0;
}

// bad == 0: the staged indicators become the resident ones; otherwise the previous state is kept -- the counts are
// rebuilt from the untouched z and exchanged like any rebuild (Phi was never touched).  Enqueues only.
static int set_z_commit(ldagpu_handle h, int bad, int32_t redraw_phi, Stage stage)
{
    const bool defer = !bad && redraw_phi != 0;
    if (stage == ST_LOCAL) {
        if (rendezvous(h)) return 1;
        if (bad) {
            if (step_counts_local(h)) return 1;
        } else {
            std::swap(h->z.p, h->z_stage.p);   // both buffers have the same size
            CK(h, launch_topic_totals(h->dm, h->n_wk.p, h->n_k.p, h->stream));
            h->last_launches += 1;
        }
    }
    if (step_counts_exchange(h, defer, stage)) return 1;
    return defer && step_phi(h, false, nullptr, true, stage) ? 1 : 0;   // UPL:1842
}

// z in corpus order
static int set_z(ldagpu_handle h, const void *z, bool is16, int32_t redraw_phi)
{
    if (!z && h->dm.N) return h->fail("null z");
    if (is16 && h->dm.K > 65536) return h->fail("16-bit topic indicators need K <= 65536");
    const size_t esz = is16 ? sizeof(uint16_t) : sizeof(int32_t);
    const Parts parts = h->parts();
    for (size_t g = 0; g < parts.size(); ++g)
        MC(h, parts[g], set_z_upload(parts[g], static_cast<const char *>(z) + (size_t)h->shard_tok0[g] * esz, is16));
    int bad = 0;
    for (ldagpu_handle c : parts) {
        int b = 0;
        MC(h, c, set_z_read_flag(c, &b));
        bad |= b;
    }
    if (run_stages(h, parts, [&](size_t g, Stage st) { return set_z_commit(parts[g], bad, redraw_phi, st); })) return 1;
    if (sync_all(h, parts)) return 1;
    return bad ? h->fail("topic indicator out of range [0, %d)%s; the previous indicators stay in place", h->dm.K,   // UPL:475-481 throws
                         h->world > 1 ? " (on this or another shard)" : "")
               : 0;
}

int ldagpu_set_z(ldagpu_handle h, const int32_t *z, int32_t redraw_phi)
{
    NEED(h);
    return set_z(h, z, false, redraw_phi);
}

int ldagpu_set_z16(ldagpu_handle h, const uint16_t *z, int32_t redraw_phi)
{
    NEED(h);
    return set_z(h, z, true, redraw_phi);
}

// the resident z of one part to the host; z16: narrowed on the device
static int get_z_one(ldagpu_handle h, int32_t *z, uint16_t *z16)
{
    if (h->dm.N && ((z16 && ensure_z16(h)) || copy_z_out(h, z, z16, 0, h->dm.N, h->stream))) return 1;
    return sync_check(h);
}

// z in corpus order
static int get_z(ldagpu_handle h, int32_t *z, uint16_t *z16)
{
    const Parts parts = h->parts();
    for (size_t g = 0; g < parts.size(); ++g) {
        const int64_t t0 = h->shard_tok0[g];
        MC(h, parts[g], get_z_one(parts[g], z ? z + t0 : nullptr, z16 ? z16 + t0 : nullptr));
    }
    return 0;
}

int ldagpu_get_z16(ldagpu_handle h, uint16_t *z)
{
    NEED(h);
    if (h->dm.K > 65536) return h->fail("16-bit topic indicators need K <= 65536");
    return get_z(h, nullptr, z);
}

int ldagpu_get_z(ldagpu_handle h, int32_t *z)
{
    NEED(h);
    return get_z(h, z, nullptr);
}

int ldagpu_sweep_get_z16(ldagpu_handle h, int32_t n, int32_t *done, uint16_t *z)
{
    NEED(h);
    if (!z && h->dm.N) return h->fail("null z");
    if (h->dm.K > 65536) return h->fail("16-bit topic indicators need K <= 65536");
    return run_sweeps(h, n, true, done, nullptr, z);
}

int ldagpu_sweep_get_z(ldagpu_handle h, int32_t n, int32_t *done, int32_t *z)
{
    NEED(h);
    if (!z && h->dm.N) return h->fail("null z");
    return run_sweeps(h, n, true, done, z, nullptr);
}

int ldagpu_sweep(ldagpu_handle h, int32_t n, int32_t *done)
{
    NEED(h);
    return run_sweeps(h, n, true, done, nullptr, nullptr);
}

int ldagpu_sample_z_given_phi(ldagpu_handle h, int32_t n, int32_t *done)
{
    NEED(h);
    return run_sweeps(h, n, false, done, nullptr, nullptr);
}

// Settings live on the parts: the setters write every part, the getters read parts[0].
int ldagpu_next_iteration(ldagpu_handle h)
{
    NEED(h);
    for (ldagpu_handle c : h->parts()) c->iteration += 1;
    return 0;
}
int ldagpu_get_iteration(ldagpu_handle h, int32_t *it) { if (!h || !it) return 1; *it = h->parts()[0]->iteration; return 0; }
int ldagpu_set_iteration(ldagpu_handle h, int32_t it)
{
    if (!h) return 1;
    for (ldagpu_handle c : h->parts()) c->iteration = it;
    return 0;
}

int ldagpu_sample_theta(ldagpu_handle h)
{
    NEED(h);
    const Parts parts = h->parts();
    for (ldagpu_handle c : parts) MC(h, c, step_theta(c));
    return sync_all(h, parts);
}
int ldagpu_sample_z(ldagpu_handle h)
{
    NEED(h);
    const Parts parts = h->parts();
    for (ldagpu_handle c : parts) MC(h, c, step_z(c));
    return sync_all(h, parts);
}
int ldagpu_rebuild_counts(ldagpu_handle h)
{
    NEED(h);
    return refresh_counts_and_phi(h, false);
}
int ldagpu_sample_phi(ldagpu_handle h)
{
    NEED(h);
    const Parts parts = h->parts();
    if (run_stages(h, parts, [&](size_t g, Stage st) {
            ldagpu_handle c = parts[g];
            if (st == ST_LOCAL && rendezvous(c)) return 1;
            return step_phi(c, mean_this_iteration(c), nullptr, false, st);
        }))
        return 1;
    for (ldagpu_handle c : parts)
        if (mean_this_iteration(c)) c->n_sampled_phi += 1;
    return sync_all(h, parts);
}

int ldagpu_get_type_topic_counts(ldagpu_handle h, int32_t *out)
{
    NEED(h);
    const Parts parts = h->parts();
    if (gather_rows(h, parts, &ldagpu_handle_s::n_wk, ncclInt32)) return 1;
    ldagpu_handle c = parts[0];
    MC(h, c, via_scratch(c, c->scratch_i32, (size_t)c->dm.V * c->dm.K, out, nullptr,
                         [&](int32_t *s) { CK(c, launch_export_counts(c->dm, c->n_wk.p, s, c->stream)); return 0; }));
    return 0;
}

int ldagpu_get_topic_totals(ldagpu_handle h, int32_t *n_k)
{
    NEED(h);
    ldagpu_handle c = h->parts()[0];
    CK(h, cudaSetDevice(c->device));
    CK(h, cudaMemcpyAsync(n_k, c->n_k.p, sizeof(int32_t) * (size_t)c->dm.K, cudaMemcpyDeviceToHost, c->stream));
    MC(h, c, sync_check(c));
    return 0;
}

// per document, in corpus order
int ldagpu_get_doc_topic_counts(ldagpu_handle h, int32_t *n_dk)
{
    NEED(h);
    const Parts parts = h->parts();
    for (size_t g = 0; g < parts.size(); ++g) {
        ldagpu_handle c = parts[g];
        const size_t cells = (size_t)c->dm.D * c->dm.K;
        if (cells == 0) continue;
        MC(h, c, via_scratch(c, c->scratch_i32, cells, n_dk + (size_t)h->shard_doc0[g] * h->dm.K, nullptr,
                             [&](int32_t *s) { CK(c, launch_doc_topic_counts(c->dm, c->doc_off.p, c->z.p, s, c->stream)); return 0; }));
    }
    return 0;
}

int ldagpu_get_phi(ldagpu_handle h, double *phi)
{
    NEED(h);
    ldagpu_handle c = h->parts()[0];   // Phi is replicated
    MC(h, c, via_scratch(c, c->scratch_f64, (size_t)c->dm.V * c->dm.K, phi, nullptr,
                         [&](double *s) { CK(c, launch_export_phi(c->dm, c->phiT.p, s, c->stream)); return 0; }));
    return 0;
}

static int set_phi_one(ldagpu_handle h, const double *phi)
{
    int rc = via_scratch(h, h->scratch_f64, (size_t)h->dm.V * h->dm.K, nullptr, phi, [&](double *s) {
        CK(h, launch_import_phi(h->dm, s, h->phiT.p, h->stream));
        return step_alias(h);
    });
    // UPL:1897-1903: setPhi resets the running mean
    if (h->phi_mean.p) CK(h, cudaMemset(h->phi_mean.p, 0, sizeof(double) * h->phi_mean.n));
    h->n_sampled_phi = 0;
    return rc;
}

int ldagpu_set_phi(ldagpu_handle h, const double *phi)
{
    NEED(h);
    for (ldagpu_handle c : h->parts()) MC(h, c, set_phi_one(c, phi));
    return 0;
}

int ldagpu_set_phi_mean_schedule(ldagpu_handle h, int32_t burn_in, int32_t thin)
{
    if (!h) return 1;
    for (ldagpu_handle c : h->parts()) {
        c->mean_burn_in = burn_in;
        c->mean_thin = thin < 1 ? 1 : thin;
    }
    return 0;
}

int ldagpu_set_phi_sampler(ldagpu_handle h, int32_t sampler, int32_t alias_poisson_threshold)
{
    if (!h) return 1;
    if (sampler != LDAGPU_PHI_GAMMA && sampler != LDAGPU_PHI_POLYA_URN) return h->fail("unknown Phi sampler");
    if (sampler == LDAGPU_PHI_POLYA_URN && (alias_poisson_threshold < 1 || alias_poisson_threshold > (1 << 20)))
        return h->fail("alias_poisson_threshold must be in [1, 2^20]");
    for (ldagpu_handle c : h->parts()) c->poisson_L = sampler == LDAGPU_PHI_POLYA_URN ? alias_poisson_threshold : 0;
    return 0;
}

int ldagpu_get_phi_mean(ldagpu_handle h, double *phi_mean, int32_t *n_sampled)
{
    NEED(h);
    const Parts parts = h->parts();
    ldagpu_handle c = parts[0];
    if (n_sampled) *n_sampled = c->n_sampled_phi;
    if (c->n_sampled_phi == 0 || !c->phi_mean.p) return 0;   // UPL:1955-1958 returns null
    if (gather_rows(h, parts, &ldagpu_handle_s::phi_mean, ncclDouble)) return 1;
    MC(h, c, via_scratch(c, c->scratch_f64, (size_t)c->dm.V * c->dm.K, phi_mean, nullptr, [&](double *s) {
           CK(c, launch_export_mean(c->dm, c->phi_mean.p, 1.0 / (double)c->n_sampled_phi, s, c->stream));
           return 0;
       }));
    return 0;
}

// theta_out != nullptr: export theta, else import theta_in; both per document, in corpus order
static int theta_io(ldagpu_handle h, double *theta_out, const double *theta_in)
{
    const Parts parts = h->parts();
    for (size_t g = 0; g < parts.size(); ++g) {
        ldagpu_handle c = parts[g];
        MC(h, c, ensure_theta(c));
        const size_t cells = (size_t)c->dm.D * c->dm.K, o = (size_t)h->shard_doc0[g] * h->dm.K;
        if (cells == 0) continue;
        MC(h, c, via_scratch(c, c->scratch_f64, cells, theta_out ? theta_out + o : nullptr, theta_in ? theta_in + o : nullptr,
                             [&](double *s) {
                                 CK(c, theta_out ? launch_export_theta(c->dm, c->theta.p, s, c->stream)
                                                 : launch_import_theta(c->dm, s, c->theta.p, c->stream));
                                 return 0;
                             }));
    }
    return 0;
}

int ldagpu_get_theta(ldagpu_handle h, double *theta)
{
    NEED(h);
    return theta_io(h, theta, nullptr);
}

int ldagpu_set_theta(ldagpu_handle h, const double *theta)
{
    NEED(h);
    return theta_io(h, nullptr, theta);
}

// this part's three partial sums of the log-likelihood into red_out[0..2] (enqueue only): document part, type part
// over the part's vocabulary rows, and the number of non-zero cells there
static int ll_partials(ldagpu_handle h)
{
    CK(h, launch_ll_doc(h->dm, h->doc_off.p, h->z.p, h->alpha_d.p, h->lgs_alpha.p, h->alpha_sum, h->red.p, N_PARTIALS, h->sm_count,
                         h->stream));
    CK(h, launch_sum_partials(h->red.p, N_PARTIALS, 1, h->red_out.p, h->stream));
    CK(h, launch_ll_type(h->dm, h->n_wk.p, h->beta, h->row0, h->row1, h->red.p, N_PARTIALS, h->stream));
    CK(h, launch_sum_partials(h->red.p, N_PARTIALS, 2, h->red_out.p + 1, h->stream));
    return 0;
}

// UPL:1698,1724-1749: parameter-sum terms, added once
static double ll_finish(ldagpu_handle h, const double part[3], const std::vector<int32_t> &nk)
{
    const double bV = h->beta * h->dm.V;
    double v = part[0] + (double)h->D_global * lgamma_stirling_host(h->alpha_sum) + part[1];
    for (int k = 0; k < h->dm.K; ++k) v -= lgamma_stirling_host(bV + nk[(size_t)k]);
    v += lgamma_stirling_host(bV) * h->dm.K;
    v -= lgamma_stirling_host(h->beta) * part[2];
    if (std::isnan(v) || std::isinf(v)) v = 0.0;   // UPL:1730-1755 returns 0
    return v;
}

static int lp_partials(ldagpu_handle h)
{
    if (ensure_theta(h)) return 1;
    CK(h, launch_lp_tokens(h->dm, h->tokens.p, h->z.p, h->phiT.p, h->red.p, N_PARTIALS, h->stream));
    CK(h, launch_sum_partials(h->red.p, N_PARTIALS, 1, h->red_out.p, h->stream));
    CK(h, launch_lp_theta(h->dm, h->doc_off.p, h->z.p, h->theta.p, h->alpha_d.p, h->red.p, N_PARTIALS, h->sm_count, h->stream));
    CK(h, launch_sum_partials(h->red.p, N_PARTIALS, 1, h->red_out.p + 1, h->stream));
    CK(h, launch_lp_phi(h->dm, h->phiT.p, h->beta, h->row0, h->row1, h->red.p, N_PARTIALS, h->stream));
    CK(h, launch_sum_partials(h->red.p, N_PARTIALS, 1, h->red_out.p + 2, h->stream));
    return 0;
}

// the three partial sums of every part, combined: an NCCL all-reduce between the ranks, a host sum in fixed shard order
// (reproducible) over the shards of a group.  nk != nullptr: also n_k, from parts[0]
static int sum_partials(ldagpu_handle h, bool ll, double part[3], std::vector<int32_t> *nk)
{
    const Parts parts = h->parts();
    for (ldagpu_handle c : parts) MC(h, c, ll ? ll_partials(c) : lp_partials(c));
    if (h->world > 1 && h->comm) NK(h, g_nccl.AllReduce(h->red_out.p, h->red_out.p, 3, ncclDouble, ncclSum, h->comm, h->stream));
    part[0] = part[1] = part[2] = 0.0;
    for (ldagpu_handle c : parts) {
        double q[3];
        CK(h, cudaSetDevice(c->device));
        CK(h, cudaMemcpyAsync(q, c->red_out.p, sizeof q, cudaMemcpyDeviceToHost, c->stream));
        if (nk && c == parts[0])
            CK(h, cudaMemcpyAsync(nk->data(), c->n_k.p, sizeof(int32_t) * nk->size(), cudaMemcpyDeviceToHost, c->stream));
        MC(h, c, sync_check(c));
        part[0] += q[0]; part[1] += q[1]; part[2] += q[2];
    }
    return 0;
}

int ldagpu_log_likelihood(ldagpu_handle h, double *ll)
{
    NEED(h);
    double part[3];
    std::vector<int32_t> nk((size_t)h->dm.K);
    if (sum_partials(h, true, part, &nk)) return 1;
    *ll = ll_finish(h->parts()[0], part, nk);
    return 0;
}

int ldagpu_log_posterior(ldagpu_handle h, double *lp)
{
    NEED(h);
    double part[3];
    if (sum_partials(h, false, part, nullptr)) return 1;
    *lp = part[0] + part[1] + part[2];
    return 0;
}

int ldagpu_abort(ldagpu_handle h)
{
    if (!h) return 1;
    for (ldagpu_handle c : h->parts()) c->abort_flag.store(1);
    return 0;
}
int ldagpu_get_abort(ldagpu_handle h, int32_t *aborted)
{
    if (!h || !aborted) return 1;
    *aborted = h->parts()[0]->abort_flag.load();
    return 0;
}

// the slowest part sets the pace of every phase
int ldagpu_get_timers(ldagpu_handle h, double *z_ms, double *counts_ms, double *phi_ms, double *comm_ms)
{
    if (!h) return 1;
    double t[4] = {0, 0, 0, 0};
    for (ldagpu_handle c : h->parts()) {
        t[0] = std::max(t[0], c->t_z); t[1] = std::max(t[1], c->t_counts);
        t[2] = std::max(t[2], c->t_phi); t[3] = std::max(t[3], c->t_comm);
    }
    if (z_ms) *z_ms = t[0];
    if (counts_ms) *counts_ms = t[1];
    if (phi_ms) *phi_ms = t[2];
    if (comm_ms) *comm_ms = t[3];
    return 0;
}

int ldagpu_get_last_call_stats(ldagpu_handle h, double *call_ms, double *z_kernel_ms, int64_t *z_kernel_launches,
                               int64_t *total_launches)
{
    if (!h) return 1;
    if (call_ms) *call_ms = h->last_call_ms;
    if (z_kernel_ms) *z_kernel_ms = h->last_zk_ms;
    if (z_kernel_launches) *z_kernel_launches = h->last_zk_launches;
    if (total_launches) *total_launches = h->last_launches;
    return 0;
}

// =============================================================================================
// Single-process multi-GPU: ldagpu_create_multi.
// The reference drives everything from ONE coordinator thread of one JVM (tui/ParallelLDA.java:173-202,
// UPL:552-943); so does this layer: the handle it returns owns one shard handle per GPU, and every entry point fans
// out over them (ldagpu_handle_s::parts) and enqueues its work on all shards before it waits for any of them.  The exchange is the peer-memory one
// (kernels_p2p.cu, kernels_phi.cu) over direct peer pointers (cudaDeviceEnablePeerAccess) -- no IPC, no NCCL,
// the same fused Phi kernels.  Results are those of the one-process-per-GPU path and of a single GPU, bit for
// bit: counters are keyed by global indices and the integer sums are order independent.
// =============================================================================================
static int multi_link_shards(ldagpu_handle P)
{
    const int G = (int)P->shards.size();
    for (int g = 0; g < G; ++g) {
        ldagpu_handle c = P->shards[(size_t)g];
        cudaSetDevice(c->device);
        c->comm = nullptr; c->D_global = P->dm.D;
        set_rank(c, g, G);
        if (init_peer_table(c)) return 1;
    }
    for (ldagpu_handle c : P->shards) {
        for (int r = 0; r < G; ++r) {
            ldagpu_handle o = P->shards[(size_t)r];
            c->pt.n_wk[r] = o->n_wk.p; c->pt.phiT[r] = o->phiT.p; c->pt.seg[r] = o->seg.p;
            c->pt.nk_parts[r] = o->nk_parts.p; c->pt.flags[r] = o->p2p_flags.p;
        }
        c->p2p = true;
        c->p2p_note = "single process, direct peer pointers";
    }
    return 0;
}

int ldagpu_create_multi(int32_t K, int32_t V, int64_t D, const int64_t *doc_offsets, const int32_t *tokens,
                        const double *alpha, double beta, uint64_t seed, int32_t scheme, int32_t n_devices,
                        const int32_t *devices, ldagpu_handle *out)
{
    if (out) *out = nullptr;
    auto bail = [&](const std::string &m) { g_create_error = m; return 1; };
    if (!out || !doc_offsets || D < 0) return bail("null argument");
    if (n_devices < 1 || PHI_SEGMENTS % n_devices != 0) return bail("n_devices must be 1, 2, 4 or 8");
    std::vector<int32_t> dev((size_t)n_devices);
    for (int g = 0; g < n_devices; ++g) dev[(size_t)g] = devices ? devices[g] : g;
    if (n_devices == 1) return ldagpu_create(K, V, D, doc_offsets, tokens, alpha, beta, seed, scheme, dev[0], 0, 0, out);
    const int ndev = ldagpu_device_count();
    if (ndev == 0) return bail("no CUDA device: libldagpu has no CPU fallback");
    for (int g = 0; g < n_devices; ++g) {
        if (dev[(size_t)g] < 0 || dev[(size_t)g] >= ndev) return bail("device ordinal out of range");
        for (int q = 0; q < g; ++q)
            if (dev[(size_t)q] == dev[(size_t)g]) return bail("the same device is listed twice");
    }
    for (int a = 0; a < n_devices; ++a)
        for (int b = 0; b < n_devices; ++b) {
            if (a == b) continue;
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, dev[(size_t)a], dev[(size_t)b]) != cudaSuccess || !can) {
                cudaGetLastError();
                return bail("no peer access between devices " + std::to_string(dev[(size_t)a]) + " and " + std::to_string(dev[(size_t)b]) +
                            ": the single-process path needs it (use one process per GPU with ldagpu_comm_init instead)");
            }
            cudaSetDevice(dev[(size_t)a]);
            cudaError_t e = cudaDeviceEnablePeerAccess(dev[(size_t)b], 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
                cudaGetLastError();
                return bail(std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
            }
            cudaGetLastError();
        }
    ldagpu_handle P = new ldagpu_handle_s();
    P->dm.K = K; P->dm.V = V; P->dm.D = D; P->dm.N = doc_offsets[D]; P->dm.Ks = K; P->dm.lg = 2;
    P->scheme = scheme; P->device = dev[0]; P->seed = seed; P->beta = beta; P->world = n_devices;
    // documents shard by TOKEN count into contiguous ranges (SURVEY 8e; north_star)
    shard_bounds_by_tokens(doc_offsets, D, n_devices, P->shard_doc0, P->shard_tok0);
    for (int g = 0; g < n_devices; ++g) {
        const int64_t d0 = P->shard_doc0[(size_t)g], d1 = P->shard_doc0[(size_t)g + 1], t0 = P->shard_tok0[(size_t)g];
        const std::vector<int64_t> loc = local_offsets(doc_offsets, d0, d1);
        ldagpu_handle c = nullptr;
        if (ldagpu_create(K, V, d1 - d0, loc.data(), tokens ? tokens + t0 : nullptr, alpha, beta, seed, scheme, dev[(size_t)g],
                          d0, t0, &c)) {
            ldagpu_destroy(P);
            return 1;   // g_create_error holds the shard's message
        }
        P->shards.push_back(c);
    }
    if (multi_link_shards(P)) {
        for (ldagpu_handle c : P->shards)
            if (!c->err.empty()) g_create_error = c->err;
        ldagpu_destroy(P);
        return 1;
    }
    *out = P;
    return 0;
}

int ldagpu_get_shards(ldagpu_handle h, int32_t *n_shards, int64_t *first_docs /*[n+1] or null*/)
{
    if (!h || !n_shards) return 1;
    *n_shards = (int32_t)h->shard_doc0.size() - 1;
    if (first_docs) std::copy(h->shard_doc0.begin(), h->shard_doc0.end(), first_docs);
    return 0;
}

// ---- hyper-parameter optimisation hooks (MSL:812-905; UPL:891-894 calls optimizeAlpha / optimizeBeta every
// hyperparam_optim_interval sweeps).  The fixed-point iteration itself is MALLET's (Dirichlet.learnParameters /
// learnSymmetricConcentration) and stays on the host; the library supplies the histograms it consumes and takes the
// new values back.
static int set_alpha_one(ldagpu_handle h, const double *alpha)
{
    for (int k = 0; k < h->dm.K; ++k)
        if (!(alpha[k] > 0.0)) return h->fail("alpha must be > 0");
    if (upload_alpha(h, alpha)) return 1;
    if (step_alias(h)) return 1;   // the sparse scheme's tables are built over alpha_k * phi_kw
    return sync_check(h);
}

int ldagpu_set_alpha(ldagpu_handle h, const double *alpha)
{
    NEED(h);
    if (!alpha) return h->fail("null alpha");
    for (ldagpu_handle c : h->parts()) MC(h, c, set_alpha_one(c, alpha));
    return 0;
}

int ldagpu_set_beta(ldagpu_handle h, double beta)
{
    if (!h) return 1;
    if (!(beta > 0.0)) return h->fail("beta must be > 0");
    for (ldagpu_handle c : h->parts()) c->beta = beta;
    return 0;
}

static int count_histograms_one(ldagpu_handle h, int32_t n_doc_bins, int32_t n_type_bins, DevBuf<unsigned long long> &buf)
{
    CK(h, buf.alloc((size_t)std::max(n_doc_bins, 0) + (size_t)std::max(n_type_bins, 0) + 1));
    CK(h, launch_count_histograms(h->dm, h->doc_off.p, h->z.p, h->n_wk.p, h->row0, h->row1, n_doc_bins > 0 ? buf.p : nullptr,
                                  n_doc_bins, n_type_bins > 0 ? buf.p + std::max(n_doc_bins, 0) : nullptr, n_type_bins, h->stream));
    return 0;
}

int ldagpu_get_count_histograms(ldagpu_handle h, int32_t n_doc_bins, int64_t *doc_topic_hist, int32_t n_type_bins,
                                int64_t *type_topic_hist)
{
    NEED(h);
    if ((n_doc_bins > 0 && !doc_topic_hist) || (n_type_bins > 0 && !type_topic_hist)) return h->fail("null histogram");
    const size_t nd = (size_t)std::max(n_doc_bins, 0), nt = (size_t)std::max(n_type_bins, 0);
    std::vector<unsigned long long> acc(nd + nt + 1, 0ull), tmp(nd + nt + 1);
    const Parts parts = h->parts();
    for (ldagpu_handle c : parts) {
        DevBuf<unsigned long long> buf;
        cudaSetDevice(c->device);
        if (count_histograms_one(c, n_doc_bins, n_type_bins, buf)) { h->err = c->err; return 1; }
        if (c->world > 1 && c->comm)
            NK(h, g_nccl.AllReduce(buf.p, buf.p, nd + nt, ncclUint64, ncclSum, c->comm, c->stream));
        CK(h, cudaMemcpyAsync(tmp.data(), buf.p, sizeof(unsigned long long) * (nd + nt), cudaMemcpyDeviceToHost, c->stream));
        if (sync_check(c)) { h->err = c->err; return 1; }
        for (size_t i = 0; i < nd + nt; ++i) acc[i] += tmp[i];
    }
    const int64_t D_all = parts[0]->D_global;
    if (nd) {
        unsigned long long others = 0;
        for (size_t i = 1; i < nd; ++i) others += acc[i];
        acc[0] = (unsigned long long)D_all * (unsigned long long)h->dm.K - others;   // pairs with n_dk = 0
        for (size_t i = 0; i < nd; ++i) doc_topic_hist[i] = (int64_t)acc[i];
    }
    if (nt) {
        unsigned long long others = 0;
        for (size_t i = 1; i < nt; ++i) others += acc[nd + i];
        acc[nd] = (unsigned long long)h->dm.V * (unsigned long long)h->dm.K - others;   // cells with n_wk = 0
        for (size_t i = 0; i < nt; ++i) type_topic_hist[i] = (int64_t)acc[nd + i];
    }
    return 0;
}

// ---- held-out evaluation (MarginalProbEstimatorPlain.evaluateLeftToRight, UPL:604-611,840-844; kernels_heldout.cu)
// replace this part's test set by documents [0, D) (offsets from 0); the old one is released only once the new one is on
// the device
static int set_test_one(ldagpu_handle c, int64_t D, const int64_t *off, const int32_t *tok, int64_t doc_base, int64_t token_base)
{
    DevBuf<int64_t> o;
    DevBuf<int32_t> t;
    if (D > 0) {
        const int64_t N = off[D];
        CK(c, o.alloc((size_t)D + 1));
        CK(c, t.alloc((size_t)std::max<int64_t>(N, 1)));
        CK(c, cudaMemcpy(o.p, off, sizeof(int64_t) * ((size_t)D + 1), cudaMemcpyHostToDevice));
        if (N) CK(c, cudaMemcpy(t.p, tok, sizeof(int32_t) * (size_t)N, cudaMemcpyHostToDevice));
    }
    c->test_doc_off = std::move(o);
    c->test_tokens = std::move(t);
    c->h_test_doc_off.assign(off, off + D + 1);
    c->test_doc_base = doc_base;
    c->test_token_base = token_base;
    return 0;
}

int ldagpu_set_test_documents(ldagpu_handle h, int64_t D_test, const int64_t *doc_offsets, const int32_t *tokens,
                              int64_t doc_base, int64_t token_base)
{
    NEED(h);
    if (heldout_refuses_k(h)) return 1;
    const int32_t V = h->dm.V;
    if (D_test < 0 || doc_base < 0 || token_base < 0) return h->fail("D_test, doc_base and token_base must be >= 0");
    static const int64_t zero = 0;
    if (D_test == 0) doc_offsets = &zero;   // removes the test set
    if (!doc_offsets) return h->fail("null doc_offsets");
    if (const char *e = csr_offsets_error(doc_offsets, D_test)) return h->fail("test doc_offsets%s", e);
    const int64_t N = doc_offsets[D_test];
    if (N > 0 && !tokens) return h->fail("null tokens");
    for (int64_t i = 0; i < N; ++i)
        if (tokens[i] < 0 || tokens[i] >= V)
            return h->fail("test token %lld: type id %d out of range [0, %d)", (long long)i, tokens[i], V);
    const Parts parts = h->parts();
    std::vector<int64_t> d0, t0;
    shard_bounds_by_tokens(doc_offsets, D_test, (int)parts.size(), d0, t0);
    for (size_t g = 0; g < parts.size(); ++g) {
        ldagpu_handle c = parts[g];
        const std::vector<int64_t> loc = local_offsets(doc_offsets, d0[g], d0[g + 1]);
        MC(h, c, set_test_one(c, d0[g + 1] - d0[g], loc.data(), tokens ? tokens + t0[g] : nullptr, doc_base + d0[g],
                              token_base + t0[g]));
    }
    h->test_doc0 = d0;
    h->test_tok0 = t0;
    h->test_doc_base = doc_base;
    h->test_token_base = token_base;
    return 0;
}

// enqueue this part's evaluation with particles R and phihat (layout hd) in c->phihat: document batches whose S fits
// HELDOUT_SCRATCH_BYTES, each one the sampling kernel and then the per-document reduction into c->ho_ll
static int heldout_enqueue(ldagpu_handle c, const Dims &hd, int32_t R)
{
    const std::vector<int64_t> &off = c->h_test_doc_off;
    const int64_t D = (int64_t)off.size() - 1;
    if (D == 0) return 0;
    const int64_t cap = std::max<int64_t>(1, HELDOUT_SCRATCH_BYTES / ((int64_t)sizeof(float) * R));
    std::vector<int64_t> b{0};
    while (b.back() < D) {
        int64_t d = b.back() + 1;   // at least one document per batch
        while (d < D && off[d + 1] - off[b.back()] <= cap) ++d;
        b.push_back(d);
    }
    int64_t most = 0;
    for (size_t i = 0; i + 1 < b.size(); ++i) most = std::max(most, off[b[i + 1]] - off[b[i]]);
    CK(c, c->ho_scores.alloc((size_t)std::max<int64_t>(most, 1) * (size_t)R));
    CK(c, c->ho_ll.alloc((size_t)D));
    HeldoutArgs a{};
    a.dm = hd;
    a.doc_off = c->test_doc_off.p;
    a.tokens = c->test_tokens.p;
    a.phihat = c->phihat.p;
    a.alpha = c->alpha_f.p;
    a.R = R;
    a.S = c->ho_scores.p;
    a.token_base = c->test_token_base;
    a.iteration = (uint32_t)c->iteration;
    a.rk = philox_keys((uint32_t)c->seed, (uint32_t)(c->seed >> 32));
    a.work_counter = c->counter.p;
    for (size_t i = 0; i + 1 < b.size(); ++i) {
        a.doc0 = b[i];
        a.doc1 = b[i + 1];
        a.tok0 = off[b[i]];
        a.batch_tokens = off[b[i + 1]] - off[b[i]];
        CK(c, cudaMemsetAsync(c->counter.p, 0, sizeof(unsigned long long), c->stream));
        CK(c, launch_heldout_l2r(a, c->sm_count, c->stream));
        CK(c, launch_heldout_reduce(a, c->alpha_sum, c->ho_ll.p + b[i], c->sm_count, c->stream));
    }
    return 0;
}

static void heldout_release(const Parts &parts)
{
    for (ldagpu_handle c : parts) {
        cudaSetDevice(c->device);
        c->phihat.release(); c->ho_scores.release(); c->ho_ll.release();
    }
}

static int heldout_run(ldagpu_handle h, const Parts &parts, int32_t R, std::vector<double> &ll)
{
    // the global counts on parts[0] (a rank: on every rank), phihat from them, copied to the other shards of a group
    if (gather_rows(h, parts, &ldagpu_handle_s::n_wk, ncclInt32)) return 1;
    ldagpu_handle c0 = parts[0];
    const Dims hd = reg_path_dims(c0->dm);
    const size_t cells = (size_t)hd.Vp * hd.Ks;
    for (ldagpu_handle c : parts) {
        CK(h, cudaSetDevice(c->device));
        MC(h, c, [&]() { CK(c, c->phihat.alloc(cells)); return 0; }());
    }
    CK(h, cudaSetDevice(c0->device));
    MC(h, c0, [&]() {
        CK(c0, launch_heldout_phihat(c0->dm, hd, c0->n_wk.p, c0->n_k.p, c0->beta, c0->phihat.p, c0->sm_count, c0->stream));
        CK(c0, cudaStreamSynchronize(c0->stream));
        return 0;
    }());
    for (size_t g = 1; g < parts.size(); ++g) {
        ldagpu_handle c = parts[g];
        CK(h, cudaSetDevice(c->device));
        CK(h, cudaMemcpyPeerAsync(c->phihat.p, c->device, c0->phihat.p, c0->device, sizeof(float) * cells, c->stream));
    }
    // every part samples its test documents before any is waited for
    for (ldagpu_handle c : parts) MC(h, c, heldout_enqueue(c, hd, R));
    for (ldagpu_handle c : parts) {
        const size_t D = c->h_test_doc_off.size() - 1, o = ll.size();
        ll.resize(o + D);
        CK(h, cudaSetDevice(c->device));
        if (D) CK(h, cudaMemcpyAsync(ll.data() + o, c->ho_ll.p, sizeof(double) * D, cudaMemcpyDeviceToHost, c->stream));
        MC(h, c, sync_check(c));
    }
    return 0;
}

// one process per GPU: every rank's per-document values to every rank, placed by global test-document index
static int heldout_allgather(ldagpu_handle h, const std::vector<double> &local, std::vector<double> &global)
{
    DevBuf<int64_t> n;
    DevBuf<double> buf;
    int64_t end = h->test_doc_base + (int64_t)local.size();
    CK(h, n.alloc(1));
    CK(h, cudaMemcpyAsync(n.p, &end, sizeof end, cudaMemcpyHostToDevice, h->stream));
    NK(h, g_nccl.AllReduce(n.p, n.p, 1, ncclInt64, ncclMax, h->comm, h->stream));
    CK(h, cudaMemcpyAsync(&end, n.p, sizeof end, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    // each cell is written by one rank and zero on the others, so the sum is exact in any order
    CK(h, buf.alloc((size_t)std::max<int64_t>(end, 1)));
    CK(h, cudaMemsetAsync(buf.p, 0, sizeof(double) * buf.n, h->stream));
    if (!local.empty())
        CK(h, cudaMemcpyAsync(buf.p + h->test_doc_base, local.data(), sizeof(double) * local.size(), cudaMemcpyHostToDevice,
                              h->stream));
    NK(h, g_nccl.AllReduce(buf.p, buf.p, buf.n, ncclDouble, ncclSum, h->comm, h->stream));
    global.assign((size_t)end, 0.0);
    if (end) CK(h, cudaMemcpyAsync(global.data(), buf.p, sizeof(double) * (size_t)end, cudaMemcpyDeviceToHost, h->stream));
    return sync_check(h);
}

int ldagpu_heldout_log_likelihood(ldagpu_handle h, int32_t n_particles, double *doc_ll, double *total)
{
    NEED(h);
    if (!total) return h->fail("null total");
    if (heldout_refuses_k(h)) return 1;
    if (n_particles < 1 || n_particles >= (1 << 24)) return h->fail("n_particles must be in [1, 2^24)");
    const Parts parts = h->parts();
    std::vector<double> ll;
    const int rc = heldout_run(h, parts, n_particles, ll);
    heldout_release(parts);
    if (rc) return 1;
    if (doc_ll && !ll.empty()) std::copy(ll.begin(), ll.end(), doc_ll);
    std::vector<double> all;
    if (h->world > 1 && h->comm) {
        if (heldout_allgather(h, ll, all)) return 1;
    } else {
        all.swap(ll);
    }
    double s = 0.0;
    for (double v : all) s += v;   // global document order
    *total = s;
    return 0;
}

}  // extern "C"
