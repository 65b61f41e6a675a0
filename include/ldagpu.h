/*
 * ldagpu.h -- C ABI of libldagpu.so, the B200-native Gibbs-sweep engine behind the reference's
 * sampler interface (schemes "gpu_ggs" / "gpu_pcgs").
 *
 * The reference (clintpgeorge/LDAGroupedGibbsSampler, 100 % Java) has no native interface; the
 * binding point is its sampler interface, so every entry point below names the Java method(s) it
 * serves.  Paths are relative to src/main/java/cc/mallet/ of the reference:
 *   LGS  = topics/LDAGibbsSampler.java        (interface, :10-47)
 *   LSWP = topics/LDASamplerWithPhi.java      (interface, :5-12)
 *   UPL  = topics/UncollapsedParallelLDA.java
 *   GGS  = topics/LDAGroupedGibbsSampler.java
 *   PCGS = topics/LDAPartiallyCollapsedGibbsSampler.java
 *   MSL  = topics/ModifiedSimpleLDA.java
 *
 * Conventions: every function returns 0 on success, non-zero on error (message through
 * ldagpu_last_error).  The caller owns every buffer it passes; the library copies in/out and owns
 * only device memory behind the opaque handle.  Matrices are flat row-major with the shape of the
 * Java array they mirror.  One caller thread per handle; ldagpu_abort may be called from any
 * thread.  There is no CPU fallback: without a CUDA device ldagpu_create fails.
 */
#ifndef LDAGPU_H
#define LDAGPU_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ldagpu_handle_s *ldagpu_handle;

#define LDAGPU_SCHEME_GGS 0  /* GGS:47-132, GGS:139-209 */
#define LDAGPU_SCHEME_PCGS 1 /* UPL:1466-1545, PCGS:48-118 */
/* PCGS with the reference's sparse z-step (topics/SpaliasUncollapsedParallelLDA.java:39-60,124-312:
 * per-type alias table over alpha_k*phi_kw + sparse cumulative sum over the topics with n_dk > 0)
 * and the PCGS Phi draw: the path for K in the thousands. */
#define LDAGPU_SCHEME_SPALIAS 2

/* version / build info ("libldagpu x.y sm_100a") */
const char *ldagpu_version(void);
/* message of the last failure on this handle (or of the last failed create when h == NULL) */
const char *ldagpu_last_error(ldagpu_handle h);
/* number of visible CUDA devices (0 if none / no driver) */
int ldagpu_device_count(void);

/*
 * addInstances (LGS:13, UPL:357-456, GGS:33-37): upload one shard of the corpus in CSR form.
 *   K, V           topics, vocabulary size
 *   D, doc_offsets local documents and their int64[D+1] token offsets (doc_offsets[0] == 0)
 *   tokens         int32[N] type ids, N = doc_offsets[D]
 *   alpha          double[K]  (MSL:61-64), beta scalar
 *   seed           Philox key of the in-sweep draws (the reference's are unseedable, UPL:1519, GGS:107)
 *   scheme         LDAGPU_SCHEME_GGS | LDAGPU_SCHEME_PCGS   (factory switch, tui/ParallelLDA.java:401-490)
 *   device         CUDA device ordinal
 *   doc_base, token_base  global index of the shard's first document / token (0 on one GPU):
 *                  random-number counters are keyed by global indices, so results do not depend
 *                  on how the corpus is sharded
 * The topic indicators start at 0; call ldagpu_init_z_java_random or ldagpu_set_z next.
 */
int ldagpu_create(int32_t K, int32_t V, int64_t D, const int64_t *doc_offsets, const int32_t *tokens,
                  const double *alpha, double beta, uint64_t seed, int32_t scheme, int32_t device,
                  int64_t doc_base, int64_t token_base, ldagpu_handle *out);
int ldagpu_destroy(ldagpu_handle h);

/*
 * The same from ONE caller thread for several GPUs of one box: the reference runs one coordinator thread in one JVM
 * (tui/ParallelLDA.java:173-202 -> UPL:552-943), so `scheme = gpu_ggs` with `gpu_devices = 0,1,...` must not need one
 * process per GPU.  Takes the WHOLE corpus; documents are sharded by token count into contiguous ranges, one per
 * device (devices == NULL: ordinals 0..n_devices-1; n_devices in {1, 2, 4, 8}); every other entry point takes the
 * returned handle and works on the whole corpus (z, theta and the document-topic matrix in corpus order).  The
 * count exchange and the Phi broadcast run inside the Phi kernels over direct peer pointers (no NCCL, no IPC), so
 * the devices need peer access (NVLink / NVSwitch); results are bit-identical to one GPU and to one process per GPU.
 */
int ldagpu_create_multi(int32_t K, int32_t V, int64_t D, const int64_t *doc_offsets, const int32_t *tokens,
                        const double *alpha, double beta, uint64_t seed, int32_t scheme, int32_t n_devices,
                        const int32_t *devices, ldagpu_handle *out);
/* how the corpus is sharded behind the handle: *n_shards, and (first_docs != NULL) the n_shards + 1 document bounds */
int ldagpu_get_shards(ldagpu_handle h, int32_t *n_shards, int64_t *first_docs);

/* multi-GPU (one process per GPU).  Rank 0 makes an id, the host program broadcasts its 128 bytes
 * (torch.distributed / any rendezvous), every rank joins.  After this, sweeps exchange counts with
 * one reduce-scatter and Phi with one all-gather per sweep (SURVEY 8e). */
int ldagpu_comm_unique_id(void *id128);
int ldagpu_comm_init(ldagpu_handle h, int32_t rank, int32_t world, const void *id128);
/* how the ranks exchange counts and Phi: 0 = single GPU, 1 = NCCL collectives (reduce-scatter / all-gather
 * around the Phi kernels), 2 = peer memory (default when the GPUs have peer access: the Phi kernels load the
 * other ranks' partial counts and store Phi into every rank's copy over NVLink themselves).  Environment:
 * LDAGPU_EXCHANGE=nccl|p2p forces one; LDAGPU_P2P_TIMEOUT_MS bounds an in-kernel wait on a dead rank (default 60000; host-side skew between the
 * ranks is absorbed by an NCCL rendezvous at the start of every exchanging call, not by these waits).
 * The stand-in for the reference's shared AtomicInteger[K][V] delta matrix (UPL:102,363-368,1107-1221). */
int ldagpu_get_exchange_mode(ldagpu_handle h, int32_t *mode);

/* initial z = MALLET Randoms(seed).nextInt(K) in document order (UPL:398-406,458-460; MSL:153-156).
 * skip = number of draws consumed by the shards before this one (token_base on a sharded corpus).
 * Rebuilds the counts and draws the initial Phi (UPL:450,1287-1294) with sweep counter 0. */
int ldagpu_init_z_java_random(ldagpu_handle h, int32_t seed);
/* setZIndicators (LGS:22, UPL:1797-1843): replace z, rebuild counts, redraw Phi (sweep counter
 * unchanged).  redraw_phi = 0 keeps the current Phi (used by tests and by checkpoint restore).
 * An indicator outside [0, K) fails the call and leaves the previous indicators and counts in place (the reference
 * throws, UPL:475-481). */
int ldagpu_set_z(ldagpu_handle h, const int32_t *z, int32_t redraw_phi);
/* getZIndicators (LGS:19, MSL:464-477) flattened in CSR order */
int ldagpu_get_z(ldagpu_handle h, int32_t *z);

/* sample(iterations) (LGS:15, UPL:552-943): n full sweeps = [theta] z, counts, Phi.
 * Stops early when ldagpu_abort was called (UPL:645,906-910); *done receives the sweeps run. */
int ldagpu_sweep(ldagpu_handle h, int32_t n, int32_t *done);
/* sample(iterations) followed by getZIndicators in one call: the indicators of the last sweep travel to the host
 * buffer z (int32[N], pinned memory for the overlap) while that sweep's count exchange and Phi draw still run.
 * This is what the Java shim's sample() does: z goes back into the documents' LabelSequences after every call
 * (MSL:464-477, util/LDAUtils.java:1552-1571 read it from there). */
int ldagpu_sweep_get_z(ldagpu_handle h, int32_t n, int32_t *done, int32_t *z);
/* 16-bit transport of the topic indicators (K <= 65 536): the same three calls with uint16 host buffers.
 * The Java int[] boundary keeps the int32 entry points (MSL:464-477, UPL:1797-1843); a host that can hold z as
 * char[] / short[] halves the PCIe bytes of every setZIndicators / sample() round trip. */
int ldagpu_set_z16(ldagpu_handle h, const uint16_t *z, int32_t redraw_phi);
int ldagpu_get_z16(ldagpu_handle h, uint16_t *z);
int ldagpu_sweep_get_z16(ldagpu_handle h, int32_t n, int32_t *done, uint16_t *z);
/* sampleZGivenPhi(iterations) (LSWP:11, UPL:975-1014): z and counts only, Phi frozen */
int ldagpu_sample_z_given_phi(ldagpu_handle h, int32_t n, int32_t *done);
/* step-wise entry points (tests, and hosts that interleave their own hooks preZ/postZ/prePhi/postPhi,
 * LGS:38-43, LSWP:9-10).  A full sweep is: next_iteration, [sample_theta], sample_z, rebuild_counts,
 * sample_phi. */
int ldagpu_next_iteration(ldagpu_handle h);
int ldagpu_sample_theta(ldagpu_handle h);   /* GGS:60-72 */
int ldagpu_sample_z(ldagpu_handle h);       /* GGS:79-130 / UPL:1491-1543 */
int ldagpu_rebuild_counts(ldagpu_handle h); /* UPL:1107-1221 net effect (= UPL:1797-1830) */
int ldagpu_sample_phi(ldagpu_handle h);     /* GGS:139-209 / PCGS:48-118 */
int ldagpu_get_iteration(ldagpu_handle h, int32_t *it); /* getCurrentIteration (LGS:18) */
int ldagpu_set_iteration(ldagpu_handle h, int32_t it);

/* getTypeTopicMatrix / getTypeTopicCounts (LGS:32, UPL:226-234): int32[V][K] (collective when sharded) */
int ldagpu_get_type_topic_counts(ldagpu_handle h, int32_t *n_wk);
/* getTopicTotals (LGS:33, MSL:971-976): int32[K] */
int ldagpu_get_topic_totals(ldagpu_handle h, int32_t *n_k);
/* getDocumentTopicMatrix (LGS:31, MSL:536-547): int32[D][K] for the local documents */
int ldagpu_get_doc_topic_counts(ldagpu_handle h, int32_t *n_dk);
/* getPhi (LSWP:6, UPL:1946-1948): double[K][V];  setPhi (LSWP:7, UPL:1897-1926) */
int ldagpu_get_phi(ldagpu_handle h, double *phi);
int ldagpu_set_phi(ldagpu_handle h, const double *phi);
/* getPhiMeans (LSWP:8, UPL:1954-1966): double[K][V] = running sum / n_sampled; n_sampled = 0 means
 * nothing accumulated yet (the Java side returns null).  Schedule: accumulate when
 * iteration > burn_in && iteration % thin == 0 (UPL:1350-1352); burn_in <= 0 disables. */
int ldagpu_set_phi_mean_schedule(ldagpu_handle h, int32_t burn_in, int32_t thin);
int ldagpu_get_phi_mean(ldagpu_handle h, double *phi_mean, int32_t *n_sampled);
/* How the rows of Phi are drawn (before ldagpu_init_z_java_random / ldagpu_set_z, which draw the first Phi):
 *   LDAGPU_PHI_GAMMA      Dirichlet = Gammas + normalise + floor (GGS:182-192, PCGS:91-101, types/ParallelDirichlet.java:46-70)
 *   LDAGPU_PHI_POLYA_URN  the Poisson Polya urn of scheme "polyaurn" (topics/PolyaUrnSpaliasLDA.java:495-507,
 *                         types/PolyaUrnDirichletFixedCoeffPoisson.java:17-44): X = Poisson(beta + n_wk), phi = X / sum X,
 *                         zeros stay zeros; alias_poisson_threshold = the reference's key of that name (default 100,
 *                         types/PoissonFixedCoeffSampler.java:45-51): counts below it are drawn exactly, from it on by
 *                         the normal approximation.  Use with LDAGPU_SCHEME_SPALIAS (the reference pairs it with the
 *                         sparse z-step); a word type whose Phi column is all zero falls back to a uniform topic
 *                         (PolyaUrnSpaliasLDA.java:275-277). */
#define LDAGPU_PHI_GAMMA 0
#define LDAGPU_PHI_POLYA_URN 1
int ldagpu_set_phi_sampler(ldagpu_handle h, int32_t sampler, int32_t alias_poisson_threshold);
/* GGS thetaMatrix (UPL:78, GGS:72): double[D][K] of the last sweep; set = test injection */
int ldagpu_get_theta(ldagpu_handle h, double *theta);
int ldagpu_set_theta(ldagpu_handle h, const double *theta);
/* modelLogLikelihood (UPL:1644-1758) -> getLogLikelihood series is kept by the host (LGS:44) */
int ldagpu_log_likelihood(ldagpu_handle h, double *ll);
/* computeLogPosterior (UPL:1573-1634); GGS uses the sweep's theta (UPL:716-720) */
int ldagpu_log_posterior(ldagpu_handle h, double *lp);

/*
 * Held-out evaluation (UPL:604-611,840-844: MarginalProbEstimatorPlain.evaluateLeftToRight, MALLET's left-to-right
 * estimator without resampling; DESIGN.md 4.8).  K <= 1024 only: a larger K fails with an error naming the limit.
 * addTestInstances (LGS): upload a test set in CSR form, as for ldagpu_create, with the global index of its first
 * document / token (doc_base, token_base; 0 unless the caller shards the test set over ranks itself).  The documents stay
 * resident; a second call replaces them, D_test = 0 removes them.  A type outside [0, V) or malformed offsets fail the
 * call and leave the previous test set in place.  A create_multi handle takes the whole test set and shards it by
 * tokens over its GPUs; with one process per GPU every rank passes its own shard.
 */
int ldagpu_set_test_documents(ldagpu_handle h, int64_t D_test, const int64_t *doc_offsets, const int32_t *tokens,
                              int64_t doc_base, int64_t token_base);
/* getHeldOutLogLikelihood (UPL:604-611,840-844), evaluateLeftToRight: the model is phi_kw = (n_wk + beta) /
 * (n_k + V beta) from the current counts and alpha; n_particles (R, MALLET's default 10) particles per document.
 * doc_ll (NULL or double[D_test] of this handle's test documents) receives ln p(w_d), *total the sum over the whole
 * test set (every rank returns the same total).  Reads the counts only: z, counts, Phi, theta, the iteration and the
 * training random streams are untouched, and two calls at the same iteration return the same values. */
int ldagpu_heldout_log_likelihood(ldagpu_handle h, int32_t n_particles, double *doc_ll, double *total);

/* Hooks for the hyper-parameter optimisation (MSL:812-905, called every hyperparam_optim_interval sweeps, UPL:891-894;
 * off by default).  MALLET's fixed-point iteration (Dirichlet.learnParameters / learnSymmetricConcentration) stays on the
 * host; the library supplies the histograms it consumes -- doc_topic_hist[c] = number of (document, topic) pairs with
 * n_dk = c (MSL:815-846 documentTopicHistogram merged over topics), type_topic_hist[c] = number of (type, topic) cells
 * with n_wk = c (MSL:860-875 countHistogram); counts beyond the last bin land in it -- and takes the new values back. */
int ldagpu_get_count_histograms(ldagpu_handle h, int32_t n_doc_bins, int64_t *doc_topic_hist, int32_t n_type_bins,
                                int64_t *type_topic_hist);
int ldagpu_set_alpha(ldagpu_handle h, const double *alpha /* [K] */);
int ldagpu_set_beta(ldagpu_handle h, double beta);

/* abort()/getAbort() (topics/AbortableSampler.java:3-6, MSL:601-608); async-safe */
int ldagpu_abort(ldagpu_handle h);
int ldagpu_get_abort(ldagpu_handle h, int32_t *aborted);

/* cumulative device time per phase in ms since creation (the reference's own timers:
 * zSamplingTimeCum = z + count merge, phiSamplingTimeCum; UPL:642-644,670-673,690-693,931-939) */
int ldagpu_get_timers(ldagpu_handle h, double *z_ms, double *counts_ms, double *phi_ms, double *comm_ms);
/* over the last ldagpu_sweep / ldagpu_sample_z_given_phi call, measured with CUDA events on the
 * library's stream: device time of the whole call, device time of the dominant kernel (the z-step
 * launches), and how many kernels the call launched */
int ldagpu_get_last_call_stats(ldagpu_handle h, double *call_ms, double *z_kernel_ms,
                               int64_t *z_kernel_launches, int64_t *total_launches);

#ifdef __cplusplus
}
#endif
#endif
