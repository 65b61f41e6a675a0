/*
 * oracle/lda_oracle.h -- TEST INFRASTRUCTURE ONLY.
 *
 * CPU restatement of one Gibbs sweep of the reference's exact-parallel LDA
 * samplers (LDAGroupedGibbsSampler = "GGS", UncollapsedParallelLDA /
 * LDAPartiallyCollapsedGibbsSampler = "PCGS") and the held-out left-to-right estimator.
 * Only tests/, __graft_entry__.smoke(), bench.py's cpu_baseline / --impl reference legs
 * and tools/heldout_bench.py may load this library; the product (libldagpu.so) never does.
 *
 * PARITY UNPINNED (against a running reference): the reference is Java 8 + MALLET 2.0.8
 * and there is no JDK in the build container, the reference holds no golden vectors for
 * GGS/PCGS, and its in-sweep RNG (ThreadLocalRandom / nanoTime-seeded xorshift) is not
 * seedable.  What IS pinned: java.util.Random known answers, Philox4x32-10 known answers,
 * the reference tests' invariants and closed forms (tests/test_oracle_*.py).
 *
 * Two arithmetic modes:
 *   faithful -- double precision, libm, the Java loop order and sequential sums.
 *   contract -- the fixed-order fp32/fp64 arithmetic the CUDA kernels implement
 *               (DESIGN.md section 4); bit-exact with the GPU by construction.
 * Both consume the same injected Philox4x32-10 stream.
 *
 * Layouts: doc_off int64[D+1] (CSR), tokens/z int32[N], n_wk int32[V][K],
 * n_k int32[K], phiT [V][K] (word-major: the transpose of the reference's phi[K][V]),
 * theta [D][K].
 */
#ifndef LDA_ORACLE_H
#define LDA_ORACLE_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { ORACLE_GGS = 0, ORACLE_PCGS = 1 };
enum { ORACLE_STREAM_Z = 1, ORACLE_STREAM_THETA = 2, ORACLE_STREAM_PHI = 3, ORACLE_STREAM_POISSON = 4, ORACLE_STREAM_HELDOUT = 5 };

void oracle_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);

/* java.util.Random(seed).nextInt(bound) stream; reference: UncollapsedParallelLDA.java:398-406,458-460 */
void oracle_java_random_next_ints(int64_t seed, int32_t bound, int64_t n, int32_t *out);
void oracle_java_random_raw_ints(int64_t seed, int64_t n, int32_t *out); /* nextInt() */

/* reference: UncollapsedParallelLDA.java:1797-1830 (setZIndicators), :471-482 */
int oracle_rebuild_counts(int64_t N, const int32_t *tokens, const int32_t *z, int32_t V, int32_t K,
                          int32_t *n_wk, int32_t *n_k);
void oracle_doc_topic_counts(int64_t D, const int64_t *doc_off, const int32_t *z, int32_t K,
                             int32_t *n_dk);

/* contract-math probes (for unit tests of the primitives) */
float oracle_c_ln_f32(float x);
double oracle_c_ln_f64(double x);
float oracle_c_exp_neg_f32(float y);
double oracle_c_exp_neg_f64(double y);
float oracle_c_cos2pi_f32(uint32_t w);
double oracle_c_cos2pi_f64(uint32_t w);
float oracle_c_gamma_f32(float a, uint64_t seed, uint64_t cell, uint32_t sweep, uint32_t stream);
double oracle_c_gamma_f64(double a, uint64_t seed, uint64_t cell, uint32_t sweep, uint32_t stream);
/* faithful (libm, double) Gamma on the same uniforms; variant = 32 or 64 picks which
 * contract's uniform construction is mirrored */
double oracle_f_gamma(double a, uint64_t seed, uint64_t cell, uint32_t sweep, uint32_t stream,
                      int variant);

/* categorical draw of the contract: a[K] * phirow[K], uniform U.  Two prefix trees, like the kernels (DESIGN.md 4.2):
 * K <= 1024 lane-contiguous (lane l of 32 owns L = 4*NT consecutive topics, one warp scan of the lane totals),
 * K > 1024 tile-major (128-topic tiles, distributed butterfly + per-tile scan).  Same selection rule -- first k
 * with cumsum_k >= U*sum in natural topic order (GGS:96-113, UPL:1507-1526) -- different fp32 rounding. */
int32_t oracle_draw_topic_contract(const float *a, const float *phirow, int32_t K, float U);

/* GGS theta draw; reference: LDAGroupedGibbsSampler.java:60-72, ParallelDirichlet.java:46-70 */
void oracle_theta_contract(int64_t D, const int64_t *doc_off, const int32_t *z, int32_t K,
                           const double *alpha, uint64_t seed, uint32_t sweep, int64_t doc_base,
                           float *theta);
void oracle_theta_faithful(int64_t D, const int64_t *doc_off, const int32_t *z, int32_t K,
                           const double *alpha, uint64_t seed, uint32_t sweep, int64_t doc_base,
                           double *theta);

/* z-step; reference: LDAGroupedGibbsSampler.java:79-130 (GGS), UncollapsedParallelLDA.java:1491-1543 (PCGS) */
void oracle_z_ggs_contract(int64_t D, const int64_t *doc_off, const int32_t *tokens, int32_t *z,
                           int32_t K, const float *theta, const float *phiT, uint64_t seed,
                           uint32_t sweep, int64_t token_base);
void oracle_z_pcgs_contract(int64_t D, const int64_t *doc_off, const int32_t *tokens, int32_t *z,
                            int32_t K, const double *alpha, const float *phiT, uint64_t seed,
                            uint32_t sweep, int64_t token_base);
void oracle_z_ggs_faithful(int64_t D, const int64_t *doc_off, const int32_t *tokens, int32_t *z,
                           int32_t K, const double *theta, const double *phiT, uint64_t seed,
                           uint32_t sweep, int64_t token_base);
void oracle_z_pcgs_faithful(int64_t D, const int64_t *doc_off, const int32_t *tokens, int32_t *z,
                            int32_t K, const double *alpha, const double *phiT, uint64_t seed,
                            uint32_t sweep, int64_t token_base);

/* Phi draw; reference: LDAGroupedGibbsSampler.java:182-192, LDAPartiallyCollapsedGibbsSampler.java:91-101,
 * MarsagliaSparseDirichlet.java:31-55 (initial Phi), ParallelDirichlet.java:46-70 */
void oracle_phi_contract(int32_t V, int32_t K, const int32_t *n_wk, double beta, uint64_t seed,
                         uint32_t sweep, float *phiT);
void oracle_phi_faithful(int32_t V, int32_t K, const int32_t *n_wk, double beta, uint64_t seed,
                         uint32_t sweep, double *phiT);

/* Poisson Polya-urn Phi draw; reference: topics/PolyaUrnSpaliasLDA.java:495-507,
 * types/PolyaUrnDirichletFixedCoeffPoisson.java:17-44, types/PoissonFixedCoeffSampler.java:45-51 (L = alias_poisson_threshold) */
int32_t oracle_poisson(double beta, int32_t n, int32_t L, uint64_t seed, uint64_t cell, uint32_t sweep, int faithful);
void oracle_phi_polya_contract(int32_t V, int32_t K, const int32_t *n_wk, double beta, int32_t L, uint64_t seed,
                               uint32_t sweep, float *phiT);
void oracle_phi_polya_faithful(int32_t V, int32_t K, const int32_t *n_wk, double beta, int32_t L, uint64_t seed,
                               uint32_t sweep, double *phiT);

/* MALLET Dirichlet.logGammaStirling (from memory of MALLET 2.0.8, see SURVEY 8c) */
double oracle_log_gamma_stirling(double z);
/* reference: UncollapsedParallelLDA.java:1644-1758 */
double oracle_log_likelihood(int64_t D, const int64_t *doc_off, const int32_t *z, int32_t K,
                             int32_t V, const int32_t *n_wk, const int32_t *n_k,
                             const double *alpha, double beta);
/* second statement of the same formula with exact lgamma instead of Stirling
 * (SerialCollapsedLDA.java:443-556 equates the two within 1e-6 in LogLikelihoodTest) */
double oracle_log_likelihood_lgamma(int64_t D, const int64_t *doc_off, const int32_t *z, int32_t K,
                                    int32_t V, const int32_t *n_wk, const int32_t *n_k,
                                    const double *alpha, double beta);
/* reference: UncollapsedParallelLDA.java:1573-1634 */
double oracle_log_posterior(int64_t D, const int64_t *doc_off, const int32_t *tokens,
                            const int32_t *z, int32_t K, int32_t V, const double *theta,
                            const double *phiT, const double *alpha, double beta);

/* held-out log-likelihood, left-to-right estimator without resampling: MALLET's MarginalProbEstimator.evaluateLeftToRight
 * (Wallach et al. 2009) as the reference's MarginalProbEstimatorPlain restates it (UncollapsedParallelLDA.java:604-611,
 * 840-844 call it).  Test set doc_off[D+1] / tokens (token_base = global index of its first token), R particles at
 * `iteration`, K <= 1024.  doc_ll[D] receives ln p(w_d); returns their sum in document order. */
double oracle_heldout_l2r_contract(int64_t D, const int64_t *doc_off, const int32_t *tokens, int32_t V, int32_t K,
                                   const int32_t *n_wk, const int32_t *n_k, const double *alpha, double beta,
                                   uint64_t seed, uint32_t iteration, int64_t token_base, int32_t R, double *doc_ll);
double oracle_heldout_l2r_faithful(int64_t D, const int64_t *doc_off, const int32_t *tokens, int32_t V, int32_t K,
                                   const int32_t *n_wk, const int32_t *n_k, const double *alpha, double beta,
                                   uint64_t seed, uint32_t iteration, int64_t token_base, int32_t R, double *doc_ll);

/* whole sweeps, contract mode: for it in first_sweep..first_sweep+n-1:
 *   [GGS: theta], z, counts, Phi     (order: UncollapsedParallelLDA.java:645-693)
 * phiT in/out, z in/out; theta (may be NULL for PCGS), n_wk, n_k out. */
void oracle_sweeps_contract(int scheme, int64_t D, int32_t V, int32_t K, const int64_t *doc_off,
                            const int32_t *tokens, int32_t *z, const double *alpha, double beta,
                            uint64_t seed, uint32_t first_sweep, int32_t n_sweeps, float *phiT,
                            float *theta, int32_t *n_wk, int32_t *n_k);
void oracle_sweeps_faithful(int scheme, int64_t D, int32_t V, int32_t K, const int64_t *doc_off,
                            const int32_t *tokens, int32_t *z, const double *alpha, double beta,
                            uint64_t seed, uint32_t first_sweep, int32_t n_sweeps, double *phiT,
                            double *theta, int32_t *n_wk, int32_t *n_k);

/* CPU baseline ("port"): the faithful sweep with the reference's threading shape --
 * document-parallel z on all threads with shared atomic +-1 deltas
 * (UncollapsedParallelLDA.java:1354-1437,1547-1557), K*V delta merge (:1107-1221),
 * topic-parallel Phi (:1240-1274).  Returns seconds for z+merge and for Phi. */
void oracle_baseline_sweeps(int scheme, int64_t D, int32_t V, int32_t K, const int64_t *doc_off,
                            const int32_t *tokens, int32_t *z, const double *alpha, double beta,
                            uint64_t seed, int32_t n_sweeps, int32_t n_threads, double *z_seconds,
                            double *phi_seconds);
int oracle_max_threads(void);
void oracle_set_num_threads(int n);

/* ---- sparse PCGS z-step ("spalias"), lda_oracle_sparse.c -------------------------------------
 * reference: topics/SpaliasUncollapsedParallelLDA.java:39-60,124-312, util/OptimizedGentleAliasMethod.java:52-107 */
void oracle_alias_build_contract(int32_t V, int32_t K, const double *alpha, const float *phiT, float *ps,
                                 int32_t *al, float *type_norm);
/* the prior part's draw of one token from its Philox words 1 (slot) and 2 (keep-or-alias uniform), one type's table */
int32_t oracle_alias_sample_contract(const float *ps, const int32_t *al, int32_t K, uint32_t w1, uint32_t w2);
void oracle_z_spalias_contract(int64_t D, const int64_t *doc_off, const int32_t *tokens, int32_t *z,
                               int32_t K, const float *phiT, const float *ps, const int32_t *al,
                               const float *type_norm, uint64_t seed, uint32_t sweep, int64_t token_base);
void oracle_z_spalias_faithful(int64_t D, int32_t V, const int64_t *doc_off, const int32_t *tokens, int32_t *z,
                               int32_t K, const double *alpha, const double *phiT, uint64_t seed,
                               uint32_t sweep, int64_t token_base);

#ifdef __cplusplus
}
#endif
#endif
