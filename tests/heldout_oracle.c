/*
 * tests/heldout_oracle.c -- TEST INFRASTRUCTURE ONLY: the CPU restatement of the held-out log-likelihood
 * (DESIGN.md 4.8), built on demand by tests/heldout_oracle.py.
 *
 * MALLET's MarginalProbEstimator.evaluateLeftToRight without resampling (Wallach et al. 2009), which the reference's
 * MarginalProbEstimatorPlain restates over plain count arrays (topics/UncollapsedParallelLDA.java:604-611,840-844
 * call it).  Model phi_kw = (n_wk + beta) / (n_k + V beta); per document and particle r, from n_dk = 0:
 * S_i = sum_k (n_dk + alpha_k) phi_kw, p_i = S_i / (i + alpha_sum), draw z_i, n_dz += 1;
 * l_d = sum_i ln((1/R) sum_r p_i^r).  Uniforms: Philox stream 5, counter (token, iteration, 5 << 24 | r).
 *
 * Two modes, as in oracle/lda_oracle.c:
 *   contract -- the fp32 / fp64 arithmetic of the kernels, bit for bit: the lane-contiguous tree of DESIGN.md 4.2 and
 *               the contract ln of oracle/contract_math.inc (included unchanged);
 *   faithful -- double precision, sequential sums over k, the reference's subtractive walk, libm log.
 * The lane tree and Philox are restated here; tests/test_oracle_heldout.py checks both against oracle/ (the same draw
 * as oracle_draw_topic_contract, the Philox known answers).
 *
 * Build: gcc -O2 -std=gnu11 -fPIC -shared -ffp-contract=off -fno-fast-math -mfma -fopenmp (no fast-math!)
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

enum { STREAM_HELDOUT = 5 };

static inline void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1)
{
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c[0];
        uint64_t p1 = (uint64_t)0xCD9E8D57u * c[2];
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
}

/* the fp64 contract math (c_ln_f64), the double instantiation of oracle/lda_oracle.c */
#define REAL double
#define UINT uint64_t
#define SINT int64_t
#define SFX(name) name##_f64
#define R(x) ((double)(x))
#define MANT_BITS 52
#define EXP_BIAS 1023
#define SQRT_HALF_BITS 0x3fe6a09e667f3bcdull
#define MANT_MASK 0x000fffffffffffffull
#define MIN_NORMAL_BITS 0x0010000000000000ull
#define DENORM_SCALE 0x1p54
#define DENORM_SHIFT 54
#define FMA fma
#define SQRT sqrt
#define RINT rint
#define LN_TERMS 11
#define EXP_DEG 14
#define TRIG_DEG 9
#define EXP_CUTOFF (-746.0)
#define LN2_HI 0x1.62e42feep-1
#define LN2_LO 0x1.a39ef35793c76p-33
#define UNI(w) (((double)(w) + 0.5) * 0x1p-32)
#define ANG_FRAC(w, odd) \
    (((double)(((w) & 0x1fffffffu) ^ ((odd) ? 0x1fffffffu : 0u)) + 0.5) * 0x1p-29)
#include "../oracle/contract_math.inc"

void heldout_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4])
{
    uint32_t c[4] = {ctr[0], ctr[1], ctr[2], ctr[3]};
    philox4x32_10(c, key[0], key[1]);
    memcpy(out, c, sizeof c);
}

double heldout_c_ln_f64(double x) { return c_ln_f64(x); }

/* The categorical draw of DESIGN.md 4.2 for K <= 1024: lane l of 32 owns the L = 4*NT consecutive topics
 * [l*L, (l+1)*L); lane-local sequential fma prefix (padding topics leave it unchanged), Kogge-Stone scan of the 32
 * lane totals, S = scan[31]; u = U*S, first lane with scan >= u, r = u - scan[l-1], first element with prefix >= r.
 * Returns the topic and, in *S_out, the total S. */
static int lanes_tiles(int32_t K) { return K <= 128 ? 1 : K <= 256 ? 2 : K <= 512 ? 4 : 8; }

int32_t heldout_draw_lanes(const float *a, const float *phirow, int32_t K, float U, float *S_out)
{
    const int L = 4 * lanes_tiles(K);
    float p[32][32], x[32], y[32];
    for (int l = 0; l < 32; ++l) {
        float run = 0.0f;
        for (int m = 0; m < L; ++m) {
            int k = l * L + m;
            if (m == 0) run = (k < K) ? a[k] * phirow[k] : 0.0f;
            else if (k < K) run = fmaf(a[k], phirow[k], run);
            p[l][m] = run;
        }
        x[l] = run;
    }
    for (int off = 1; off < 32; off <<= 1) {
        for (int l = 0; l < 32; ++l) y[l] = (l >= off) ? x[l] + x[l - off] : x[l];
        memcpy(x, y, sizeof x);
    }
    const float S = x[31];
    if (S_out) *S_out = S;
    const float u = U * S;
    int ls = 31;
    for (int l = 0; l < 32; ++l)
        if (x[l] >= u) { ls = l; break; }
    const float r = u - (ls > 0 ? x[ls - 1] : 0.0f);
    int ms = L - 1;
    for (int m = 0; m < L; ++m)
        if (p[ls][m] >= r) { ms = m; break; }
    const int32_t k = ls * L + ms;
    return k < K ? k : K - 1;
}

static inline float heldout_uniform_f32(uint64_t seed, uint64_t token, uint32_t iteration, uint32_t r)
{
    uint32_t w[4] = {(uint32_t)token, (uint32_t)(token >> 32), iteration, ((uint32_t)STREAM_HELDOUT << 24) | r};
    philox4x32_10(w, (uint32_t)seed, (uint32_t)(seed >> 32));
    return ((float)(w[0] >> 9) + 0.5f) * 0x1p-23f;
}

/* the reference's walk: subtract scores until the sample is used up (the reference overruns instead of clamping) */
static inline int32_t walk_faithful(const double *score, double sum, double U, int32_t K)
{
    double sample = U * sum;
    int32_t nt = -1;
    while (sample > 0.0 && nt < K - 1) {
        nt++;
        sample -= score[nt];
    }
    return nt < 0 ? 0 : nt;
}

static double alpha_sum_of(const double *alpha, int32_t K)
{
    double s = 0.0;
    for (int k = 0; k < K; ++k) s += alpha[k];
    return s;
}

static int64_t longest(int64_t D, const int64_t *doc_off)
{
    int64_t m = 0;
    for (int64_t d = 0; d < D; ++d)
        if (doc_off[d + 1] - doc_off[d] > m) m = doc_off[d + 1] - doc_off[d];
    return m > 0 ? m : 1;
}

/* Test set (doc_off[D+1], tokens; token_base = global index of its first token), model n_wk int32[V][K], n_k int32[K],
 * R particles at `iteration`.  doc_ll[D] receives ln p(w_d); returns their sum in document order. */
double heldout_l2r_contract(int64_t D, const int64_t *doc_off, const int32_t *tokens, int32_t V, int32_t K,
                            const int32_t *n_wk, const int32_t *n_k, const double *alpha, double beta, uint64_t seed,
                            uint32_t iteration, int64_t token_base, int32_t R, double *doc_ll)
{
    float *ph = (float *)malloc(sizeof(float) * (size_t)V * (size_t)K);
    const double vbeta = (double)V * beta, alpha_sum = alpha_sum_of(alpha, K);
    for (int64_t w = 0; w < V; ++w)
        for (int k = 0; k < K; ++k)
            ph[w * K + k] = (float)(((double)n_wk[w * K + k] + beta) / ((double)n_k[k] + vbeta));
    const int64_t max_len = longest(D, doc_off);
#pragma omp parallel
    {
        int32_t *cnt = (int32_t *)malloc(sizeof(int32_t) * (size_t)K);
        float *a = (float *)malloc(sizeof(float) * (size_t)K);
        double *acc = (double *)malloc(sizeof(double) * (size_t)max_len);
#pragma omp for schedule(dynamic, 4)
        for (int64_t d = 0; d < D; ++d) {
            const int64_t t0 = doc_off[d], n = doc_off[d + 1] - t0;
            for (int64_t i = 0; i < n; ++i) acc[i] = 0.0;
            for (int32_t r = 0; r < R; ++r) {
                memset(cnt, 0, sizeof(int32_t) * (size_t)K);
                for (int k = 0; k < K; ++k) a[k] = (float)alpha[k];
                for (int64_t i = 0; i < n; ++i) {
                    const float U = heldout_uniform_f32(seed, (uint64_t)(token_base + t0 + i), iteration, (uint32_t)r);
                    float S = 0.0f;
                    const int32_t k = heldout_draw_lanes(a, ph + (size_t)tokens[t0 + i] * K, K, U, &S);
                    acc[i] = acc[i] + (double)S;   /* particle order */
                    cnt[k] += 1;
                    a[k] = (float)cnt[k] + (float)alpha[k];
                }
            }
            double ll = 0.0;
            for (int64_t i = 0; i < n; ++i) ll = ll + c_ln_f64(acc[i] / ((double)R * ((double)i + alpha_sum)));
            doc_ll[d] = ll;
        }
        free(acc);
        free(a);
        free(cnt);
    }
    free(ph);
    double total = 0.0;
    for (int64_t d = 0; d < D; ++d) total += doc_ll[d];
    return total;
}

double heldout_l2r_faithful(int64_t D, const int64_t *doc_off, const int32_t *tokens, int32_t V, int32_t K,
                            const int32_t *n_wk, const int32_t *n_k, const double *alpha, double beta, uint64_t seed,
                            uint32_t iteration, int64_t token_base, int32_t R, double *doc_ll)
{
    double *ph = (double *)malloc(sizeof(double) * (size_t)V * (size_t)K);
    const double vbeta = (double)V * beta, alpha_sum = alpha_sum_of(alpha, K);
    for (int64_t w = 0; w < V; ++w)
        for (int k = 0; k < K; ++k) ph[w * K + k] = ((double)n_wk[w * K + k] + beta) / ((double)n_k[k] + vbeta);
    const int64_t max_len = longest(D, doc_off);
#pragma omp parallel
    {
        int32_t *cnt = (int32_t *)malloc(sizeof(int32_t) * (size_t)K);
        double *score = (double *)malloc(sizeof(double) * (size_t)K);
        double *prob = (double *)malloc(sizeof(double) * (size_t)max_len);
#pragma omp for schedule(dynamic, 4)
        for (int64_t d = 0; d < D; ++d) {
            const int64_t t0 = doc_off[d], n = doc_off[d + 1] - t0;
            for (int64_t i = 0; i < n; ++i) prob[i] = 0.0;
            for (int32_t r = 0; r < R; ++r) {
                memset(cnt, 0, sizeof(int32_t) * (size_t)K);
                for (int64_t i = 0; i < n; ++i) {
                    const double *row = ph + (size_t)tokens[t0 + i] * K;
                    double sum = 0.0;
                    for (int k = 0; k < K; ++k) { score[k] = ((double)cnt[k] + alpha[k]) * row[k]; sum += score[k]; }
                    prob[i] += sum / ((double)i + alpha_sum);
                    const double U = (double)heldout_uniform_f32(seed, (uint64_t)(token_base + t0 + i), iteration, (uint32_t)r);
                    cnt[walk_faithful(score, sum, U, K)] += 1;
                }
            }
            double ll = 0.0;
            for (int64_t i = 0; i < n; ++i) ll += log(prob[i] / (double)R);
            doc_ll[d] = ll;
        }
        free(prob);
        free(score);
        free(cnt);
    }
    free(ph);
    double total = 0.0;
    for (int64_t d = 0; d < D; ++d) total += doc_ll[d];
    return total;
}
