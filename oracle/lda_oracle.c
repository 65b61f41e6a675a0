/*
 * oracle/lda_oracle.c -- TEST INFRASTRUCTURE ONLY.  See lda_oracle.h for scope and the
 * "parity unpinned" statement.  Every function cites the reference file:line it follows
 * (paths relative to /root/reference/src/main/java/cc/mallet/).
 *
 * Build: make -C oracle   (gcc -O2 -ffp-contract=off -mfma -fopenmp; no fast-math!)
 */
#include "lda_oracle.h"

#include <float.h>
#include <math.h>
#include <omp.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

/* ------------------------------------------------------------------------------------------
 * Philox4x32-10 (Salmon et al., SC'11).  Injected in place of the reference's unseedable
 * ThreadLocalRandom / XORShiftRandom (util/ParallelRandoms.java:16-24, util/XORShiftRandom.java:7).
 * ------------------------------------------------------------------------------------------ */
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

void oracle_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4])
{
    uint32_t c[4] = {ctr[0], ctr[1], ctr[2], ctr[3]};
    philox4x32_10(c, key[0], key[1]);
    memcpy(out, c, sizeof c);
}

/* ------------------------------------------------------------------------------------------
 * Contract math, two instantiations
 * ------------------------------------------------------------------------------------------ */
#define REAL float
#define UINT uint32_t
#define SINT int32_t
#define SFX(name) name##_f32
#define R(x) ((float)(x))
#define MANT_BITS 23
#define EXP_BIAS 127
#define SQRT_HALF_BITS 0x3f3504f3u
#define MANT_MASK 0x007fffffu
#define MIN_NORMAL_BITS 0x00800000u
#define DENORM_SCALE 0x1p23f
#define DENORM_SHIFT 23
#define FMA fmaf
#define SQRT sqrtf
#define RINT rintf
#define LN_TERMS 5
#define EXP_DEG 7
#define TRIG_DEG 5
#define EXP_CUTOFF (-104.0f)
#define LN2_HI 0x1.62ep-1f
#define LN2_LO 0x1.0bfbe8p-15f
#define UNI(w) (((float)((w) >> 9) + 0.5f) * 0x1p-23f)
#define ANG_FRAC(w, odd) \
    (((float)((((w) >> 6) & 0x7fffffu) ^ ((odd) ? 0x7fffffu : 0u)) + 0.5f) * 0x1p-23f)
#include "contract_math.inc"
#undef REAL
#undef UINT
#undef SINT
#undef SFX
#undef R
#undef MANT_BITS
#undef EXP_BIAS
#undef SQRT_HALF_BITS
#undef MANT_MASK
#undef MIN_NORMAL_BITS
#undef DENORM_SCALE
#undef DENORM_SHIFT
#undef FMA
#undef SQRT
#undef RINT
#undef LN_TERMS
#undef EXP_DEG
#undef TRIG_DEG
#undef EXP_CUTOFF
#undef LN2_HI
#undef LN2_LO
#undef UNI
#undef ANG_FRAC

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
#include "contract_math.inc"
#undef REAL
#undef UINT
#undef SINT
#undef SFX
#undef R
#undef MANT_BITS
#undef EXP_BIAS
#undef SQRT_HALF_BITS
#undef MANT_MASK
#undef MIN_NORMAL_BITS
#undef DENORM_SCALE
#undef DENORM_SHIFT
#undef FMA
#undef SQRT
#undef RINT
#undef LN_TERMS
#undef EXP_DEG
#undef TRIG_DEG
#undef EXP_CUTOFF
#undef LN2_HI
#undef LN2_LO
#undef UNI
#undef ANG_FRAC

#define F32_TRUE_MIN 0x1p-149f

float oracle_c_ln_f32(float x) { return c_ln_f32(x); }
double oracle_c_ln_f64(double x) { return c_ln_f64(x); }
float oracle_c_exp_neg_f32(float y) { return c_exp_neg_f32(y); }
double oracle_c_exp_neg_f64(double y) { return c_exp_neg_f64(y); }
float oracle_c_cos2pi_f32(uint32_t w) { return c_cos2pi_f32(w); }
double oracle_c_cos2pi_f64(uint32_t w) { return c_cos2pi_f64(w); }

float oracle_c_gamma_f32(float a, uint64_t seed, uint64_t cell, uint32_t sweep, uint32_t stream)
{
    return c_gamma_f32(a, (uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)cell,
                       (uint32_t)(cell >> 32), sweep, stream, NULL);
}
double oracle_c_gamma_f64(double a, uint64_t seed, uint64_t cell, uint32_t sweep, uint32_t stream)
{
    return c_gamma_f64(a, (uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)cell,
                       (uint32_t)(cell >> 32), sweep, stream, NULL);
}

/* ------------------------------------------------------------------------------------------
 * Faithful Gamma: the reference's control flow in double with libm
 * (util/ParallelRandoms.java:60-70,148-159), uniforms/normal from the same Philox words the
 * contract uses.  variant 32: 23-bit uniforms and 26-bit angle (the fp32 contract's inputs);
 * variant 64: 32-bit uniforms and angle.
 * ------------------------------------------------------------------------------------------ */
static inline double f_uniform(uint32_t w, int variant)
{
    return variant == 32 ? ((double)(w >> 9) + 0.5) * 0x1p-23 : ((double)w + 0.5) * 0x1p-32;
}
static inline double f_turn(uint32_t w, int variant)
{
    /* the angle (in turns) whose cosine the contract evaluates */
    if (variant == 32) {
        uint32_t o = w >> 29, b = (w >> 6) & 0x7fffffu;
        return ((double)o + ((double)b + 0.5) * 0x1p-23) * 0.125;
    }
    return ((double)w + 0.5) * 0x1p-32;
}
static double f_gamma(double a, uint32_t k0, uint32_t k1, uint32_t c0, uint32_t c1, uint32_t c2,
                      uint32_t stream, int variant)
{
    int boost = a < 1.0;
    double aa = boost ? 1.0 + a : a;
    double d = aa - (1.0 / 3.0);
    double c = 1.0 / sqrt(9.0 * d);
    for (uint32_t attempt = 0;; ++attempt) {
        uint32_t w[4] = {c0, c1, c2, (stream << 24) | attempt};
        philox4x32_10(w, k0, k1);
        double u1 = f_uniform(w[0], variant);
        double x = sqrt(-2.0 * log(u1)) * cos(2.0 * M_PI * f_turn(w[1], variant));
        double v = 1.0 + c * x;
        if (v <= 0.0) continue;
        v = v * v * v;
        double u = f_uniform(w[2], variant);
        if (u < (1.0 - 0.0331 * (x * x) * (x * x)) ||
            log(u) < (0.5 * x * x + d * (1.0 - v + log(v)))) {
            double g = d * v;
            if (boost) g = g * pow(f_uniform(w[3], variant), 1.0 / a);
            return g;
        }
    }
}
double oracle_f_gamma(double a, uint64_t seed, uint64_t cell, uint32_t sweep, uint32_t stream,
                      int variant)
{
    return f_gamma(a, (uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)cell,
                   (uint32_t)(cell >> 32), sweep, stream, variant);
}

/* ------------------------------------------------------------------------------------------
 * java.util.Random (JDK 8 specification) -- the reference draws the initial z with
 * MALLET Randoms(seed).nextInt(numTopics) in document order, token order
 * (topics/UncollapsedParallelLDA.java:398-406,458-460; topics/ModifiedSimpleLDA.java:137,153-156).
 * ------------------------------------------------------------------------------------------ */
typedef struct { uint64_t s; } jrandom;
static void jr_seed(jrandom *r, int64_t seed) { r->s = ((uint64_t)seed ^ 0x5DEECE66Dull) & ((1ull << 48) - 1); }
static int32_t jr_next(jrandom *r, int bits)
{
    r->s = (r->s * 0x5DEECE66Dull + 0xBull) & ((1ull << 48) - 1);
    return (int32_t)(uint32_t)(r->s >> (48 - bits));
}
static int32_t jr_next_int(jrandom *r, int32_t bound)
{
    int32_t x = jr_next(r, 31);
    int32_t m = bound - 1;
    if ((bound & m) == 0) return (int32_t)(((int64_t)bound * (int64_t)x) >> 31);
    for (int32_t u = x;; u = jr_next(r, 31)) {
        x = u % bound;
        /* Java: u - x + m < 0 in wrapping int arithmetic */
        int32_t t = (int32_t)((uint32_t)u - (uint32_t)x + (uint32_t)m);
        if (t >= 0) break;
    }
    return x;
}
void oracle_java_random_next_ints(int64_t seed, int32_t bound, int64_t n, int32_t *out)
{
    jrandom r; jr_seed(&r, seed);
    for (int64_t i = 0; i < n; ++i) out[i] = jr_next_int(&r, bound);
}
void oracle_java_random_raw_ints(int64_t seed, int64_t n, int32_t *out)
{
    jrandom r; jr_seed(&r, seed);
    for (int64_t i = 0; i < n; ++i) out[i] = jr_next(&r, 32);
}

/* ------------------------------------------------------------------------------------------
 * Counts.  reference: topics/UncollapsedParallelLDA.java:1797-1830 (setZIndicators rebuild),
 * :471-482 (updateTypeTopicCount: both layouts + tokensPerTopic).  One [V][K] layout here.
 * Returns non-zero on an out-of-range topic/type (the reference would throw).
 * ------------------------------------------------------------------------------------------ */
int oracle_rebuild_counts(int64_t N, const int32_t *tokens, const int32_t *z, int32_t V, int32_t K,
                          int32_t *n_wk, int32_t *n_k)
{
    memset(n_wk, 0, sizeof(int32_t) * (size_t)V * (size_t)K);
    memset(n_k, 0, sizeof(int32_t) * (size_t)K);
    for (int64_t i = 0; i < N; ++i) {
        int32_t w = tokens[i], k = z[i];
        if (w < 0 || w >= V || k < 0 || k >= K) return 1;
        n_wk[(size_t)w * K + k] += 1;
        n_k[k] += 1;
    }
    return 0;
}

/* reference: topics/ModifiedSimpleLDA.java:536-547 (getDocumentTopicMatrix) */
void oracle_doc_topic_counts(int64_t D, const int64_t *doc_off, const int32_t *z, int32_t K,
                             int32_t *n_dk)
{
    memset(n_dk, 0, sizeof(int32_t) * (size_t)D * (size_t)K);
    for (int64_t d = 0; d < D; ++d)
        for (int64_t i = doc_off[d]; i < doc_off[d + 1]; ++i) n_dk[(size_t)d * K + z[i]] += 1;
}

/* ------------------------------------------------------------------------------------------
 * Contract categorical draw (DESIGN.md section 4.2).  Restates the reference's
 *   sum = sum_k score_k; sample = U*sum; walk k until sample - cumsum_k <= 0
 * (topics/LDAGroupedGibbsSampler.java:96-113, topics/UncollapsedParallelLDA.java:1507-1526)
 * as "first k with cumsum_k >= U*sum" over a fixed fp32 prefix tree:
 *   tile = 128 topics, lane l of 32 owns 4 consecutive topics of the tile; lane-local sequential
 *     prefix p0 = s0, p_i = fma(a_i, phi_i, p_{i-1}), lane total t = p3;
 *   tile totals, 8 tiles at a time, by a distributed butterfly over the 32 lanes: xor 16 (lanes
 *     with bit 4 clear keep tiles 0-3, the others tiles 4-7), xor 8 (2 tiles kept), xor 4 (1 tile
 *     kept: lane l now works for tile (l>>2)&7), xor 2, xor 1;
 *   cumulative tile totals: Kogge-Stone over the tile index (lane offsets 4, 8, 16), plus the
 *     carry of the previous groups of 8 tiles;
 *   inside the chosen tile: Kogge-Stone inclusive scan of its 32 lane totals.
 * Search tile -> lane -> element; clamp to K-1.
 * ------------------------------------------------------------------------------------------ */
static int32_t draw_topic_contract_tiles(const float *a, const float *phirow, int32_t K, float U,
                                         float *scratch /* NT*128 + ceil(NT/8)*33 floats */)
{
    int NT = (K + 127) / 128;
    int NG = (NT + 7) / 8;
    float *p = scratch;                 /* [NT][32][4] lane-local prefixes */
    float *Bf = scratch + NT * 128;     /* [NG][32] cumulative tile totals as the lanes hold them */
    float *carry = Bf + NG * 32;        /* [NG] cumulative total before each group */
    for (int j = 0; j < NT; ++j)
        for (int l = 0; l < 32; ++l) {
            float run = 0.0f;
            for (int i = 0; i < 4; ++i) {
                int k = 128 * j + 4 * l + i;
                /* one product, then three fused multiply-adds (padding topics add +0) */
                if (i == 0) run = (k < K) ? a[k] * phirow[k] : 0.0f;
                else if (k < K) run = fmaf(a[k], phirow[k], run);
                p[(j * 32 + l) * 4 + i] = run;
            }
        }
    float cr = 0.0f;
    for (int g = 0; g < NG; ++g) {
        float t[8][32], uA[32][4], vB[32][2], wC[32], wD[32], T[32], x[32], y[32];
        for (int tau = 0; tau < 8; ++tau)
            for (int l = 0; l < 32; ++l) {
                int j = 8 * g + tau;
                t[tau][l] = j < NT ? p[(j * 32 + l) * 4 + 3] : 0.0f;
            }
        for (int l = 0; l < 32; ++l) {
            int hi = (l >> 4) & 1;
            for (int i = 0; i < 4; ++i) uA[l][i] = t[4 * hi + i][l] + t[4 * hi + i][l ^ 16];
        }
        for (int l = 0; l < 32; ++l) {
            int h = (l >> 3) & 1;
            for (int i = 0; i < 2; ++i) vB[l][i] = uA[l][2 * h + i] + uA[l ^ 8][2 * h + i];
        }
        for (int l = 0; l < 32; ++l) { int h = (l >> 2) & 1; wC[l] = vB[l][h] + vB[l ^ 4][h]; }
        for (int l = 0; l < 32; ++l) wD[l] = wC[l] + wC[l ^ 2];
        for (int l = 0; l < 32; ++l) T[l] = wD[l] + wD[l ^ 1];
        memcpy(x, T, sizeof x);
        for (int off = 4; off < 32; off <<= 1) {
            for (int l = 0; l < 32; ++l) y[l] = (l >= off) ? x[l] + x[l - off] : x[l];
            memcpy(x, y, sizeof x);
        }
        carry[g] = cr;
        for (int l = 0; l < 32; ++l) Bf[g * 32 + l] = (g == 0) ? x[l] : cr + x[l];
        cr = Bf[g * 32 + 31];
    }
    float S = cr;
    float u = U * S;
    int js = NT - 1;
    float base = 0.0f;
    int found = 0;
    for (int g = 0; g < NG && !found; ++g)
        for (int l = 0; l < 32; ++l)
            if (Bf[g * 32 + l] >= u) {
                int tau = l >> 2;
                js = 8 * g + tau;
                base = tau > 0 ? Bf[g * 32 + 4 * tau - 1] : carry[g];
                found = 1;
                break;
            }
    if (!found || js > NT - 1) { /* unreachable for finite inputs (u <= S); kept total */
        js = NT - 1;
        int g = js / 8, tau = js % 8;
        base = tau > 0 ? Bf[g * 32 + 4 * tau - 1] : carry[g];
    }
    float r = u - base;
    float x[32], y[32];
    for (int l = 0; l < 32; ++l) x[l] = p[(js * 32 + l) * 4 + 3];
    for (int off = 1; off < 32; off <<= 1) {
        for (int l = 0; l < 32; ++l) y[l] = (l >= off) ? x[l] + x[l - off] : x[l];
        memcpy(x, y, sizeof x);
    }
    int ls = 31;
    for (int l = 0; l < 32; ++l)
        if (x[l] >= r) { ls = l; break; }
    float r2 = r - (ls > 0 ? x[ls - 1] : 0.0f);
    int is = 3;
    for (int i = 0; i < 4; ++i)
        if (p[(js * 32 + ls) * 4 + i] >= r2) { is = i; break; }
    int32_t k = 128 * js + 4 * ls + is;
    return k < K ? k : K - 1;
}

/* ------------------------------------------------------------------------------------------
 * Categorical draw of the contract for K <= 1024 (DESIGN.md 4.2, "lane-contiguous" tree; the
 * register path of the z kernel).  NT = 1, 2, 4 or 8 tiles (the smallest with 128*NT >= K),
 * L = 4*NT; lane l of 32 owns the L CONSECUTIVE topics [l*L, (l+1)*L):
 *   lane-local sequential prefix p_0 = a*phi, p_m = fma(a_m, phi_m, p_{m-1}) (padding topics k >= K
 *     leave the prefix unchanged);
 *   Kogge-Stone inclusive scan of the 32 lane totals (offsets 1, 2, 4, 8, 16): S = scan[31];
 *   u = U*S; lane = first l with scan[l] >= u; r = u - scan[l-1]; element = first m with p_m >= r.
 * Same selection rule as the reference's walk (first k with cumsum_k >= U*sum), natural topic order.
 * S_out (may be NULL) receives S: the held-out estimator averages it.
 * ------------------------------------------------------------------------------------------ */
static int lanes_tiles(int32_t K) { return K <= 128 ? 1 : K <= 256 ? 2 : K <= 512 ? 4 : 8; }

static int32_t draw_topic_contract_lanes(const float *a, const float *phirow, int32_t K, float U, float *S_out)
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
    float S = x[31];
    if (S_out) *S_out = S;
    float u = U * S;
    int ls = 31;
    for (int l = 0; l < 32; ++l)
        if (x[l] >= u) { ls = l; break; }
    float r = u - (ls > 0 ? x[ls - 1] : 0.0f);
    int ms = L - 1;
    for (int m = 0; m < L; ++m)
        if (p[ls][m] >= r) { ms = m; break; }
    int32_t k = ls * L + ms;
    return k < K ? k : K - 1;
}

/* two regimes, like the kernels: K <= 1024 keeps the row in registers (lane-contiguous tree),
 * larger K walks it in shared memory tile by tile (tile tree) */
static int32_t draw_topic_contract(const float *a, const float *phirow, int32_t K, float U, float *scratch)
{
    return K <= 1024 ? draw_topic_contract_lanes(a, phirow, K, U, NULL)
                     : draw_topic_contract_tiles(a, phirow, K, U, scratch);
}

int32_t oracle_draw_topic_contract(const float *a, const float *phirow, int32_t K, float U)
{
    int NT = (K + 127) / 128;
    float *scratch = (float *)malloc(sizeof(float) * (size_t)NT * 161);
    int32_t k = draw_topic_contract(a, phirow, K, U, scratch);
    free(scratch);
    return k;
}

static inline float z_uniform_f32(uint64_t seed, uint64_t token, uint32_t sweep)
{
    uint32_t w[4] = {(uint32_t)token, (uint32_t)(token >> 32), sweep, (uint32_t)ORACLE_STREAM_Z << 24};
    philox4x32_10(w, (uint32_t)seed, (uint32_t)(seed >> 32));
    return ((float)(w[0] >> 9) + 0.5f) * 0x1p-23f;
}
static inline double z_uniform_f64(uint64_t seed, uint64_t token, uint32_t sweep)
{
    /* same 23 bits the contract uses, so faithful and contract walk with the same U */
    return (double)z_uniform_f32(seed, token, sweep);
}
/* held-out evaluation: particle r of the test token at `iteration` (DESIGN.md 4.8); both modes use this fp32 value */
static inline float heldout_uniform_f32(uint64_t seed, uint64_t token, uint32_t iteration, uint32_t r)
{
    uint32_t w[4] = {(uint32_t)token, (uint32_t)(token >> 32), iteration, ((uint32_t)ORACLE_STREAM_HELDOUT << 24) | r};
    philox4x32_10(w, (uint32_t)seed, (uint32_t)(seed >> 32));
    return ((float)(w[0] >> 9) + 0.5f) * 0x1p-23f;
}

/* ------------------------------------------------------------------------------------------
 * GGS theta draw, contract: theta_d ~ Dir(n_d + alpha) from the document's counts BEFORE any of
 * its tokens is resampled (topics/LDAGroupedGibbsSampler.java:60-72); Dirichlet = K Gammas,
 * normalise, floor (types/ParallelDirichlet.java:46-70).  fp32; normalising sum in the lane/tile
 * order of DESIGN.md 4.3 (lane-sequential, then xor-butterfly).  Empty documents are skipped
 * by the reference (LDAGroupedGibbsSampler.java:52-53): their row stays zero.
 * ------------------------------------------------------------------------------------------ */
void oracle_theta_contract(int64_t D, const int64_t *doc_off, const int32_t *z, int32_t K,
                           const double *alpha, uint64_t seed, uint32_t sweep, int64_t doc_base,
                           float *theta)
{
    int NT = (K + 127) / 128;
#pragma omp parallel
    {
        int32_t *cnt = (int32_t *)malloc(sizeof(int32_t) * (size_t)K);
#pragma omp for schedule(dynamic, 16)
        for (int64_t d = 0; d < D; ++d) {
            float *th = theta + (size_t)d * K;
            if (doc_off[d + 1] == doc_off[d]) {
                memset(th, 0, sizeof(float) * (size_t)K);
                continue;
            }
            memset(cnt, 0, sizeof(int32_t) * (size_t)K);
            for (int64_t i = doc_off[d]; i < doc_off[d + 1]; ++i) cnt[z[i]] += 1;
            for (int k = 0; k < K; ++k) {
                float a = (float)cnt[k] + (float)alpha[k];
                uint64_t cell = (uint64_t)(doc_base + d) * (uint64_t)K + (uint64_t)k;
                th[k] = c_gamma_f32(a, (uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)cell,
                                    (uint32_t)(cell >> 32), sweep, ORACLE_STREAM_THETA, NULL);
            }
            float acc[32], t[32];
            for (int l = 0; l < 32; ++l) {
                float s = 0.0f;
                if (K <= 1024) {   /* lane l owns the consecutive topics [l*L, (l+1)*L) */
                    const int L = 4 * lanes_tiles(K);
                    for (int m = 0; m < L; ++m) {
                        int k = l * L + m;
                        if (k < K) s = s + th[k];
                    }
                } else {
                    for (int j = 0; j < NT; ++j)
                        for (int i = 0; i < 4; ++i) {
                            int k = 128 * j + 4 * l + i;
                            if (k < K) s = s + th[k];
                        }
                }
                acc[l] = s;
            }
            for (int off = 16; off >= 1; off >>= 1) {
                for (int l = 0; l < 32; ++l) t[l] = acc[l] + acc[l ^ off];
                memcpy(acc, t, sizeof acc);
            }
            float sum = acc[0];
            if (sum != 0.0f) {
                float inv = 1.0f / sum;   /* one division per document, then K products */
                for (int k = 0; k < K; ++k) {
                    float v = th[k] * inv;
                    th[k] = (v <= 0.0f) ? F32_TRUE_MIN : v;
                }
            }
        }
        free(cnt);
    }
}

/* GGS theta draw, faithful: double, sequential sum, floor at Double.MIN_VALUE
 * (types/ParallelDirichlet.java:53-66); the Gamma shape goes through MALLET's
 * partition*magnitude round trip (ParallelDirichlet.java:55; Dirichlet(double[]) ctor, SURVEY 8c). */
void oracle_theta_faithful(int64_t D, const int64_t *doc_off, const int32_t *z, int32_t K,
                           const double *alpha, uint64_t seed, uint32_t sweep, int64_t doc_base,
                           double *theta)
{
#pragma omp parallel
    {
        int32_t *cnt = (int32_t *)malloc(sizeof(int32_t) * (size_t)K);
#pragma omp for schedule(dynamic, 16)
        for (int64_t d = 0; d < D; ++d) {
            double *th = theta + (size_t)d * K;
            if (doc_off[d + 1] == doc_off[d]) {
                memset(th, 0, sizeof(double) * (size_t)K);
                continue;
            }
            memset(cnt, 0, sizeof(int32_t) * (size_t)K);
            for (int64_t i = doc_off[d]; i < doc_off[d + 1]; ++i) cnt[z[i]] += 1;
            double magnitude = 0.0;
            for (int k = 0; k < K; ++k) magnitude += (double)cnt[k] + (double)(float)alpha[k];
            double sum = 0.0;
            for (int k = 0; k < K; ++k) {
                /* the fp32 contract rounds alpha to float; mirror that input, not the arithmetic */
                double pk = (double)cnt[k] + (double)(float)alpha[k];
                double shape = (pk / magnitude) * magnitude;
                uint64_t cell = (uint64_t)(doc_base + d) * (uint64_t)K + (uint64_t)k;
                th[k] = f_gamma(shape, (uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)cell,
                                (uint32_t)(cell >> 32), sweep, ORACLE_STREAM_THETA, 32);
                sum += th[k];
            }
            if (sum != 0.0)
                for (int k = 0; k < K; ++k) {
                    th[k] /= sum;
                    if (th[k] <= 0.0) th[k] = 0x1p-1074; /* Double.MIN_VALUE */
                }
        }
        free(cnt);
    }
}

/* ------------------------------------------------------------------------------------------
 * z-step, contract mode
 * ------------------------------------------------------------------------------------------ */
/* GGS: score_k = theta_dk * phi[k][w]; tokens independent given theta
 * (topics/LDAGroupedGibbsSampler.java:79-130; the loop never reads localTopicCounts for scoring) */
void oracle_z_ggs_contract(int64_t D, const int64_t *doc_off, const int32_t *tokens, int32_t *z,
                           int32_t K, const float *theta, const float *phiT, uint64_t seed,
                           uint32_t sweep, int64_t token_base)
{
    int NT = (K + 127) / 128;
#pragma omp parallel
    {
        float *scratch = (float *)malloc(sizeof(float) * (size_t)NT * 161);
#pragma omp for schedule(dynamic, 16)
        for (int64_t d = 0; d < D; ++d) {
            const float *th = theta + (size_t)d * K;
            for (int64_t i = doc_off[d]; i < doc_off[d + 1]; ++i) {
                float U = z_uniform_f32(seed, (uint64_t)(token_base + i), sweep);
                z[i] = draw_topic_contract(th, phiT + (size_t)tokens[i] * K, K, U, scratch);
            }
        }
        free(scratch);
    }
}

/* PCGS: score_k = (n_dk^{-i} + alpha_k) * phi[k][w], sequential within a document
 * (topics/UncollapsedParallelLDA.java:1479-1543) */
void oracle_z_pcgs_contract(int64_t D, const int64_t *doc_off, const int32_t *tokens, int32_t *z,
                            int32_t K, const double *alpha, const float *phiT, uint64_t seed,
                            uint32_t sweep, int64_t token_base)
{
    int NT = (K + 127) / 128;
#pragma omp parallel
    {
        float *scratch = (float *)malloc(sizeof(float) * (size_t)NT * 161);
        int32_t *cnt = (int32_t *)malloc(sizeof(int32_t) * (size_t)K);
        float *a = (float *)malloc(sizeof(float) * (size_t)K);
#pragma omp for schedule(dynamic, 16)
        for (int64_t d = 0; d < D; ++d) {
            if (doc_off[d + 1] == doc_off[d]) continue;
            memset(cnt, 0, sizeof(int32_t) * (size_t)K);
            for (int64_t i = doc_off[d]; i < doc_off[d + 1]; ++i) cnt[z[i]] += 1;
            for (int k = 0; k < K; ++k) a[k] = (float)cnt[k] + (float)alpha[k];
            for (int64_t i = doc_off[d]; i < doc_off[d + 1]; ++i) {
                int32_t old = z[i];
                cnt[old] -= 1;
                a[old] = (float)cnt[old] + (float)alpha[old];
                float U = z_uniform_f32(seed, (uint64_t)(token_base + i), sweep);
                int32_t nw = draw_topic_contract(a, phiT + (size_t)tokens[i] * K, K, U, scratch);
                z[i] = nw;
                cnt[nw] += 1;
                a[nw] = (float)cnt[nw] + (float)alpha[nw];
            }
        }
        free(a);
        free(cnt);
        free(scratch);
    }
}

/* ------------------------------------------------------------------------------------------
 * z-step, faithful mode: double scores, sequential sum, subtractive walk, exactly the Java loop
 * ------------------------------------------------------------------------------------------ */
static inline int32_t walk_faithful(const double *score, double sum, double U, int32_t K)
{
    double sample = U * sum;
    int32_t nt = -1;
    while (sample > 0.0 && nt < K - 1) { /* the reference overruns the array instead of clamping */
        nt++;
        sample -= score[nt];
    }
    return nt < 0 ? 0 : nt;
}

void oracle_z_ggs_faithful(int64_t D, const int64_t *doc_off, const int32_t *tokens, int32_t *z,
                           int32_t K, const double *theta, const double *phiT, uint64_t seed,
                           uint32_t sweep, int64_t token_base)
{
#pragma omp parallel
    {
        double *score = (double *)malloc(sizeof(double) * (size_t)K);
#pragma omp for schedule(dynamic, 16)
        for (int64_t d = 0; d < D; ++d) {
            const double *th = theta + (size_t)d * K;
            for (int64_t i = doc_off[d]; i < doc_off[d + 1]; ++i) {
                const double *ph = phiT + (size_t)tokens[i] * K;
                double sum = 0.0;
                for (int k = 0; k < K; ++k) { score[k] = th[k] * ph[k]; sum += score[k]; }
                z[i] = walk_faithful(score, sum, z_uniform_f64(seed, (uint64_t)(token_base + i), sweep), K);
            }
        }
        free(score);
    }
}

void oracle_z_pcgs_faithful(int64_t D, const int64_t *doc_off, const int32_t *tokens, int32_t *z,
                            int32_t K, const double *alpha, const double *phiT, uint64_t seed,
                            uint32_t sweep, int64_t token_base)
{
#pragma omp parallel
    {
        double *score = (double *)malloc(sizeof(double) * (size_t)K);
        int32_t *cnt = (int32_t *)malloc(sizeof(int32_t) * (size_t)K);
#pragma omp for schedule(dynamic, 16)
        for (int64_t d = 0; d < D; ++d) {
            if (doc_off[d + 1] == doc_off[d]) continue;
            memset(cnt, 0, sizeof(int32_t) * (size_t)K);
            for (int64_t i = doc_off[d]; i < doc_off[d + 1]; ++i) cnt[z[i]] += 1;
            for (int64_t i = doc_off[d]; i < doc_off[d + 1]; ++i) {
                const double *ph = phiT + (size_t)tokens[i] * K;
                cnt[z[i]] -= 1;
                double sum = 0.0;
                for (int k = 0; k < K; ++k) { score[k] = ((double)cnt[k] + alpha[k]) * ph[k]; sum += score[k]; }
                int32_t nw = walk_faithful(score, sum, z_uniform_f64(seed, (uint64_t)(token_base + i), sweep), K);
                z[i] = nw;
                cnt[nw] += 1;
            }
        }
        free(cnt);
        free(score);
    }
}

/* ------------------------------------------------------------------------------------------
 * Held-out log-likelihood (DESIGN.md 4.8).  MALLET's MarginalProbEstimator.evaluateLeftToRight
 * without resampling (Wallach et al. 2009), which the reference's MarginalProbEstimatorPlain
 * restates over plain count arrays (topics/UncollapsedParallelLDA.java:604-611,840-844 call it).
 * phihat_kw = (n_wk + beta) / (n_k + V beta); per document and particle r, from n_dk = 0:
 * S_i = sum_k (n_dk + alpha_k) phihat_kw, draw z_i, n_dz += 1;
 * l_d = sum_i ln((1/R) sum_r S_i^r / (i + alpha_sum)).  K <= 1024 (the lane-contiguous draw).
 * ------------------------------------------------------------------------------------------ */
static double alpha_sum_of(const double *alpha, int32_t K)
{
    double s = 0.0;
    for (int k = 0; k < K; ++k) s += alpha[k];
    return s;
}

static int64_t longest_doc(int64_t D, const int64_t *doc_off)
{
    int64_t m = 0;
    for (int64_t d = 0; d < D; ++d)
        if (doc_off[d + 1] - doc_off[d] > m) m = doc_off[d + 1] - doc_off[d];
    return m > 0 ? m : 1;
}

/* contract: fp32 phihat (one fp64 division per cell) and scores, the draw's own S summed over the particles in fp64 in
 * particle order, the contract ln of the fp64 mean */
double oracle_heldout_l2r_contract(int64_t D, const int64_t *doc_off, const int32_t *tokens, int32_t V, int32_t K,
                                   const int32_t *n_wk, const int32_t *n_k, const double *alpha, double beta,
                                   uint64_t seed, uint32_t iteration, int64_t token_base, int32_t R, double *doc_ll)
{
    float *ph = (float *)malloc(sizeof(float) * (size_t)V * (size_t)K);
    const double vbeta = (double)V * beta, alpha_sum = alpha_sum_of(alpha, K);
    for (int64_t w = 0; w < V; ++w)
        for (int k = 0; k < K; ++k)
            ph[w * K + k] = (float)(((double)n_wk[w * K + k] + beta) / ((double)n_k[k] + vbeta));
    const int64_t max_len = longest_doc(D, doc_off);
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
                    const int32_t k = draw_topic_contract_lanes(a, ph + (size_t)tokens[t0 + i] * K, K, U, &S);
                    acc[i] = acc[i] + (double)S;
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

/* faithful: fp64 phihat and scores, sequential sums over k, the reference's walk, libm log; the same uniforms */
double oracle_heldout_l2r_faithful(int64_t D, const int64_t *doc_off, const int32_t *tokens, int32_t V, int32_t K,
                                   const int32_t *n_wk, const int32_t *n_k, const double *alpha, double beta,
                                   uint64_t seed, uint32_t iteration, int64_t token_base, int32_t R, double *doc_ll)
{
    double *ph = (double *)malloc(sizeof(double) * (size_t)V * (size_t)K);
    const double vbeta = (double)V * beta, alpha_sum = alpha_sum_of(alpha, K);
    for (int64_t w = 0; w < V; ++w)
        for (int k = 0; k < K; ++k) ph[w * K + k] = ((double)n_wk[w * K + k] + beta) / ((double)n_k[k] + vbeta);
    const int64_t max_len = longest_doc(D, doc_off);
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

/* ------------------------------------------------------------------------------------------
 * Phi draw, contract (DESIGN.md 4.4): g = Gamma(beta + n_wk) in fp64 (cell = w*K + k), rounded to
 * fp32; per-topic sum S_k in fp64 over the ROUNDED values in a fixed three-level order:
 *   row blocks of 8 words summed sequentially, blocks of one of 8 vocabulary segments summed
 *   sequentially, the 8 segment sums combined as ((0+1)+(2+3))+((4+5)+(6+7));
 * phi = (float)(g32 * (1 / S_k)), floored at the smallest fp32 subnormal.
 * Reference: topics/LDAGroupedGibbsSampler.java:182-192, topics/LDAPartiallyCollapsedGibbsSampler.java:91-101,
 * types/ParallelDirichlet.java:46-70; the initial Phi of every scheme:
 * topics/UncollapsedParallelLDA.java:1287-1294 + types/MarsagliaSparseDirichlet.java:31-55.
 * ------------------------------------------------------------------------------------------ */
#define PHI_ROW_BLOCK 8
#define PHI_SEGMENTS 8
void oracle_phi_contract(int32_t V, int32_t K, const int32_t *n_wk, double beta, uint64_t seed,
                         uint32_t sweep, float *phiT)
{
    int64_t unit = (int64_t)PHI_ROW_BLOCK * PHI_SEGMENTS;
    int64_t Vp = ((int64_t)V + unit - 1) / unit * unit;
    int64_t seg_rows = Vp / PHI_SEGMENTS;
    int64_t blocks_per_seg = seg_rows / PHI_ROW_BLOCK;
    int64_t nblocks = Vp / PHI_ROW_BLOCK;
    double *partial = (double *)calloc((size_t)nblocks * (size_t)K, sizeof(double));
#pragma omp parallel for schedule(dynamic, 4)
    for (int64_t b = 0; b < nblocks; ++b) {
        double *ps = partial + (size_t)b * K;
        for (int64_t w = b * PHI_ROW_BLOCK; w < (b + 1) * PHI_ROW_BLOCK && w < V; ++w)
            for (int k = 0; k < K; ++k) {
                uint64_t cell = (uint64_t)w * (uint64_t)K + (uint64_t)k;
                double a = beta + (double)n_wk[cell];
                double g = c_gamma_f64(a, (uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)cell,
                                       (uint32_t)(cell >> 32), sweep, ORACLE_STREAM_PHI, NULL);
                float g32 = (float)g;
                phiT[cell] = g32;
                ps[k] = ps[k] + (double)g32;
            }
    }
    double *S = (double *)malloc(sizeof(double) * (size_t)K);
    for (int k = 0; k < K; ++k) {
        double seg[PHI_SEGMENTS];
        for (int s = 0; s < PHI_SEGMENTS; ++s) {
            double acc = 0.0;
            for (int64_t b = s * blocks_per_seg; b < (s + 1) * blocks_per_seg; ++b)
                acc = acc + partial[(size_t)b * K + k];
            seg[s] = acc;
        }
        S[k] = ((seg[0] + seg[1]) + (seg[2] + seg[3])) + ((seg[4] + seg[5]) + (seg[6] + seg[7]));
    }
#pragma omp parallel for schedule(static)
    for (int64_t w = 0; w < V; ++w)
        for (int k = 0; k < K; ++k) {
            if (S[k] == 0.0) continue;
            /* one reciprocal per topic, one product per cell (contract 4.4) */
            float v = (float)((double)phiT[(size_t)w * K + k] * (1.0 / S[k]));
            phiT[(size_t)w * K + k] = (v <= 0.0f) ? F32_TRUE_MIN : v;
        }
    free(S);
    free(partial);
}

/* ------------------------------------------------------------------------------------------
 * Poisson Polya-urn Phi draw (SURVEY 8f row 4).  Reference: topics/PolyaUrnSpaliasLDA.java:495-507 ->
 * types/PolyaUrnDirichletFixedCoeffPoisson.java:17-44: X_w = Poisson(beta + n_wk) through
 * types/PoissonFixedCoeffSampler.java:45-51 (alias table over the pmf truncated to [0, 2L) for n < L, the normal
 * approximation of types/PolyaUrnDirichlet.java:102-107 from L on), phi = X / sum X, zeros allowed.
 * Contract (contract_math.cuh c_poisson): one Philox block per cell (stream 4); n < L: inversion by sequential
 * search with one 52-bit uniform; n >= L: floor(sqrt(lambda) x + lambda + 1/2), x = Box-Muller normal, >= 0.
 * ------------------------------------------------------------------------------------------ */
static inline double uniform52(uint32_t hi, uint32_t lo)
{
    uint64_t n = ((uint64_t)hi << 20) | (uint64_t)(lo >> 12);
    return ((double)n + 0.5) * 0x1p-52;
}

static int32_t poisson_contract(double beta, int32_t n, int32_t L, double p0, const uint32_t w[4])
{
    double lambda = beta + (double)n;
    if (n < L) {
        double u = uniform52(w[0], w[1]);
        double p = n == 0 ? p0 : c_exp_neg_f64(-lambda);
        double F = p;
        int32_t k = 0, kmax = 2 * L - 1;
        while (u > F && k < kmax) {
            ++k;
            p = p * (lambda / (double)k);
            F = F + p;
        }
        return k;
    }
    double u1 = ((double)w[0] + 0.5) * 0x1p-32;
    double x = sqrt(-2.0 * c_ln_f64(u1)) * c_cos2pi_f64(w[1]);
    double v = fma(sqrt(lambda), x, lambda) + 0.5;
    double r = floor(v);
    return r > 0.0 ? (int32_t)r : 0;
}

/* the same draw with libm (faithful mode): exp / log / cos from glibc, same uniforms */
static int32_t poisson_faithful(double beta, int32_t n, int32_t L, const uint32_t w[4])
{
    double lambda = beta + (double)n;
    if (n < L) {
        double u = uniform52(w[0], w[1]);
        double p = exp(-lambda), F = p;
        int32_t k = 0, kmax = 2 * L - 1;
        while (u > F && k < kmax) { ++k; p *= lambda / (double)k; F += p; }
        return k;
    }
    double u1 = ((double)w[0] + 0.5) * 0x1p-32;
    double x = sqrt(-2.0 * log(u1)) * cos(2.0 * M_PI * f_turn(w[1], 64));
    long r = lround(floor(sqrt(lambda) * x + lambda + 0.5));
    return r > 0 ? (int32_t)r : 0;
}

int32_t oracle_poisson(double beta, int32_t n, int32_t L, uint64_t seed, uint64_t cell, uint32_t sweep, int faithful)
{
    uint32_t w[4] = {(uint32_t)cell, (uint32_t)(cell >> 32), sweep, (uint32_t)ORACLE_STREAM_POISSON << 24};
    philox4x32_10(w, (uint32_t)seed, (uint32_t)(seed >> 32));
    return faithful ? poisson_faithful(beta, n, L, w) : poisson_contract(beta, n, L, c_exp_neg_f64(-beta), w);
}

void oracle_phi_polya_contract(int32_t V, int32_t K, const int32_t *n_wk, double beta, int32_t L, uint64_t seed,
                               uint32_t sweep, float *phiT)
{
    const double p0 = c_exp_neg_f64(-beta);
    double *S = (double *)calloc((size_t)K, sizeof(double));
    /* the draws are integers: any summation order gives the same (exact) column sums as the kernels' fixed tree */
    for (int64_t w = 0; w < V; ++w)
        for (int k = 0; k < K; ++k) {
            uint64_t cell = (uint64_t)w * (uint64_t)K + (uint64_t)k;
            uint32_t r[4] = {(uint32_t)cell, (uint32_t)(cell >> 32), sweep, (uint32_t)ORACLE_STREAM_POISSON << 24};
            philox4x32_10(r, (uint32_t)seed, (uint32_t)(seed >> 32));
            float x = (float)poisson_contract(beta, n_wk[cell], L, p0, r);
            phiT[cell] = x;
            S[k] += (double)x;
        }
    for (int64_t w = 0; w < V; ++w)
        for (int k = 0; k < K; ++k) {
            if (S[k] == 0.0) continue;   /* a topic that drew nothing keeps its zero row (PolyaUrnDirichletFixedCoeffPoisson.java:33) */
            phiT[(size_t)w * K + k] = (float)((double)phiT[(size_t)w * K + k] * (1.0 / S[k]));
        }
    free(S);
}

void oracle_phi_polya_faithful(int32_t V, int32_t K, const int32_t *n_wk, double beta, int32_t L, uint64_t seed,
                               uint32_t sweep, double *phiT)
{
    for (int k = 0; k < K; ++k) {   /* per topic, as loopOverTopics: draw the row, sum, divide */
        double sum = 0.0;
        for (int64_t w = 0; w < V; ++w) {
            uint64_t cell = (uint64_t)w * (uint64_t)K + (uint64_t)k;
            uint32_t r[4] = {(uint32_t)cell, (uint32_t)(cell >> 32), sweep, (uint32_t)ORACLE_STREAM_POISSON << 24};
            philox4x32_10(r, (uint32_t)seed, (uint32_t)(seed >> 32));
            double x = (double)poisson_faithful(beta, n_wk[cell], L, r);
            phiT[cell] = x;
            sum += x;
        }
        if (sum > 0)
            for (int64_t w = 0; w < V; ++w) phiT[(size_t)w * K + k] /= sum;
    }
}

/* Phi draw, faithful: per topic, V Gammas in double, sequential sum, normalise, floor at
 * Double.MIN_VALUE; shape through partition*magnitude (types/ParallelDirichlet.java:46-70). */
void oracle_phi_faithful(int32_t V, int32_t K, const int32_t *n_wk, double beta, uint64_t seed,
                         uint32_t sweep, double *phiT)
{
#pragma omp parallel for schedule(dynamic, 1)
    for (int k = 0; k < K; ++k) {
        double magnitude = 0.0;
        for (int64_t w = 0; w < V; ++w) magnitude += beta + (double)n_wk[(size_t)w * K + k];
        double sum = 0.0;
        for (int64_t w = 0; w < V; ++w) {
            uint64_t cell = (uint64_t)w * (uint64_t)K + (uint64_t)k;
            double pk = beta + (double)n_wk[cell];
            double shape = (pk / magnitude) * magnitude;
            double g = f_gamma(shape, (uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)cell,
                               (uint32_t)(cell >> 32), sweep, ORACLE_STREAM_PHI, 64);
            phiT[cell] = g;
            sum += g;
        }
        if (sum != 0.0)
            for (int64_t w = 0; w < V; ++w) {
                double v = phiT[(size_t)w * K + k] / sum;
                phiT[(size_t)w * K + k] = (v <= 0.0) ? 0x1p-1074 : v;
            }
    }
}

/* ------------------------------------------------------------------------------------------
 * Log-likelihood.  MALLET 2.0.8 Dirichlet.logGammaStirling, restated from its published form
 * (the jar is absent: pom.xml:130-141; SURVEY 8c): shift z up to >= 2, Stirling series with
 * 1/(12z) - 1/(360 z^3) + 1/(1260 z^5), subtract the logs of the shifted values.
 * ------------------------------------------------------------------------------------------ */
double oracle_log_gamma_stirling(double z)
{
    int shift = 0;
    while (z < 2) { z++; shift++; }
    double result = 0.5 * log(2 * M_PI) + (z - 0.5) * log(z) - z + 1 / (12 * z) -
                    1 / (360 * z * z * z) + 1 / (1260 * z * z * z * z * z);
    while (shift > 0) { shift--; z--; result -= log(z); }
    return result;
}

typedef double (*lg_fn)(double);
static double lgamma_exact(double x) { return lgamma(x); }

/* reference: topics/UncollapsedParallelLDA.java:1644-1758, same summation order */
static double log_likelihood_impl(int64_t D, const int64_t *doc_off, const int32_t *z, int32_t K,
                                  int32_t V, const int32_t *n_wk, const int32_t *n_k,
                                  const double *alpha, double beta, lg_fn lg)
{
    double ll = 0.0, alpha_sum = 0.0;
    int32_t *tc = (int32_t *)calloc((size_t)K, sizeof(int32_t));
    double *tlg = (double *)malloc(sizeof(double) * (size_t)K);
    for (int k = 0; k < K; ++k) { tlg[k] = lg(alpha[k]); alpha_sum += alpha[k]; }
    for (int64_t d = 0; d < D; ++d) {
        for (int64_t i = doc_off[d]; i < doc_off[d + 1]; ++i) tc[z[i]]++;
        for (int k = 0; k < K; ++k)
            if (tc[k] > 0) ll += lg(alpha[k] + tc[k]) - tlg[k];
        ll -= lg(alpha_sum + (double)(doc_off[d + 1] - doc_off[d]));
        memset(tc, 0, sizeof(int32_t) * (size_t)K);
    }
    ll += (double)D * lg(alpha_sum);
    int64_t nnz = 0;
    for (int64_t w = 0; w < V; ++w)
        for (int k = 0; k < K; ++k) {
            int32_t c = n_wk[(size_t)w * K + k];
            if (c == 0) continue;
            nnz++;
            ll += lg(beta + c);
        }
    for (int k = 0; k < K; ++k) ll -= lg(beta * V + n_k[k]);
    ll += lg(beta * V) * K;
    ll -= lg(beta) * (double)nnz;
    free(tlg);
    free(tc);
    return ll;
}
double oracle_log_likelihood(int64_t D, const int64_t *doc_off, const int32_t *z, int32_t K,
                             int32_t V, const int32_t *n_wk, const int32_t *n_k,
                             const double *alpha, double beta)
{
    return log_likelihood_impl(D, doc_off, z, K, V, n_wk, n_k, alpha, beta, oracle_log_gamma_stirling);
}
double oracle_log_likelihood_lgamma(int64_t D, const int64_t *doc_off, const int32_t *z, int32_t K,
                                    int32_t V, const int32_t *n_wk, const int32_t *n_k,
                                    const double *alpha, double beta)
{
    return log_likelihood_impl(D, doc_off, z, K, V, n_wk, n_k, alpha, beta, lgamma_exact);
}

/* reference: topics/UncollapsedParallelLDA.java:1573-1634 (computeLogPosterior), summation order kept:
 * per document, (topic, type) pairs in topic-major order; then the theta term; finally the
 * (beta-1) sum over all K*V cells topic-major. */
typedef struct { int32_t k, w; } kw_pair;
static int kw_cmp(const void *a, const void *b)
{
    const kw_pair *x = (const kw_pair *)a, *y = (const kw_pair *)b;
    if (x->k != y->k) return x->k < y->k ? -1 : 1;
    return x->w < y->w ? -1 : (x->w > y->w);
}
double oracle_log_posterior(int64_t D, const int64_t *doc_off, const int32_t *tokens,
                            const int32_t *z, int32_t K, int32_t V, const double *theta,
                            const double *phiT, const double *alpha, double beta)
{
    const double EPS = 1e-12;
    double lp = 0.0;
    int64_t maxlen = 0;
    for (int64_t d = 0; d < D; ++d)
        if (doc_off[d + 1] - doc_off[d] > maxlen) maxlen = doc_off[d + 1] - doc_off[d];
    kw_pair *pairs = (kw_pair *)malloc(sizeof(kw_pair) * (size_t)(maxlen + 1));
    double *ndj = (double *)malloc(sizeof(double) * (size_t)K);
    for (int64_t d = 0; d < D; ++d) {
        int64_t len = doc_off[d + 1] - doc_off[d];
        for (int k = 0; k < K; ++k) ndj[k] = 0.0;
        for (int64_t i = 0; i < len; ++i) {
            pairs[i].k = z[doc_off[d] + i];
            pairs[i].w = tokens[doc_off[d] + i];
            ndj[pairs[i].k] += 1.0;
        }
        qsort(pairs, (size_t)len, sizeof(kw_pair), kw_cmp);
        for (int64_t i = 0; i < len;) {
            int64_t j = i;
            while (j < len && pairs[j].k == pairs[i].k && pairs[j].w == pairs[i].w) ++j;
            lp += (double)(j - i) * log(phiT[(size_t)pairs[i].w * K + pairs[i].k] + EPS);
            i = j;
        }
        for (int k = 0; k < K; ++k)
            lp += (ndj[k] + alpha[k] - 1.0) * log(theta[(size_t)d * K + k] + EPS);
    }
    double bm1 = beta - 1.0;
    for (int k = 0; k < K; ++k)
        for (int64_t w = 0; w < V; ++w) lp += bm1 * log(phiT[(size_t)w * K + k] + EPS);
    free(ndj);
    free(pairs);
    return lp;
}

/* ------------------------------------------------------------------------------------------
 * Whole sweeps.  Order of one iteration: topics/UncollapsedParallelLDA.java:645-693
 * (loopOverBatches -> updateCounts -> samplePhi).
 * ------------------------------------------------------------------------------------------ */
void oracle_sweeps_contract(int scheme, int64_t D, int32_t V, int32_t K, const int64_t *doc_off,
                            const int32_t *tokens, int32_t *z, const double *alpha, double beta,
                            uint64_t seed, uint32_t first_sweep, int32_t n_sweeps, float *phiT,
                            float *theta, int32_t *n_wk, int32_t *n_k)
{
    int64_t N = doc_off[D];
    float *th = theta;
    if (scheme == ORACLE_GGS && !th) th = (float *)malloc(sizeof(float) * (size_t)D * (size_t)K);
    for (int32_t s = 0; s < n_sweeps; ++s) {
        uint32_t it = first_sweep + (uint32_t)s;
        if (scheme == ORACLE_GGS) {
            oracle_theta_contract(D, doc_off, z, K, alpha, seed, it, 0, th);
            oracle_z_ggs_contract(D, doc_off, tokens, z, K, th, phiT, seed, it, 0);
        } else {
            oracle_z_pcgs_contract(D, doc_off, tokens, z, K, alpha, phiT, seed, it, 0);
        }
        oracle_rebuild_counts(N, tokens, z, V, K, n_wk, n_k);
        oracle_phi_contract(V, K, n_wk, beta, seed, it, phiT);
    }
    if (th != theta) free(th);
}

void oracle_sweeps_faithful(int scheme, int64_t D, int32_t V, int32_t K, const int64_t *doc_off,
                            const int32_t *tokens, int32_t *z, const double *alpha, double beta,
                            uint64_t seed, uint32_t first_sweep, int32_t n_sweeps, double *phiT,
                            double *theta, int32_t *n_wk, int32_t *n_k)
{
    int64_t N = doc_off[D];
    double *th = theta;
    if (scheme == ORACLE_GGS && !th) th = (double *)malloc(sizeof(double) * (size_t)D * (size_t)K);
    for (int32_t s = 0; s < n_sweeps; ++s) {
        uint32_t it = first_sweep + (uint32_t)s;
        if (scheme == ORACLE_GGS) {
            oracle_theta_faithful(D, doc_off, z, K, alpha, seed, it, 0, th);
            oracle_z_ggs_faithful(D, doc_off, tokens, z, K, th, phiT, seed, it, 0);
        } else {
            oracle_z_pcgs_faithful(D, doc_off, tokens, z, K, alpha, phiT, seed, it, 0);
        }
        oracle_rebuild_counts(N, tokens, z, V, K, n_wk, n_k);
        oracle_phi_faithful(V, K, n_wk, beta, seed, it, phiT);
    }
    if (th != theta) free(th);
}

/* ------------------------------------------------------------------------------------------
 * CPU baseline with the reference's data structures and threading shape.
 *   phi[K][V] topic-major rows (UncollapsedParallelLDA.java:69), so a token touches K rows;
 *   a shared K*V matrix of atomic +-1 deltas (:102,363-368,1547-1557);
 *   fork-join halving of the document range is replaced by an OpenMP dynamic loop over the same
 *   leaf size (document_sampler_split_limit = 100 documents, configuration/LDAConfiguration.java:51);
 *   updateCounts scans all K*V deltas, one topic per task (:1107-1138,1203-1221) -- the reference
 *   runs that on 2 threads (:1085); here it uses n_threads, which favours the baseline;
 *   Phi: one task per topic on n_threads (the reference default is topic_batches=2; BASELINE.md
 *   sets topic_batches = #cores).
 * ------------------------------------------------------------------------------------------ */
void oracle_baseline_sweeps(int scheme, int64_t D, int32_t V, int32_t K, const int64_t *doc_off,
                            const int32_t *tokens, int32_t *z, const double *alpha, double beta,
                            uint64_t seed, int32_t n_sweeps, int32_t n_threads, double *z_seconds,
                            double *phi_seconds)
{
    if (n_threads <= 0) n_threads = omp_get_max_threads();
    size_t KV = (size_t)K * (size_t)V;
    double *phi = (double *)malloc(sizeof(double) * KV);       /* [K][V] */
    int32_t *delta = (int32_t *)calloc(KV, sizeof(int32_t));   /* [K][V] */
    int32_t *ttc = (int32_t *)calloc(KV, sizeof(int32_t));     /* topicTypeCountMapping [K][V] */
    int32_t *n_k = (int32_t *)calloc((size_t)K, sizeof(int32_t));
    int64_t N = doc_off[D];
    for (int64_t i = 0; i < N; ++i) { ttc[(size_t)z[i] * V + tokens[i]]++; n_k[z[i]]++; }
    double zt = 0.0, pt = 0.0;
    for (int32_t s = -1; s < n_sweeps; ++s) {
        if (s >= 0) {
            double t0 = omp_get_wtime();
            int64_t nleaf = (D + 99) / 100;
#pragma omp parallel num_threads(n_threads)
            {
                double *score = (double *)malloc(sizeof(double) * (size_t)K);
                double *th = (double *)malloc(sizeof(double) * (size_t)K);
                int32_t *cnt = (int32_t *)malloc(sizeof(int32_t) * (size_t)K);
#pragma omp for schedule(dynamic, 1)
                for (int64_t leaf = 0; leaf < nleaf; ++leaf) {
                    int64_t d1 = (leaf + 1) * 100 < D ? (leaf + 1) * 100 : D;
                    for (int64_t d = leaf * 100; d < d1; ++d) {
                        if (doc_off[d + 1] == doc_off[d]) continue;
                        memset(cnt, 0, sizeof(int32_t) * (size_t)K);
                        for (int64_t i = doc_off[d]; i < doc_off[d + 1]; ++i) cnt[z[i]]++;
                        if (scheme == ORACLE_GGS) {
                            double sum = 0.0;
                            for (int k = 0; k < K; ++k) {
                                uint64_t cell = (uint64_t)d * (uint64_t)K + (uint64_t)k;
                                th[k] = f_gamma((double)cnt[k] + alpha[k], (uint32_t)seed,
                                                (uint32_t)(seed >> 32), (uint32_t)cell,
                                                (uint32_t)(cell >> 32), (uint32_t)(s + 1),
                                                ORACLE_STREAM_THETA, 64);
                                sum += th[k];
                            }
                            for (int k = 0; k < K; ++k) th[k] /= sum;
                        }
                        for (int64_t i = doc_off[d]; i < doc_off[d + 1]; ++i) {
                            int32_t w = tokens[i], old = z[i];
                            cnt[old]--;
#pragma omp atomic
                            delta[(size_t)old * V + w] -= 1;
                            double sum = 0.0;
                            if (scheme == ORACLE_GGS)
                                for (int k = 0; k < K; ++k) { score[k] = th[k] * phi[(size_t)k * V + w]; sum += score[k]; }
                            else
                                for (int k = 0; k < K; ++k) { score[k] = ((double)cnt[k] + alpha[k]) * phi[(size_t)k * V + w]; sum += score[k]; }
                            int32_t nw = walk_faithful(score, sum, z_uniform_f64(seed, (uint64_t)i, (uint32_t)(s + 1)), K);
                            z[i] = nw;
                            cnt[nw]++;
#pragma omp atomic
                            delta[(size_t)nw * V + w] += 1;
                        }
                    }
                }
                free(cnt); free(th); free(score);
            }
            /* updateCounts: full K*V scan, one topic per task */
#pragma omp parallel for schedule(dynamic, 1) num_threads(n_threads)
            for (int k = 0; k < K; ++k)
                for (int64_t w = 0; w < V; ++w) {
                    int32_t dl = delta[(size_t)k * V + w];
                    if (dl != 0) { ttc[(size_t)k * V + w] += dl; n_k[k] += dl; delta[(size_t)k * V + w] = 0; }
                }
            zt += omp_get_wtime() - t0;
        }
        double t1 = omp_get_wtime();
#pragma omp parallel for schedule(dynamic, 1) num_threads(n_threads)
        for (int k = 0; k < K; ++k) {
            double sum = 0.0;
            double *row = phi + (size_t)k * V;
            for (int64_t w = 0; w < V; ++w) {
                uint64_t cell = (uint64_t)w * (uint64_t)K + (uint64_t)k;
                row[w] = f_gamma(beta + (double)ttc[(size_t)k * V + w], (uint32_t)seed,
                                 (uint32_t)(seed >> 32), (uint32_t)cell, (uint32_t)(cell >> 32),
                                 (uint32_t)(s + 1), ORACLE_STREAM_PHI, 64);
                sum += row[w];
            }
            for (int64_t w = 0; w < V; ++w) { row[w] /= sum; if (row[w] <= 0) row[w] = 0x1p-1074; }
        }
        if (s >= 0) pt += omp_get_wtime() - t1; /* the initial Phi (s = -1) is set-up, not timed */
    }
    *z_seconds = zt;
    *phi_seconds = pt;
    free(n_k); free(ttc); free(delta); free(phi);
}

int oracle_max_threads(void) { return omp_get_max_threads(); }
/* torchrun exports OMP_NUM_THREADS=1 to its workers: the checker on rank 0 may take the host back */
void oracle_set_num_threads(int n) { if (n > 0) omp_set_num_threads(n); }
