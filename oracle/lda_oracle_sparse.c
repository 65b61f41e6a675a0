/*
 * oracle/lda_oracle_sparse.c -- TEST INFRASTRUCTURE ONLY (see lda_oracle.h).
 *
 * CPU restatement of the reference's sparse PCGS z-step ("spalias"):
 *   topics/SpaliasUncollapsedParallelLDA.java:39-60   per-type alias table over alpha_k * phi[k][w]
 *   topics/SpaliasUncollapsedParallelLDA.java:124-245 the token loop (sparse cumulative sum over the
 *                                                     topics with n_dk > 0, one uniform per token)
 *   topics/SpaliasUncollapsedParallelLDA.java:262-279 sampleNewTopic (prior vs likelihood branch)
 *   topics/SpaliasUncollapsedParallelLDA.java:295-312 insert / remove of the non-zero topic list
 *   util/OptimizedGentleAliasMethod.java:52-79        alias table construction
 *   util/OptimizedGentleAliasMethod.java:100-107      generateSample(u)
 *
 * Two modes as in lda_oracle.c: "faithful" (double, the Java statements as written) and "contract"
 * (the fixed fp32/fp64 operation order of the CUDA kernels, DESIGN.md 4.6; bit-exact with the GPU).
 * Both use the injected Philox stream (stream 1 = z, counter = global token index): word 0 of a token's block for the
 * branch and the likelihood part, words 1 and 2 for the alias draw, where the reference reuses its one uniform
 * (same distribution, DESIGN.md 4.6).
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "lda_oracle.h"

/* util/OptimizedGentleAliasMethod.java:52-79, in the precision the contract fixes:
 * pi_k = alpha_k * phi_k (fp32 product), normaliser = fp64 sum of the products (32 strided partial sums + butterfly),
 * b_i = pi_i / norm - 1/K in fp64, stack algorithm as written, ps stored as fp32. */
static void alias_build_contract(int32_t K, const float *alpha_f, const float *phirow, float *ps,
                                 int32_t *al, float *type_norm, double *bs, int32_t *lows, int32_t *highs)
{
    /* normaliser: 32 strided fp64 partial sums (lane l takes topics l, l+32, ...), xor butterfly */
    double acc[32], tmp[32];
    for (int l = 0; l < 32; ++l) {
        double s = 0.0;
        for (int k = l; k < K; k += 32) s = s + (double)(alpha_f[k] * phirow[k]);
        acc[l] = s;
    }
    for (int off = 16; off >= 1; off >>= 1) {
        for (int l = 0; l < 32; ++l) tmp[l] = acc[l] + acc[l ^ off];
        memcpy(acc, tmp, sizeof acc);
    }
    const double norm = acc[0];
    *type_norm = (float)norm;
    int low = 0, high = 0;
    const double k1 = 1.0 / (double)K;
    for (int i = 0; i < K; ++i) {
        al[i] = i;
        ps[i] = 0.0f;
        /* an all-zero Phi column (Polya-urn Phi draw) has no prior part: the table is never consulted */
        bs[i] = norm > 0.0 ? ((double)(alpha_f[i] * phirow[i]) / norm) - k1 : 0.0;
        if (bs[i] < 0.0) lows[low++] = i; else highs[high++] = i;
    }
    int steps = 0; /* the reference never increments it (OptimizedGentleAliasMethod.java:67): kept for fidelity */
    while (steps <= K && low > 0 && high > 0) {
        int l = lows[--low];
        int h = highs[high - 1];
        double c = bs[l], d = bs[h];
        bs[l] = 0;
        bs[h] = c + d;
        if (bs[h] <= 0) high--;
        if (bs[h] < 0) lows[low++] = h;
        al[l] = h;
        ps[l] = (float)(1.0 + (double)K * c);
    }
}

void oracle_alias_build_contract(int32_t V, int32_t K, const double *alpha, const float *phiT, float *ps,
                                 int32_t *al, float *type_norm)
{
    float *af = (float *)malloc(sizeof(float) * (size_t)K);
    for (int k = 0; k < K; ++k) af[k] = (float)alpha[k];
#pragma omp parallel
    {
        double *bs = (double *)malloc(sizeof(double) * (size_t)K);
        int32_t *lows = (int32_t *)malloc(sizeof(int32_t) * (size_t)K);
        int32_t *highs = (int32_t *)malloc(sizeof(int32_t) * (size_t)K);
#pragma omp for schedule(dynamic, 16)
        for (int64_t w = 0; w < V; ++w)
            alias_build_contract(K, af, phiT + (size_t)w * K, ps + (size_t)w * K, al + (size_t)w * K,
                                 type_norm + w, bs, lows, highs);
        free(highs); free(lows); free(bs);
    }
    free(af);
}

static inline float uniform23(uint32_t w) { return ((float)(w >> 9) + 0.5f) * 0x1p-23f; }

/* the alias slot floor(w1 K / 2^32) (the kernel's __umulhi): every slot is hit by floor(2^32/K) or ceil(2^32/K) words */
static inline int32_t alias_slot(uint32_t w1, int32_t K) { return (int32_t)(((uint64_t)w1 * (uint32_t)K) >> 32); }

/* util/OptimizedGentleAliasMethod.java:100-107 on two Philox words of the token (DESIGN.md 4.6): slot from w1, keep
 * it if uniform23(w2) <= ps (fp32 compare), else its alias */
int32_t oracle_alias_sample_contract(const float *ps, const int32_t *al, int32_t K, uint32_t w1, uint32_t w2)
{
    const int32_t i = alias_slot(w1, K);
    return uniform23(w2) > ps[i] ? al[i] : i;
}

/* the token's Philox block: word 0 -> branch / likelihood uniform, words 1 and 2 -> alias draw */
static inline void z_words(uint64_t seed, uint64_t token, uint32_t sweep, uint32_t out[4])
{
    uint32_t ctr[4] = {(uint32_t)token, (uint32_t)(token >> 32), sweep, (uint32_t)ORACLE_STREAM_Z << 24};
    uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    oracle_philox4x32_10(ctr, key, out);
}

/* Sparse z-step, contract (DESIGN.md 4.6).  Per token of a document, in order:
 *   remove the token from its topic (swap-remove from the list when the count reaches 0);
 *   s_i = float(cnt_i) * phiT[w][nz_i] over the list in list order; cumulative sums in blocks of 256
 *   entries (8 consecutive entries per lane: lane-local prefix, Kogge-Stone over the 32 lane totals,
 *   block carries added sequentially); sum = last carry;
 *   u = uniform23(word 0); tot = tn + sum; if u < tn / tot: alias draw on words 1 and 2
 *   else: first i with u*tot - tn <= cum_i (last entry if none);
 *   add the token to its new topic (append to the list when it was 0). */
void oracle_z_spalias_contract(int64_t D, const int64_t *doc_off, const int32_t *tokens, int32_t *z,
                               int32_t K, const float *phiT, const float *ps, const int32_t *al,
                               const float *type_norm, uint64_t seed, uint32_t sweep, int64_t token_base)
{
#pragma omp parallel
    {
        int32_t *nz = (int32_t *)malloc(sizeof(int32_t) * (size_t)(K + 32));
        int32_t *cnt = (int32_t *)malloc(sizeof(int32_t) * (size_t)(K + 32));
        float *cum = (float *)malloc(sizeof(float) * (size_t)(K + 256));
#pragma omp for schedule(dynamic, 16)
        for (int64_t d = 0; d < D; ++d) {
            int64_t t0 = doc_off[d], t1 = doc_off[d + 1];
            if (t0 == t1) continue;
            int nnz = 0;
            for (int64_t t = t0; t < t1; ++t) { /* SpaliasUncollapsedParallelLDA.java:147-153 */
                int k = z[t], i;
                for (i = 0; i < nnz; ++i) if (nz[i] == k) break;
                if (i == nnz) { nz[nnz] = k; cnt[nnz] = 0; nnz++; }
                cnt[i]++;
            }
            for (int64_t t = t0; t < t1; ++t) {
                const int32_t w = tokens[t], old = z[t];
                const float *ph = phiT + (size_t)w * K;
                int i;
                for (i = 0; i < nnz; ++i) if (nz[i] == old) break;
                cnt[i]--;
                if (cnt[i] == 0) { nz[i] = nz[nnz - 1]; cnt[i] = cnt[nnz - 1]; nnz--; } /* :295-304 */
                /* cumulative sums, contract 4.6: blocks of 256 list entries; lane l of 32 owns entries
                 * 8l..8l+7 of the block: lane-local sequential prefix q, Kogge-Stone inclusive scan I of the
                 * 32 lane totals, cum = carry + (I[l-1] + q); the carry moves on by the block total */
                float carry = 0.0f, sum = 0.0f;
                for (int b0 = 0; b0 < nnz; b0 += 256) {
                    float q[32][8], x[32], y[32];
                    for (int l = 0; l < 32; ++l)
                        for (int e = 0; e < 8; ++e) {
                            int i = b0 + 8 * l + e;
                            float sv = (i < nnz) ? (float)cnt[i] * ph[nz[i]] : 0.0f;
                            q[l][e] = (e == 0) ? sv : q[l][e - 1] + sv;
                        }
                    for (int l = 0; l < 32; ++l) x[l] = q[l][7];
                    for (int off = 1; off < 32; off <<= 1) {
                        for (int l = 0; l < 32; ++l) y[l] = (l >= off) ? x[l] + x[l - off] : x[l];
                        memcpy(x, y, sizeof x);
                    }
                    for (int l = 0; l < 32; ++l) {
                        float E = l > 0 ? x[l - 1] : 0.0f;
                        for (int e = 0; e < 8; ++e) {
                            int i = b0 + 8 * l + e;
                            if (i < nnz) cum[i] = carry + (E + q[l][e]);
                        }
                    }
                    carry = carry + x[31];
                    sum = carry;
                }
                uint32_t r[4];
                z_words(seed, (uint64_t)(token_base + t), sweep, r);
                const float u = uniform23(r[0]);
                const float tn = type_norm[w];
                const float tot = tn + sum;
                int32_t nw;
                if (!(tot > 0.0f)) {
                    /* no prior mass and no document mass for this type: uniform topic
                     * (topics/PolyaUrnSpaliasLDA.java:275-277) */
                    nw = alias_slot(r[1], K);
                } else if (u < tn / tot || nnz == 0) {
                    nw = oracle_alias_sample_contract(ps + (size_t)w * K, al + (size_t)w * K, K, r[1], r[2]);
                } else {
                    const float ul = u * tot - tn;
                    int slot = nnz - 1;
                    for (int j = 0; j < nnz; ++j) if (ul <= cum[j]) { slot = j; break; }
                    nw = nz[slot];
                }
                z[t] = nw;
                for (i = 0; i < nnz; ++i) if (nz[i] == nw) break;
                if (i == nnz) { nz[nnz] = nw; cnt[nnz] = 0; nnz++; } /* :306-312 */
                cnt[i]++;
            }
        }
        free(cum); free(cnt); free(nz);
    }
}

/* Faithful: the Java statements in double.  phiT [V][K] double, alias tables built in double. */
static void alias_build_faithful(int32_t K, const double *alpha, const double *phirow, double *ps, int32_t *al,
                                 double *type_norm, double *bs, int32_t *lows, int32_t *highs)
{
    double norm = 0.0;
    for (int k = 0; k < K; ++k) norm += phirow[k] * alpha[k];
    *type_norm = norm;
    int low = 0, high = 0;
    const double k1 = 1.0 / K;
    for (int i = 0; i < K; ++i) {
        al[i] = i; ps[i] = 0.0;
        bs[i] = norm > 0.0 ? (phirow[i] * alpha[i] / norm) - k1 : 0.0;
        if (bs[i] < 0.0) lows[low++] = i; else highs[high++] = i;
    }
    while (low > 0 && high > 0) {
        int l = lows[--low], h = highs[high - 1];
        double c = bs[l], d = bs[h];
        bs[l] = 0; bs[h] = c + d;
        if (bs[h] <= 0) high--;
        if (bs[h] < 0) lows[low++] = h;
        al[l] = h; ps[l] = 1.0 + ((double)K) * c;
    }
}

void oracle_z_spalias_faithful(int64_t D, int32_t V, const int64_t *doc_off, const int32_t *tokens, int32_t *z,
                               int32_t K, const double *alpha, const double *phiT, uint64_t seed,
                               uint32_t sweep, int64_t token_base)
{
    double *ps = (double *)malloc(sizeof(double) * (size_t)V * K);
    int32_t *al = (int32_t *)malloc(sizeof(int32_t) * (size_t)V * K);
    double *tn = (double *)malloc(sizeof(double) * (size_t)V);
#pragma omp parallel
    {
        double *bs = (double *)malloc(sizeof(double) * (size_t)K);
        int32_t *lows = (int32_t *)malloc(sizeof(int32_t) * (size_t)K);
        int32_t *highs = (int32_t *)malloc(sizeof(int32_t) * (size_t)K);
#pragma omp for schedule(dynamic, 16)
        for (int64_t w = 0; w < V; ++w)
            alias_build_faithful(K, alpha, phiT + (size_t)w * K, ps + (size_t)w * K, al + (size_t)w * K, tn + w,
                                 bs, lows, highs);
        free(highs); free(lows); free(bs);
    }
#pragma omp parallel
    {
        int32_t *nz = (int32_t *)malloc(sizeof(int32_t) * (size_t)K);
        int32_t *back = (int32_t *)malloc(sizeof(int32_t) * (size_t)K);
        int32_t *cnt = (int32_t *)calloc((size_t)K, sizeof(int32_t));
        double *cum = (double *)malloc(sizeof(double) * (size_t)K);
#pragma omp for schedule(dynamic, 16)
        for (int64_t d = 0; d < D; ++d) {
            int64_t t0 = doc_off[d], t1 = doc_off[d + 1];
            if (t0 == t1) continue;
            int nnz = 0;
            for (int64_t t = t0; t < t1; ++t) {
                int k = z[t];
                if (++cnt[k] == 1) { nz[nnz] = k; back[k] = nnz; nnz++; }
            }
            for (int64_t t = t0; t < t1; ++t) {
                const int32_t w = tokens[t], old = z[t];
                const double *ph = phiT + (size_t)w * K;
                if (--cnt[old] == 0) { int i = back[old]; nz[i] = nz[--nnz]; back[nz[i]] = i; }
                double sum = 0.0;
                for (int i = 0; i < nnz; ++i) { sum += cnt[nz[i]] * ph[nz[i]]; cum[i] = sum; }
                uint32_t r[4];
                z_words(seed, (uint64_t)(token_base + t), sweep, r);
                const double u = (double)uniform23(r[0]);
                const double u_sigma = u * (tn[w] + sum);
                int32_t nw;
                if (!(tn[w] + sum > 0.0)) {
                    nw = alias_slot(r[1], K);   /* PolyaUrnSpaliasLDA.java:275-277 */
                } else if (u < (tn[w] / (tn[w] + sum)) || nnz == 0) {
                    /* the reference rescales u to u' = u + sum*u/tn, slot = floor(u'K), fraction against ps: given
                     * the branch, slot and fraction are independent uniforms, here drawn from words 1 and 2 */
                    const int i = alias_slot(r[1], K);
                    nw = (double)uniform23(r[2]) > ps[(size_t)w * K + i] ? al[(size_t)w * K + i] : i;
                } else {
                    double ul = u_sigma - tn[w];
                    int slot = nnz - 1;
                    for (int i = 0; i < nnz; ++i) if (ul <= cum[i]) { slot = i; break; }
                    nw = nz[slot];
                }
                z[t] = nw;
                if (++cnt[nw] == 1) { nz[nnz] = nw; back[nw] = nnz; nnz++; }
            }
            for (int i = 0; i < nnz; ++i) cnt[nz[i]] = 0;
        }
        free(cum); free(cnt); free(back); free(nz);
    }
    free(tn); free(al); free(ps);
}
