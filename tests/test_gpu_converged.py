"""The regime long runs spend their sweeps in, against the contract oracle and against scipy.

Every other GPU parity test starts from a random z and runs a few sweeps, so its counts stay near uniform: n_dk ~ N_d / K,
n_wk ~ count(w) / K.  A chain that has mixed looks different: documents dominated by one or two topics, frequent word types
in a few topics with n_wk in the thousands to millions, most zero-count theta cells at the 2^-149 floor, the Polya urn on
its normal branch, short sparse topic lists.  This file checks that regime:

1. whole sweeps from a burned-in state (a few hundred device sweeps on an LDA-generated corpus), bit-exact;
2. whole sweeps from a planted state with extreme counts (n_wk ~ 2e6, n_dk ~ 6e4), bit-exact, and the initial Phi within
   1e-5 of the faithful (double, libm) draw on the same uniforms;
3. Dirichlet marginals at large shapes (theta at fp32 shape 12 000, Phi at fp64 shape 4 096) against scipy's Beta
   distribution -- an independent reference, so it also sees a flaw the kernels and the oracle would share;
4. the count histograms with fewer bins than the largest count, and the log-likelihood, on the planted state.

Each test asserts the regime it claims (statistics of the state it checked), so that a change of corpus or seed cannot
quietly turn it into an early-sweep test."""
import numpy as np
import pytest

from test_gpu_edges import _check_sweeps, _sampler

pytestmark = pytest.mark.gpu

FLOOR = 2.0 ** -149
BURN_IN = 200


def _doc_stats(oracle, off, z, K):
    """(mean over non-empty documents of max_k n_dk / N_d, median number of distinct topics per document)"""
    n_dk = oracle.doc_topic_counts(off, z, K)
    lens = np.diff(off)
    ne = lens > 0
    return float((n_dk[ne].max(axis=1) / lens[ne]).mean()), float(np.median((n_dk[ne] > 0).sum(axis=1)))


def _regime(oracle, scheme, off, tokens, z, theta, V, K):
    top, distinct = _doc_stats(oracle, off, z, K)
    n_wk, _ = oracle.rebuild_counts(tokens, z, V, K)
    st = dict(top_share=top, distinct=distinct, nonzero_nwk=float((n_wk > 0).mean()),
              cells_ge_L=int((n_wk >= 100).sum()))
    if scheme == "gpu_ggs":
        st["theta_floor"] = float((theta[np.diff(off) > 0] == np.float32(FLOOR)).mean())
    return st


# ---------------------------------------------------------------------------------------------------------------------
# 1. whole sweeps from a burned-in state
# ---------------------------------------------------------------------------------------------------------------------
# (corpus: documents, vocabulary, mean length; alpha).  GGS K = 100 has NIPS-like long documents (all chunked: theta from
# the stand-alone kernel); the K = 1000 / 1500 corpora mix documents of one work item (fused theta at K = 1000) with
# chunked ones.  GGS runs at alpha = 0.01, where a zero-count theta cell lands on the floor about a third of the time.
CONVERGED = {("gpu_ggs", 100): ((300, 2000, 1267.0), 0.01), ("gpu_ggs", 1000): ((8000, 2000, 40.0), 0.01),
             ("gpu_ggs", 1500): ((8000, 2000, 40.0), 0.01), ("gpu_pcgs", 400): ((8000, 3000, 50.0), 0.05),
             ("gpu_spalias", 1500): ((8000, 2000, 40.0), 0.005), ("gpu_polyaurn", 300): ((8000, 3000, 50.0), 0.05)}


@pytest.mark.parametrize("scheme,K", list(CONVERGED))
def test_sweeps_from_a_burned_in_state(oracle, scheme, K):
    """BURN_IN device sweeps on an LDA-generated corpus (50 true topics, so the chain concentrates), then two more device
    sweeps against the oracle started from the device's z, Phi and iteration.  The regime is asserted against the same
    statistics of the random initial state."""
    import ldagroupedgibbssampler_b200 as L
    (D, V, mean_len), alpha = CONVERGED[(scheme, K)]
    beta, seed = 0.01, 2019
    off, tokens = L.synth_corpus(D, V, mean_len, seed=20190529)
    a = np.full(K, alpha)
    s = _sampler(scheme, off, tokens, V, K, alpha, beta, seed)
    z0 = s.get_z_flat()
    th0 = oracle.theta_contract(off, z0, K, a, seed, 1) if scheme == "gpu_ggs" else None
    s.sample(BURN_IN)
    it = s.getCurrentIteration()
    assert it == BURN_IN
    z = s.get_z_flat()
    phi = s.getPhi().T.astype(np.float32).copy()
    th = s.getTheta().astype(np.float32) if scheme == "gpu_ggs" else None
    init = _regime(oracle, scheme, off, tokens, z0, th0, V, K)
    burnt = _regime(oracle, scheme, off, tokens, z, th, V, K)
    print(f"\n{scheme} K={K} N={len(tokens)} initial {init}\n{scheme} K={K} after {it} sweeps {burnt}")
    s.sample(2)
    _check_sweeps(oracle, s, scheme, off, tokens, z, phi, V, K, a, beta, seed, 2, first_sweep=it + 1)
    s.close()

    # the state the two sweeps started from is the regime this test claims
    assert burnt["top_share"] >= 2 * init["top_share"]
    assert burnt["nonzero_nwk"] <= 0.5 * init["nonzero_nwk"]
    if scheme == "gpu_ggs":
        assert burnt["theta_floor"] >= 0.2 and burnt["theta_floor"] >= init["theta_floor"]
    if scheme == "gpu_polyaurn":
        assert burnt["cells_ge_L"] >= max(200, 2 * init["cells_ge_L"])
    if scheme == "gpu_spalias":
        assert burnt["distinct"] <= 0.5 * init["distinct"]


# ---------------------------------------------------------------------------------------------------------------------
# 2. a planted state with extreme counts
# ---------------------------------------------------------------------------------------------------------------------
HOT_TOKENS, HOT_DOCS = 2 ** 21, 4096          # word type 0: 512 tokens in each of 4 096 documents
BIG_DOC, BIG_TOPIC_TOKENS = 65536, 60000


def _planted(K, V=1000, seed=0):
    """(doc_off, tokens, z): word type 0 with 2^21 tokens, 99.5 % of them in topic K // 3, in 4 096 documents (512 of them
    each, plus 64 filler tokens: sorted, so the z-step meets runs of 512 equal types); one document of 65 536 tokens with
    60 000 in topic K - 1; 1 000 one-topic documents; 2 000 uniform filler documents.  Document order is shuffled."""
    rng = np.random.default_rng(seed)
    docs = []
    hot = K // 3
    for _ in range(HOT_DOCS):
        w = np.concatenate([np.zeros(HOT_TOKENS // HOT_DOCS, np.int32), rng.integers(1, V, 64)])
        zz = np.where(w == 0, np.where(rng.random(len(w)) < 0.995, hot, rng.integers(0, K, len(w))),
                      rng.integers(0, K, len(w)))
        docs.append((w, zz))
    w = rng.integers(1, V, BIG_DOC)
    zz = rng.integers(0, K, BIG_DOC)
    zz[rng.permutation(BIG_DOC)[:BIG_TOPIC_TOKENS]] = K - 1
    docs.append((w, zz))
    for _ in range(1000):
        n = int(rng.integers(1, 49))
        docs.append((rng.integers(0, V, n), np.full(n, rng.integers(0, K))))
    for _ in range(2000):
        n = int(rng.integers(1, 200))
        docs.append((rng.integers(0, V, n), rng.integers(0, K, n)))
    off = np.zeros(len(docs) + 1, np.int64)
    tokens, z = [], []
    for i, d in enumerate(rng.permutation(len(docs))):
        w, zz = docs[d]
        o = np.argsort(w, kind="stable")
        tokens.append(w[o])
        z.append(zz[o])
        off[i + 1] = off[i] + len(w)
    return off, np.concatenate(tokens).astype(np.int32), np.concatenate(z).astype(np.int32), V


def _planted_sampler(oracle, scheme, K, alpha, beta, seed):
    off, tokens, z0, V = _planted(K)
    s = _sampler(scheme, off, tokens, V, K, alpha, beta, seed, init_z=False)
    s.set_z_flat(z0)
    n_wk = s.getTypeTopicMatrix()
    n_dk = s.getDocumentTopicMatrix()
    print(f"\n{scheme} K={K} N={len(tokens)} uploaded: max n_wk {n_wk.max()}, max n_dk {n_dk.max()}, "
          f"one-topic documents {int(((n_dk > 0).sum(axis=1) == 1).sum())}")
    assert n_wk.max() >= 2_000_000 and n_wk[0].argmax() == K // 3
    assert n_dk.max() >= BIG_TOPIC_TOKENS and n_dk[:, K - 1].max() >= BIG_TOPIC_TOKENS
    return s, off, tokens, z0, V, n_wk


@pytest.mark.parametrize("scheme,K", [("gpu_ggs", 100), ("gpu_ggs", 1000), ("gpu_pcgs", 400), ("gpu_spalias", 1500),
                                      ("gpu_polyaurn", 300)])
def test_planted_extreme_counts(oracle, scheme, K):
    """The initial Phi drawn by set_z: the fp64 Gamma at shape ~2e6 (the Polya urn: the Poisson normal branch at
    lambda ~2e6), bit-exact against the contract and within 1e-5 of the faithful draw on the same uniforms.  Then one
    whole sweep: GGS draws theta at fp32 shape ~6e4 in the stand-alone kernel, PCGS scores float(n_dk) + alpha at 6e4."""
    alpha, beta, seed = 50.0 / K, 0.01, 2024
    a = np.full(K, alpha)
    s, off, tokens, z0, V, n_wk = _planted_sampler(oracle, scheme, K, alpha, beta, seed)
    phi0 = s.getPhi().T.astype(np.float32).copy()
    if scheme == "gpu_polyaurn":
        assert np.array_equal(phi0, oracle.phi_polya_contract(n_wk, beta, seed, 0))
        assert np.allclose(phi0, oracle.phi_polya_faithful(n_wk, beta, seed, 0), rtol=1e-5, atol=1e-12)
    else:
        assert np.array_equal(phi0, oracle.phi_contract(n_wk, beta, seed, 0))
        phif = oracle.phi_faithful(n_wk, beta, seed, 0)
        big = phif > 1e-30
        assert ((np.abs(phi0 - phif)[big] / phif[big]) > 1e-5).sum() <= 3          # accept/reject flips only
    s.sample(1)
    _check_sweeps(oracle, s, scheme, off, tokens, z0, phi0, V, K, a, beta, seed, 1)
    if scheme == "gpu_ggs":
        th = s.getTheta()
        thf = oracle.theta_faithful(off, z0, K, a, seed, 1)
        big = thf > 1e-8
        assert (np.abs(th - thf)[big] > 1e-5 * thf[big] + 1e-9).sum() <= 3         # the bar of the parity tests
    s.close()


# ---------------------------------------------------------------------------------------------------------------------
# 3. Dirichlet marginals at large shapes, against scipy
# ---------------------------------------------------------------------------------------------------------------------
def _beta_check(x, a, b):
    """KS p > 1e-5 against Beta(a, b), and the sample mean within 4 standard errors of a / (a + b)."""
    from scipy import stats
    x = np.asarray(x, np.float64)
    p = stats.kstest(x, stats.beta(a, b).cdf).pvalue
    mean, var = a / (a + b), a * b / ((a + b) ** 2 * (a + b + 1))
    z = (x.mean() - mean) / np.sqrt(var / len(x))
    print(f"  Beta({a:.4g}, {b:.4g}), n={len(x)}: KS p = {p:.3g}, mean off by {z:+.2f} sigma")
    assert p > 1e-5
    assert abs(z) < 4


def test_dirichlet_marginals_at_large_shapes():
    """theta and Phi of the device against scipy's Beta distribution, no oracle.
    theta, K = 1000 and 100: 2 000 documents of 20 000 tokens (12 000 at topic 0, 8 000 at topic K - 1, so both ends of
    the row layout are read) are split into work items, so the stand-alone kernel draws their theta; 2 000 documents of
    32 tokens at one mid topic are one work item each, so the z kernel draws theirs.  theta_d ~ Dir(n_d + alpha), so
    theta_d0 ~ Beta(12 000 + alpha, 8 000 + (K - 1) alpha) and the short documents' mid cell ~ Beta(32 + alpha,
    (K - 1) alpha).
    Phi, K = 1000: every topic has the same count column (word 0: 4 096, five words at a few hundred, the rest at 2;
    ~10^4 tokens a topic, ~10^7 in all), so phi[:, w] are K iid draws of Beta(beta + c_w, sum_{v != w} (beta + c_v))."""
    alpha, beta, seed = 0.1, 0.01, 77
    n_long, n_short, len_long, len_short = 2000, 2000, 20000, 32
    V = 500
    off = np.zeros(n_long + n_short + 1, np.int64)
    np.cumsum(np.r_[np.full(n_long, len_long), np.full(n_short, len_short)], out=off[1:])
    N = int(off[-1])
    tokens = np.random.default_rng(1).integers(0, V, N).astype(np.int32)
    for K in (1000, 100):
        mid = K // 2
        z = np.full(N, mid, np.int32)
        zl = z[:n_long * len_long].reshape(n_long, len_long)
        zl[:, :12000] = 0
        zl[:, 12000:] = K - 1
        s = _sampler("gpu_ggs", off, tokens, V, K, alpha, beta, seed, init_z=False)
        s.set_z_flat(z)
        s.sample(1)
        th = s.getTheta()
        s.close()
        print(f"\ntheta, K={K}")
        _beta_check(th[:n_long, 0], 12000 + alpha, 8000 + (K - 1) * alpha)
        _beta_check(th[:n_long, K - 1], 8000 + alpha, 12000 + (K - 1) * alpha)
        _beta_check(th[n_long:, mid], len_short + alpha, (K - 1) * alpha)

    # Phi: topic k holds c_w tokens of every word w, in one document
    K = 1000
    c = np.full(2000, 2, np.int64)
    c[0] = 4096
    c[1:6] = [200, 300, 400, 500, 700]
    V = len(c)
    per_topic = np.repeat(np.arange(V, dtype=np.int32), c)
    tokens = np.tile(per_topic, K)
    z = np.repeat(np.arange(K, dtype=np.int32), len(per_topic))
    off = np.arange(K + 1, dtype=np.int64) * len(per_topic)
    s = _sampler("gpu_ggs", off, tokens, V, K, alpha, beta, seed, init_z=False)
    s.set_z_flat(z)
    assert len(tokens) > 10_000_000
    assert np.array_equal(s.getTypeTopicMatrix(), np.repeat(c[:, None].astype(np.int32), K, axis=1))
    phi = s.getPhi()                                                     # [K][V]
    s.close()
    print(f"Phi, K={K}, {len(tokens)} tokens")
    tot = float((beta + c).sum())
    for w in range(6):
        _beta_check(phi[:, w], beta + c[w], tot - (beta + c[w]))


# ---------------------------------------------------------------------------------------------------------------------
# 4. count histograms and the log-likelihood at large counts
# ---------------------------------------------------------------------------------------------------------------------
def _clipped_hist(values, nbins):
    """numpy's histogram of the values with everything beyond the last bin in the last bin"""
    h = np.bincount(values.ravel(), minlength=nbins).astype(np.int64)
    h[nbins - 1] = h[nbins - 1:].sum()
    return h[:nbins]


def test_histograms_and_log_likelihood_at_large_counts(oracle):
    """ldagpu_get_count_histograms with fewer bins than the largest count (1 000 type bins against n_wk ~ 2e6, 1 000
    document bins against n_dk ~ 6e4): counts beyond the last bin land in it.  The log-likelihood of the planted state
    within 1e-9 of the oracle and within 1e-6 of the statement with the exact lgamma."""
    from ldagroupedgibbssampler_b200._lib import ptr
    K, alpha, beta, seed = 1000, 0.05, 0.01, 3
    s, off, tokens, z0, V, n_wk = _planted_sampler(oracle, "gpu_ggs", K, alpha, beta, seed)
    n_dk = s.getDocumentTopicMatrix()
    nd_bins, nt_bins = 1000, 1000
    assert n_wk.max() > 1000 * nt_bins and n_dk.max() > 50 * nd_bins
    dh, th = np.zeros(nd_bins, np.int64), np.zeros(nt_bins, np.int64)
    s._ck(s._L.ldagpu_get_count_histograms(s._h, nd_bins, ptr(dh), nt_bins, ptr(th)))
    want_th = _clipped_hist(n_wk, nt_bins)
    want_dh = _clipped_hist(n_dk, nd_bins)
    print(f"\nlast type bin {th[-1]} (cells >= {nt_bins - 1}), last document bin {dh[-1]}")
    assert want_th[-1] > 0 and want_dh[-1] > 0
    assert np.array_equal(th, want_th)
    assert np.array_equal(dh, want_dh)

    a = np.full(K, alpha)
    n_k = s.getTopicTotals()
    ll = s.modelLogLikelihood()
    want = oracle.log_likelihood(off, z0, K, V, n_wk, n_k, a, beta)
    exact = oracle.log_likelihood(off, z0, K, V, n_wk, n_k, a, beta, exact_lgamma=True)
    print(f"LL {ll!r}, oracle {want!r}, exact lgamma {exact!r}")
    assert abs(ll - want) <= 1e-9 * abs(want)
    assert abs(ll - exact) <= 1e-6 * abs(exact)
    s.close()
