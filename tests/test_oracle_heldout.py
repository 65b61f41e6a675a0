"""The oracle's held-out left-to-right estimator (oracle_heldout_l2r_*, DESIGN.md 4.8): closed forms, exact enumeration,
and the contract mode against the faithful mode.  CPU only."""
import itertools
import math

import numpy as np
import pytest

from conftest import make_corpus

BETA = 0.01


def _counts(rng, V, K, scale=30):
    n_wk = rng.integers(0, scale, (V, K)).astype(np.int32)
    return n_wk, n_wk.sum(axis=0).astype(np.int32)


def _phihat(n_wk, n_k, beta):
    V = n_wk.shape[0]
    return (n_wk.astype(np.float64) + beta) / (n_k.astype(np.float64) + V * beta)


def test_one_token_documents(oracle):
    """A one-token document has no draw to average over: l_d = ln(sum_k alpha_k phihat_kw / alpha_sum) in both modes.
    In contract mode that sum is the total S of the K <= 1024 draw, which must be the fp64 sum within 1e-5 relative at
    every row layout (K from 1 to 1024, padding topics included)."""
    rng = np.random.default_rng(1)
    V = 40
    off = np.arange(V + 1, dtype=np.int64)
    tokens = np.arange(V, dtype=np.int32)
    for K in (7, 1, 3, 31, 100, 128, 129, 256, 257, 400, 512, 513, 1000, 1024):
        n_wk, n_k = _counts(rng, V, K)
        alpha = rng.uniform(0.05, 2.0, K)
        ph = _phihat(n_wk, n_k, BETA)
        closed = np.log((alpha[None, :] * ph).sum(axis=1) / alpha.sum())
        _, f = oracle.heldout_l2r("faithful", off, tokens, n_wk, n_k, alpha, BETA, 5, 3, R=4)
        _, c = oracle.heldout_l2r("contract", off, tokens, n_wk, n_k, alpha, BETA, 5, 3, R=4)
        np.testing.assert_allclose(f, closed, rtol=1e-12, atol=0, err_msg=f"K = {K}")
        if K == 7:
            np.testing.assert_allclose(c, closed, rtol=1e-6, atol=0)   # fp32 phihat and scores
        assert np.abs(np.expm1(c - closed)).max() <= 1e-5, K       # S / sum_k alpha_k phihat_kw - 1


def _enumerate(ph, alpha, words):
    """Exact moments of the estimator's per-particle values p_2 (and p_3) under its own sampling distribution:
    z_1 ~ (alpha + 0) phi_{., w1}, z_2 ~ (alpha + e_{z1}) phi_{., w2}.  Returns p_1 and the list of
    (probability, p_2[, p_3]) over the enumerated draws."""
    K = len(alpha)
    asum = alpha.sum()

    def scores(cnt, w):
        return (cnt + alpha) * ph[w]

    p1 = scores(np.zeros(K), words[0]).sum() / asum
    out = []
    for zs in itertools.product(range(K), repeat=len(words) - 1):
        cnt = np.zeros(K)
        prob, vals = 1.0, []
        for i, w in enumerate(words):
            s = scores(cnt, w)
            if i > 0:
                vals.append(s.sum() / (i + asum))
            if i < len(words) - 1:
                prob *= s[zs[i]] / s.sum()
                cnt[zs[i]] += 1
        out.append((prob, vals))
    return p1, out


@pytest.mark.parametrize("n_tok", [2, 3])
def test_faithful_against_exact_enumeration(oracle, n_tok):
    """R = 4096 particles against exact enumeration over the topics of the earlier tokens (K = 4).  For two tokens the
    particle mean of p_2 is an unbiased estimate of p(w_2 | w_1); for three tokens the estimate exp(l_d) / p_1 =
    mean(p_2) * mean(p_3) is compared with E[p_2] E[p_3], the value it converges to, and sigma comes from the enumerated
    variances and covariance (delta method).  Bound: 5 sigma, on each of 12 documents."""
    rng = np.random.default_rng(7 + n_tok)
    V, K, R = 6, 4, 4096
    n_wk, n_k = _counts(rng, V, K, scale=12)
    alpha = rng.uniform(0.2, 1.5, K)
    ph = _phihat(n_wk, n_k, BETA)
    docs = [rng.integers(0, V, n_tok).astype(np.int32) for _ in range(12)]
    off = np.arange(0, n_tok * len(docs) + 1, n_tok, dtype=np.int64)
    tokens = np.concatenate(docs)
    _, ll = oracle.heldout_l2r("faithful", off, tokens, n_wk, n_k, alpha, BETA, 11, 2, R=R)
    for d, words in enumerate(docs):
        p1, cases = _enumerate(ph, alpha, words)
        pr = np.array([c[0] for c in cases])
        vals = np.array([c[1] for c in cases])      # [cases][n_tok - 1]
        assert abs(pr.sum() - 1.0) < 1e-12
        mean = pr @ vals
        cov = (vals - mean).T @ np.diag(pr) @ (vals - mean)
        est = math.exp(ll[d]) / p1
        if n_tok == 2:
            target, var = mean[0], cov[0, 0]
        else:
            g = np.array([mean[1], mean[0]])            # gradient of m2 * m3
            target, var = mean[0] * mean[1], g @ cov @ g
        sigma = math.sqrt(var / R)
        assert abs(est - target) <= 5 * sigma + 1e-15, (d, est, target, sigma)


def _trained_counts(oracle, off, tokens, V, K, alpha, seed, sweeps):
    z = oracle.java_next_ints(seed, K, int(off[-1]))
    n_wk, _ = oracle.rebuild_counts(tokens, z, V, K)
    phi = oracle.phi_contract(n_wk, BETA, seed, 0)
    st = oracle.sweeps("contract", oracle.PCGS, off, tokens, z, V, K, alpha, BETA, seed, 1, sweeps, phi)
    return st["n_wk"], st["n_k"]


@pytest.mark.parametrize("case", ["cats_K10", "synth_K100", "synth_K400", "synth_K1000"])
def test_contract_against_faithful(oracle, cats, case):
    """Same uniforms, fp32 contract against fp64 faithful, R = 10, on counts after five PCGS sweeps.  Measured on exactly
    these cases when this test was written (cats: its training documents as test set; synthetic: 600 training documents,
    400 ragged test documents with empties).  A document whose draws all agree differs by rounding only, <= 3.3e-9
    relative; a flipped draw moves it by 1e-4 .. 1.5e-3.  Flipped documents: 0 of 23 (cats, K = 10), 0 of 400 (K = 100),
    2 of 400 (K = 400), 6 of 400 (K = 1000).  Totals apart by 1.3e-9, 2.2e-10, 5.0e-6 and 1.1e-6 relative.
    Tolerances: every document within 1e-2 relative, at most 3 % of the documents beyond 1e-6, the total within 5e-5
    relative (ten times the largest measured)."""
    if case == "cats_K10":
        off, tokens = cats
        V, K = int(tokens.max()) + 1, 10
        toff, ttok = off, tokens
    else:
        K = int(case.split("K")[1])
        V = 500
        off, tokens = make_corpus(600, V, 60, 3, sort_docs=False, empty_every=9)
        toff, ttok = make_corpus(400, V, 40, 4, sort_docs=False, empty_every=7)
    alpha = np.full(K, 50.0 / K if K > 10 else 0.1)
    n_wk, n_k = _trained_counts(oracle, off, tokens, V, K, alpha, 7, 5)
    tc, c = oracle.heldout_l2r("contract", toff, ttok, n_wk, n_k, alpha, BETA, 7, 5, R=10)
    tf, f = oracle.heldout_l2r("faithful", toff, ttok, n_wk, n_k, alpha, BETA, 7, 5, R=10)
    empty = np.diff(toff) == 0
    assert np.all(c[empty] == 0.0) and np.all(f[empty] == 0.0)
    rel = np.abs(c - f) / np.maximum(np.abs(f), 1e-300)
    assert rel.max() <= 1e-2
    assert (rel > 1e-6).mean() <= 0.03
    assert abs(tc - tf) <= 5e-5 * abs(tf)
    assert tc == np.cumsum(c)[-1]


def test_evaluation_is_reproducible_and_keyed(oracle):
    """Same iteration: the same values; another iteration or a shifted token base: other uniforms."""
    rng = np.random.default_rng(3)
    V, K = 50, 20
    n_wk, n_k = _counts(rng, V, K)
    off, tokens = make_corpus(30, V, 20, 5, sort_docs=False)
    alpha = np.full(K, 0.3)
    a = oracle.heldout_l2r("contract", off, tokens, n_wk, n_k, alpha, BETA, 9, 4, R=3)
    b = oracle.heldout_l2r("contract", off, tokens, n_wk, n_k, alpha, BETA, 9, 4, R=3)
    c = oracle.heldout_l2r("contract", off, tokens, n_wk, n_k, alpha, BETA, 9, 5, R=3)
    d = oracle.heldout_l2r("contract", off, tokens, n_wk, n_k, alpha, BETA, 9, 4, R=3, token_base=1)
    assert np.array_equal(a[1], b[1])
    assert not np.array_equal(a[1], c[1])
    assert not np.array_equal(a[1], d[1])


def test_test_set_keeps_the_training_alphabet(tmp_path):
    """LDAConfiguration.loadTestDataset: the test set is read with the training alphabet frozen, so words the training
    set does not hold are dropped and the alphabet does not grow; the test_dataset key is read from a .cfg"""
    from ldagroupedgibbssampler_b200.sampler import LDAConfiguration
    train = tmp_path / "train.txt"
    test = tmp_path / "test.txt"
    train.write_text("d1\tX\tthe cat sat on the mat\nd2\tX\ta dog sat\n", encoding="utf-8")
    test.write_text("t1\tX\tthe zebra sat\nt2\tX\tunknown words only\nt3\tX\tdog dog cat\n", encoding="utf-8")
    cfg_file = tmp_path / "run.cfg"
    cfg_file.write_text(f"scheme = gpu_pcgs\ndataset = {train}\ntest_dataset = {test}\n", encoding="utf-8")
    cfg = LDAConfiguration.from_cfg(str(cfg_file))
    assert cfg.test_dataset == str(test)
    tr = cfg.loadDataset()
    n_types = tr.getNumTypes()
    te = cfg.loadTestDataset(tr.getDataAlphabet())
    a = tr.getDataAlphabet()
    assert a.size() == n_types
    assert [list(d) for d in te.docs] == [[a.lookupIndex("the"), a.lookupIndex("sat")], [],
                                          [a.lookupIndex("dog"), a.lookupIndex("dog"), a.lookupIndex("cat")]]
