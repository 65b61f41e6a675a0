"""CPU tests of the oracle's sampler-level functions: the reference tests' own invariants and
distribution checks (SURVEY section 4), contract-vs-faithful agreement, golden regression."""
import numpy as np
import pytest
from scipy import stats

from conftest import make_corpus


# RandomTesting.java:39-89 / SparseDirichletDrawTest.java:15-123: KS p > 1e-5 for the Gamma sampler
@pytest.mark.parametrize("alpha", [0.05, 0.5001, 1.0001, 2.0001, 64.0001, 1024.0001])
def test_gamma_ks(oracle, alpha):
    L = oracle.lib()
    n = 4000
    for fn, arg in ((L.oracle_c_gamma_f32, np.float32(alpha)), (L.oracle_c_gamma_f64, alpha)):
        g = np.array([fn(arg, 2019, i, 7, 3) for i in range(n)])
        assert stats.kstest(g, "gamma", args=(float(arg),)).pvalue > 1e-5
    gf = np.array([L.oracle_f_gamma(alpha, 2019, i, 7, 3, 64) for i in range(n)])
    assert stats.kstest(gf, "gamma", args=(alpha,)).pvalue > 1e-5


def test_gamma_contract_matches_faithful(oracle):
    # same Philox words, contract arithmetic vs libm: identical up to rounding
    L = oracle.lib()
    for a in (0.01, 0.3, 1.0, 7.01, 500.0):
        c = np.array([L.oracle_c_gamma_f64(a, 11, i, 1, 3) for i in range(3000)])
        f = np.array([L.oracle_f_gamma(a, 11, i, 1, 3, 64) for i in range(3000)])
        ok = np.abs(c - f) <= 1e-9 * np.abs(f) + 1e-300
        assert ok.mean() > 0.999      # the rest are accept/reject flips at the test boundary
        a32 = float(np.float32(a))
        c32 = np.array([L.oracle_c_gamma_f32(a32, 11, i, 1, 2) for i in range(3000)], np.float64)
        f32 = np.array([L.oracle_f_gamma(a32, 11, i, 1, 2, 32) for i in range(3000)])
        big = f32 > 1e-20   # below that, fp32 exponent arithmetic of U^(1/a) dominates (DESIGN.md 4.5)
        ok = np.abs(c32 - f32)[big] <= 2e-5 * f32[big]
        assert ok.mean() > 0.995


def test_dirichlet_theta_moments(oracle):
    # Dirichlet(n + alpha) mean = (n_k + alpha_k) / sum; check over many documents (KS on a marginal)
    K, D = 8, 3000
    off = np.arange(D + 1, dtype=np.int64) * 10
    z = np.tile(np.array([0, 0, 0, 1, 1, 2, 3, 3, 3, 3], np.int32), D)
    alpha = np.full(K, 0.5)
    th = oracle.theta_contract(off, z, K, alpha, 5, 1)
    assert np.allclose(th.sum(axis=1), 1.0, atol=1e-5)
    p = np.array([3, 2, 1, 4, 0, 0, 0, 0]) + 0.5
    assert np.allclose(th.mean(axis=0), p / p.sum(), atol=0.01)
    # marginal of component 0 is Beta(p0, sum - p0)
    assert stats.kstest(th[:, 0].astype(np.float64), "beta", args=(p[0], p.sum() - p[0])).pvalue > 1e-5
    thf = oracle.theta_faithful(off, z, K, alpha, 5, 1)
    assert np.allclose(th, thf, rtol=1e-4, atol=1e-7)


def test_empty_documents(oracle):
    # GGS:52-53 / UPL:1474: empty documents are skipped
    off, tokens = make_corpus(40, 50, 12, seed=2, empty_every=7)
    K = 10
    z = oracle.java_next_ints(1, K, len(tokens))
    th = oracle.theta_contract(off, z, K, np.full(K, 0.1), 9, 1)
    lens = np.diff(off)
    assert np.all(th[lens == 0] == 0) and np.all(th[lens > 0].sum(axis=1) > 0.999)
    n_wk, _ = oracle.rebuild_counts(tokens, z, 50, K)
    phi = oracle.phi_contract(n_wk, 0.01, 9, 0)
    z1 = oracle.z_ggs_contract(off, tokens, z, K, th, phi, 9, 1)
    z2 = oracle.z_pcgs_contract(off, tokens, z, K, np.full(K, 0.1), phi, 9, 1)
    assert len(z1) == len(z2) == len(tokens) and z1.max() < K and z2.max() < K


@pytest.mark.parametrize("scheme", ["ggs", "pcgs"])
def test_sweep_invariants(oracle, scheme):
    # ParanoidUncollapsedParallelLDA.java:14-55, UPL:299-351: counts consistent, Phi rows sane
    off, tokens = make_corpus(60, 200, 40, seed=5)
    V, K, beta = 200, 33, 0.01
    alpha = np.full(K, 50.0 / K)
    N = len(tokens)
    z = oracle.java_next_ints(2019, K, N)
    n_wk, n_k = oracle.rebuild_counts(tokens, z, V, K)
    assert n_wk.sum() == N and n_k.sum() == N and np.array_equal(n_wk.sum(axis=0), n_k)
    phi = oracle.phi_contract(n_wk, beta, 2019, 0)
    sch = oracle.GGS if scheme == "ggs" else oracle.PCGS
    st = oracle.sweeps("contract", sch, off, tokens, z, V, K, alpha, beta, 2019, 1, 4, phi)
    assert st["n_wk"].min() >= 0 and st["n_wk"].sum() == N and st["n_k"].sum() == N
    assert np.array_equal(st["n_wk"].sum(axis=0), st["n_k"])
    nw2, nk2 = oracle.rebuild_counts(tokens, st["z"], V, K)
    assert np.array_equal(nw2, st["n_wk"]) and np.array_equal(nk2, st["n_k"])
    cs = st["phiT"].astype(np.float64).sum(axis=0)
    assert np.all(np.abs(cs - 1.0) < 1e-4) and st["phiT"].min() > 0
    ndk = oracle.doc_topic_counts(off, st["z"], K)
    assert np.array_equal(ndk.sum(axis=1), np.diff(off))


def test_z_given_phi_leaves_phi_unchanged_and_is_deterministic(oracle):
    # SpaliasUncollapsedTest.java:117-124
    off, tokens = make_corpus(30, 80, 25, seed=8)
    K, V = 12, 80
    alpha = np.full(K, 0.3)
    z = oracle.java_next_ints(3, K, len(tokens))
    n_wk, _ = oracle.rebuild_counts(tokens, z, V, K)
    phi = oracle.phi_contract(n_wk, 0.1, 3, 0)
    keep = phi.copy()
    a = oracle.z_pcgs_contract(off, tokens, z, K, alpha, phi, 3, 1)
    b = oracle.z_pcgs_contract(off, tokens, z, K, alpha, phi, 3, 1)
    assert np.array_equal(a, b) and np.array_equal(phi, keep)
    assert not np.array_equal(a, oracle.z_pcgs_contract(off, tokens, z, K, alpha, phi, 3, 2))


def test_contract_vs_faithful_one_step(oracle):
    """Same uniforms, same inputs: the fp32 prefix tree and the Java double walk pick the same topic
    except when U*sum falls within rounding distance of a boundary; Phi agrees to 1e-5."""
    off, tokens = make_corpus(80, 300, 60, seed=13)
    V, K, beta = 300, 100, 0.01
    alpha = np.full(K, 0.5)
    z = oracle.java_next_ints(2019, K, len(tokens))
    n_wk, n_k = oracle.rebuild_counts(tokens, z, V, K)
    phic = oracle.phi_contract(n_wk, beta, 2019, 0)
    phif = oracle.phi_faithful(n_wk, beta, 2019, 0)
    big = phif > 1e-30
    rel = np.abs(phic.astype(np.float64) - phif)[big] / phif[big]
    assert (rel > 1e-5).sum() <= 2          # accept/reject flips only
    assert np.all(phic[~big] <= 1.0000001e-30) and phic.min() > 0
    thc = oracle.theta_contract(off, z, K, alpha, 2019, 1)
    zc = oracle.z_ggs_contract(off, tokens, z, K, thc, phic, 2019, 1)
    zf = oracle.z_ggs_faithful(off, tokens, z, K, thc.astype(np.float64), phic.astype(np.float64), 2019, 1)
    assert (zc == zf).mean() > 0.999
    pc = oracle.z_pcgs_contract(off, tokens, z, K, alpha, phic, 2019, 1)
    pf = oracle.z_pcgs_faithful(off, tokens, z, K, alpha.astype(np.float32).astype(np.float64),
                                phic.astype(np.float64), 2019, 1)
    # PCGS is sequential: one differing draw changes later scores of that document only
    assert (pc == pf).mean() > 0.99


def test_log_likelihood_two_statements(oracle, cats):
    # LogLikelihoodTest.java:22-122 / TestInitialization.java:24 equate the Stirling LL of
    # UncollapsedParallelLDA with SerialCollapsedLDA's within 1e-6 (relative, here vs exact lgamma)
    off, tokens = cats
    K, V = 20, 303
    z = oracle.java_next_ints(2019, K, len(tokens))
    n_wk, n_k = oracle.rebuild_counts(tokens, z, V, K)
    for alpha, beta in ((5.0, 7.0), (0.1, 0.01), (2.5, 0.5)):
        a = oracle.log_likelihood(off, z, K, V, n_wk, n_k, np.full(K, alpha), beta)
        b = oracle.log_likelihood(off, z, K, V, n_wk, n_k, np.full(K, alpha), beta, exact_lgamma=True)
        assert abs(a - b) <= 1e-6 * abs(b)
        assert a < 0


def test_log_posterior_closed_form(oracle):
    # tiny case worked by hand: UPL:1573-1634
    off = np.array([0, 2, 3], np.int64)
    tokens = np.array([0, 1, 1], np.int32)
    z = np.array([0, 1, 1], np.int32)
    K, V = 2, 2
    theta = np.array([[0.25, 0.75], [0.5, 0.5]])
    phiT = np.array([[0.6, 0.1], [0.4, 0.9]])     # [V][K]
    alpha, beta = np.array([2.0, 3.0]), 1.5
    e = 1e-12
    want = (np.log(0.6 + e) + np.log(0.9 + e) + np.log(0.9 + e)
            + (1 + 2 - 1) * np.log(0.25 + e) + (1 + 3 - 1) * np.log(0.75 + e)
            + (0 + 2 - 1) * np.log(0.5 + e) + (1 + 3 - 1) * np.log(0.5 + e)
            + (beta - 1) * np.log(phiT + e).sum())
    got = oracle.log_posterior(off, tokens, z, K, V, theta, phiT, alpha, beta)
    assert abs(got - want) < 1e-12


def test_golden_regression(oracle, cats, golden):
    """The oracle must keep producing the committed vectors (cats, K=20, alpha=5, beta=7, seed 2019)."""
    off, tokens = cats
    K, V, beta, seed = 20, 303, 7.0, 2019
    al = np.full(K, 5.0)
    z0 = oracle.java_next_ints(seed, K, len(tokens))
    assert np.array_equal(z0, golden["z0"])
    n_wk0, n_k0 = oracle.rebuild_counts(tokens, z0, V, K)
    assert np.array_equal(n_k0, golden["n_k0"])
    for mode in ("contract", "faithful"):
        phi0 = oracle.phi_contract(n_wk0, beta, seed, 0) if mode == "contract" else oracle.phi_faithful(n_wk0, beta, seed, 0)
        for sch, name in ((oracle.GGS, "ggs"), (oracle.PCGS, "pcgs")):
            st = oracle.sweeps(mode, sch, off, tokens, z0, V, K, al, beta, seed, 1, 3, phi0)
            if mode == "contract":
                # pure IEEE arithmetic: bit-exact on any x86-64 host
                assert np.array_equal(st["z"], golden[f"{mode}_{name}_z3"])
                assert np.array_equal(st["n_k"], golden[f"{mode}_{name}_nk3"])
                assert np.array_equal(st["phiT"][::37, ::3], golden[f"{mode}_{name}_phi3_sample"])
            else:
                # libm may differ in the last bit between hosts: compare within tolerance
                assert (st["z"] == golden[f"{mode}_{name}_z3"]).mean() > 0.98
                assert np.allclose(st["phiT"].sum(axis=0), golden[f"{mode}_{name}_phi3_colsum"], rtol=1e-9)
            ll = oracle.log_likelihood(off, st["z"], K, V, st["n_wk"], st["n_k"], al, beta)
            tol = 1e-12 if mode == "contract" else 2e-2
            assert abs(ll - golden[f"{mode}_{name}_ll"][2]) <= tol * abs(ll)


@pytest.mark.parametrize("scheme", ["ggs", "pcgs"])
def test_contract_and_faithful_chains_agree_statistically(oracle, cats, scheme):
    """Multi-chain posterior-statistics check (north_star level 3): the contract arithmetic and the
    Java-order double arithmetic target the same posterior.  Compare the log-likelihood reached
    after burn-in over several seeds."""
    off, tokens = cats
    K, V, beta = 5, 303, 0.5
    al = np.full(K, 0.5)
    sch = oracle.GGS if scheme == "ggs" else oracle.PCGS
    res = {"contract": [], "faithful": []}
    for seed in range(6):
        z0 = oracle.java_next_ints(seed + 1, K, len(tokens))
        n_wk0, _ = oracle.rebuild_counts(tokens, z0, V, K)
        for mode in res:
            phi0 = (oracle.phi_contract if mode == "contract" else oracle.phi_faithful)(n_wk0, beta, seed, 0)
            st = oracle.sweeps(mode, sch, off, tokens, z0, V, K, al, beta, seed, 1, 60, phi0)
            lls = []
            for it in range(61, 81):
                st = oracle.sweeps(mode, sch, off, tokens, st["z"], V, K, al, beta, seed, it, 1, st["phiT"])
                lls.append(oracle.log_likelihood(off, st["z"], K, V, st["n_wk"], st["n_k"], al, beta))
            res[mode].append(np.mean(lls))
    c, f = np.array(res["contract"]), np.array(res["faithful"])
    spread = max(c.std(), f.std(), 1.0)
    assert abs(c.mean() - f.mean()) < 4 * spread / np.sqrt(len(c)) + 5e-4 * abs(f.mean())


# ---- sparse PCGS z-step ("spalias") ---------------------------------------------------------------
def test_alias_tables_reproduce_the_prior(oracle):
    """WalkerAliasTableTest / OptimizedGentleAliasMethod.main: the table must encode alpha_k*phi_kw / norm, at a small
    K and at the K = 10 000 of the wiki-shaped workloads."""
    V = 40
    for K in (37, 10_000):
        rng = np.random.default_rng(1)
        phi = rng.dirichlet(np.full(V, 0.05), size=K).T.astype(np.float32).copy()      # [V][K]
        alpha = rng.random(K) + 0.01
        ps, al, tn = oracle.alias_build_contract(phi, alpha)
        for w in range(V):
            own = al[w] == np.arange(K)
            keep = np.where(own, 1.0, ps[w].astype(np.float64))
            p = keep / K
            np.add.at(p, al[w], (1.0 - keep) / K)
            want = alpha.astype(np.float32).astype(np.float64) * phi[w]
            assert abs(tn[w] - want.sum()) <= 1e-6 * want.sum(), (K, w)
            assert np.allclose(p, want / want.sum(), atol=2e-6), (K, w)
            assert ps[w].min() >= 0 and ps[w].max() <= 1.0 + 1e-6 and al[w].min() >= 0 and al[w].max() < K, (K, w)


@pytest.mark.parametrize("K", [1, 5, 1500, 10_000])
def test_alias_draw_induces_the_prior_exactly(oracle, K):
    """The prior part's draw over all its inputs, with no sampling: Philox word 1 picks slot floor(w1 K / 2^32), word 2
    keeps it when uniform23(w2) <= ps, else the alias is taken.  Slot i is hit by exactly ceil((i+1) 2^32/K) -
    ceil(i 2^32/K) words; (n + 1/2) 2^-23 <= ps holds for n <= ps 2^23 - 1/2.  The distribution these counts give
    must be alpha_k phi_kw / norm.  The resolution does not depend on the prior's share of the token's mass (DESIGN.md
    4.6).  The oracle's draw is checked at every boundary of the counting, for a flat and a skewed Phi column."""
    rng = np.random.default_rng(K)
    phi = np.stack([rng.gamma(1.0, size=K), rng.gamma(0.05, size=K)]).astype(np.float32)      # [V][K]
    phi /= phi.sum(axis=1, keepdims=True)
    alpha = np.full(K, 0.005)
    ps, al, _ = oracle.alias_build_contract(phi, alpha)
    i = np.arange(K, dtype=np.int64)
    first = -((-i << 32) // K)                               # first word of slot i: ceil(i 2^32 / K)
    hits = np.diff(np.append(first, 1 << 32))
    assert hits.sum() == 1 << 32 and set(np.unique(hits)) <= {(1 << 32) // K, -(-(1 << 32) // K)}
    for w in range(phi.shape[0]):
        kept = np.clip(np.floor(ps[w].astype(np.float64) * 2.0**23 - 0.5) + 1, 0, 1 << 23)   # 23-bit values kept
        keep = kept / 2.0**23
        p = hits * keep
        np.add.at(p, al[w], hits * (1.0 - keep))
        p /= 2.0**32
        want = np.float32(0.005) * phi[w].astype(np.float64)
        want /= want.sum()
        tv = 0.5 * np.abs(p - want).sum()
        assert tv <= 1e-5, f"K = {K}, column {w}: TV {tv:.3g}"
        draw = oracle.lib().oracle_alias_sample_contract
        for s in {0, 1, K // 2, K - 2, K - 1} & set(range(K)):
            lo, hi = int(first[s]), int(first[s] + hits[s] - 1)
            for w1 in (lo, hi):
                if kept[s] > 0:
                    assert draw(ps[w], al[w], K, w1, (int(kept[s]) - 1) << 9) == s
                if kept[s] < 1 << 23:
                    assert draw(ps[w], al[w], K, w1, int(kept[s]) << 9) == al[w, s]


def test_spalias_contract_vs_faithful_and_invariants(oracle):
    off, tokens = make_corpus(80, 150, 30, seed=11, empty_every=9)
    V, K, beta = 150, 64, 0.05
    alpha = np.full(K, 0.2)
    z = oracle.java_next_ints(5, K, len(tokens))
    n_wk, _ = oracle.rebuild_counts(tokens, z, V, K)
    phi = oracle.phi_contract(n_wk, beta, 5, 0)
    a = oracle.z_spalias_contract(off, tokens, z, K, alpha, phi, 5, 1)
    b = oracle.z_spalias_faithful(off, tokens, z, K, alpha.astype(np.float32).astype(np.float64),
                                  phi.astype(np.float64), 5, 1)
    assert a.min() >= 0 and a.max() < K and (a == b).mean() > 0.99
    assert np.array_equal(a, oracle.z_spalias_contract(off, tokens, z, K, alpha, phi, 5, 1))
    st = oracle.sweeps("contract", oracle.SPALIAS, off, tokens, z, V, K, alpha, beta, 5, 1, 3, phi)
    assert st["n_wk"].sum() == len(tokens) and np.array_equal(st["n_wk"].sum(axis=0), st["n_k"])


def test_spalias_contract_multi_block_lists(oracle):
    """Documents whose non-zero topic list exceeds one 256-entry block of the contract's cumulative sum
    (random start, K = 3000, ~700-token documents): the block carries must keep the contract on the
    faithful walk.  A single rounding flip reorders the document's list (swap-remove / append) and so
    changes every later draw of THAT document, hence the comparison per document."""
    off, tokens = make_corpus(12, 200, 700, seed=23)
    V, K, beta = 200, 3000, 0.05
    alpha = np.full(K, 0.02)
    z = oracle.java_next_ints(7, K, len(tokens))
    assert max(len(np.unique(z[off[d]:off[d + 1]])) for d in range(len(off) - 1)) > 2 * 256
    n_wk, _ = oracle.rebuild_counts(tokens, z, V, K)
    phi = oracle.phi_contract(n_wk, beta, 7, 0)
    a = oracle.z_spalias_contract(off, tokens, z, K, alpha, phi, 7, 1)
    b = oracle.z_spalias_faithful(off, tokens, z, K, alpha.astype(np.float32).astype(np.float64),
                                  phi.astype(np.float64), 7, 1)
    assert a.min() >= 0 and a.max() < K
    same = [np.array_equal(a[off[d]:off[d + 1]], b[off[d]:off[d + 1]]) for d in range(len(off) - 1)]
    assert sum(same) >= len(same) - 2


def test_spalias_targets_the_same_conditional_as_dense_pcgs(oracle):
    """One token resampled many times: the sparse mixture (alias prior + sparse likelihood) and the dense
    walk must give the same distribution over topics (chi-square on a single-document corpus)."""
    K, V = 12, 5
    rng = np.random.default_rng(3)
    phi = rng.dirichlet(np.full(V, 0.5), size=K).T.astype(np.float32).copy()
    alpha = np.full(K, 0.3)
    base = np.array([0, 0, 3, 3, 3, 7], np.int32)            # the other tokens of the document
    n = 4000
    off = np.arange(n + 1, dtype=np.int64) * (len(base) + 1)
    tokens = np.tile(np.concatenate([[2], np.zeros(len(base), np.int32)]), n).astype(np.int32)
    z0 = np.tile(np.concatenate([[5], base]), n).astype(np.int32)
    zs = oracle.z_spalias_contract(off, tokens, z0, K, alpha, phi, 9, 1)[:: len(base) + 1]
    zd = oracle.z_pcgs_contract(off, tokens, z0, K, alpha, phi, 9, 1)[:: len(base) + 1]
    cnt = np.bincount(base, minlength=K)
    p = (cnt + alpha) * phi[2]
    p /= p.sum()
    for draw in (zs, zd):
        obs = np.bincount(draw, minlength=K)
        keep = p * n > 5
        chi2 = ((obs[keep] - p[keep] * n) ** 2 / (p[keep] * n)).sum()
        assert chi2 < stats.chi2.ppf(1 - 1e-5, keep.sum() - 1)


def test_spalias_and_dense_chains_agree_statistically(oracle, cats):
    off, tokens = cats
    K, V, beta = 8, 303, 0.5
    al = np.full(K, 0.5)
    res = {oracle.PCGS: [], oracle.SPALIAS: []}
    for seed in range(5):
        z0 = oracle.java_next_ints(seed + 1, K, len(tokens))
        n_wk0, _ = oracle.rebuild_counts(tokens, z0, V, K)
        phi0 = oracle.phi_contract(n_wk0, beta, seed, 0)
        for sch in res:
            st = oracle.sweeps("contract", sch, off, tokens, z0, V, K, al, beta, seed, 1, 50, phi0)
            lls = []
            for it in range(51, 66):
                st = oracle.sweeps("contract", sch, off, tokens, st["z"], V, K, al, beta, seed, it, 1, st["phiT"])
                lls.append(oracle.log_likelihood(off, st["z"], K, V, st["n_wk"], st["n_k"], al, beta))
            res[sch].append(np.mean(lls))
    a, b = np.array(res[oracle.PCGS]), np.array(res[oracle.SPALIAS])
    spread = max(a.std(), b.std(), 1.0)
    assert abs(a.mean() - b.mean()) < 4 * spread / np.sqrt(len(a)) + 5e-4 * abs(a.mean())
