"""GPU parity tests: libldagpu.so (through its C ABI) against the CPU oracle on the same seeded inputs.

Bar: integer state (z, n_wk, n_k, n_dk) bit-exact; theta and Phi bit-exact against the oracle's
contract mode (same IEEE operation sequence) and within 1e-5 relative against its faithful (libm,
double, Java loop order) mode; log-likelihood / log-posterior within 1e-9 relative (stated 1e-5)."""
import numpy as np
import pytest

from conftest import make_corpus

pytestmark = pytest.mark.gpu


def _sampler(scheme, off, tokens, V, K, alpha, beta, seed, init_z=True):
    import ldagroupedgibbssampler_b200 as L
    cfg = L.LDAConfiguration(scheme=scheme, topics=K, alpha=alpha, beta=beta, seed=seed, exec_time=0)
    s = L.GpuLDASampler(cfg)
    s.addInstances(L.InstanceList.from_csr(off, tokens, V), init_z=init_z)
    return s


def test_library_and_device():
    import ldagroupedgibbssampler_b200 as L
    lib = L.load()
    assert lib.ldagpu_device_count() >= 1
    assert b"sm_100a" in lib.ldagpu_version()


@pytest.mark.parametrize("K", [3, 20, 100, 129, 400, 1000])
def test_initial_state_matches_oracle(oracle, K):
    """addInstances: java.util.Random initial z, counts, initial Phi (UPL:357-456)."""
    off, tokens = make_corpus(50, 300, 30, seed=K, empty_every=9)
    V, beta, seed = 300, 0.01, 2019
    s = _sampler("gpu_ggs", off, tokens, V, K, 0.1, beta, seed)
    z0 = oracle.java_next_ints(seed, K, len(tokens))
    assert np.array_equal(s.get_z_flat(), z0)
    n_wk, n_k = oracle.rebuild_counts(tokens, z0, V, K)
    assert np.array_equal(s.getTypeTopicMatrix(), n_wk)
    assert np.array_equal(s.getTopicTotals(), n_k)
    assert np.array_equal(s.getDocumentTopicMatrix(), oracle.doc_topic_counts(off, z0, K))
    phi = oracle.phi_contract(n_wk, beta, seed, 0)
    got = s.getPhi().T.astype(np.float32)
    assert np.array_equal(got, phi)            # bit-exact Phi draw
    s.close()


@pytest.mark.parametrize("K,V,D,mean_len", [(20, 303, 23, 300), (100, 500, 40, 700), (400, 2000, 200, 60),
                                            (1000, 3000, 150, 90), (7, 50, 30, 5)])
def test_theta_and_z_ggs_bit_exact(oracle, K, V, D, mean_len):
    off, tokens = make_corpus(D, V, mean_len, seed=K + 1, empty_every=11)
    alpha, beta, seed = 50.0 / K, 0.01, 77
    s = _sampler("gpu_ggs", off, tokens, V, K, alpha, beta, seed)
    z0 = s.get_z_flat()
    phi = s.getPhi().T.astype(np.float32).copy()
    s._step("next_iteration")
    s._step("sample_theta")
    th = oracle.theta_contract(off, z0, K, np.full(K, alpha), seed, 1)
    got_th = s.getTheta().astype(np.float32)
    assert np.array_equal(got_th, th)
    # against the faithful (double, libm) draw on the same uniforms
    thf = oracle.theta_faithful(off, z0, K, np.full(K, alpha), seed, 1)
    big = thf > 1e-8
    assert np.all(np.abs(got_th[big] - thf[big]) <= 1e-5 * thf[big] + 1e-9)
    s._step("sample_z")
    z1 = oracle.z_ggs_contract(off, tokens, z0, K, th, phi, seed, 1)
    assert np.array_equal(s.get_z_flat(), z1)
    s.close()


def test_z_ggs_with_injected_theta_and_phi(oracle):
    """north_star: sampled z bit-exact against the harness with injected RNG; theta/Phi injected (UPL:1897-1926)."""
    off, tokens = make_corpus(64, 400, 50, seed=21, sort_docs=False)
    K, V, seed = 100, 400, 5
    rng = np.random.default_rng(0)
    theta = rng.dirichlet(np.full(K, 0.2), size=len(off) - 1)
    phi = rng.dirichlet(np.full(V, 0.05), size=K)             # [K][V]
    s = _sampler("gpu_ggs", off, tokens, V, K, 0.1, 0.01, seed)
    z0 = s.get_z_flat()
    s.setPhi(phi)
    s.setTheta(theta)
    s._step("next_iteration")
    s._step("sample_z")
    want = oracle.z_ggs_contract(off, tokens, z0, K, theta.astype(np.float32),
                                 np.ascontiguousarray(phi.T.astype(np.float32)), seed, 1)
    got = s.get_z_flat()
    assert np.array_equal(got, want)
    # and close to the Java-order double walk on the same uniforms
    zf = oracle.z_ggs_faithful(off, tokens, z0, K, theta.astype(np.float32).astype(np.float64),
                               np.ascontiguousarray(phi.T.astype(np.float32).astype(np.float64)), seed, 1)
    assert (got == zf).mean() > 0.999
    s.close()


@pytest.mark.parametrize("K,V,D,mean_len", [(20, 303, 23, 300), (400, 1500, 120, 160), (129, 200, 60, 20), (1000, 800, 40, 50)])
def test_z_pcgs_bit_exact(oracle, K, V, D, mean_len):
    off, tokens = make_corpus(D, V, mean_len, seed=K + 5, empty_every=13)
    alpha, seed = 50.0 / K, 31
    s = _sampler("gpu_pcgs", off, tokens, V, K, alpha, 0.01, seed)
    z0 = s.get_z_flat()
    phi = s.getPhi().T.astype(np.float32).copy()
    s._step("next_iteration")
    s._step("sample_z")
    want = oracle.z_pcgs_contract(off, tokens, z0, K, np.full(K, alpha), phi, seed, 1)
    assert np.array_equal(s.get_z_flat(), want)
    s.close()


@pytest.mark.parametrize("scheme,osch", [("gpu_ggs", 0), ("gpu_pcgs", 1)])
def test_whole_sweeps_bit_exact_cats(oracle, cats, golden, scheme, osch):
    """BASELINE.json configs[0]: cats, K=20, alpha=5, beta=7, seed 2019 -- three full sweeps."""
    off, tokens = cats
    K, V, alpha, beta, seed = 20, 303, 5.0, 7.0, 2019
    s = _sampler(scheme, off, tokens, V, K, alpha, beta, seed)
    assert np.array_equal(s.get_z_flat(), golden["z0"])
    s.sample(3)
    name = "ggs" if osch == 0 else "pcgs"
    assert np.array_equal(s.get_z_flat(), golden[f"contract_{name}_z3"])
    assert np.array_equal(s.getTopicTotals(), golden[f"contract_{name}_nk3"])
    phi = s.getPhi().T.astype(np.float32)
    assert np.array_equal(phi[::37, ::3], golden[f"contract_{name}_phi3_sample"])
    ll = s.modelLogLikelihood()
    assert abs(ll - golden[f"contract_{name}_ll"][2]) <= 1e-9 * abs(ll)
    if osch == 0:
        assert np.array_equal(s.getTheta().astype(np.float32)[::5, ::3], golden["contract_ggs_theta3_sample"])
    assert s.getCurrentIteration() == 3
    s.close()


# K boundaries of the register path: 1 and 2 topics, full tiles (128, 512: no padding), 513 (the first K with 8 tiles;
# GGS switches to its 8-tile launch shape), 1024 (the largest K there: the clamp to K - 1 falls in a full lane)
@pytest.mark.parametrize("scheme,osch,K", [("gpu_ggs", 0, 100), ("gpu_pcgs", 1, 400), ("gpu_ggs", 0, 1000),
                                           ("gpu_ggs", 0, 1), ("gpu_ggs", 0, 2), ("gpu_ggs", 0, 128), ("gpu_ggs", 0, 512),
                                           ("gpu_ggs", 0, 513), ("gpu_ggs", 0, 1024), ("gpu_pcgs", 1, 256),
                                           ("gpu_pcgs", 1, 513), ("gpu_pcgs", 1, 1024)])
def test_whole_sweeps_bit_exact_synthetic(oracle, scheme, osch, K):
    import ldagroupedgibbssampler_b200 as L
    V = 1200
    off, tokens = L.synth_corpus(300, V, 80.0, seed=4)
    alpha, beta, seed = 50.0 / K, 0.01, 2019
    s = _sampler(scheme, off, tokens, V, K, alpha, beta, seed)
    z0 = s.get_z_flat()
    phi0 = s.getPhi().T.astype(np.float32).copy()
    s.sample(2)
    st = oracle.sweeps("contract", osch, off, tokens, z0, V, K, np.full(K, alpha), beta, seed, 1, 2, phi0)
    assert np.array_equal(s.get_z_flat(), st["z"])
    assert np.array_equal(s.getTypeTopicMatrix(), st["n_wk"])
    assert np.array_equal(s.getTopicTotals(), st["n_k"])
    assert np.array_equal(s.getPhi().T.astype(np.float32), st["phiT"])
    # Phi within 1e-5 of the faithful double-precision draw from the same counts (flips aside)
    phif = oracle.phi_faithful(st["n_wk"], beta, seed, 2)
    got = s.getPhi().T
    big = phif > 1e-30
    assert ((np.abs(got - phif)[big] / phif[big]) > 1e-5).sum() <= 3
    want_ll = oracle.log_likelihood(off, st["z"], K, V, st["n_wk"], st["n_k"], np.full(K, alpha), beta)
    assert abs(s.modelLogLikelihood() - want_ll) <= 1e-9 * abs(want_ll)
    if osch == 0:
        want_lp = oracle.log_posterior(off, tokens, st["z"], K, V, st["theta"].astype(np.float64),
                                       st["phiT"].astype(np.float64), np.full(K, alpha), beta)
        assert abs(s.computeLogPosterior() - want_lp) <= 1e-9 * abs(want_lp)
    else:
        # PCGS diagnostics draw theta ~ Dir(n_d + alpha) from the current z first (UPL:710-714)
        th = oracle.theta_contract(off, st["z"], K, np.full(K, alpha), seed, s.getCurrentIteration())
        want_lp = oracle.log_posterior(off, tokens, st["z"], K, V, th.astype(np.float64),
                                       st["phiT"].astype(np.float64), np.full(K, alpha), beta)
        assert abs(s.computeLogPosterior() - want_lp) <= 1e-9 * abs(want_lp)
        assert np.array_equal(s.getTheta().astype(np.float32), th)
    s.close()


def test_sample_with_z_read_back_and_pipelined_set_z(oracle):
    """ldagpu_sweep_get_z: z of the last sweep arrives in the host buffer; ldagpu_set_z uploads in chunks with
    the range check inside the count kernel."""
    off, tokens = make_corpus(3000, 500, 60, seed=21)        # > 8 Mi tokens is not needed: one chunk here
    K, V, alpha, beta = 64, 500, 0.2, 0.01
    a = _sampler("gpu_ggs", off, tokens, V, K, alpha, beta, 5)
    b = _sampler("gpu_ggs", off, tokens, V, K, alpha, beta, 5)
    zbuf = np.full(len(tokens), -1, np.int32)
    a.sample(3, z_out=zbuf)
    b.sample(3)
    assert np.array_equal(zbuf, a.get_z_flat()) and np.array_equal(zbuf, b.get_z_flat())
    assert np.array_equal(a.getTypeTopicMatrix(), b.getTypeTopicMatrix())
    data = a.getData()                                        # LGS:26: documents with their current z
    assert len(data) == len(off) - 1 and all(len(t.instance) == len(t.topicSequence) for t in data)
    assert np.array_equal(np.concatenate([t.topicSequence for t in data]), zbuf)
    assert np.array_equal(np.concatenate([t.instance for t in data]), tokens)
    zbuf2 = np.zeros(len(tokens), np.int32)
    a.sample(0, z_out=zbuf2)                                  # no sweep: plain copy of the current z
    assert np.array_equal(zbuf2, zbuf)
    # set_z: counts follow the uploaded z; an out-of-range indicator is reported, not counted
    n_wk, n_k = oracle.rebuild_counts(tokens, zbuf, V, K)
    b.set_z_flat(zbuf, redraw_phi=False)
    assert np.array_equal(b.getTypeTopicMatrix(), n_wk) and np.array_equal(b.getTopicTotals(), n_k)
    bad = zbuf.copy(); bad[len(bad) // 2] = K
    with pytest.raises(Exception, match="out of range"):
        b.set_z_flat(bad, redraw_phi=False)
    with pytest.raises(ValueError):
        a.sample(1, z_out=np.zeros(3, np.int32))
    a.close(); b.close()


@pytest.mark.parametrize("scheme", ["gpu_ggs", "gpu_pcgs", "gpu_spalias"])
def test_checkpoint_resume_is_exact(oracle, scheme):
    """State = (z, Phi, iteration): a fresh handle restored from it continues exactly like the original run
    (all random-number counters are keyed by indices and the iteration, nothing else carries over)."""
    off, tokens = make_corpus(150, 300, 40, seed=9)
    K, V, alpha, beta, seed = 96, 300, 0.3, 0.01, 11
    a = _sampler(scheme, off, tokens, V, K, alpha, beta, seed)
    a.sample(2)
    z2, phi2, it2 = a.get_z_flat(), a.getPhi(), a.getCurrentIteration()
    a.sample(2)
    b = _sampler(scheme, off, tokens, V, K, alpha, beta, seed)
    b.set_z_flat(z2, redraw_phi=False)
    b.setPhi(phi2, None, None)
    b._L.ldagpu_set_iteration(b._h, it2)
    b.sample(2)
    assert np.array_equal(a.get_z_flat(), b.get_z_flat())
    assert np.array_equal(a.getTypeTopicMatrix(), b.getTypeTopicMatrix())
    assert np.array_equal(a.getPhi(), b.getPhi())
    a.close(); b.close()


def test_diagnostic_files(oracle, tmp_path):
    """log-posterior.txt / log-likelihood.txt as the reference's sweep loop appends them
    (UPL:707-823,838-850; util/LDAUtils.java:955-979)."""
    import ldagroupedgibbssampler_b200 as L
    off, tokens = make_corpus(40, 120, 30, seed=5)
    cfg = L.LDAConfiguration(scheme="gpu_ggs", topics=8, alpha=0.5, beta=0.01, seed=3, exec_time=0,
                             start_diagnostic=3, compute_likelihood=True, topic_interval=2,
                             logging_path=str(tmp_path / "run"))
    s = L.GpuLDASampler(cfg, device=0)
    s.addInstances(L.InstanceList.from_csr(off, tokens, 120))
    s.sample(6)
    lp = [ln.split("\t") for ln in open(tmp_path / "run" / "log-posterior.txt").read().splitlines()]
    assert [int(r[0]) for r in lp] == [3, 4, 5, 6] and all(len(r) == 3 for r in lp)
    assert abs(float(lp[-1][1]) - s.computeLogPosterior()) <= 1e-6 * abs(float(lp[-1][1])) + 1e-6
    ll = [ln.split("\t") for ln in open(tmp_path / "run" / "log-likelihood.txt").read().splitlines()]
    assert [int(r[0]) for r in ll] == [2, 4, 6]
    assert float(ll[-1][1]) == s.getLogLikelihood()[-1] == s.modelLogLikelihood()
    assert len(s.getLogLikelihood()) == 4          # iteration 0 (UPL:587-593) + 2, 4, 6
    s.close()


@pytest.mark.parametrize("scheme,osch,K", [("gpu_ggs", 0, 1025), ("gpu_pcgs", 1, 1500), ("gpu_ggs", 0, 2600),
                                           ("gpu_pcgs", 1, 2049), ("gpu_ggs", 0, 2048), ("gpu_pcgs", 1, 2048),
                                           ("gpu_ggs", 0, 27000), ("gpu_pcgs", 1, 18000)])
def test_large_k_dense_path_bit_exact(oracle, scheme, osch, K):
    """K > 1024: Phi^T row staged in shared memory, tile totals in groups of 8 tiles with a carry.  K = 2048 is whole
    groups of 8 tiles (no partial group for the carry); 27 000 (GGS) and 18 000 (PCGS) are the largest K that fit."""
    off, tokens = make_corpus(40, 300, 30, seed=K, empty_every=9)
    V, alpha, beta, seed = 300, 50.0 / K, 0.01, 5
    s = _sampler(scheme, off, tokens, V, K, alpha, beta, seed)
    z0 = s.get_z_flat()
    phi0 = s.getPhi().T.astype(np.float32).copy()
    s.sample(2)
    st = oracle.sweeps("contract", osch, off, tokens, z0, V, K, np.full(K, alpha), beta, seed, 1, 2, phi0)
    assert np.array_equal(s.get_z_flat(), st["z"])
    assert np.array_equal(s.getTypeTopicMatrix(), st["n_wk"])
    assert np.array_equal(s.getPhi().T.astype(np.float32), st["phiT"])
    if osch == 0:
        assert np.array_equal(s.getTheta().astype(np.float32), st["theta"])
    want_ll = oracle.log_likelihood(off, st["z"], K, V, st["n_wk"], st["n_k"], np.full(K, alpha), beta)
    assert abs(s.modelLogLikelihood() - want_ll) <= 1e-9 * abs(want_ll)
    s.close()


@pytest.mark.parametrize("K,V,D,mean_len", [(20, 303, 23, 300), (300, 800, 120, 60), (1500, 400, 60, 40), (4000, 300, 50, 150),
                                            (1, 120, 30, 40), (5, 200, 40, 50)])
def test_sparse_pcgs_bit_exact(oracle, K, V, D, mean_len):
    """gpu_spalias: alias tables and sparse z-step bit-exact against the oracle, whole sweeps included; the diagnostic
    theta (rows in natural topic order here, Ks = round_up(K, 32)) and the log-posterior too."""
    off, tokens = make_corpus(D, V, mean_len, seed=K + 2, empty_every=11)
    alpha, beta, seed = 50.0 / K, 0.01, 17
    s = _sampler("gpu_spalias", off, tokens, V, K, alpha, beta, seed)
    z0 = s.get_z_flat()
    phi0 = s.getPhi().T.astype(np.float32).copy()
    s._step("next_iteration")
    s._step("sample_z")
    want = oracle.z_spalias_contract(off, tokens, z0, K, np.full(K, alpha), phi0, seed, 1)
    assert np.array_equal(s.get_z_flat(), want)
    s.set_z_flat(z0, redraw_phi=False)
    s._L.ldagpu_set_iteration(s._h, 0)
    s.sample(3)
    st = oracle.sweeps("contract", oracle.SPALIAS, off, tokens, z0, V, K, np.full(K, alpha), beta, seed, 1, 3, phi0)
    assert np.array_equal(s.get_z_flat(), st["z"])
    assert np.array_equal(s.getTypeTopicMatrix(), st["n_wk"]) and np.array_equal(s.getTopicTotals(), st["n_k"])
    assert np.array_equal(s.getPhi().T.astype(np.float32), st["phiT"])
    want_ll = oracle.log_likelihood(off, st["z"], K, V, st["n_wk"], st["n_k"], np.full(K, alpha), beta)
    assert abs(s.modelLogLikelihood() - want_ll) <= 1e-9 * abs(want_ll)
    lp = s.computeLogPosterior()
    th = oracle.theta_contract(off, st["z"], K, np.full(K, alpha), seed, s.getCurrentIteration())
    assert np.array_equal(s.getTheta().astype(np.float32), th)
    want_lp = oracle.log_posterior(off, tokens, st["z"], K, V, th.astype(np.float64), st["phiT"].astype(np.float64),
                                   np.full(K, alpha), beta)
    assert abs(lp - want_lp) <= 1e-9 * abs(want_lp)
    s.close()


def test_set_z_round_trip_and_invariants(oracle):
    """TestInitialization.java:458-555: setZIndicators reproduces counts and LL; ParanoidTest invariants."""
    off, tokens = make_corpus(80, 250, 35, seed=3)
    K, V, alpha, beta = 50, 250, 1.0, 0.01
    a = _sampler("gpu_pcgs", off, tokens, V, K, alpha, beta, 1)
    a.sample(5)
    N = len(tokens)
    n_wk, n_k = a.getTypeTopicMatrix(), a.getTopicTotals()
    assert n_wk.min() >= 0 and n_wk.sum() == N and n_k.sum() == N and np.array_equal(n_wk.sum(axis=0), n_k)
    assert np.array_equal(a.getDocumentTopicMatrix().sum(axis=1), np.diff(off))
    phi = a.getPhi()
    assert np.all(np.abs(phi.sum(axis=1) - 1) < 1e-4) and phi.min() > 0
    b = _sampler("gpu_pcgs", off, tokens, V, K, alpha, beta, 999)
    b.setZIndicators(a.getZIndicators())
    assert np.array_equal(b.getTypeTopicMatrix(), n_wk) and np.array_equal(b.getTopicTotals(), n_k)
    assert abs(a.modelLogLikelihood() - b.modelLogLikelihood()) <= 1e-12 * abs(a.modelLogLikelihood())
    # zbar / theta estimate closed forms (ModifiedSimpleLDATest.java:29-110)
    ndk = a.getDocumentTopicMatrix().astype(np.float64)
    assert np.allclose(a.getZbar().sum(axis=1), 1.0)
    assert np.allclose(a.getThetaEstimate(), (ndk + alpha) / (ndk + alpha).sum(axis=1, keepdims=True))
    # sampleZGivenPhi leaves Phi unchanged (SpaliasUncollapsedTest.java:117-124)
    before = b.getPhi()
    b.sampleZGivenPhi(2)
    assert np.array_equal(before, b.getPhi())
    assert b.getTypeTopicMatrix().sum() == N
    a.close(); b.close()


def test_errors_and_abort(oracle):
    import ldagroupedgibbssampler_b200 as L
    off, tokens = make_corpus(10, 20, 8, seed=1)
    s = _sampler("gpu_ggs", off, tokens, 20, 5, 0.1, 0.01, 1)
    bad = s.get_z_flat().copy()
    bad[0] = 5
    with pytest.raises(L.LdaGpuError):
        s.set_z_flat(bad)                      # UPL:475-481 throws on an invalid topic
    with pytest.raises(ValueError):
        s.set_z_flat(bad[:-1])                 # UPL:1828-1830
    s.abort()
    assert s.getAbort()
    it = s.getCurrentIteration()
    s.sample(3)
    assert s.getCurrentIteration() == it       # aborted: no sweep ran (UPL:645)
    s.close()
    cfg = L.LDAConfiguration(scheme="gpu_ggs", topics=5, alpha=0.1, beta=0.01)
    t = L.GpuLDASampler(cfg)
    bad_tokens = tokens.copy(); bad_tokens[3] = 20
    with pytest.raises(L.LdaGpuError):
        t.addInstances(L.InstanceList.from_csr(off, bad_tokens, 20))


def test_phi_mean_schedule():
    import ldagroupedgibbssampler_b200 as L
    off, tokens = make_corpus(30, 60, 20, seed=2)
    cfg = L.LDAConfiguration(scheme="gpu_pcgs", topics=8, alpha=0.5, beta=0.1, seed=4, save_phi_mean=True,
                             phi_mean_burnin=50, phi_mean_thin=2, exec_time=0)
    s = L.GpuLDASampler(cfg)
    s.addInstances(L.InstanceList.from_csr(off, tokens, 60))
    assert s.getPhiMeans() is None
    acc, n = np.zeros((8, 60)), 0

    class Hooked(L.GpuLDASampler):
        def postPhi(self_inner):
            nonlocal acc, n
            it = self_inner.getCurrentIteration()
            if it > 5 and it % 2 == 0:          # burn-in = 50 % of 10 sweeps, thin 2 (UPL:1350-1352)
                acc += self_inner.getPhi(); n += 1

    h = Hooked(cfg)
    h.addInstances(L.InstanceList.from_csr(off, tokens, 60))
    h.sample(10)
    s.sample(10)
    assert n == 3
    assert np.allclose(s.getPhiMeans(), acc / n, rtol=1e-12)
    assert np.allclose(h.getPhiMeans(), acc / n, rtol=1e-12)
    s.close(); h.close()


def test_count_rebuild_large_properties():
    """K3 at a size the oracle would not finish quickly: size-independent properties."""
    import ldagroupedgibbssampler_b200 as L
    V, K = 20000, 1000
    off, tokens = L.synth_corpus(40000, V, 90.0, seed=9)
    s = _sampler("gpu_ggs", off, tokens, V, K, 0.05, 0.01, 7)
    s.sample(1)
    N = len(tokens)
    n_k = s.getTopicTotals()
    z = s.get_z_flat()
    assert n_k.sum() == N and np.array_equal(n_k, np.bincount(z, minlength=K))
    n_wk = s.getTypeTopicMatrix()
    assert np.array_equal(n_wk.sum(axis=0), n_k)
    assert np.array_equal(n_wk.sum(axis=1), np.bincount(tokens, minlength=V))
    # idempotence: rebuilding from the same z changes nothing
    s._step("rebuild_counts")
    assert np.array_equal(s.getTypeTopicMatrix(), n_wk)
    phi = s.getPhi()
    assert np.all(np.abs(phi.sum(axis=1) - 1) < 1e-4)
    s.close()
