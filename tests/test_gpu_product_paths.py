"""GPU parity tests for the product paths that bench.py times (VERDICT round 1, "untested product paths"):

* the sparse z-step's global-memory slow path (documents with more than 256 distinct topics),
* the 8-chunk pipelined ldagpu_set_z (N >= 8 Mi tokens) and its 16-bit twin,
* the BASELINE.json shapes themselves: NIPS-shaped K=100 and a PubMed-shaped K=1000 slice, whole sweeps
  against the oracle's contract mode,
* the fused theta draw: documents of one work item (theta drawn inside the z kernel) mixed with documents
  split into chunks (theta from the stand-alone kernel),
* the GPU against the stored FAITHFUL-mode goldens of the cats corpus (the reference's arithmetic).

All through the C ABI; integer state bit-exact, theta / Phi bit-exact against the contract oracle."""
import ctypes as C

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


def test_sparse_slow_path_more_than_256_topics_per_document(oracle):
    """kernels_sparse.cu: a document whose non-zero topic list outgrows the 256 shared-memory entries continues on
    the per-warp lists in global memory (reference: SpaliasUncollapsedParallelLDA.java:124-293)."""
    K, V, D, mean_len = 4000, 600, 40, 2000
    off, tokens = make_corpus(D, V, mean_len, seed=5, empty_every=13)
    alpha, beta, seed = 50.0 / K, 0.01, 23
    s = _sampler("gpu_spalias", off, tokens, V, K, alpha, beta, seed)
    z0 = s.get_z_flat()
    nnz = [len(np.unique(z0[off[d]:off[d + 1]])) for d in range(D)]
    assert max(nnz) > 600, "the corpus must exercise the global-memory lists"
    phi0 = s.getPhi().T.astype(np.float32).copy()
    s._step("next_iteration")
    s._step("sample_z")
    want = oracle.z_spalias_contract(off, tokens, z0, K, np.full(K, alpha), phi0, seed, 1)
    assert np.array_equal(s.get_z_flat(), want)
    # whole sweeps on the same path
    s.set_z_flat(z0, redraw_phi=False)
    s._L.ldagpu_set_iteration(s._h, 0)
    s.sample(2)
    st = oracle.sweeps("contract", oracle.SPALIAS, off, tokens, z0, V, K, np.full(K, alpha), beta, seed, 1, 2, phi0)
    assert np.array_equal(s.get_z_flat(), st["z"])
    assert np.array_equal(s.getTypeTopicMatrix(), st["n_wk"]) and np.array_equal(s.getTopicTotals(), st["n_k"])
    s.close()


def test_sparse_alias_tables_in_several_rounds(oracle, monkeypatch):
    """kernels_sparse.cu launch_alias_build: when the active vocabulary exceeds the scratch slots the classify + pair
    kernels run in rounds over slices of the active types (LDAGPU_ALIAS_SLOTS caps the slots; by default a round
    covers 151 552 types).  The tables -- and so every sampled topic -- must not depend on the number of rounds
    (reference: SpaliasUncollapsedParallelLDA.java:39-60 builds one table per type, independently)."""
    K, V, D, mean_len = 1200, 900, 300, 120
    off, tokens = make_corpus(D, V, mean_len, seed=8)
    alpha, beta, seed = 50.0 / K, 0.01, 31
    assert len(np.unique(tokens)) > 3 * 128, "several rounds of 128 slots"
    monkeypatch.setenv("LDAGPU_ALIAS_SLOTS", "128")
    s = _sampler("gpu_spalias", off, tokens, V, K, alpha, beta, seed)
    monkeypatch.delenv("LDAGPU_ALIAS_SLOTS")
    z0 = s.get_z_flat()
    phi0 = s.getPhi().T.astype(np.float32).copy()
    s.sample(2)
    launches = s.getLastCallStats()[3]
    st = oracle.sweeps("contract", oracle.SPALIAS, off, tokens, z0, V, K, np.full(K, alpha), beta, seed, 1, 2, phi0)
    assert np.array_equal(s.get_z_flat(), st["z"])
    assert np.array_equal(s.getTypeTopicMatrix(), st["n_wk"]) and np.array_equal(s.getTopicTotals(), st["n_k"])
    # the same corpus with one round per build: the same chain, fewer launches
    t = _sampler("gpu_spalias", off, tokens, V, K, alpha, beta, seed)
    t.sample(2)
    assert np.array_equal(t.get_z_flat(), st["z"]) and t.getLastCallStats()[3] < launches
    s.close(); t.close()


def test_set_z_eight_chunks_and_16_bit_upload():
    """ldagpu_set_z pipelines the upload in 8 chunks from N >= 8 Mi tokens on (engine.cu); the counts must equal a
    plain histogram.  ldagpu_set_z16 / ldagpu_sweep_get_z16 move the same indicators as uint16."""
    import ldagroupedgibbssampler_b200 as L
    K, V = 8, 5000
    off, tokens = L.synth_corpus(96000, V, 90.0, seed=3)
    N = len(tokens)
    assert N >= (8 << 20) + 100000
    s = _sampler("gpu_pcgs", off, tokens, V, K, 0.5, 0.1, 1, init_z=False)
    rng = np.random.default_rng(0)
    z = rng.integers(0, K, N).astype(np.int32)
    s.set_z_flat(z, redraw_phi=False)
    want = np.bincount(tokens.astype(np.int64) * K + z, minlength=V * K).reshape(V, K).astype(np.int32)
    assert np.array_equal(s.get_z_flat(), z)
    assert np.array_equal(s.getTypeTopicMatrix(), want)
    assert np.array_equal(s.getTopicTotals(), want.sum(axis=0))
    # an out-of-range indicator in the LAST chunk is refused and the previous state stays in place (UPL:475-481 throws)
    bad = z.copy()
    bad[N - 5] = K
    with pytest.raises(L.LdaGpuError):
        s.set_z_flat(bad, redraw_phi=False)
    assert np.array_equal(s.get_z_flat(), z)
    assert np.array_equal(s.getTypeTopicMatrix(), want)
    # 16-bit twin
    z2 = rng.integers(0, K, N).astype(np.uint16)
    s.set_z16_flat(z2, redraw_phi=False)
    want2 = np.bincount(tokens.astype(np.int64) * K + z2, minlength=V * K).reshape(V, K).astype(np.int32)
    assert np.array_equal(s.get_z_flat(), z2.astype(np.int32))
    assert np.array_equal(s.getTypeTopicMatrix(), want2)
    out16 = np.zeros(N, np.uint16)
    s.sample(1, z_out=out16)
    assert np.array_equal(out16.astype(np.int32), s.get_z_flat())
    s.close()


def test_nips_shaped_whole_sweeps_bit_exact(oracle):
    """BASELINE.json configs[1]: 1 500 documents of ~1 267 tokens, V = 12 419, GGS K = 100 (every document is split
    into chunks: theta comes from the stand-alone kernel)."""
    import ldagroupedgibbssampler_b200 as L
    K, V, alpha, beta, seed = 100, 12419, 1.0, 0.01, 2019
    off, tokens = L.synth_corpus(1500, V, 1267.0, seed=20190529)
    s = _sampler("gpu_ggs", off, tokens, V, K, alpha, beta, seed)
    z0 = s.get_z_flat()
    assert np.array_equal(z0, oracle.java_next_ints(seed, K, len(tokens)))
    phi0 = s.getPhi().T.astype(np.float32).copy()
    s.sample(2)
    st = oracle.sweeps("contract", oracle.GGS, off, tokens, z0, V, K, np.full(K, alpha), beta, seed, 1, 2, phi0)
    assert np.array_equal(s.get_z_flat(), st["z"])
    assert np.array_equal(s.getTypeTopicMatrix(), st["n_wk"]) and np.array_equal(s.getTopicTotals(), st["n_k"])
    assert np.array_equal(s.getPhi().T.astype(np.float32), st["phiT"])
    assert np.array_equal(s.getTheta().astype(np.float32), st["theta"])
    s.close()


def test_enron_shaped_pcgs_sweep_bit_exact(oracle):
    """BASELINE.json configs[2] shape (V = 28 102, K = 400, ~161 tokens per document), a 6 000-document slice."""
    import ldagroupedgibbssampler_b200 as L
    K, V, alpha, beta, seed = 400, 28102, 0.125, 0.01, 2019
    off, tokens = L.synth_corpus(6000, V, 161.0, seed=20190529)
    s = _sampler("gpu_pcgs", off, tokens, V, K, alpha, beta, seed)
    z0 = s.get_z_flat()
    phi0 = s.getPhi().T.astype(np.float32).copy()
    s.sample(2)
    st = oracle.sweeps("contract", oracle.PCGS, off, tokens, z0, V, K, np.full(K, alpha), beta, seed, 1, 2, phi0)
    assert np.array_equal(s.get_z_flat(), st["z"])
    assert np.array_equal(s.getTypeTopicMatrix(), st["n_wk"]) and np.array_equal(s.getTopicTotals(), st["n_k"])
    assert np.array_equal(s.getPhi().T.astype(np.float32), st["phiT"])
    s.close()


def test_pubmed_shaped_slice_whole_sweep_bit_exact(oracle):
    """BASELINE.json configs[3] shape: V = 141 043, K = 1000, ~90 tokens per document; a 60 000-document slice
    (5.4 M tokens), one whole sweep with the theta draw fused into the z kernel."""
    import ldagroupedgibbssampler_b200 as L
    K, V, alpha, beta, seed = 1000, 141043, 0.05, 0.01, 2019
    off, tokens = L.synth_corpus(60000, V, 90.0, seed=20190529)
    s = _sampler("gpu_ggs", off, tokens, V, K, alpha, beta, seed)
    z0 = s.get_z_flat()
    n_wk0, _ = oracle.rebuild_counts(tokens, z0, V, K)
    phi0 = oracle.phi_contract(n_wk0, beta, seed, 0)
    s.sample(1)
    st = oracle.sweeps("contract", oracle.GGS, off, tokens, z0, V, K, np.full(K, alpha), beta, seed, 1, 1, phi0)
    assert np.array_equal(s.get_z_flat(), st["z"])
    assert np.array_equal(s.getTopicTotals(), st["n_k"])
    assert np.array_equal(s.getTypeTopicMatrix(), st["n_wk"])
    d_sel = np.arange(0, 60000, 997)
    assert np.array_equal(s.getTheta().astype(np.float32)[d_sel], st["theta"][d_sel])
    got = s.getPhi().T.astype(np.float32)
    assert np.array_equal(got[::13], st["phiT"][::13])
    s.close()


@pytest.mark.parametrize("K", [100, 300, 1000])
def test_fused_theta_mixed_document_lengths(oracle, K):
    """Documents of one work item draw theta inside the z kernel, longer ones are split into chunks and read the
    theta row the stand-alone kernel wrote: both in one corpus, empty documents included."""
    rng = np.random.default_rng(K)
    lens = np.concatenate([rng.integers(1, 60, 300), rng.integers(300, 900, 12), np.zeros(5, np.int64),
                           rng.integers(1, 33, 100)])
    rng.shuffle(lens)
    off = np.zeros(len(lens) + 1, np.int64)
    np.cumsum(lens, out=off[1:])
    V = 700
    tokens = rng.integers(0, V, int(off[-1])).astype(np.int32)
    for d in range(len(lens)):
        tokens[off[d]:off[d + 1]].sort()
    alpha, beta, seed = 50.0 / K, 0.01, 5
    s = _sampler("gpu_ggs", off, tokens, V, K, alpha, beta, seed)
    z0 = s.get_z_flat()
    phi0 = s.getPhi().T.astype(np.float32).copy()
    s.sample(3)
    st = oracle.sweeps("contract", oracle.GGS, off, tokens, z0, V, K, np.full(K, alpha), beta, seed, 1, 3, phi0)
    assert np.array_equal(s.get_z_flat(), st["z"])
    assert np.array_equal(s.getTheta().astype(np.float32), st["theta"])
    assert np.array_equal(s.getPhi().T.astype(np.float32), st["phiT"])
    s.close()


@pytest.mark.parametrize("scheme,name", [("gpu_ggs", "ggs"), ("gpu_pcgs", "pcgs")])
def test_gpu_against_faithful_goldens_cats(cats, golden, scheme, name):
    """The stored faithful-mode goldens (double, libm, the Java loop order) on the bundled cats corpus, K = 20,
    alpha = 5, beta = 7, seed 2019, 3 sweeps: the GPU's topic indicators agree with them (>= 99 % stated; they are
    identical today) and the log-likelihood series within 1e-9 relative."""
    off, tokens = cats
    K, V, alpha, beta, seed = 20, 303, 5.0, 7.0, 2019
    s = _sampler(scheme, off, tokens, V, K, alpha, beta, seed)
    assert np.array_equal(s.get_z_flat(), golden["z0"])
    lls = []
    for _ in range(3):
        s.sample(1)
        lls.append(s.modelLogLikelihood())
    agree = float((s.get_z_flat() == golden[f"faithful_{name}_z3"]).mean())
    assert agree >= 0.99, agree
    assert np.allclose(lls, golden[f"faithful_{name}_ll"], rtol=1e-9, atol=0)
    assert np.abs(s.getTopicTotals() - golden[f"faithful_{name}_nk3"]).max() <= 0.01 * len(tokens)
    got_phi = s.getPhi().T[::37, ::3]
    assert np.allclose(got_phi, golden[f"faithful_{name}_phi3_sample"], rtol=1e-5, atol=1e-30)
    s.close()


def test_two_handles_on_one_device_and_large_smem_paths():
    """Launch configuration is cached per device, not per process (ADVICE round 1): two live handles whose kernels
    need the > 48 KB shared-memory opt-in (PCGS K = 1000, GGS K = 1000) keep working side by side."""
    off, tokens = make_corpus(60, 400, 40, seed=2)
    a = _sampler("gpu_pcgs", off, tokens, 400, 1000, 0.05, 0.01, 3)
    b = _sampler("gpu_ggs", off, tokens, 400, 1000, 0.05, 0.01, 3)
    a.sample(2)
    b.sample(2)
    a.sample(1)
    assert a.getTopicTotals().sum() == len(tokens) and b.getTopicTotals().sum() == len(tokens)
    a.close()
    b.close()


@pytest.mark.parametrize("K,V,D,mean_len", [(30, 120, 60, 40), (300, 800, 120, 60), (1500, 400, 60, 40)])
def test_polya_urn_scheme_bit_exact(oracle, K, V, D, mean_len):
    """scheme gpu_polyaurn (the reference's "polyaurn": topics/PolyaUrnSpaliasLDA.java): the Poisson Polya-urn Phi draw
    (exact zeros in Phi) and the sparse z-step on top of it, whole sweeps, against the oracle's contract mode."""
    off, tokens = make_corpus(D, V, mean_len, seed=K + 5, empty_every=11)
    alpha, beta, seed = 50.0 / K, 0.01, 29
    s = _sampler("gpu_polyaurn", off, tokens, V, K, alpha, beta, seed)
    z0 = s.get_z_flat()
    nw0, _ = oracle.rebuild_counts(tokens, z0, V, K)
    phi0 = oracle.phi_polya_contract(nw0, beta, seed, 0)
    got0 = s.getPhi().T.astype(np.float32)
    assert np.array_equal(got0, phi0)                    # initial Phi: the urn too (UPL:450 -> loopOverTopics override)
    assert (got0 == 0).mean() > 0.5                      # sparse rows
    if K <= 300:
        # word types of the corpus whose Phi column is all zero: their tokens take the tot = 0 fallback (DESIGN.md 4.6)
        assert not got0[np.unique(tokens)].any(axis=1).all()
    s.sample(3)
    st = oracle.sweeps("contract", oracle.POLYAURN, off, tokens, z0, V, K, np.full(K, alpha), beta, seed, 1, 3, phi0)
    assert np.array_equal(s.get_z_flat(), st["z"])
    assert np.array_equal(s.getTypeTopicMatrix(), st["n_wk"]) and np.array_equal(s.getTopicTotals(), st["n_k"])
    assert np.array_equal(s.getPhi().T.astype(np.float32), st["phiT"])
    # against the faithful (libm) urn on the same uniforms
    pf = oracle.phi_polya_faithful(st["n_wk"], beta, seed, 3)
    assert np.allclose(s.getPhi().T, pf, rtol=1e-5, atol=1e-12)
    s.close()


def test_polya_urn_large_counts_normal_branch(oracle):
    """cells with n >= alias_poisson_threshold take the normal approximation (PoissonFixedCoeffSampler.java:45-51)"""
    import ldagroupedgibbssampler_b200 as L
    V, K = 6, 4
    off = np.array([0, 3000, 6000], np.int64)
    tokens = np.sort(np.concatenate([np.arange(3000) % V, np.arange(3000) % V])).astype(np.int32).reshape(2, 3000)
    tokens = np.concatenate([np.sort(tokens[0]), np.sort(tokens[1])]).astype(np.int32)
    cfg = L.LDAConfiguration(scheme="gpu_polyaurn", topics=K, alpha=0.5, beta=0.01, seed=3, exec_time=0,
                             alias_poisson_threshold=20)
    s = L.GpuLDASampler(cfg)
    s.addInstances(L.InstanceList.from_csr(off, tokens, V))
    z0 = s.get_z_flat()
    nw0, _ = oracle.rebuild_counts(tokens, z0, V, K)
    assert nw0.max() > 100
    assert np.array_equal(s.getPhi().T.astype(np.float32), oracle.phi_polya_contract(nw0, 0.01, 3, 0, L=20))
    s.close()


def test_hyperparameter_hooks(oracle):
    """MSL:812-905 hooks: the histograms of n_dk and n_wk equal numpy's, set_alpha / set_beta reach the kernels (theta and
    Phi follow the oracle with the new values), and hyperparam_optim_interval runs the host-side fixed point."""
    import ldagroupedgibbssampler_b200 as L
    off, tokens = make_corpus(300, 400, 60, seed=12, empty_every=17)
    K, V, alpha, beta, seed = 50, 400, 0.2, 0.05, 8
    s = _sampler("gpu_ggs", off, tokens, V, K, alpha, beta, seed)
    s.sample(3)
    dh, th, dl, ts = s._count_histograms()
    n_dk, n_wk = s.getDocumentTopicMatrix(), s.getTypeTopicMatrix()
    assert np.array_equal(dh, np.bincount(n_dk.ravel(), minlength=len(dh)))
    assert np.array_equal(th, np.bincount(n_wk.ravel(), minlength=len(th)))
    assert dl.sum() == len(off) - 1 and ts.sum() == K
    # new hyper-parameters reach the kernels
    new_alpha = np.linspace(0.05, 0.6, K)
    s._ck(s._L.ldagpu_set_alpha(s._h, new_alpha.ctypes.data))
    s._ck(s._L.ldagpu_set_beta(s._h, 0.2))
    z3 = s.get_z_flat()
    s._step("next_iteration")
    s._step("sample_theta")
    assert np.array_equal(s.getTheta().astype(np.float32), oracle.theta_contract(off, z3, K, new_alpha, seed, 4))
    s._step("sample_phi")
    assert np.array_equal(s.getPhi().T.astype(np.float32), oracle.phi_contract(n_wk, 0.2, seed, 4))
    want_ll = oracle.log_likelihood(off, z3, K, V, n_wk, s.getTopicTotals(), new_alpha, 0.2)
    assert abs(s.modelLogLikelihood() - want_ll) <= 1e-9 * abs(want_ll)
    s.close()
    # the optimisation loop itself (symmetric alpha): runs every 2 sweeps, values stay positive and finite and move
    cfg = L.LDAConfiguration(scheme="gpu_pcgs", topics=K, alpha=alpha, beta=beta, seed=seed, exec_time=0,
                             hyperparam_optim_interval=2)
    o = L.GpuLDASampler(cfg)
    o.addInstances(L.InstanceList.from_csr(off, tokens, V))
    o.sample(6)
    assert np.all(np.isfinite(o.alpha)) and np.all(o.alpha > 0) and np.isfinite(o.beta) and o.beta > 0
    assert abs(o.alpha[0] - alpha) > 1e-6 and np.allclose(o.alpha, o.alpha[0])
    o.close()
