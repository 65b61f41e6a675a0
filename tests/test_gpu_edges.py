"""Parity at the edges the other GPU tests leave open, against the contract oracle (DESIGN.md 4):

* an asymmetric alpha through every z-step: on the register path (K <= 1024, GGS / PCGS) rows are stored in a permuted
  column order and alpha in natural order, so each kernel that reads alpha must convert -- a symmetric alpha hides a
  wrong conversion;
* K at the limits the kernels accept, and the refusal just beyond them;
* random-number counters above 2^32: theta cell (doc_base + d) * K + k and token token_base + t, on one GPU through
  presharded bases;
* the full-size PubMed-shaped GGS sweep (1024-token work items, a theta matrix of more than 2^31 cells), checked on
  sampled document windows;
* degenerate scores on injected state (S = 0, a single non-zero topic at either end, products that underflow) and whole
  sweeps at extreme hyper-parameters.

Tests without the gpu mark check the oracle itself and the argument checks of ldagpu_create, which run before any
device is touched."""
import numpy as np
import pytest

from conftest import make_corpus

gpu = pytest.mark.gpu

GGS, PCGS, SPALIAS, POLYAURN = 0, 1, 2, 3
OSCH = {"gpu_ggs": GGS, "gpu_pcgs": PCGS, "gpu_spalias": SPALIAS, "gpu_polyaurn": POLYAURN}


def _sampler(scheme, off, tokens, V, K, alpha, beta, seed, **add):
    import ldagroupedgibbssampler_b200 as L
    cfg = L.LDAConfiguration(scheme=scheme, topics=K, alpha=alpha, beta=beta, seed=seed, exec_time=0)
    s = L.GpuLDASampler(cfg)
    s.addInstances(L.InstanceList.from_csr(off, tokens, V), **add)
    return s


def _set_alpha(s, alpha):
    alpha = np.ascontiguousarray(alpha, np.float64)
    s._ck(s._L.ldagpu_set_alpha(s._h, alpha.ctypes.data))
    s.alpha = alpha


def _corpus(lens, V, seed):
    """Documents of the given lengths, word types uniform over V, sorted inside each document."""
    rng = np.random.default_rng(seed)
    lens = np.asarray(lens, np.int64)
    off = np.zeros(len(lens) + 1, np.int64)
    np.cumsum(lens, out=off[1:])
    tokens = rng.integers(0, V, int(off[-1])).astype(np.int32)
    for d in range(len(lens)):
        tokens[off[d]:off[d + 1]].sort()
    return off, tokens


def _mixed_lengths(seed):
    """Short documents (one GGS work item: theta drawn inside the z kernel), long ones (split into chunks: theta from
    the stand-alone kernel) and empty ones, shuffled."""
    rng = np.random.default_rng(seed)
    lens = np.concatenate([rng.integers(1, 60, 200), rng.integers(300, 900, 8), np.zeros(4, np.int64),
                           rng.integers(1, 33, 60)])
    rng.shuffle(lens)
    return lens


def _check_sweeps(oracle, s, scheme, off, tokens, z0, phi0, V, K, alpha, beta, seed, n, first_sweep=1):
    """The handle ran n whole sweeps from (z0, phi0), the first of them numbered first_sweep: z, counts, Phi (and GGS
    theta) bit-exact, LL and LP within 1e-9."""
    osch = OSCH[scheme]
    st = oracle.sweeps("contract", osch, off, tokens, z0, V, K, alpha, beta, seed, first_sweep, n, phi0)
    assert np.array_equal(s.get_z_flat(), st["z"])
    assert np.array_equal(s.getTypeTopicMatrix(), st["n_wk"])
    assert np.array_equal(s.getTopicTotals(), st["n_k"])
    assert np.array_equal(s.getPhi().T.astype(np.float32), st["phiT"])
    if osch == GGS:
        assert np.array_equal(s.getTheta().astype(np.float32), st["theta"])
    want_ll = oracle.log_likelihood(off, st["z"], K, V, st["n_wk"], st["n_k"], alpha, beta)
    assert abs(s.modelLogLikelihood() - want_ll) <= 1e-9 * abs(want_ll)
    lp = s.computeLogPosterior()
    if osch == GGS:
        th = st["theta"]
    else:
        # the other schemes draw a diagnostic theta ~ Dir(n_d + alpha) first, counter = current iteration
        th = oracle.theta_contract(off, st["z"], K, alpha, seed, s.getCurrentIteration())
        assert np.array_equal(s.getTheta().astype(np.float32), th)
    want_lp = oracle.log_posterior(off, tokens, st["z"], K, V, th.astype(np.float64), st["phiT"].astype(np.float64),
                                   alpha, beta)
    assert abs(lp - want_lp) <= 1e-9 * abs(want_lp)
    return st


# ---------------------------------------------------------------------------------------------------------------------
# 1. asymmetric alpha
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("scheme,K", [("gpu_ggs", 129), ("gpu_ggs", 300), ("gpu_ggs", 1000), ("gpu_ggs", 1025),
                                      ("gpu_ggs", 2600), ("gpu_pcgs", 200), ("gpu_pcgs", 1000), ("gpu_pcgs", 1500),
                                      ("gpu_spalias", 300), ("gpu_spalias", 1500), ("gpu_spalias", 4000)])
def test_asymmetric_alpha_whole_sweeps(oracle, scheme, K):
    """alpha_k = a permutation of geomspace(0.01, 2, K), set after addInstances (the initial state does not read it):
    PCGS alpha_s, the GGS theta tables and drain, the alias tables and the LL / LP kernels must all read alpha_k for
    topic k whatever column the row layout puts it in."""
    if scheme == "gpu_ggs" and K <= 1024:
        V = 700
        off, tokens = _corpus(_mixed_lengths(K), V, seed=K)
    else:
        V = 400
        off, tokens = make_corpus(60, V, 50, seed=K, empty_every=9)
    alpha = np.random.default_rng(K).permutation(np.geomspace(0.01, 2.0, K))
    beta, seed = 0.01, 13
    s = _sampler(scheme, off, tokens, V, K, 0.1, beta, seed)
    _set_alpha(s, alpha)
    z0 = s.get_z_flat()
    phi0 = s.getPhi().T.astype(np.float32).copy()
    s.sample(2)
    st = _check_sweeps(oracle, s, scheme, off, tokens, z0, phi0, V, K, alpha, beta, seed, 2)
    # the order of alpha matters on this input: the test can fail
    rev = oracle.sweeps("contract", OSCH[scheme], off, tokens, z0, V, K, alpha[::-1].copy(), beta, seed, 1, 2, phi0)
    assert not np.array_equal(rev["z"], st["z"])
    s.close()


# ---------------------------------------------------------------------------------------------------------------------
# 2. K limits (the boundary values themselves are inputs of the parametrized tests in test_gpu_parity.py)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scheme,K_max", [("gpu_ggs", 27000), ("gpu_pcgs", 18000)])
def test_create_refuses_k_beyond_dense_limit(scheme, K_max):
    """One Phi^T row and one document vector per warp must fit in shared memory: ldagpu_create refuses the first K
    beyond the limit with its message, before it looks for a device."""
    import ldagroupedgibbssampler_b200 as L
    off, tokens = make_corpus(4, 20, 5, seed=1)
    cfg = L.LDAConfiguration(scheme=scheme, topics=K_max + 1, alpha=0.1, beta=0.01, seed=1, exec_time=0)
    s = L.GpuLDASampler(cfg)
    with pytest.raises(L.LdaGpuError, match="K is too large for the dense z-step"):
        s.addInstances(L.InstanceList.from_csr(off, tokens, 20))


# ---------------------------------------------------------------------------------------------------------------------
# 3. counters above 2^32
# ---------------------------------------------------------------------------------------------------------------------
def test_oracle_counters_use_the_high_word(oracle):
    """The oracle's theta cell and token counters carry their high word into Philox: bases 2^32 apart give the same
    low words and different draws."""
    K = 256                       # 2^32 / K is an integer: doc_base + 2^24 moves every cell by exactly 2^32
    off, tokens = make_corpus(20, 60, 30, seed=3)
    z = np.random.default_rng(0).integers(0, K, len(tokens)).astype(np.int32)
    alpha = np.full(K, 0.3)
    lo = oracle.theta_contract(off, z, K, alpha, 7, 1, doc_base=5)
    hi = oracle.theta_contract(off, z, K, alpha, 7, 1, doc_base=5 + (1 << 24))
    nonempty = np.diff(off) > 0
    assert np.all(np.any(lo[nonempty] != hi[nonempty], axis=1))
    phiT = np.random.default_rng(1).dirichlet(np.full(K, 0.5), size=60).astype(np.float32)
    z_lo = oracle.z_ggs_contract(off, tokens, z, K, lo, phiT, 7, 1, token_base=0)
    z_hi = oracle.z_ggs_contract(off, tokens, z, K, lo, phiT, 7, 1, token_base=1 << 32)
    assert (z_lo != z_hi).mean() > 0.5


@gpu
@pytest.mark.parametrize("scheme,K", [("gpu_ggs", 1000), ("gpu_ggs", 1500), ("gpu_pcgs", 400), ("gpu_spalias", 1500)])
def test_counters_above_32_bits(oracle, scheme, K):
    """A shard whose theta cells (doc_base + d) * K + k and token indices token_base + t cross 2^32 in its middle: step
    by step, then one whole sweep.  GGS at K = 1000 has documents of <= 32 and > 32 tokens (32-token work items on a
    corpus this small), so the whole sweep draws theta both inside the z kernel and in the stand-alone kernel; K = 1500
    takes theta_kernel_big."""
    rng = np.random.default_rng(K)
    lens = np.concatenate([rng.integers(1, 33, 150), rng.integers(33, 200, 30), np.zeros(3, np.int64)])
    rng.shuffle(lens)
    V = 500
    off, tokens = _corpus(lens, V, seed=K + 1)
    D, N = len(off) - 1, len(tokens)
    doc_base, token_base = 2 ** 32 // K - D // 2, 2 ** 32 - N // 2
    assert doc_base * K < 2 ** 32 < (doc_base + D - 1) * K and token_base + N > 2 ** 32
    alpha, beta, seed = np.full(K, 50.0 / K), 0.01, 2019
    s = _sampler(scheme, off, tokens, V, K, 50.0 / K, beta, seed, init_z=False,
                 presharded=(doc_base, token_base, token_base + N))
    z0 = rng.integers(0, K, N).astype(np.int32)
    s.set_z_flat(z0)
    n_wk0, _ = oracle.rebuild_counts(tokens, z0, V, K)
    phi0 = s.getPhi().T.astype(np.float32).copy()
    assert np.array_equal(phi0, oracle.phi_contract(n_wk0, beta, seed, 0))   # keyed by w * K + k: no base
    s._step("next_iteration")
    if scheme == "gpu_ggs":
        s._step("sample_theta")
        th = oracle.theta_contract(off, z0, K, alpha, seed, 1, doc_base=doc_base)
        assert np.array_equal(s.getTheta().astype(np.float32), th)
        s._step("sample_z")
        want = oracle.z_ggs_contract(off, tokens, z0, K, th, phi0, seed, 1, token_base=token_base)
        at_zero = oracle.z_ggs_contract(off, tokens, z0, K, oracle.theta_contract(off, z0, K, alpha, seed, 1), phi0,
                                        seed, 1)
    elif scheme == "gpu_pcgs":
        s._step("sample_z")
        want = oracle.z_pcgs_contract(off, tokens, z0, K, alpha, phi0, seed, 1, token_base=token_base)
        at_zero = oracle.z_pcgs_contract(off, tokens, z0, K, alpha, phi0, seed, 1)
    else:
        s._step("sample_z")
        want = oracle.z_spalias_contract(off, tokens, z0, K, alpha, phi0, seed, 1, token_base=token_base)
        at_zero = oracle.z_spalias_contract(off, tokens, z0, K, alpha, phi0, seed, 1)
    assert np.array_equal(s.get_z_flat(), want)
    assert not np.array_equal(want, at_zero)
    # the same sweep as one sample(1): z-step (GGS: fused and stand-alone theta), count rebuild, Phi draw
    s.set_z_flat(z0, redraw_phi=False)
    s._L.ldagpu_set_iteration(s._h, 0)
    s.sample(1)
    n_wk1, n_k1 = oracle.rebuild_counts(tokens, want, V, K)
    assert np.array_equal(s.get_z_flat(), want)
    assert np.array_equal(s.getTypeTopicMatrix(), n_wk1) and np.array_equal(s.getTopicTotals(), n_k1)
    assert np.array_equal(s.getPhi().T.astype(np.float32), oracle.phi_contract(n_wk1, beta, seed, 1))
    if scheme == "gpu_ggs":
        assert np.array_equal(s.getTheta().astype(np.float32), th)
    s.close()


# ---------------------------------------------------------------------------------------------------------------------
# 4. the PubMed-shaped GGS sweep at full size
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_pubmed_full_size_sweep_on_sampled_documents(oracle):
    """bench.py's default workload (8.2 M documents, 738 M tokens, K = 1000) is the only size at which GGS work items
    hold 1024 tokens and theta has more than 2^31 cells.  One sweep with the streamed z read-back (8 parts); windows of
    documents are recomputed by the oracle from the initial z and Phi: the first and last documents, both sides of the
    document where the theta cell passes 2^32, the longest documents (chunked: stand-alone theta), the part boundaries
    of the read-back and seeded random windows.  theta itself (65 GB as doubles) is not read back."""
    import torch

    import ldagroupedgibbssampler_b200 as L
    free, _ = torch.cuda.mem_get_info()
    if free < 64 * 2 ** 30:
        pytest.skip(f"needs 64 GB of free device memory (the sampler holds about 45 GB), {free / 2 ** 30:.0f} GB free")
    D, V, mean_len, K, alpha, beta = 8_200_000, 141_043, 90.0, 1000, 0.05, 0.01
    CORPUS_SEED, SEED = 20190529, 2019
    off, tokens = L.synth_corpus(D, V, mean_len, seed=CORPUS_SEED)
    N = len(tokens)
    lens = np.diff(off)
    s = _sampler("gpu_ggs", off, tokens, V, K, alpha, beta, SEED)
    z0 = s.get_z_flat()
    phi0 = np.ascontiguousarray(s.getPhi().T.astype(np.float32))
    buf = np.full(N, -1, np.int32)
    s.sample(1, z_out=buf)
    assert np.array_equal(buf, s.get_z_flat())
    assert np.array_equal(s.getTopicTotals(), np.bincount(buf, minlength=K))

    longest = np.argsort(lens, kind="stable")[-20:]
    assert lens[longest].min() > 1024, "the longest documents must be split into work items"
    d_cross = -(-2 ** 32 // K)
    windows = [(0, 16), (D - 16, D), (d_cross - 8, d_cross + 8)]
    windows += [(int(d), int(d) + 1) for d in longest]
    for p in range(1, 8):                                       # engine.cu build_items: 8 parts of ~N/8 tokens
        d = int(np.searchsorted(off, N // 8 * p, side="right")) - 1
        windows.append((d - 8, d + 8))
    rng = np.random.default_rng(SEED)
    windows += [(int(d), int(d) + 16) for d in rng.integers(0, D - 16, 50)]
    a = np.full(K, alpha)
    for d0, d1 in windows:
        t0, t1 = int(off[d0]), int(off[d1])
        sub_off = off[d0:d1 + 1] - t0
        th = oracle.theta_contract(sub_off, z0[t0:t1], K, a, SEED, 1, doc_base=d0)
        want = oracle.z_ggs_contract(sub_off, tokens[t0:t1], z0[t0:t1], K, th, phi0, SEED, 1, token_base=t0)
        assert np.array_equal(buf[t0:t1], want), (d0, d1)
    s.close()


# ---------------------------------------------------------------------------------------------------------------------
# 5. degenerate scores
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("scheme", ["gpu_ggs", "gpu_pcgs"])
def test_degenerate_scores_injected(oracle, scheme):
    """Injected Phi with word types whose scores are all zero (S = 0), non-zero only at topic K - 1 or only at topic 0,
    or 2^-149 everywhere (the products underflow); GGS theta rows one-hot at either end or in the middle, and uniform.
    S = 0 takes topic 0 (DESIGN.md 4.2: the first k with cumsum_k >= U * S = 0)."""
    K, V, D = 300, 200, 80
    off, tokens = make_corpus(D, V, 40, seed=3)      # types 0..3 are the most frequent
    rng = np.random.default_rng(5)
    phi = rng.dirichlet(np.full(V, 0.05), size=K)    # [K][V]
    phi[:, 0] = 0.0
    phi[:, 1] = 0.0
    phi[K - 1, 1] = 0.25
    phi[:, 2] = 0.0
    phi[0, 2] = 0.25
    phi[:, 3] = 2.0 ** -149
    theta = rng.dirichlet(np.full(K, 0.2), size=D)
    for i, d in enumerate(range(0, D, 4)):
        theta[d] = 0.0
        theta[d, (0, K - 1, K // 2)[i % 3]] = 1.0
    theta[1::4] = 1.0 / K
    alpha, seed = 0.1, 9
    s = _sampler(scheme, off, tokens, V, K, alpha, 0.01, seed)
    z0 = s.get_z_flat()
    s.setPhi(phi)
    phiT = np.ascontiguousarray(phi.T.astype(np.float32))
    if scheme == "gpu_ggs":
        s.setTheta(theta)
    s._step("next_iteration")
    s._step("sample_z")
    if scheme == "gpu_ggs":
        want = oracle.z_ggs_contract(off, tokens, z0, K, theta.astype(np.float32), phiT, seed, 1)
    else:
        want = oracle.z_pcgs_contract(off, tokens, z0, K, np.full(K, alpha), phiT, seed, 1)
    got = s.get_z_flat()
    assert np.array_equal(got, want)
    assert np.all(got[tokens == 0] == 0)                 # S = 0
    assert np.all(got[tokens == 2] == 0)
    assert np.any(got[tokens == 1] == K - 1)
    s.close()


@gpu
@pytest.mark.parametrize("scheme,K,alpha,beta", [("gpu_ggs", 1000, 1e-4, 0.01), ("gpu_ggs", 1000, 200.0, 0.01),
                                                 ("gpu_pcgs", 400, 0.125, 1e-6), ("gpu_pcgs", 400, 0.125, 50.0)])
def test_whole_sweeps_extreme_hyperparameters(oracle, scheme, K, alpha, beta):
    """alpha = 1e-4: almost every theta cell underflows to the 2^-149 floor; alpha = 200: flat theta; beta = 1e-6 / 50:
    Phi close to the counts / close to uniform."""
    import ldagroupedgibbssampler_b200 as L
    V = 1200
    off, tokens = L.synth_corpus(300, V, 80.0, seed=4)
    seed = 2019
    s = _sampler(scheme, off, tokens, V, K, alpha, beta, seed)
    z0 = s.get_z_flat()
    phi0 = s.getPhi().T.astype(np.float32).copy()
    s.sample(2)
    _check_sweeps(oracle, s, scheme, off, tokens, z0, phi0, V, K, np.full(K, alpha), beta, seed, 2)
    s.close()
