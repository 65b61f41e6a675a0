"""Held-out evaluation on the GPU (DESIGN.md 4.8): ldagpu_set_test_documents / ldagpu_heldout_log_likelihood against the
contract oracle bit for bit, against the faithful oracle within the tolerance of tests/test_oracle_heldout.py, free of side
effects on training, refusals, the sample() series, and a two-GPU shard group against one GPU."""
import ctypes as C

import numpy as np
import pytest

import ldagroupedgibbssampler_b200 as L
from ldagroupedgibbssampler_b200._lib import LdaGpuError, ptr
from conftest import make_corpus

pytestmark = pytest.mark.gpu

SEED, BETA, V = 4242, 0.01, 700


def _sampler(scheme, K, off, tokens, V=V, alpha=None, sweeps=2, **kw):
    cfg = L.LDAConfiguration(scheme=scheme, topics=K, alpha=alpha if alpha else 50.0 / K, beta=BETA, seed=SEED,
                             exec_time=0)
    s = L.GpuLDASampler(cfg, **kw)
    s.addInstances(L.InstanceList.from_csr(off, tokens, V))
    if sweeps:
        s.sample(sweeps)
    return s


def _test_set(seed=21, D=120, mean_len=35, V=V, empty_every=6):
    """ragged test documents with empty ones, types in random order (runs of equal types are rare but present)"""
    return make_corpus(D, V, mean_len, seed, sort_docs=False, empty_every=empty_every)


def _expect(oracle, s, toff, ttok, R):
    """the contract oracle on the sampler's current counts, alpha, beta and iteration"""
    return oracle.heldout_l2r("contract", toff, ttok, s.getTypeTopicMatrix(), s.getTopicTotals(), s.alpha, s.beta,
                              SEED, s.getCurrentIteration(), R=R)


def _check(oracle, s, toff, ttok, R):
    s.addTestInstances(L.InstanceList.from_csr(toff, ttok, s.numTypes))
    total, ll = s.heldOutLogLikelihood(R)
    t_o, ll_o = _expect(oracle, s, toff, ttok, R)
    assert np.array_equal(ll, ll_o), np.flatnonzero(ll != ll_o)[:10]
    assert total == t_o
    assert np.all(ll[np.diff(toff) == 0] == 0.0)
    return total, ll


@pytest.mark.parametrize("scheme", ["gpu_ggs", "gpu_pcgs"])
@pytest.mark.parametrize("K", [3, 100, 128, 129, 400, 1000, 1024])
def test_bit_exact_dense(oracle, scheme, K):
    off, tokens = make_corpus(300, V, 50, 11, sort_docs=False)
    s = _sampler(scheme, K, off, tokens)
    toff, ttok = _test_set()
    _check(oracle, s, toff, ttok, 10)


@pytest.mark.parametrize("K", [100, 1000])
def test_bit_exact_sparse_natural_order(oracle, K):
    """gpu_spalias keeps n_wk in natural topic order (row stride round_up(K, 32)): phihat is rebuilt in the register
    path's layout"""
    off, tokens = make_corpus(300, V, 50, 12, sort_docs=False)
    s = _sampler("gpu_spalias", K, off, tokens)
    toff, ttok = _test_set(seed=22)
    _check(oracle, s, toff, ttok, 10)


@pytest.mark.parametrize("K", [3, 129, 1000])
def test_one_particle(oracle, K):
    off, tokens = make_corpus(300, V, 50, 13, sort_docs=False)
    s = _sampler("gpu_pcgs", K, off, tokens)
    toff, ttok = _test_set(seed=23, D=200)
    _check(oracle, s, toff, ttok, 1)


def test_runs_of_equal_types_and_long_documents(oracle):
    """sorted documents (long runs share one row fetch) and documents of several thousand tokens"""
    off, tokens = make_corpus(300, V, 50, 14)
    s = _sampler("gpu_ggs", 400, off, tokens)
    toff, ttok = make_corpus(12, V, 3000, 24, sort_docs=True, empty_every=5)
    _check(oracle, s, toff, ttok, 10)


def test_from_a_burned_in_state(oracle):
    """200 device sweeps on an LDA-generated corpus (the pattern of test_gpu_converged.py), so that n_wk is
    concentrated, then the evaluation against the oracle on the device's counts"""
    V2 = 2000
    off, tokens = L.synth_corpus(3000, V2, 60.0, seed=31)
    s = _sampler("gpu_pcgs", 400, off, tokens, V=V2, alpha=0.05, sweeps=0)
    start = (s.getTypeTopicMatrix() > 0).mean()
    s.sample(200)
    assert (s.getTypeTopicMatrix() > 0).mean() < 0.5 * start   # the counts have concentrated
    toff, ttok = L.synth_corpus(300, V2, 60.0, seed=32, doc_first=3000)
    _check(oracle, s, toff, ttok, 10)


def test_asymmetric_alpha(oracle):
    off, tokens = make_corpus(300, V, 50, 15, sort_docs=False)
    s = _sampler("gpu_ggs", 250, off, tokens)
    s.alpha = np.random.default_rng(5).uniform(0.01, 0.8, 250)
    s._ck(s._L.ldagpu_set_alpha(s._h, ptr(s.alpha)))
    toff, ttok = _test_set(seed=25)
    _check(oracle, s, toff, ttok, 10)


def test_several_scratch_batches(oracle):
    """R * N_test floats beyond the 1 GiB bound of the score buffer: the test set is evaluated in document batches"""
    R = 1000
    off, tokens = make_corpus(200, 60, 40, 16, sort_docs=False)
    s = _sampler("gpu_pcgs", 3, off, tokens, V=60)
    toff, ttok = make_corpus(3000, 60, 100, 26, sort_docs=False, empty_every=50)
    assert R * int(toff[-1]) * 4 > 2 ** 30
    _check(oracle, s, toff, ttok, R)


def test_faithful_cats(oracle, cats):
    """cats corpus, K = 10, R = 10: the device against the faithful (fp64, libm) oracle, within the tolerances that
    tests/test_oracle_heldout.py::test_contract_against_faithful measured"""
    off, tokens = cats
    Vc = int(tokens.max()) + 1
    s = _sampler("gpu_pcgs", 10, off, tokens, V=Vc, alpha=0.1, sweeps=5)
    s.addTestInstances(L.InstanceList.from_csr(off, tokens, Vc))
    total, ll = s.heldOutLogLikelihood(10)
    tf, f = oracle.heldout_l2r("faithful", off, tokens, s.getTypeTopicMatrix(), s.getTopicTotals(), s.alpha, s.beta,
                               SEED, s.getCurrentIteration(), R=10)
    rel = np.abs(ll - f) / np.abs(f)
    assert rel.max() <= 1e-2 and (rel > 1e-6).mean() <= 0.03
    assert abs(total - tf) <= 5e-5 * abs(tf)


def _state(s, with_theta):
    st = dict(z=s.get_z_flat(), n_wk=s.getTypeTopicMatrix(), n_k=s.getTopicTotals(), phi=s.getPhi(),
              it=s.getCurrentIteration(), ll=s.modelLogLikelihood())
    if with_theta:
        st["theta"] = s.getTheta()
    return st


@pytest.mark.parametrize("scheme", ["gpu_ggs", "gpu_spalias"])
def test_no_side_effects(oracle, scheme):
    """sweeps, two evaluations, more sweeps: the same state as the same run without the evaluations, and the two
    evaluations at the same iteration agree"""
    off, tokens = make_corpus(300, V, 50, 17, sort_docs=False)
    toff, ttok = _test_set(seed=27)
    a = _sampler(scheme, 200, off, tokens, sweeps=3)
    b = _sampler(scheme, 200, off, tokens, sweeps=3)
    a.addTestInstances(L.InstanceList.from_csr(toff, ttok, V))
    e1, e2 = a.heldOutLogLikelihood(10), a.heldOutLogLikelihood(10)
    assert e1[0] == e2[0] and np.array_equal(e1[1], e2[1])
    a.sample(3)
    b.sample(3)
    sa, sb = _state(a, scheme == "gpu_ggs"), _state(b, scheme == "gpu_ggs")
    for k in sa:
        assert np.array_equal(sa[k], sb[k]), k


def test_refusals_keep_the_previous_test_set(oracle):
    off, tokens = make_corpus(300, V, 50, 18, sort_docs=False)
    s = _sampler("gpu_pcgs", 100, off, tokens)
    toff, ttok = _test_set(seed=28)
    before = _check(oracle, s, toff, ttok, 10)
    bad = ttok.copy()
    bad[5] = V
    with pytest.raises(LdaGpuError, match="out of range"):
        s.addTestInstances(L.InstanceList.from_csr(toff, bad, V))
    bad_off = toff.copy()
    bad_off[3], bad_off[4] = bad_off[4] + 1, bad_off[3]
    with pytest.raises(LdaGpuError, match="non-decreasing"):
        s.addTestInstances(L.InstanceList.from_csr(bad_off, ttok, V))
    assert s._L.ldagpu_set_test_documents(s._h, 2, ptr(np.array([1, 2, 3], np.int64)), ptr(ttok), 0, 0) != 0
    # the refused uploads left the first test set in place
    out = np.zeros(len(toff) - 1)
    total = C.c_double(0)
    s._ck(s._L.ldagpu_heldout_log_likelihood(s._h, 10, ptr(out), C.byref(total)))
    assert total.value == before[0] and np.array_equal(out, before[1])
    with pytest.raises(LdaGpuError, match="n_particles"):
        s.heldOutLogLikelihood(0)
    big = _sampler("gpu_ggs", 1500, off, tokens, sweeps=0)
    with pytest.raises(LdaGpuError, match="K <= 1024"):
        big.addTestInstances(L.InstanceList.from_csr(toff, ttok, V))
    # D_test = 0 removes the test set: the total is 0
    s._ck(s._L.ldagpu_set_test_documents(s._h, 0, None, None, 0, 0))
    s._ck(s._L.ldagpu_heldout_log_likelihood(s._h, 10, None, C.byref(total)))
    assert total.value == 0.0


def test_sample_fills_the_series_on_the_likelihood_grid(oracle):
    off, tokens = make_corpus(300, V, 50, 19, sort_docs=False)
    toff, ttok = _test_set(seed=29)
    cfg = L.LDAConfiguration(scheme="gpu_ggs", topics=50, beta=BETA, seed=SEED, exec_time=0, compute_likelihood=True,
                             topic_interval=5)
    s = L.GpuLDASampler(cfg)
    s.addInstances(L.InstanceList.from_csr(off, tokens, V))
    assert s.getHeldOutLogLikelihood() == []
    s.addTestInstances(L.InstanceList.from_csr(toff, ttok, V))
    s.sample(20)
    series = s.getHeldOutLogLikelihood()
    assert len(series) == len(s.getLogLikelihood()) == 5   # before the first sweep, then every 5 sweeps
    assert series[-1] == _expect(oracle, s, toff, ttok, 10)[0]
    assert series[-1] == s.heldOutLogLikelihood()[0]
    # without a test set the series stays empty
    t = L.GpuLDASampler(cfg)
    t.addInstances(L.InstanceList.from_csr(off, tokens, V))
    t.sample(10)
    assert t.getHeldOutLogLikelihood() == []


@pytest.mark.parametrize("scheme", ["gpu_ggs", "gpu_spalias"])
def test_shard_group_matches_one_gpu(oracle, scheme):
    """ldagpu_create_multi on 2 GPUs (the test set sharded by tokens over them) returns the bits of one GPU"""
    if L.load().ldagpu_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    off, tokens = L.synth_corpus(400, V, 70.0, seed=8)
    toff, ttok = _test_set(seed=30, D=300)
    one = _sampler(scheme, 100, off, tokens, sweeps=3)
    two = _sampler(scheme, 100, off, tokens, sweeps=3, devices=[0, 1])
    r1 = _check(oracle, one, toff, ttok, 10)
    r2 = _check(oracle, two, toff, ttok, 10)
    assert r1[0] == r2[0] and np.array_equal(r1[1], r2[1])
