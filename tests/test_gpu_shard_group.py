"""A shard group (`ldagpu_create_multi` on 2 GPUs) against a plain single-GPU handle, bit for bit, for the entry points
that tests/singleproc_multigpu_check.py does not run on a group: the Phi mean, the count histograms, set_alpha /
set_beta, set_theta, abort and the Polya-urn Phi sampler.  Needs >= 2 GPUs; skipped otherwise."""
import ctypes as C

import numpy as np
import pytest

import ldagroupedgibbssampler_b200 as L
from ldagroupedgibbssampler_b200._lib import ptr

pytestmark = pytest.mark.gpu

K, V, SEED = 100, 900, 2019


@pytest.fixture(scope="module", autouse=True)
def two_gpus():
    if L.load().ldagpu_device_count() < 2:
        pytest.skip("needs 2 GPUs")


def pair(scheme="gpu_ggs", K=K, V=V):
    """The same corpus on one GPU and as a group of two shards."""
    off, tokens = L.synth_corpus(400, V, 70.0, seed=8)
    cfg = L.LDAConfiguration(scheme=scheme, topics=K, alpha=50.0 / K, beta=0.01, seed=SEED, exec_time=0,
                             alias_poisson_threshold=4)
    out = []
    for kw in (dict(device=0), dict(devices=[0, 1])):
        s = L.GpuLDASampler(cfg, **kw)
        s.addInstances(L.InstanceList.from_csr(off, tokens, V))
        out.append(s)
    assert out[1].getExchangeMode() == "p2p"
    return out


def same_state(a, b):
    assert np.array_equal(a.get_z_flat(), b.get_z_flat())
    assert np.array_equal(a.getTypeTopicMatrix(), b.getTypeTopicMatrix())
    assert np.array_equal(a.getTopicTotals(), b.getTopicTotals())
    assert np.array_equal(a.getPhi(), b.getPhi())
    assert a.getCurrentIteration() == b.getCurrentIteration()


def test_phi_mean_schedule_and_reset_by_set_phi():
    one, grp = pair()
    for s in (one, grp):
        s._ck(s._L.ldagpu_set_phi_mean_schedule(s._h, 2, 2))
        s.sample(7)
    m1, mg = one.getPhiMeans(), grp.getPhiMeans()
    assert m1 is not None and np.array_equal(m1, mg)
    phi = one.getPhi()
    for s in (one, grp):
        s.setPhi(phi)
        assert s.getPhiMeans() is None
        s._step("rebuild_counts")
        s._step("sample_phi")   # iteration 7: not on the thinning grid
        s.sample(1)
    m1, mg = one.getPhiMeans(), grp.getPhiMeans()
    assert m1 is not None and np.array_equal(m1, mg)
    same_state(one, grp)


def test_count_histograms():
    one, grp = pair()
    for s in (one, grp):
        s.sample(2)
    for h1, hg in zip(one._count_histograms(), grp._count_histograms()):
        assert np.array_equal(h1, hg)
    dh, th = one._count_histograms()[:2]
    assert dh.sum() == 400 * K and th.sum() == V * K


def test_set_alpha_asymmetric_and_set_beta_then_sweeps():
    one, grp = pair()
    alpha = np.linspace(0.05, 1.5, K)
    for s in (one, grp):
        s.sample(1)
        s.alpha = alpha.copy()
        s._ck(s._L.ldagpu_set_alpha(s._h, ptr(s.alpha)))
        s._ck(s._L.ldagpu_set_beta(s._h, 0.03))
        s.sample(2)
    same_state(one, grp)
    ll1, llg = one.modelLogLikelihood(), grp.modelLogLikelihood()   # partial sums added in another order
    assert abs(ll1 - llg) <= 1e-9 * abs(ll1)


def test_set_theta_then_sample_z():
    one, grp = pair()
    theta = np.random.default_rng(5).gamma(0.5, size=(400, K))
    theta /= theta.sum(axis=1, keepdims=True)
    for s in (one, grp):
        s.setTheta(theta)
        s._step("sample_z")
    assert np.array_equal(one.getTheta(), grp.getTheta())
    assert np.array_equal(one.get_z_flat(), grp.get_z_flat())


def test_abort_before_a_call_runs_no_sweep():
    one, grp = pair()
    for s in (one, grp):
        s.sample(1)
        z0, it0 = s.get_z_flat(), s.getCurrentIteration()
        s.abort()
        assert s.getAbort()
        done = C.c_int32(-1)
        s._ck(s._L.ldagpu_sweep(s._h, 3, C.byref(done)))
        assert done.value == 0 and s.getCurrentIteration() == it0
        assert np.array_equal(s.get_z_flat(), z0)
    same_state(one, grp)


def test_polya_urn_scheme():
    one, grp = pair("gpu_polyaurn", K=200, V=700)
    same_state(one, grp)
    for s in (one, grp):
        s.sample(3)
    same_state(one, grp)
