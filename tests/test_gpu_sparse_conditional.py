"""The sparse z-step's draw on the device against the exact float64 conditional, at K = 10 000 and alpha = 0.005, the
shape of the wiki-shaped workloads.

The parity tests compare the kernel with the CPU oracle bit for bit. A flaw in how the draw uses its uniforms is
then shared by both and invisible there. Here one token is drawn 2^26 times from a planted state whose conditional is
known in closed form, and the topic counts are compared with it.

Planted state: V = 2 (word A under test, filler word B). A's Phi column is a flat Gamma(1) column except at one topic
k*, where phi_{k*,A} = 1/2; B takes the rest of every topic. Every document is A followed by c tokens of B, all with
z = k*. When token 0 is drawn, the document's non-zero list is {k*: c}, so its conditional is
    p_k  ~  alpha_k phi_kA + [k = k*] c phi_{k*,A},
and the scale of the flat part sets the prior's share tn / tot of the mass: the alias draw serves that share. One token
of k* alone cannot push the share below alpha / (1 + alpha), so the smallest share takes c = 20. c = 0 (one-token
documents, an empty list) is the control at share 1. p is formed in float64 from the device's own fp32 Phi and fp32
alpha.

Every repetition restores the planted z without redrawing Phi, sets the sweep number and runs one z-only sweep: the
sweep number keys fresh uniforms. Nothing on this path allocates a D x K array: theta is allocated only for GGS or when
it is read or set."""
import numpy as np
import pytest
from scipy import stats

pytestmark = pytest.mark.gpu

K, ALPHA, BETA, SEED = 10_000, 0.005, 0.01, 2026
K_STAR, PHI_STAR = 4321, 0.5
DOCS, DRAWS = 1 << 20, 1 << 26


def _planted_phi(share, c):
    """Phi [K][2]: A's column flat (Gamma(1)) with phi_{k*,A} = PHI_STAR, scaled so that tn / (tn + c PHI_STAR) = share."""
    rng = np.random.default_rng(7)
    col = rng.gamma(1.0, size=K)
    col[K_STAR] = 0.0
    flat = 10.0 if c == 0 else share * c * PHI_STAR / (ALPHA * (1.0 - share)) - PHI_STAR
    assert flat > 0, "share too small for c tokens at k*"
    col *= flat / col.sum()
    col[K_STAR] = PHI_STAR
    return np.stack([col, 1.0 - col], axis=1)


def _pooled_chi2(obs, p, n):
    """Chi-square of the counts against n p, topics pooled in order of expectation until every bin expects >= 5."""
    e = n * p
    order = np.argsort(e, kind="stable")
    bins = np.empty(K, np.int64)
    nb, acc = 0, 0.0           # nb = closed bins
    for k in order:
        bins[k] = nb
        acc += e[k]
        if acc >= 5.0:
            nb, acc = nb + 1, 0.0
    if acc > 0.0:              # the last, short bin joins the one before
        bins[bins == nb] = nb - 1
    eb = np.bincount(bins, e, nb)
    ob = np.bincount(bins, obs.astype(np.float64), nb)
    chi2 = float(((ob - eb) ** 2 / eb).sum())
    return chi2, nb - 1, float(stats.chi2.sf(chi2, nb - 1))


@pytest.mark.parametrize("scheme,share,c", [("gpu_spalias", 1.0, 0), ("gpu_spalias", 0.1, 1), ("gpu_spalias", 0.01, 2),
                                            ("gpu_spalias", 0.001, 20), ("gpu_pcgs", 1.0, 0)])
def test_draw_matches_the_exact_conditional(scheme, share, c):
    """gpu_pcgs, the dense shared-memory path, is the calibration: it draws from the same conditional with one 23-bit
    uniform over the whole mass. It runs at share 1, where that grid gives every topic ~840 points. At share 0.01 it
    gives the flat topics ~8 points each, and its own rounding would then show up in the statistic."""
    import ldagroupedgibbssampler_b200 as L
    A, B = 0, 1
    off = np.arange(DOCS + 1, dtype=np.int64) * (1 + c)
    tokens = np.tile(np.array([A] + [B] * c, np.int32), DOCS)
    z_planted = np.full(len(tokens), K_STAR, np.int32)
    cfg = L.LDAConfiguration(scheme=scheme, topics=K, alpha=ALPHA, beta=BETA, seed=SEED, exec_time=0)
    s = L.GpuLDASampler(cfg)
    s.addInstances(L.InstanceList.from_csr(off, tokens, 2))
    s.setPhi(_planted_phi(share, c))
    phi_a = s.getPhi()[:, A]                       # the device's fp32 values
    p = float(np.float32(ALPHA)) * phi_a
    tn = p.sum()
    p[K_STAR] += c * phi_a[K_STAR]
    p /= p.sum()
    got_share = tn / (tn + c * phi_a[K_STAR])
    first = off[:-1]
    obs = np.zeros(K, np.int64)
    for rep in range(DRAWS // DOCS):
        s.set_z_flat(z_planted, redraw_phi=False)
        s._ck(s._L.ldagpu_set_iteration(s._h, rep))    # the z-only sweep runs as sweep rep + 1
        s.sampleZGivenPhi(1)
        obs += np.bincount(s.get_z_flat()[first], minlength=K)
    s.close()
    n = int(obs.sum())
    assert n == DRAWS
    chi2, df, pval = _pooled_chi2(obs, p, n)
    e_star, sd_star = n * p[K_STAR], np.sqrt(n * p[K_STAR] * (1.0 - p[K_STAR]))
    msg = (f"{scheme}, share tn/tot = {got_share:.4g} (c = {c}), {n} draws: chi2 = {chi2:.1f} on {df} df "
           f"(excess {chi2 - df:.0f}, null sd {np.sqrt(2 * df):.0f}), p = {pval:.3g}; "
           f"k*: {obs[K_STAR]} drawn, {e_star:.1f} +- {sd_star:.1f} expected")
    print(msg)
    assert abs(obs[K_STAR] - e_star) <= 5.0 * sd_star, msg
    assert pval > 1e-6, msg
