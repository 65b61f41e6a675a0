"""One process, several GPUs (ldagpu_create_multi): the reference runs one coordinator thread in one JVM
(tui/ParallelLDA.java:173-202), so `gpu_devices = 0,1,..` must give what one GPU gives.  Runs every scheme on
`--gpus` devices from THIS process and compares with the CPU oracle on the whole corpus, bit for bit:
whole sweeps, a z-only sweep, the step-wise count rebuild + Phi draw, setZIndicators (32- and 16-bit, the
refused out-of-range case included), theta / document-topic accessors in corpus order, log-likelihood and
log-posterior, checkpoint/resume, and the held-out evaluation of a test set (DESIGN.md 4.8).

    python tests/singleproc_multigpu_check.py --gpus 2
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("LDAGPU_P2P_TIMEOUT_MS", "10000")   # a broken exchange should fail this check in seconds
import ldagroupedgibbssampler_b200 as L  # noqa: E402
from oracle import oracle as O  # noqa: E402


def stalled_shard(gpus):
    """A shard that never publishes its Phi rows (fault injection, LDAGPU_FAULT_STALL_SHARD): the bounded in-kernel
    waits of the others must end in the library's error, within the timeout, not in a hung GPU."""
    import time
    assert os.environ.get("LDAGPU_FAULT_STALL_SHARD") is not None and int(os.environ["LDAGPU_P2P_TIMEOUT_MS"]) <= 2000
    off, tokens = L.synth_corpus(400, 900, 70.0, seed=8)
    cfg = L.LDAConfiguration(scheme="gpu_ggs", topics=100, alpha=0.5, beta=0.01, seed=1, exec_time=0)
    s = L.GpuLDASampler(cfg, devices=list(range(gpus)))
    s.addInstances(L.InstanceList.from_csr(off, tokens, 900))
    t0 = time.time()
    try:
        s.sample(1)
    except L.LdaGpuError as e:
        dt = time.time() - t0
        print("stalled shard reported after %.2f s: %s" % (dt, e))
        assert "timed out" in str(e) and dt < 30
        print("stalled_shard ok")
        return
    print("no error raised")
    sys.exit(1)


def heldout(s, V, K, beta, seed):
    """Held-out evaluation on the group: the test set is sharded by tokens over the shards and phihat is built once and
    copied to the others.  The per-document values and the total must equal the oracle's contract mode on the device's
    counts bit for bit -- the values one GPU gives -- and two evaluations at the same iteration must agree.  K > 1024 is
    refused with an error naming the limit."""
    toff, ttok = L.synth_corpus(150, V, 50.0, seed=9, doc_first=400)
    if K > 1024:
        try:
            s.addTestInstances(L.InstanceList.from_csr(toff, ttok, V))
            return dict(heldout_refused=False)
        except L.LdaGpuError as e:
            return dict(heldout_refused="K <= 1024" in str(e))
    s.addTestInstances(L.InstanceList.from_csr(toff, ttok, V))
    tot, dll = s.heldOutLogLikelihood(10)
    tot2, dll2 = s.heldOutLogLikelihood(10)
    want_t, want_d = O.heldout_l2r("contract", toff, ttok, s.getTypeTopicMatrix(), s.getTopicTotals(), s.alpha, beta, seed,
                                   s.getCurrentIteration(), R=10)
    return dict(heldout=tot == want_t and np.array_equal(dll, want_d),
                heldout_repeatable=tot2 == tot and np.array_equal(dll2, dll))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=2)
    ap.add_argument("--stress", type=int, default=0, help="extra sweeps with host-side jitter between calls")
    ap.add_argument("--stalled-shard", action="store_true",
                    help="run with LDAGPU_FAULT_STALL_SHARD / a short LDAGPU_P2P_TIMEOUT_MS: expect the error, not a hang")
    args = ap.parse_args()
    if args.stalled_shard:
        return stalled_shard(args.gpus)
    devices = list(range(args.gpus))
    ok = True
    for scheme, osch, K, V in (("gpu_ggs", O.GGS, 100, 900), ("gpu_pcgs", O.PCGS, 400, 1300), ("gpu_ggs", O.GGS, 1000, 2100),
                               ("gpu_spalias", O.SPALIAS, 1500, 700)):
        alpha, beta, seed = 50.0 / K, 0.01, 2019
        off, tokens = L.synth_corpus(400, V, 70.0, seed=8)
        cfg = L.LDAConfiguration(scheme=scheme, topics=K, alpha=alpha, beta=beta, seed=seed, exec_time=0)
        s = L.GpuLDASampler(cfg, devices=devices)
        s.addInstances(L.InstanceList.from_csr(off, tokens, V))
        al = np.full(K, alpha)
        z0 = O.java_next_ints(seed, K, len(tokens))
        nw0, _ = O.rebuild_counts(tokens, z0, V, K)
        phi0 = O.phi_contract(nw0, beta, seed, 0)
        checks = dict(z0=np.array_equal(s.get_z_flat(), z0), phi0=np.array_equal(s.getPhi().T.astype(np.float32), phi0),
                      mode=s.getExchangeMode() == ("p2p" if args.gpus > 1 else "single"))
        s.sample(2)
        st = O.sweeps("contract", osch, off, tokens, z0, V, K, al, beta, seed, 1, 2, phi0)
        want_ll = O.log_likelihood(off, st["z"], K, V, st["n_wk"], st["n_k"], al, beta)
        checks.update(z=np.array_equal(s.get_z_flat(), st["z"]), n_wk=np.array_equal(s.getTypeTopicMatrix(), st["n_wk"]),
                      n_k=np.array_equal(s.getTopicTotals(), st["n_k"]),
                      phi=np.array_equal(s.getPhi().T.astype(np.float32), st["phiT"]),
                      ll=abs(s.modelLogLikelihood() - want_ll) <= 1e-9 * abs(want_ll),
                      n_dk=np.array_equal(s.getDocumentTopicMatrix(), O.doc_topic_counts(off, st["z"], K)))
        if osch == O.GGS:
            checks["theta"] = np.array_equal(s.getTheta().astype(np.float32), st["theta"])
            want_lp = O.log_posterior(off, tokens, st["z"], K, V, st["theta"].astype(np.float64),
                                      st["phiT"].astype(np.float64), al, beta)
            checks["lp"] = abs(s.computeLogPosterior() - want_lp) <= 1e-9 * abs(want_lp)
        # the evaluation changes no state, so the checks below are unaffected
        checks.update(heldout(s, V, K, beta, seed))
        # z-only sweep (Phi frozen): stand-alone count exchange, no Phi draw
        s.sampleZGivenPhi(1)
        z3 = s.get_z_flat()
        nw3, nk3 = O.rebuild_counts(tokens, z3, V, K)
        checks["zonly_phi_kept"] = np.array_equal(s.getPhi().T.astype(np.float32), st["phiT"])
        checks["zonly_n_wk"] = np.array_equal(s.getTypeTopicMatrix(), nw3)
        checks["zonly_n_k"] = np.array_equal(s.getTopicTotals(), nk3)
        # step-wise API: count rebuild with its own exchange, then a Phi draw on already-merged counts
        s._step("rebuild_counts")
        s._step("sample_phi")
        checks["step_n_wk"] = np.array_equal(s.getTypeTopicMatrix(), nw3)
        checks["step_phi"] = np.array_equal(s.getPhi().T.astype(np.float32), O.phi_contract(nw3, beta, seed, 3))
        # setZIndicators, both widths; an out-of-range indicator on the LAST shard is refused everywhere
        rng = np.random.default_rng(1)
        zr = rng.integers(0, K, len(tokens)).astype(np.int32)
        s.set_z_flat(zr, redraw_phi=False)
        nwr, nkr = O.rebuild_counts(tokens, zr, V, K)
        checks["setz"] = np.array_equal(s.getTypeTopicMatrix(), nwr) and np.array_equal(s.get_z_flat(), zr)
        bad = zr.copy(); bad[-3] = K
        try:
            s.set_z_flat(bad, redraw_phi=False)
            checks["setz_refused"] = False
        except L.LdaGpuError:
            checks["setz_refused"] = np.array_equal(s.get_z_flat(), zr) and np.array_equal(s.getTypeTopicMatrix(), nwr) \
                and np.array_equal(s.getTopicTotals(), nkr)
        s.set_z16_flat(z3.astype(np.uint16), redraw_phi=False)
        out16 = np.zeros(len(tokens), np.uint16)
        # checkpoint / resume: (z, Phi, iteration) into a fresh multi-GPU sampler continues bit-identically
        phi_ck, it_ck = s.getPhi(), s.getCurrentIteration()
        s.sample(2, z_out=out16)
        checks["z16_out"] = np.array_equal(out16.astype(np.int32), s.get_z_flat())
        r = L.GpuLDASampler(cfg, devices=devices)
        r.addInstances(L.InstanceList.from_csr(off, tokens, V), init_z=False)
        r.set_z_flat(z3, redraw_phi=False)
        r.setPhi(phi_ck)
        r._L.ldagpu_set_iteration(r._h, it_ck)
        r.sample(2)
        checks["resume"] = np.array_equal(r.get_z_flat(), s.get_z_flat()) and np.array_equal(r.getPhi(), s.getPhi())
        r.close()
        if args.stress:
            # exchange-protocol stress: many short calls with host-side jitter between them; the epoch flags must keep
            # every shard in step (a lost or early signal shows up as a wrong count or a timeout)
            import time
            zt = s.get_z_flat()
            pt = s.getPhi().T.astype(np.float32).copy()
            it0 = s.getCurrentIteration()
            for i in range(args.stress):
                if i % 3 == 0:
                    time.sleep(float(rng.uniform(0, 0.003)))
                s.sample(1)
                if i % 7 == 3:
                    s._step("rebuild_counts")
            stt = O.sweeps("contract", osch, off, tokens, zt, V, K, al, beta, seed, it0 + 1, args.stress, pt)
            checks["stress"] = np.array_equal(s.get_z_flat(), stt["z"]) and np.array_equal(s.getTypeTopicMatrix(), stt["n_wk"])
        print(scheme, K, f"{args.gpus} GPUs, one process:", checks, flush=True)
        ok &= all(bool(v) for v in checks.values())
        s.close()
    # the sparse scheme keeps n_wk in natural topic order, phihat is in the register path's layout: held-out only
    K, V = 1000, 700
    s = L.GpuLDASampler(L.LDAConfiguration(scheme="gpu_spalias", topics=K, alpha=50.0 / K, beta=0.01, seed=2019, exec_time=0),
                        devices=devices)
    s.addInstances(L.InstanceList.from_csr(*L.synth_corpus(400, V, 70.0, seed=8), V))
    s.sample(2)
    checks = heldout(s, V, K, 0.01, 2019)
    print("gpu_spalias", K, f"{args.gpus} GPUs, one process:", checks, flush=True)
    ok &= all(checks.values())
    s.close()
    if not ok:
        sys.exit(1)
    print("singleproc_multigpu_check ok, gpus =", args.gpus)


if __name__ == "__main__":
    main()
