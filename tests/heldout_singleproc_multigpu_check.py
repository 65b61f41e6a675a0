"""Held-out evaluation on several GPUs of ONE process (ldagpu_create_multi, `gpu_devices = 0,1,..`): the test set is
sharded by tokens over the shards and phihat is built once and copied to the others.  For every scheme, after two sweeps
on `--gpus` devices, the per-document values and the total must equal, bit for bit, the CPU contract restatement on the
device's counts (tests/heldout_oracle.c) -- the values one GPU gives -- and two evaluations at the same iteration must
agree.  K > 1024 is refused with an error naming the limit.

    python tests/heldout_singleproc_multigpu_check.py --gpus 2        (1, 2, 4 or 8)
"""
import argparse
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
os.environ.setdefault("LDAGPU_P2P_TIMEOUT_MS", "10000")   # a broken exchange should fail this check in seconds
import heldout_oracle as H  # noqa: E402
import ldagroupedgibbssampler_b200 as L  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=2)
    args = ap.parse_args()
    devices = list(range(args.gpus))
    ok = True
    for scheme, K, V in (("gpu_ggs", 100, 900), ("gpu_pcgs", 400, 1300), ("gpu_ggs", 1000, 2100),
                         ("gpu_spalias", 1000, 700), ("gpu_spalias", 1500, 700)):
        alpha, beta, seed = 50.0 / K, 0.01, 2019
        off, tokens = L.synth_corpus(400, V, 70.0, seed=8)
        toff, ttok = L.synth_corpus(150, V, 50.0, seed=9, doc_first=400)
        cfg = L.LDAConfiguration(scheme=scheme, topics=K, alpha=alpha, beta=beta, seed=seed, exec_time=0)
        s = L.GpuLDASampler(cfg, devices=devices)
        s.addInstances(L.InstanceList.from_csr(off, tokens, V))
        s.sample(2)
        checks = {}
        if K <= 1024:
            s.addTestInstances(L.InstanceList.from_csr(toff, ttok, V))
            tot, dll = s.heldOutLogLikelihood(10)
            tot2, dll2 = s.heldOutLogLikelihood(10)
            want_t, want_d = H.heldout_l2r("contract", toff, ttok, s.getTypeTopicMatrix(), s.getTopicTotals(), s.alpha,
                                           beta, seed, s.getCurrentIteration(), R=10)
            checks.update(heldout=tot == want_t and np.array_equal(dll, want_d),
                          repeatable=tot2 == tot and np.array_equal(dll2, dll))
        else:
            try:
                s.addTestInstances(L.InstanceList.from_csr(toff, ttok, V))
                checks["heldout_refused"] = False
            except L.LdaGpuError as e:
                checks["heldout_refused"] = "K <= 1024" in str(e)
        print(scheme, K, f"{args.gpus} GPUs, one process:", checks, flush=True)
        ok &= all(bool(v) for v in checks.values())
        s.close()
    if not ok:
        sys.exit(1)
    print("heldout_singleproc_multigpu_check ok, gpus =", args.gpus)


if __name__ == "__main__":
    main()
