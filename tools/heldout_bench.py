"""Time one held-out evaluation (ldagpu_heldout_log_likelihood, DESIGN.md 4.8) and print one JSON line.

    python tools/heldout_bench.py [--particles 10] [--repeats 3] [--device 0]

Two shapes (corpus.SHAPES): a 10 % PubMed-shaped test split (820 000 documents of mean length 90, ~74 M tokens, V = 141 043,
K = 1000) held out from a 1.6 M-document PubMed-shaped training slice, and a 10 % NIPS-shaped split (150 documents of mean
length 1267, V = 12 419, K = 100) held out from the other 1350 documents.  The model is whatever the counts are after two
sweeps from the random start (the estimator's cost does not depend on the counts' values).  Per shape: the wall time of
the synchronous call (median of --repeats, after one warm-up call; it includes the phihat build and the copies back) and
tokens x particles per second.  For comparison, as bench.py's cpu_baseline does, the rate of the faithful CPU
restatement (tests/heldout_oracle.c) on the first documents of the split (at most 2 M token-particles, all host
threads).  The card's name and power limit are read in the same run.  Writes nothing."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import heldout_oracle as O  # noqa: E402  (the CPU restatement, tests/heldout_oracle.c)
import ldagroupedgibbssampler_b200 as L  # noqa: E402
from ldagroupedgibbssampler_b200.corpus import SHAPES  # noqa: E402


def card(device):
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(device)],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception as e:   # the numbers stay usable without the card's name
        return f"unknown ({e})", "unknown"


def run_shape(shape, train_docs, test_docs, R, repeats, device, seed=20190529):
    sh = SHAPES[shape]
    V, K = sh["V"], sh["K"]
    off, tokens = L.synth_corpus(train_docs, V, sh["mean_len"], seed=seed)
    toff, ttok = L.synth_corpus(test_docs, V, sh["mean_len"], seed=seed, doc_first=train_docs)
    cfg = L.LDAConfiguration(scheme="gpu_pcgs", topics=K, alpha=sh["alpha"], beta=sh["beta"], seed=1, exec_time=0)
    s = L.GpuLDASampler(cfg, device=device)
    s.addInstances(L.InstanceList.from_csr(off, tokens, V))
    s.sample(2)
    s.addTestInstances(L.InstanceList.from_csr(toff, ttok, V))
    total = s.heldOutLogLikelihood(R)[0]   # warm-up (module load, first allocations)
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        t = s.heldOutLogLikelihood(R)[0]
        times.append(time.perf_counter() - t0)
        assert t == total   # same iteration: the same value
    sec = float(np.median(times))
    n_test = int(toff[-1])
    res = dict(shape=shape, K=K, V=V, test_docs=test_docs, test_tokens=n_test, particles=R,
               eval_ms=round(sec * 1e3, 2), eval_ms_all=[round(x * 1e3, 2) for x in times],
               token_particles_per_s=n_test * R / sec, heldout_ll=total)
    # faithful CPU oracle on a bounded sample of the same split, counts from the device
    n_wk, n_k = s.getTypeTopicMatrix(), s.getTopicTotals()
    d = int(np.searchsorted(toff, 2_000_000 // R, side="right")) - 1
    d = max(1, min(d, test_docs))
    t0 = time.perf_counter()
    O.heldout_l2r("faithful", toff[: d + 1], ttok[: toff[d]], n_wk, n_k, s.alpha, s.beta, 1, s.getCurrentIteration(), R=R)
    cpu = time.perf_counter() - t0
    res.update(cpu_faithful_docs=d, cpu_faithful_token_particles_per_s=int(toff[d]) * R / cpu,
               cpu_threads=os.cpu_count())
    s.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--particles", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--device", type=int, default=0)
    args = ap.parse_args()
    name, power = card(args.device)
    out = dict(metric="heldout_eval", card=name, power_limit=power,
               pubmed=run_shape("pubmed", 1_600_000, 820_000, args.particles, args.repeats, args.device),
               nips=run_shape("nips", 1350, 150, args.particles, args.repeats, args.device))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
