#!/usr/bin/env python
"""bench.py -- token-topic samples/sec of one Gibbs sweep (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload pubmed|pubmed8|nips|enron|wiki8|wiki8_polya] [--scaling strong|weak]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the CPU port of the reference's sampler, same metric and config
    python bench.py ... --dump-outputs DIR    # also write the sampler state after the last timed step (one process)

A "step" is one full sweep ([theta +] z with the count rebuild, [exchange], Phi draw) over the corpus.
Default workload: BASELINE.json configs[3] -- the WHOLE PubMed-shaped corpus (8.2 M documents, ~738 M tokens,
V = 141 043), GGS K = 1000.  It fits one B200 (tokens + z 5.9 GB, theta 33.6 GB, Phi^T + n_wk 1.2 GB), so N = 1
runs all of it and N GPUs share the same fixed corpus: `scaling` is "strong".  Phi^T is 578 MB, larger than the
126 MB L2, so no L2 flush is needed between steps.  `--workload pubmed8 / wiki8` keep the round-1 weak-scaling
shards (one eighth of the corpus per GPU).

value   device-resident: K sweeps inside ONE ldagpu_sweep call, timed with CUDA events on the library's
        stream, max over ranks.
e2e     the same metric through the sampler API with host buffers: every step uploads z from pinned
        host memory (setZIndicators path, keeps Phi), runs sample(1, z_out=...) which reads z back, and
        reads the topic totals.  K <= 65 536: z travels as uint16 (ldagpu_set_z16 / ldagpu_sweep_get_z16).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # D = documents of the WHOLE corpus for scaling "strong", documents per GPU for scaling "weak"
    "pubmed": dict(desc="PubMed-shaped GGS K=1000, V=141043, the whole 8.2M-doc corpus (BASELINE.json configs[3])",
                   D=8200000, V=141043, mean_len=90.0, K=1000, scheme="gpu_ggs", alpha=0.05, beta=0.01, scaling="strong"),
    "pubmed8": dict(desc="PubMed-shaped GGS K=1000, V=141043, per-GPU shard = 1/8 of the 8.2M-doc corpus",
                    D=1025000, V=141043, mean_len=90.0, K=1000, scheme="gpu_ggs", alpha=0.05, beta=0.01, scaling="weak"),
    "nips": dict(desc="NIPS-shaped GGS K=100 (BASELINE.json configs[1])",
                 D=1500, V=12419, mean_len=1267.0, K=100, scheme="gpu_ggs", alpha=1.0, beta=0.01, scaling="strong"),
    "enron": dict(desc="Enron-shaped PCGS K=400 (BASELINE.json configs[2])",
                  D=39861, V=28102, mean_len=161.0, K=400, scheme="gpu_pcgs", alpha=0.125, beta=0.01, scaling="strong"),
    "wiki8": dict(desc="Wikipedia-shaped sparse PCGS K=10000, V=100000, per-GPU shard = 1/8 of the ~4M-doc corpus "
                       "(BASELINE.json configs[4] at 8 GPUs)",
                  D=500000, V=100000, mean_len=250.0, K=10000, scheme="gpu_spalias", alpha=0.005, beta=0.01, scaling="weak"),
    "wiki8_polya": dict(desc="Wikipedia-shaped K=10000, V=100000, per-GPU shard = 1/8 of the ~4M-doc corpus, sparse z-step with "
                             "the Poisson Polya-urn Phi draw (the reference's scheme polyaurn: sparse rows of Phi)",
                        D=500000, V=100000, mean_len=250.0, K=10000, scheme="gpu_polyaurn", alpha=0.005, beta=0.01, scaling="weak"),
}
METRIC = "token-topic samples/sec per Gibbs sweep"
UNIT = "tokens/s"
SEED = 2019
CORPUS_SEED = 20190529


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def profile_record(workload):
    """What the committed `ncu --set full` capture of the z-step kernel says for this workload shape
    (profiles/z_kernel_traffic.json: DRAM and L2->SM bytes per token, the binding unit).  None when there is no
    capture for the shape."""
    p = os.path.join(ROOT, "profiles", "z_kernel_traffic.json")
    if os.path.exists(p):
        return json.load(open(p)).get(workload)
    return None


DUMP_Z = 4 << 20           # topic indicators kept (float32: 16 MiB)
DUMP_CELLS = 2 << 20       # cells of the n_wk rows (float64: 16 MiB) and of the same Phi^T rows (float32: 8 MiB)


def dump_outputs(s, out_dir):
    """What a caller of sample() receives after the last timed sweep, as DIR/<name>.npy: the topic indicators z,
    the type-topic counts n_wk and Phi^T (the same rows of both, [rows][K]), the topic totals n_k and the model
    log-likelihood.  Arrays larger than the caps above are a sample drawn from SEED, the same one for the same
    corpus shape, so two builds run with the same arguments can be compared output for output.  theta is left out:
    it is D x K (33.6 GB on the default workload), the library exports it only whole, and z is drawn from it."""
    rng = np.random.default_rng(SEED)

    def pick(n, cap):
        return np.arange(n) if n <= cap else np.sort(rng.choice(n, cap, replace=False))

    z = s.get_z_flat()
    z = z[pick(len(z), DUMP_Z)]
    rows = pick(s.numTypes, max(1, DUMP_CELLS // s.numTopics))
    n_wk = s.getTypeTopicMatrix()[rows]
    phiT = s.getPhi().T[rows]
    out = {"z": z.astype(np.float32), "n_wk_rows": n_wk.astype(np.float64), "phiT_rows": phiT.astype(np.float32),
           "n_k": s.getTopicTotals().astype(np.float64),
           "log_likelihood": np.array([s.modelLogLikelihood()], np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def make_config(name, wl, scaling):
    """Identical keys in both arms (ours and --impl reference)."""
    ks = (wl["K"] + 31) // 32 * 32
    return {"workload": wl["desc"], "name": name, "scheme": wl["scheme"], "K": wl["K"], "V": wl["V"],
            "docs": wl["D"], "docs_are": "whole corpus" if scaling == "strong" else "per GPU",
            "mean_doc_len": wl["mean_len"], "alpha": wl["alpha"], "beta": wl["beta"], "scaling": scaling,
            "corpus_seed": CORPUS_SEED, "seed": SEED,
            "l2": ("inputs larger than L2 (Phi^T %.0f MB, corpus + theta several GB), no flush"
                   if wl["V"] * 4 * wl["K"] > 126e6 else
                   "Phi^T %.0f MB is L2-resident, no flush -- the HBM roofline is a loose bound here")
                  % (wl["V"] * 4 * ks / 1e6)}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self, gpu_indices):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9 or not c[0].isdigit() or int(c[0]) not in gpu_indices:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2]))
            except ValueError:
                continue
            for n, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        os.unlink(self.f.name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def bind_to_gpu_numa_node(local_rank):
    """Run this rank's host thread (and so the first touch of its pinned buffers) on the NUMA node of its GPU."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(local_rank)],
                             capture_output=True, text=True, timeout=10).stdout.strip().lower()
        bdf = out[-12:] if len(out) >= 12 else out          # 00000000:1b:00.0 -> 0000:1b:00.0
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


def cpu_baseline(wl, off, tokens, budget_tokens, n_total_tokens, threads):
    """The reference's sampler restated on the CPU (oracle, faithful mode, the reference's threading
    shape) on a bounded sample: whole documents up to `budget_tokens` tokens, one sweep, `threads` host
    threads.  z cost is per token, Phi cost is per sweep (K*V Gammas, independent of the sample), so
    the rate on the whole workload is N / (N * z_sec_per_token + phi_sec): an EXTRAPOLATION, flagged as such.
    Returns (record, wall seconds of this sample)."""
    from oracle import oracle as O
    w0 = time.perf_counter()
    d1 = int(np.searchsorted(off, budget_tokens, side="right")) - 1
    d1 = max(1, min(d1, len(off) - 1))
    o, t = off[: d1 + 1].copy(), tokens[: off[d1]].copy()
    K, V = wl["K"], wl["V"]
    z = O.java_next_ints(SEED, K, len(t))
    if wl["scheme"] in ("gpu_spalias", "gpu_polyaurn"):
        # the reference's own sparse sampler (SpaliasUncollapsedParallelLDA), restated in double: per sweep
        # alias tables for all V types + Phi draw (both O(K*V)); per token the sparse walk
        alpha = np.full(K, wl["alpha"])
        n_wk, _ = O.rebuild_counts(t, z, V, K)
        t0 = time.perf_counter()
        phi = O.phi_faithful(n_wk, wl["beta"], SEED, 0)
        ps = time.perf_counter() - t0
        del n_wk
        t0 = time.perf_counter()
        O.z_spalias_faithful(o[:1], t[:0], z[:0], K, alpha, phi, SEED, 1)      # alias build only
        ab = time.perf_counter() - t0
        t0 = time.perf_counter()
        O.z_spalias_faithful(o, t, z, K, alpha, phi, SEED, 1)
        zs = max(time.perf_counter() - t0 - ab, 1e-9)
        nt = O.lib().oracle_max_threads()
        per_tok = zs / max(len(t), 1)
        value = n_total_tokens / (n_total_tokens * per_tok + ps + ab)
        what = (f"token loop {zs:.3f}s ({per_tok * 1e9:.1f} ns/token), alias tables {ab:.3f}s and Phi draw {ps:.3f}s "
                f"(both full K*V); C restatement (oracle/lda_oracle_sparse.c)")
    else:
        sch = O.GGS if wl["scheme"] == "gpu_ggs" else O.PCGS
        zs, ps, nt = O.baseline_sweeps(sch, o, t, z, V, K, np.full(K, wl["alpha"]), wl["beta"], SEED, 1, n_threads=threads)
        per_tok = zs / max(len(t), 1)
        value = n_total_tokens / (n_total_tokens * per_tok + ps)
        what = (f"z+merge {zs:.3f}s ({per_tok * 1e9:.1f} ns/token), Phi draw {ps:.3f}s (full K*V); C restatement "
                f"(oracle/lda_oracle.c oracle_baseline_sweeps)")
    rec = {"value": value, "unit": UNIT, "cores": nt, "kind": "port", "extrapolated": True,
           "sample": f"{d1} documents / {len(t)} tokens of the same corpus, 1 sweep: {what}; rate extrapolated to the "
                     f"{n_total_tokens}-token workload; no JDK in the image, so this is the C port, not the Java reference"}
    return rec, time.perf_counter() - w0


def reference_arm(args, name, wl, scaling):
    """--impl reference: the reference's own CPU implementation of the path (C port of the Java sampler; no JDK in
    the image) on all host threads, rank 0 only.  Loads the oracle and the host-only corpus generator -- never
    libldagpu.so."""
    threads = os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = str(threads)      # torchrun exports OMP_NUM_THREADS=1 to its workers
    os.environ.pop("OMP_PROC_BIND", None)
    from ldagroupedgibbssampler_b200._lib import synth_corpus
    n_gpus = max(args.gpus, 1)
    docs_total = wl["D"] * (n_gpus if scaling == "weak" else 1)
    n_total = int(round(docs_total * wl["mean_len"]))
    sample_docs = int(min(wl["D"], max(2000, 1.3 * args.cpu_sample_tokens / wl["mean_len"])))
    off, tokens = synth_corpus(sample_docs, wl["V"], wl["mean_len"], seed=CORPUS_SEED)
    vals, walls = [], []
    for i in range(args.warmup + args.steps):
        r, wall = cpu_baseline(wl, off, tokens, args.cpu_sample_tokens, n_total, threads)
        if i >= args.warmup:
            vals.append(r); walls.append(wall)
    v = float(np.mean([x["value"] for x in vals]))
    cb = dict(vals[-1]); cb["value"] = v
    return {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * float(np.mean(walls)), "ms_per_step_is": "wall time of one bounded-sample step "
            "(the extrapolated whole-workload sweep would take %.1f s)" % (n_total / v),
            "extrapolated": True, "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": make_config(name, wl, scaling),
            "cpu_baseline": cb,
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="pubmed", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default=None, choices=["strong", "weak"],
                    help="strong: N GPUs share the workload's documents; weak: every GPU gets that many (default per workload)")
    ap.add_argument("--docs", type=int, default=0, help="override the workload's document count (debugging)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="N=1: skip the NIPS-/Enron-/Wikipedia-shaped side measurements")
    ap.add_argument("--cpu-sample-tokens", type=int, default=3_000_000)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the state of the last one as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and (args.impl != "ours" or world > 1):
        ap.error("--dump-outputs needs --impl ours in one process")
    wl = dict(WORKLOADS[args.workload])
    if args.docs:
        wl["D"] = args.docs
    scaling = args.scaling or wl["scaling"]

    if args.impl == "reference":
        return reference_arm(args, args.workload, wl, scaling) if rank == 0 else None

    # ----------------------------------------------------------------------------------------
    import torch
    import torch.distributed as dist

    import ldagroupedgibbssampler_b200 as L

    if world > 1:
        dist.init_process_group("nccl" if torch.cuda.is_available() else "gloo")
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(local_rank)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def all_max(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def measure(name, wl, scaling, steps, warmup, with_e2e, with_clocks, with_props=True, dump_dir=None):
        """One workload on this process group: device-resident sweeps, then the end-to-end loop."""
        if scaling == "strong":
            d0, d1 = wl["D"] * rank // world, wl["D"] * (rank + 1) // world      # this rank's documents of the fixed corpus
        else:
            d0, d1 = rank * wl["D"], (rank + 1) * wl["D"]
        t0 = time.time()
        off, tokens = L.synth_corpus(d1 - d0, wl["V"], wl["mean_len"], seed=CORPUS_SEED, doc_first=d0)
        n_local = len(tokens)
        if world > 1:
            sizes = [torch.zeros(1, dtype=torch.int64, device="cuda") for _ in range(world)]
            dist.all_gather(sizes, torch.tensor([n_local], dtype=torch.int64, device="cuda"))
            sizes = [int(s.item()) for s in sizes]
        else:
            sizes = [n_local]
        token_base, n_total = sum(sizes[:rank]), sum(sizes)
        gen_s = time.time() - t0

        cfg = L.LDAConfiguration(scheme=wl["scheme"], topics=wl["K"], alpha=wl["alpha"], beta=wl["beta"], seed=SEED,
                                 exec_time=0)
        s = L.GpuLDASampler(cfg, device=local_rank)
        comm_id = None
        if world > 1:
            box = [L.GpuLDASampler.make_comm_id() if rank == 0 else None]
            dist.broadcast_object_list(box, src=0)
            comm_id = box[0]
        s.addInstances(L.InstanceList.from_csr(off, tokens, wl["V"]), rank=rank, world=world, comm_id=comm_id,
                       presharded=(d0, token_base, n_total))

        # ---- device-resident: warm-up, then exactly K sweeps in one library call ---------------
        s.sample(warmup, chunk=0)
        it0 = s.getCurrentIteration()
        clocks = ClockSampler()
        barrier()
        if rank == 0 and with_clocks:
            clocks.start()
        w0 = time.perf_counter()
        s.sample(steps, chunk=0)
        barrier()
        wall_ms = (time.perf_counter() - w0) * 1e3
        call_ms, zk_ms, zk_launches, launches = s.getLastCallStats()
        if s.getCurrentIteration() - it0 != steps:
            raise RuntimeError(f"{name}: the timed call ran {s.getCurrentIteration() - it0} sweeps, not {steps}")
        ck = clocks.stop(set(range(world))) if (rank == 0 and with_clocks) else None
        if dump_dir:
            dump_outputs(s, dump_dir)
        need_more = 1.0 if (rank == 0 and with_clocks and (ck.get("samples") or 0) < 3) else 0.0
        wall_ms = all_max(wall_ms)
        if all_max(need_more) > 0:
            # the timed region was shorter than nvidia-smi's sampling period (small workloads): sample the clocks
            # over an untimed repeat of the same sweeps, long enough for a few samples
            reps = max(steps, int(0.8 / max(wall_ms / 1e3 / steps, 1e-6)))
            clocks2 = ClockSampler()
            barrier()
            if rank == 0:
                clocks2.start()
                time.sleep(0.15)
            s.sample(reps, chunk=0)
            barrier()
            if rank == 0:
                ck = clocks2.stop(set(range(world)))
                ck["note"] = (f"timed region ({wall_ms:.1f} ms) shorter than the sampling period: clocks sampled over an "
                              f"untimed repeat of {reps} sweeps of the same workload")
        dev_ms = all_max(call_ms)
        zk_ms_per_launch = all_max(zk_ms / max(zk_launches, 1))
        res = {"value": n_total * steps / (dev_ms / 1e3), "ms_per_step": dev_ms / steps, "clocks": ck,
               "launches": int(launches), "zk_ms_per_launch": zk_ms_per_launch, "zk_share": zk_ms / max(call_ms, 1e-9),
               "n_total": n_total, "sizes": sizes, "gen_s": gen_s, "wall_ms_per_step": wall_ms / steps,
               "exchange": s.getExchangeMode(), "timers": dict(zip(("z", "counts", "phi", "comm"), s.getTimers()))}

        # ---- roofline inputs: how many Phi^T row fetches a token costs on this corpus ------------------------
        ns = min(n_local, 30_000_000)
        if ns > 1:
            ds = int(np.searchsorted(off, ns, side="right")) - 1
            ns = int(off[ds])
            tk = tokens[:ns]
            pos = np.arange(ns, dtype=np.int64) - np.repeat(off[:ds], np.diff(off[: ds + 1]))
            head = np.ones(ns, bool)
            head[1:] = tk[1:] != tk[:-1]
            head |= (pos & 31) == 0        # a run ends at the 32-token block of the warp
            res["fetches_per_token"] = float(head.mean())
        mean_nnz = None
        if wl["scheme"] in ("gpu_spalias", "gpu_polyaurn"):
            # SURVEY 8(d) sparse z-step: 12 + 8*nnz_d + 16 bytes per token, nnz_d measured on a sample of documents
            zf, dsamp = s.get_z_flat(), min(len(off) - 1, 20000)
            nnz = np.array([len(np.unique(zf[off[d]:off[d + 1]])) for d in range(dsamp)], np.float64)
            lens = np.diff(off[: dsamp + 1]).astype(np.float64)
            mean_nnz = float((nnz * lens).sum() / max(lens.sum(), 1.0))
        res["mean_nnz"] = mean_nnz

        # ---- end to end through the sampler API with pinned host buffers -----------------------
        if with_e2e:
            z16 = wl["K"] <= 65536
            zbuf = torch.empty(max(n_local, 1), dtype=torch.uint16 if z16 else torch.int32, pin_memory=True)
            znp = zbuf.numpy()[:n_local]
            znp[:] = s.get_z_flat().astype(znp.dtype)
            import ctypes as C
            lib = L.load()
            set_z = lib.ldagpu_set_z16 if z16 else lib.ldagpu_set_z

            def e2e_step():
                s._ck(set_z(s._h, C.c_void_p(zbuf.data_ptr()), 0))                 # H2D z (+ count rebuild, Phi kept)
                s.sample(1, z_out=znp, chunk=0)                                     # sweep; D2H z under the Phi draw
                return s.getTopicTotals()                                           # D2H n_k

            for _ in range(max(1, min(warmup, 2))):
                e2e_step()
            barrier()
            e0 = time.perf_counter()
            for _ in range(steps):
                e2e_step()
            barrier()
            e2e_ms = all_max((time.perf_counter() - e0) * 1e3)
            esz = 2 if z16 else 4
            res["e2e"] = {"value": n_total * steps / (e2e_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": esz * n_local,
                          "d2h_bytes_per_step": esz * n_local + 4 * wl["K"], "ms_per_step": e2e_ms / steps,
                          "z_dtype": "uint16" if z16 else "int32", "numa_node": numa,
                          "what": "per step: ldagpu_set_z16 from pinned host z (upload pipelined with the widening and the "
                                  "count rebuild), sample(1, z_out=pinned host z) = ldagpu_sweep_get_z16 (z narrowed and read "
                                  "back in document-aligned parts under the z-step of the following parts; small corpora and "
                                  "the PCGS schemes: under the Phi draw), getTopicTotals; host wall clock, max over ranks; "
                                  "bytes are per rank"}
        # ---- size-independent properties of the sampler state at the workload's full size (untimed) ----------------
        if with_props:
            K, V = wl["K"], wl["V"]
            zf = s.get_z_flat()
            n_k = np.asarray(s.getTopicTotals(), np.int64)
            hist = np.bincount(zf, minlength=K).astype(np.int64)
            if world > 1:
                ht = torch.from_numpy(hist).cuda()
                dist.all_reduce(ht)
                hist = ht.cpu().numpy()
            props = {"tokens": int(n_total),
                     "z_in_range": bool(n_local == 0 or (int(zf.min()) >= 0 and int(zf.max()) < K)),
                     "n_k_is_histogram_of_z": bool(np.array_equal(n_k, hist)),
                     "sum_n_k_is_N": int(n_k.sum()) == int(n_total)}
            if world == 1 and K * V <= 200_000_000:
                n_wk = s.getTypeTopicMatrix()
                props["n_wk_column_sums_are_n_k"] = bool(np.array_equal(n_wk.sum(axis=0, dtype=np.int64), n_k))
                props["n_wk_row_sums_are_type_counts"] = bool(np.array_equal(
                    n_wk.sum(axis=1, dtype=np.int64), np.bincount(tokens, minlength=V).astype(np.int64)))
                s._step("rebuild_counts")                      # idempotence: the rebuild from the same z changes nothing
                props["count_rebuild_idempotent"] = bool(np.array_equal(s.getTypeTopicMatrix(), n_wk))
                del n_wk
                phi = s.getPhi()
                props["phi_rows_sum_to_1"] = bool(np.all(np.abs(phi.sum(axis=1) - 1.0) < 1e-4))
                if wl["scheme"] != "gpu_polyaurn":             # the urn keeps exact zeros (DESIGN 4.7)
                    props["phi_positive"] = bool(phi.min() > 0.0)
                del phi
            del zf
            bad = [k for k, v in props.items() if v is False]
            if bad:
                raise RuntimeError(f"{name}: state properties violated at full size: {bad}")
            res["properties"] = props
        s.close()
        return res, off, tokens

    config = make_config(args.workload, wl, scaling)
    res, off, tokens = measure(args.workload, wl, scaling, args.steps, args.warmup, True, True,
                               dump_dir=args.dump_outputs)

    # ---- roofline of the dominant kernel (z-step; GGS: with the fused theta draw) ---------------------
    peak, peak_src = peaks()
    n_launch = max(res["sizes"])                               # one launch processes the rank's tokens
    t_s = res["zk_ms_per_launch"] / 1e3
    ks = (wl["K"] + 127) // 128 * 128 if wl["K"] <= 1024 else (wl["K"] + 31) // 32 * 32
    prof = profile_record(args.workload) or {}
    if res["mean_nnz"] is not None:
        bytes_per_token = 28 + 8 * res["mean_nnz"]
        kernel = "z_spalias_kernel"
    else:
        bytes_per_token = 4 * wl["K"] + 12                      # SURVEY 8(d): one fp32 K-vector + w + z in + z out
        kernel = "z_kernel"
    model_bytes = bytes_per_token * n_launch
    dram_pt = prof.get("dram_bytes_per_token")
    traffic = dram_pt * n_launch if dram_pt else None
    achieved = (traffic / t_s / 1e9) if traffic else None
    fpt = res.get("fetches_per_token")
    roofline = {"bound": "hbm", "kernel": kernel, "unit": "GB/s", "peak": peak, "peak_source": peak_src,
                "achieved": achieved, "frac": (achieved / peak) if achieved else None,
                "achieved_is": "DRAM bytes the kernel really moves (ncu dram__bytes_read+write per token of the committed "
                               "capture of this kernel on this workload shape, x the tokens of one launch) / the launch "
                               "duration measured live with CUDA events" if achieved else
                               "no committed ncu capture for this workload shape: frac left null rather than guessed",
                "traffic": traffic, "traffic_source": prof.get("source"),
                "kernel_ms_per_launch": res["zk_ms_per_launch"], "kernel_share_of_step": res["zk_share"],
                "achieved_model": model_bytes / t_s / 1e9, "frac_model": model_bytes / t_s / 1e9 / peak,
                "model": "SURVEY 8(d) algorithmic figure: %.0f bytes per token x %d tokens per launch; it charges one Phi^T "
                         "row per TOKEN, so it exceeds the HBM peak whenever rows are shared or cached -- kept for "
                         "reference, not a roofline fraction" % (bytes_per_token, n_launch),
                "algorithmic_bytes_per_launch": model_bytes, "bytes_per_token": bytes_per_token,
                "mean_nnz_d": res["mean_nnz"], "fetches_per_token": fpt,
                "dedup_bytes": (fpt * 4 * ks * n_launch) if (fpt and res["mean_nnz"] is None) else None,
                "dedup_is": "row fetches the kernel issues (one per run of equal word types inside a 32-token block, "
                            "counted on this corpus) x 4*Ks bytes: the L2->SM traffic of the launch",
                "binding": prof.get("binding")}
    if roofline["dedup_bytes"]:
        roofline["l2_to_sm_gbs"] = roofline["dedup_bytes"] / t_s / 1e9

    out = {"metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
           "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": config,
           "run": {"exchange": res["exchange"], "tokens_total": res["n_total"], "tokens_per_gpu": res["sizes"],
                   "corpus_gen_s": round(res["gen_s"], 1), "wall_ms_per_step": res["wall_ms_per_step"]},
           "clocks": res["clocks"], "e2e": res["e2e"], "gpu_launches": res["launches"], "roofline": roofline,
           "timers_ms": res["timers"],
           "properties": dict(res["properties"], what="checked after the timed loops on the state of the whole workload, "
                                                       "untimed; a violated property aborts the run")}

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"], _ = cpu_baseline(wl, off, tokens, args.cpu_sample_tokens, res["n_total"], os.cpu_count() or 1)
    del off, tokens

    # ---- the other BASELINE.json configs on one GPU, measured in the same run (N = 1 only) ------------------------
    if world == 1 and not args.no_secondary and not args.docs:
        sec = {}
        for nm in ("nips", "enron", "wiki8", "wiki8_polya"):
            if nm == args.workload:
                continue
            w2 = dict(WORKLOADS[nm])
            try:
                big = nm.startswith("wiki8")
                r2, _, _ = measure(nm, w2, w2["scaling"], 5 if big else 50, 2 if big else 5, False, False)
                sec[nm] = {"config": make_config(nm, w2, w2["scaling"]), "value": r2["value"], "unit": UNIT,
                           "ms_per_step": r2["ms_per_step"], "steps": 5 if big else 50,
                           "tokens_total": r2["n_total"], "z_kernel_ms_per_launch": r2["zk_ms_per_launch"],
                           "fetches_per_token": r2.get("fetches_per_token"), "mean_nnz_d": r2["mean_nnz"],
                           "timers_ms_since_create": r2["timers"], "properties": r2.get("properties")}
            except Exception as e:   # a side measurement must not take the headline down with it
                sec[nm] = {"error": str(e)[:200]}
        out["secondary"] = sec

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return out if rank == 0 else None


if __name__ == "__main__":
    # Libraries (NCCL's version banner, for one) write to the process's stdout; the contract is ONE JSON
    # line there.  Point fd 1 at stderr while the benchmark runs and restore it for the result.
    sys.stdout.flush()
    _saved_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        _result = main()
    finally:
        sys.stdout.flush()
        os.dup2(_saved_stdout, 1)
        os.close(_saved_stdout)
    if _result is not None:
        print(json.dumps(_result), flush=True)
