"""Run under torchrun on >= 2 GPUs: the sharded library run (NCCL reduce-scatter / all-gather inside
libldagpu) must give bit-identical z, counts, Phi and (1e-9) log-likelihood to the CPU oracle run on
the whole corpus -- results do not depend on the number of GPUs (SURVEY 8e "Determinism").

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29511 tests/multigpu_check.py
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ldagroupedgibbssampler_b200 as L  # noqa: E402
from ldagroupedgibbssampler_b200._lib import ptr  # noqa: E402
from oracle import oracle as O  # noqa: E402


def stress(rank, world, local, sweeps):
    """Exchange-protocol stress in place of racecheck (compute-sanitizer is closed on this pool): an Enron-shaped PCGS
    slice, `sweeps` single-sweep calls with random per-rank host sleeps between them (every rank its own random stream, so
    the ranks arrive skewed), stand-alone count rebuilds and Phi redraws mixed in, and the final state must equal the
    oracle's on the whole corpus bit for bit -- in whichever exchange mode LDAGPU_EXCHANGE selects."""
    import faulthandler
    import time
    if os.environ.get("LDAGPU_STRESS_DUMP_AFTER"):   # where is every rank if the run stalls?
        faulthandler.dump_traceback_later(float(os.environ["LDAGPU_STRESS_DUMP_AFTER"]), exit=True)
    K, V, alpha, beta, seed = 400, 28102, 0.125, 0.01, 2019
    off, tokens = L.synth_corpus(3000, V, 161.0, seed=20190529)
    cfg = L.LDAConfiguration(scheme="gpu_pcgs", topics=K, alpha=alpha, beta=beta, seed=seed, exec_time=0)
    s = L.GpuLDASampler(cfg, device=local)
    box = [L.GpuLDASampler.make_comm_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    s.addInstances(L.InstanceList.from_csr(off, tokens, V), rank=rank, world=world, comm_id=box[0])
    rng = np.random.default_rng(1000 + rank)
    t_loop = time.time()
    for i in range(sweeps):
        if rng.random() < 0.4:
            time.sleep(float(rng.uniform(0, 0.004)))
        s.sample(1)
        if i % 17 == 5:                       # same call sequence on every rank, different timing
            s._step("rebuild_counts")
        if i % 29 == 7:
            s.getTopicTotals()
    print(f"[rank {rank}] stress loop done after {time.time() - t_loop:.1f} s", flush=True)
    zs = [None] * world
    dist.all_gather_object(zs, s.get_z_flat())
    z = np.concatenate(zs)
    n_wk, phi = s.getTypeTopicMatrix(), s.getPhi().T.astype(np.float32)
    mode = s.getExchangeMode()
    s.close()
    faulthandler.cancel_dump_traceback_later()
    ok = True
    if rank == 0:
        O.set_num_threads(os.cpu_count() or 1)
        z0 = O.java_next_ints(seed, K, len(tokens))
        nw0, _ = O.rebuild_counts(tokens, z0, V, K)
        st = O.sweeps("contract", O.PCGS, off, tokens, z0, V, K, np.full(K, alpha), beta, seed, 1, sweeps,
                      O.phi_contract(nw0, beta, seed, 0))
        checks = dict(z=np.array_equal(z, st["z"]), n_wk=np.array_equal(n_wk, st["n_wk"]), phi=np.array_equal(phi, st["phiT"]))
        print(f"stress: {sweeps} sweeps, world {world}, exchange {mode}:", checks, flush=True)
        ok = all(checks.values())
    return ok


def accessors(rank, world, local):
    """The accessors that gather rows or sums across the ranks -- the Phi mean under a burn-in / thin schedule, both
    count histograms -- and set_alpha (asymmetric) / set_beta followed by sweeps, against one GPU running the whole
    corpus in rank 0's process."""
    K, V = 100, 900
    off, tokens = L.synth_corpus(400, V, 70.0, seed=8)
    cfg = L.LDAConfiguration(scheme="gpu_ggs", topics=K, alpha=0.5, beta=0.01, seed=2019, exec_time=0)
    s = L.GpuLDASampler(cfg, device=local)
    box = [L.GpuLDASampler.make_comm_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    s.addInstances(L.InstanceList.from_csr(off, tokens, V), rank=rank, world=world, comm_id=box[0])
    runs = [s]
    if rank == 0:
        ref = L.GpuLDASampler(cfg, device=local)
        ref.addInstances(L.InstanceList.from_csr(off, tokens, V))
        runs.append(ref)
    # the same bin counts on every rank: the histograms are summed over the ranks
    dh = np.zeros(int(np.diff(off).max()) + 1, np.int64)
    th = np.zeros(int(np.bincount(tokens, minlength=V).max()) + 1, np.int64)
    out = []
    for r in runs:
        r._ck(r._L.ldagpu_set_phi_mean_schedule(r._h, 2, 2))
        r.sample(4)
        r.alpha = np.linspace(0.05, 1.5, K)
        r._ck(r._L.ldagpu_set_alpha(r._h, ptr(r.alpha)))
        r._ck(r._L.ldagpu_set_beta(r._h, 0.03))
        r.sample(3)
        r._ck(r._L.ldagpu_get_count_histograms(r._h, len(dh), ptr(dh), len(th), ptr(th)))
        out.append(dict(mean=r.getPhiMeans(), dh=dh.copy(), th=th.copy(), phi=r.getPhi(), n_wk=r.getTypeTopicMatrix(),
                        z=r.get_z_flat()))
    zs = [None] * world
    dist.all_gather_object(zs, out[0]["z"])
    out[0]["z"] = np.concatenate(zs)
    s.close()
    if rank != 0:
        return True
    ref.close()
    got, want = out
    checks = {k: want[k] is not None and np.array_equal(got[k], want[k]) for k in want}
    print("accessors, world", world, checks, flush=True)
    return all(checks.values())


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl")
    ok = True
    O.set_num_threads(max(1, (os.cpu_count() or 1) // world))   # torchrun exports OMP_NUM_THREADS=1
    if "--stress" in sys.argv:
        ok = stress(rank, world, local, int(sys.argv[sys.argv.index("--stress") + 1]))
        t = torch.tensor([1 if ok else 0], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        dist.destroy_process_group()
        if int(t.item()) != 1:
            sys.exit(1)
        if rank == 0:
            print("multigpu stress ok, world =", world)
        return
    for scheme, osch, K, V in (("gpu_ggs", O.GGS, 100, 900), ("gpu_pcgs", O.PCGS, 400, 1300), ("gpu_ggs", O.GGS, 1000, 2100),
                               ("gpu_spalias", O.SPALIAS, 1500, 700)):
        alpha, beta, seed = 50.0 / K, 0.01, 2019
        off, tokens = L.synth_corpus(400, V, 70.0, seed=8)
        cfg = L.LDAConfiguration(scheme=scheme, topics=K, alpha=alpha, beta=beta, seed=seed, exec_time=0)
        s = L.GpuLDASampler(cfg, device=local)
        box = [L.GpuLDASampler.make_comm_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        s.addInstances(L.InstanceList.from_csr(off, tokens, V), rank=rank, world=world, comm_id=box[0])
        s.sample(2)
        ll = s.modelLogLikelihood()
        n_wk, n_k, phi = s.getTypeTopicMatrix(), s.getTopicTotals(), s.getPhi().T.astype(np.float32)
        zs = [None] * world
        dist.all_gather_object(zs, s.get_z_flat())
        z = np.concatenate(zs)
        z0 = O.java_next_ints(seed, K, len(tokens))
        nw0, _ = O.rebuild_counts(tokens, z0, V, K)
        st = O.sweeps("contract", osch, off, tokens, z0, V, K, np.full(K, alpha), beta, seed, 1, 2,
                      O.phi_contract(nw0, beta, seed, 0))
        want_ll = O.log_likelihood(off, st["z"], K, V, st["n_wk"], st["n_k"], np.full(K, alpha), beta)
        checks = dict(z=np.array_equal(z, st["z"]), n_wk=np.array_equal(n_wk, st["n_wk"]),
                      n_k=np.array_equal(n_k, st["n_k"]), phi=np.array_equal(phi, st["phiT"]),
                      ll=abs(ll - want_ll) <= 1e-9 * abs(want_ll))
        # z-only sweep (Phi frozen): stand-alone count exchange, no Phi draw
        s.sampleZGivenPhi(1)
        zs = [None] * world
        dist.all_gather_object(zs, s.get_z_flat())
        z3 = np.concatenate(zs)
        nw3, nk3 = O.rebuild_counts(tokens, z3, V, K)
        checks["zonly_phi_kept"] = np.array_equal(s.getPhi().T.astype(np.float32), st["phiT"])
        checks["zonly_n_wk"] = np.array_equal(s.getTypeTopicMatrix(), nw3)
        checks["zonly_n_k"] = np.array_equal(s.getTopicTotals(), nk3)
        # step-wise API: count rebuild with its own exchange, then a Phi draw on already-merged counts
        s._step("rebuild_counts")
        s._step("sample_phi")
        checks["step_n_wk"] = np.array_equal(s.getTypeTopicMatrix(), nw3)
        checks["step_phi"] = np.array_equal(s.getPhi().T.astype(np.float32), O.phi_contract(nw3, beta, seed, 3))
        if rank == 0:
            print(scheme, K, s.getExchangeMode(), checks, flush=True)
        ok &= all(checks.values())
        s.close()
    ok &= accessors(rank, world, local)
    t = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    dist.destroy_process_group()
    if int(t.item()) != 1:
        sys.exit(1)
    if rank == 0:
        print("multigpu_check ok, world =", world)


if __name__ == "__main__":
    main()
