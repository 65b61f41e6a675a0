"""Held-out evaluation with one process per GPU.  Run it under torchrun on >= 2 GPUs, in either exchange mode
(LDAGPU_EXCHANGE=p2p|nccl).
- Every rank uploads its token-balanced shard of the test set.
- phihat comes from the n_wk all-gathered over the ranks.
- The per-document values are all-gathered, so every rank returns the total of the whole test set.
The concatenated per-document values and every rank's total must equal, bit for bit, the CPU contract restatement
(tests/heldout_oracle.c) on the global counts.  K > 1024 is refused on every rank.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \\
        --master-port 29512 tests/heldout_multigpu_check.py
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import heldout_oracle as H  # noqa: E402
import ldagroupedgibbssampler_b200 as L  # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl")
    ok = True
    for scheme, K, V in (("gpu_ggs", 100, 900), ("gpu_pcgs", 400, 1300), ("gpu_ggs", 1000, 2100),
                         ("gpu_spalias", 1500, 700)):
        alpha, beta, seed = 50.0 / K, 0.01, 2019
        off, tokens = L.synth_corpus(400, V, 70.0, seed=8)
        toff, ttok = L.synth_corpus(150, V, 50.0, seed=9, doc_first=400)
        cfg = L.LDAConfiguration(scheme=scheme, topics=K, alpha=alpha, beta=beta, seed=seed, exec_time=0)
        s = L.GpuLDASampler(cfg, device=local)
        box = [L.GpuLDASampler.make_comm_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        s.addInstances(L.InstanceList.from_csr(off, tokens, V), rank=rank, world=world, comm_id=box[0])
        s.sample(2)
        checks = {}
        if K <= 1024:
            s.addTestInstances(L.InstanceList.from_csr(toff, ttok, V))
            tot, dll = s.heldOutLogLikelihood(10)
            n_wk, n_k, it = s.getTypeTopicMatrix(), s.getTopicTotals(), s.getCurrentIteration()   # collective
            parts = [None] * world
            dist.all_gather_object(parts, (tot, dll))
            if rank == 0:
                want_t, want_d = H.heldout_l2r("contract", toff, ttok, n_wk, n_k, s.alpha, beta, seed, it, R=10)
                checks.update(total=all(p[0] == want_t for p in parts),
                              doc_ll=np.array_equal(np.concatenate([p[1] for p in parts]), want_d))
        else:
            try:
                s.addTestInstances(L.InstanceList.from_csr(toff, ttok, V))
                checks["heldout_refused"] = False
            except L.LdaGpuError as e:
                checks["heldout_refused"] = "K <= 1024" in str(e)
        if rank == 0:
            print(scheme, K, s.getExchangeMode(), checks, flush=True)
        ok &= all(bool(v) for v in checks.values())
        s.close()
    t = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    dist.destroy_process_group()
    if int(t.item()) != 1:
        sys.exit(1)
    if rank == 0:
        print("heldout_multigpu_check ok, world =", world)


if __name__ == "__main__":
    main()
