"""Run under torchrun with >= 2 ranks, one GPU each (tests/test_gpu_maxsim_topk.py launches it): ShardedKnn(kind="maxsim")
over a document-sharded token corpus -- through the peer-mapped exchange and through the NCCL allgather + merge, in the
knn_dev, knn_dev_pipelined and knn forms -- must equal the unsharded maxsim_topk_batch on the whole corpus, in indices
and score bits, on every rank."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import torch
    import torch.distributed as dist
    import innr_b200 as ib
    from innr_b200 import sharded, synth
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    ib.init(local)
    ex = sharded.PeerExchange.for_process_group(dist)
    dev = torch.device(f"cuda:{local}")
    failures = []

    def same(a, b):
        return bool(torch.equal(a[0].cpu().view(torch.int64), torch.from_numpy(np.ascontiguousarray(b[0]).view(np.int64)))) \
            and a[1].cpu().numpy().tobytes() == np.ascontiguousarray(b[1]).tobytes()

    n_docs, nt, dim, n_q = 20_001, 40, 128, 32
    lo, hi = sharded.shard_range(n_docs, rank, world)
    shard = ib.TokenCorpus.generate(synth.SALT_CORPUS, lo, hi - lo, nt, dim, index_base=lo)
    whole = ib.TokenCorpus.generate(synth.SALT_CORPUS, 0, n_docs, nt, dim)
    for metric in ("dot", "cosine"):
        cos = metric == "cosine"
        peer = sharded.ShardedKnn(shard, "maxsim", metric, exchange=ex, query_tokens=n_q)
        nccl = sharded.ShardedKnn(shard, "maxsim", metric, query_tokens=n_q)
        for nq, k in ((1, 10), (3, 100), (2, 200)):
            qs = synth.ghash_f32(synth.SALT_QUERY, 77 * nq + k, nq * n_q * dim).reshape(nq, n_q, dim)
            want = ib.maxsim_topk_batch(qs, whole, k, cosine=cos)
            dq = torch.from_numpy(qs).to(dev)
            for name, sk in (("peer", peer), ("nccl", nccl)):
                got = [t.clone() for t in sk.knn_dev(dq, nq, k)]
                torch.cuda.synchronize()
                if not same(got, want):
                    failures.append((name, metric, nq, k))
                if not same([torch.from_numpy(x.view(np.int64)) if x.dtype == np.uint64 else torch.from_numpy(x)
                             for x in sk.knn(qs, k)], want):
                    failures.append((name + "-host", metric, nq, k))
        # pipelined: the exchange of call i runs on the side stream behind the scan of call i + 1
        qs = synth.ghash_f32(synth.SALT_QUERY, 9000, 5 * n_q * dim).reshape(5, n_q, dim)
        dqs = torch.from_numpy(qs).to(dev)
        main = torch.cuda.current_stream()
        got, pending = [], None
        for i in range(5):
            cur = peer.knn_dev_pipelined(dqs[i:i + 1], 1, 10)
            if pending is not None:
                main.wait_event(pending[2])
                got.append((pending[0].clone(), pending[1].clone()))
            pending = cur
        main.wait_event(pending[2])
        got.append((pending[0].clone(), pending[1].clone()))
        peer.drain()
        torch.cuda.synchronize()
        for i in range(5):
            if not same(got[i], ib.maxsim_topk_batch(qs[i:i + 1], whole, 10, cosine=cos)):
                failures.append(("pipelined", metric, i))
    if ex.status() != 0:
        failures.append(("timeout",))
    bad = torch.tensor([len(failures)], device=dev)
    dist.all_reduce(bad)
    if failures:
        print(f"rank {rank}: FAILURES {failures}", flush=True)
    dist.destroy_process_group()
    if int(bad.item()):
        sys.exit(1)
    if rank == 0:
        print("mp_maxsim_check ok", flush=True)


if __name__ == "__main__":
    main()
