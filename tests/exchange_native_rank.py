"""One rank of test_gpu_exchange_run's real-rank case (torchrun, NCCL): on the same contexts,
NativePatternExchange (pf_exchange_run over torch.distributed) and PatternExchange give the same
global pattern counts and the same writer totals.  argv[1]: 1 = consider_missing."""
import os
import sys

import torch
import torch.distributed as dist

from panfeed_b200 import capi, dist as pfdist


def main():
    cm = bool(int(sys.argv[1]))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    dev = torch.device("cuda", local)
    S, C = 64, 6
    hb = capi.synth_batch(local, 20261020, S, C, first_cluster=rank * C, total_clusters=world * C, gene_len=600)
    ctx = capi.Context(31, S, consider_missing=cm, maf=0.01, device=local)
    ctx.submit(hb)
    ctx.collect()
    py_ex = pfdist.PatternExchange(ctx, dev)
    py = py_ex.run(want_writer=True)
    nat_ex = pfdist.NativePatternExchange(ctx, dev)
    nat = nat_ex.run(want_writer=True)
    for name in ("cluster", "kmer"):
        assert py[name]["n_global"] == nat[name]["n_global"], name
        assert (py[name]["n_owned"], py[name]["owned_base"]) == (nat[name]["n_owned"], nat[name]["owned_base"])
        w = torch.tensor([int(py[name]["writer"].sum()), int(nat[name]["writer"].sum())], device=dev,
                         dtype=torch.int64)
        dist.all_reduce(w)
        assert int(w[0]) == int(w[1]) == nat[name]["n_global"], (name, w.tolist())
    nat_ex.close()
    py_ex.close()
    if rank == 0:
        print(f"native == python: cluster {nat['cluster']['n_global']} kmer {nat['kmer']['n_global']}")
    ctx.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
