"""On-hardware check of the multi-GPU pattern exchange (SURVEY.md §8(e)).

The reference keeps ONE `patterns` set in its single writer process
(`/root/reference/panfeed/__main__.py:70`, `panfeed.py:210-212`); here every
rank numbers its own patterns (K4) and `dist.PatternExchange` (pf_exchange_run)
makes the numbering global over NCCL.  `check_exchange` proves, on the ranks and the
communicator that are actually running, that the global numbering is the one a
single context over all clusters would produce:

  1. every local pattern's full key equals the key its owner stored under the
     returned global id (k-mer keys of the cluster-absent mode compared through
     the NaN plane their last word names, local id -> global id);
  2. the global table holds every full (ternary) pattern exactly once;
  3. rank 0 runs ALL clusters of the sample through one context: the same
     number of patterns in both namespaces and the same set of full patterns.

With more_clusters_per_rank, the same contexts then take that many clusters more per rank and
the same PatternExchange runs again: the receive buffers the first exchange sized (and the
other ranks mapped) have to grow, and the checks apply to the second result.

Used by `bench.py` before the timed region at N > 1 and by
`tests/test_gpu_multirank.py`; works at world size 1 too (degenerate routing).
"""
import numpy as np
import torch
import torch.distributed as dist

from . import capi
from .dist import PatternExchange


def _gather(obj, world):
    if world == 1:
        return [obj]
    out = [None] * world
    dist.all_gather_object(out, obj)
    return out


def check_exchange(local_device, consider_missing, seed=20261018, n_samples=256,
                   clusters_per_rank=6, gene_len=400, k=31, maf=0.01, more_clusters_per_rank=0):
    """Raises AssertionError on any mismatch; returns the pattern counts."""
    world = dist.get_world_size() if dist.is_initialized() else 1
    rank = dist.get_rank() if dist.is_initialized() else 0
    dev = torch.device("cuda", local_device)
    S, cpr, more = n_samples, clusters_per_rank, more_clusters_per_rank
    W = (S + 31) // 32
    total = world * (cpr + more)
    hb = capi.synth_batch(local_device, seed, S, cpr, first_cluster=rank * cpr,
                          total_clusters=total, gene_len=gene_len)
    ctx = capi.Context(k, S, consider_missing=consider_missing, maf=maf, device=local_device)
    ex = None
    try:
        ctx.submit(hb)
        ctx.collect()
        ex = PatternExchange(ctx, dev)
        out = ex.run(want_unique=True)
        grown = {}
        if more:
            grown = {"kmer_patterns_local_first_exchange": len(out["kmer"]["local_to_global"])}
            ctx.submit(capi.synth_batch(local_device, seed, S, more, first_cluster=world * cpr + rank * more,
                                        total_clusters=total, gene_len=gene_len))
            ctx.collect()
            out = ex.run(want_unique=True)
        # the transport asked for: pf_exchange_run still falls back to the all-to-all on every rank
        # when a peer buffer cannot be mapped
        transport = "local copy" if world == 1 else "nccl all-to-all" if ex.no_peer else "peer memory"
        n_cl = len(out["cluster"]["local_to_global"])
        n_km = len(out["kmer"]["local_to_global"])
        local_cl = ctx.export_patterns(True, 0, n_cl)
        local_km = ctx.export_patterns(False, 0, n_km)
        l2g_cl = out["cluster"]["local_to_global"].cpu().numpy().astype(np.int64)
        l2g_km = out["kmer"]["local_to_global"].cpu().numpy().astype(np.int64)
        # global tables = owned keys in rank order (global id = base[owner] + unique index)
        glob_cl = np.concatenate(_gather(out["cluster"]["owned_keys"], world))
        glob_km = np.concatenate(_gather(out["kmer"]["owned_keys"], world))
        assert len(glob_cl) == out["cluster"]["n_global"], "cluster namespace: n_global != sum of owned"
        assert len(glob_km) == out["kmer"]["n_global"], "k-mer namespace: n_global != sum of owned"
        # 1. local key == key stored under its global id
        assert np.array_equal(glob_cl[l2g_cl], local_cl), "cluster pattern ids point at other keys"
        if consider_missing:
            want = local_km.copy()
            want[:, W] = l2g_cl[local_km[:, W].astype(np.int64)]
            assert np.array_equal(glob_km[l2g_km], want), "k-mer pattern ids point at other keys (NaN plane)"
        else:
            assert np.array_equal(glob_km[l2g_km], local_km), "k-mer pattern ids point at other keys"
        # 2. no duplicates in the global tables
        assert len(np.unique(glob_cl, axis=0)) == len(glob_cl), "duplicate cluster pattern in the global table"
        assert len(np.unique(glob_km, axis=0)) == len(glob_km), "duplicate k-mer pattern in the global table"

        def full(km, cl):
            if consider_missing:
                return {row[:W].tobytes() + cl[int(row[W])].tobytes() for row in km}
            return {row[:W].tobytes() for row in km}

        # 3. one context over all clusters (rank 0)
        if rank == 0:
            hb_all = capi.synth_batch(local_device, seed, S, total, first_cluster=0,
                                      total_clusters=total, gene_len=gene_len)
            one = capi.Context(k, S, consider_missing=consider_missing, maf=maf, device=local_device)
            try:
                one.submit(hb_all)
                r = one.collect()
            finally:
                one.close()
            assert len(r["new_cluster_patterns"]) == len(glob_cl), \
                f"cluster patterns: {len(glob_cl)} global vs {len(r['new_cluster_patterns'])} in one context"
            assert len(r["new_kmer_patterns"]) == len(glob_km), \
                f"k-mer patterns: {len(glob_km)} global vs {len(r['new_kmer_patterns'])} in one context"
            assert {x.tobytes() for x in r["new_cluster_patterns"]} == {x.tobytes() for x in glob_cl}
            assert full(r["new_kmer_patterns"], r["new_cluster_patterns"]) == full(glob_km, glob_cl), \
                "the global k-mer pattern set differs from the single-context one"
        return {"world": world, "consider_missing": bool(consider_missing),
                "cluster_patterns_global": int(len(glob_cl)), "kmer_patterns_global": int(len(glob_km)),
                "kmer_patterns_local": int(n_km), "ok": True,
                "transport": transport, **grown}
    finally:
        if ex is not None:
            ex.close()
        ctx.close()
