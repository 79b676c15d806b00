"""Multi-GPU: cluster sharding and the global pattern dedup exchange
(SURVEY.md §8(e)).

Gene clusters are independent for K1-K3 and for the rows of kmers_to_hashes /
kmers.tsv, so whole clusters are sharded over ranks with no data-path
collective.  The only global state of the reference is the `patterns` set its
single writer owns (`/root/reference/panfeed/__main__.py:70`,
`panfeed.py:210-212`); here every rank dedups locally (K4) and one exchange
makes the numbering global:

    owner(pattern) = hash(full key) % world                (x_classify kernel)
    the full keys to their owners: written straight into the owners' receive buffers, which the
      ranks of a box map once over CUDA IPC (x_scatter, NVLink peer stores); where a buffer
      cannot be mapped: x_pack + all-to-all(v)             (NCCL, torch.distributed)
    owner dedups on the full key, numbers its uniques       (k4_probe + scan + x_finish)
    all-gather of the unique counts -> base[owner] (exclusive scan, on the device)
    the unique indices back; local order + base[owner]      (x_unpack kernel)

The library runs all of it in one call, pf_exchange_run: the transport choice, the peer
mappings, the buffer growth and the agreement points are its own.  PatternExchange hands it the
collectives of torch.distributed (all_gather_into_tensor, all_to_all_single on the context's
stream) as a pf_comm.  Bit 31 of an owner's unique index marks the ONE sender whose copy of the
pattern was the first at its owner: that rank writes the pattern's hashes_to_patterns row
(`writer` table), so every pattern is written exactly once.

With --consider-missing a k-mer pattern key ends with the id of the cluster
pattern that gives its NaN plane, so cluster patterns are exchanged first and the
k-mer keys are rewritten with the GLOBAL cluster-pattern id before hashing.
"""
import os
import time

import numpy as np
import torch
import torch.distributed as dist

KMER, CLUSTER = 0, 1


def shard_clusters(weights, world):
    """Greedy longest-processing-time partition of clusters by weight (sum of
    sequence lengths).  -> list (per rank) of ascending cluster indices."""
    weights = np.asarray(weights, dtype=np.int64)
    order = np.argsort(-weights, kind="stable")
    load = np.zeros(world, np.int64)
    shards = [[] for _ in range(world)]
    for c in order:
        r = int(np.argmin(load))
        shards[r].append(int(c))
        load[r] += int(weights[c])
    return [sorted(s) for s in shards]


def any_rank(flag, device):
    """True on every rank if `flag` is true on any rank: an all_reduce (MAX) over the default
    group, on `device` (the rank's GPU under NCCL, the CPU under gloo).  A collective: every
    rank calls it at the same point."""
    t = torch.tensor([1 if flag else 0], dtype=torch.int32, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return bool(t.item())


class _DeviceBytes:
    """A device buffer of the library (raw address) as seen by torch: __cuda_array_interface__."""

    def __init__(self, ptr, n, typestr="|u1"):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2}


def _device_view(ptr, n, device, typestr="|u1", dtype=torch.uint8):
    if n == 0 or not ptr:
        return torch.empty(0, dtype=dtype, device=device)
    return torch.as_tensor(_DeviceBytes(ptr, n, typestr), device=device)


class PatternExchange:
    """Global numbering of the patterns of all ranks in ONE library call (pf_exchange_run) over the
    collectives of torch.distributed (NCCL; plain copies at world 1).  `run()` returns, per
    namespace, the local->global id table, the writer flags and the counts.  PF_EXCHANGE_PEER=0
    asks for the all-to-all transport of the keys instead of peer memory."""

    def __init__(self, ctx, device, group=None):
        from . import capi
        self.ctx, self.device, self.group = ctx, device, group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.no_peer = os.environ.get("PF_EXCHANGE_PEER", "1") == "0"
        self._error = None
        # (the ctypes callbacks must stay referenced as long as the library may call them)
        self._ag = capi.ALL_GATHER_FN(self._all_gather)
        self._a2a = capi.ALL_TO_ALL_V_FN(self._all_to_all_v)
        self.comm = capi.Comm(self.rank, self.world, None, self._ag, self._a2a)
        self._ran = False

    def _on(self, stream):
        return torch.cuda.stream(torch.cuda.ExternalStream(stream, device=self.device))

    def _all_gather(self, send, recv, nbytes, stream, user):
        try:
            with self._on(stream):
                inp = _device_view(send, nbytes, self.device)
                out = _device_view(recv, nbytes * self.world, self.device)
                if self.world == 1:
                    out.copy_(inp)
                else:
                    dist.all_gather_into_tensor(out, inp, group=self.group)
            return 0
        except Exception as e:          # (no exception may cross the C frames)
            self._error = e
            return -1

    def _all_to_all_v(self, send, send_bytes, recv, recv_bytes, stream, user):
        try:
            sb = [int(send_bytes[r]) for r in range(self.world)]
            rb = [int(recv_bytes[r]) for r in range(self.world)]
            with self._on(stream):
                inp = _device_view(send, sum(sb), self.device)
                out = _device_view(recv, sum(rb), self.device)
                if self.world == 1:
                    out.copy_(inp)
                else:
                    dist.all_to_all_single(out, inp, output_split_sizes=rb, input_split_sizes=sb, group=self.group)
            return 0
        except Exception as e:
            self._error = e
            return -1

    def run(self, want_unique=False, want_writer=False):
        from . import capi
        t0 = time.perf_counter()
        flags = (capi.PF_EXCHANGE_WRITER if want_writer else 0) | (capi.PF_EXCHANGE_KEEP_UNIQUE if want_unique else 0) \
            | (capi.PF_EXCHANGE_NO_PEER if self.no_peer else 0)
        self._error = None
        try:
            res = self.ctx.exchange_run(self.comm, flags)
        except capi.PfError:
            if self._error is not None:
                raise RuntimeError(f"pattern exchange: a collective failed: {self._error!r}") from self._error
            raise
        self._ran = True
        ms = (time.perf_counter() - t0) * 1e3
        out = {}
        for name, ns in (("cluster", CLUSTER), ("kmer", KMER)):
            r = res[name]
            n = int(r["n_local"])
            # copies: the library's tables are reused by its next exchange
            l2g = _device_view(r["local_to_global"], n, self.device, "<i4", torch.int32).clone()
            writer = _device_view(r["writer"], n, self.device).clone() if want_writer else None
            out[name] = {"local_to_global": l2g, "writer": writer, "n_global": int(r["n_global"]),
                         "n_owned": int(r["n_owned"]), "owned_base": int(r["owned_base"]),
                         "bytes_sent": int(r["bytes_sent"]), "ms": {"total_both_namespaces": ms, "stages": None}}
            if want_unique:
                out[name]["owned_keys"] = self.ctx.exchange_unique_keys(ns == CLUSTER)
        return out

    def close(self):
        """Unmap the peers' receive buffers; collective: every rank has unmapped before any rank
        goes on to destroy its context (and with it the buffer the others had mapped)."""
        if self._ran:
            self.ctx.exchange_release(self.comm)
            self._ran = False
