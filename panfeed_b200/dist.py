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
    reverse all-to-all of the unique indices; local order + base[owner]   (x_unpack kernel)

Everything (library kernels and NCCL) is enqueued on the context's own stream, so
nothing waits on the host but the bucket sizes NCCL needs as split sizes (one small
all-to-all for both namespaces when the k-mer keys do not depend on the cluster
ids) and the final counts.  Bit 31 of a returned index marks the ONE sender whose copy
of the pattern was the first at its owner: that rank writes the pattern's
hashes_to_patterns row (`writer` table), so every pattern is written exactly once.

With --consider-missing a k-mer pattern key ends with the id of the cluster
pattern that gives its NaN plane, so cluster patterns are exchanged first and the
k-mer keys are rewritten with the GLOBAL cluster-pattern id before hashing.

torch is plumbing here (device buffers + the collective); the kernels are in
libpanfeed_b200.so behind pf_exchange_*.
"""
import ctypes as C

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


class DeviceBackend:
    """pf_exchange_* on one pf_ctx; buffers are torch tensors on its device."""

    def __init__(self, ctx, device):
        self.ctx, self.device = ctx, device
        self.consider_missing = bool(ctx.consider_missing)

    def stream(self):
        return torch.cuda.ExternalStream(self.ctx.stream_handle(), device=self.device)

    def key_words(self, ns):
        return self.ctx.W if ns == CLUSTER else self.ctx.Wk

    def n_local(self, ns):
        st = self.ctx.stats()
        return int(st["cluster_patterns"] if ns == CLUSTER else st["kmer_patterns"])

    def pack(self, ns, world, mask_remap, send):
        counts = (C.c_uint64 * world)()
        self.ctx._check(self.ctx.lib.pf_exchange_pack(
            self.ctx.h, ns, world, mask_remap.data_ptr() if mask_remap is not None else None,
            send.data_ptr() if send.numel() else None, send.shape[0], counts))
        return [int(c) for c in counts]

    # -- peer-memory path: keys go straight into the owners' receive buffers --
    def classify(self, ns, world, mask_remap):
        counts = (C.c_uint64 * world)()
        self.ctx._check(self.ctx.lib.pf_exchange_classify(
            self.ctx.h, ns, world, mask_remap.data_ptr() if mask_remap is not None else None, counts))
        return [int(c) for c in counts]

    def recv_buffer(self, ns, min_rows):
        """-> (device pointer, capacity in rows, 64-byte CUDA IPC handle) of this rank's receive
        buffer; grows (and changes its handle) when min_rows exceeds the capacity."""
        ptr, cap, handle = C.c_void_p(), C.c_uint64(), (C.c_ubyte * 64)()
        self.ctx._check(self.ctx.lib.pf_exchange_recv_buffer(self.ctx.h, ns, int(min_rows), C.byref(ptr),
                                                             C.byref(cap), handle))
        return int(ptr.value), int(cap.value), bytes(handle)

    def open_peer(self, handle):
        mapped = C.c_void_p()
        self.ctx._check(self.ctx.lib.pf_exchange_open_peer(self.ctx.h, (C.c_ubyte * 64).from_buffer_copy(handle),
                                                           C.byref(mapped)))
        return int(mapped.value)

    def close_peer(self, mapped):
        self.ctx._check(self.ctx.lib.pf_exchange_close_peer(self.ctx.h, C.c_void_p(mapped)))

    def scatter(self, ns, world, mask_remap, ptrs, row0):
        self.ctx._check(self.ctx.lib.pf_exchange_scatter(
            self.ctx.h, ns, world, mask_remap.data_ptr() if mask_remap is not None else None,
            (C.c_void_p * world)(*ptrs), (C.c_uint64 * world)(*row0)))

    def dedup(self, ns, recv, unique_index, n_unique, keep_unique=False):
        """Asynchronous: n_unique is a one-element int32 device tensor.  keep_unique: the owner
        keeps a compact copy of its unique keys for unique_keys() (tests, self-check).
        recv: a [rows, words] tensor or (device pointer, rows)."""
        if isinstance(recv, tuple):
            self.ctx._check(self.ctx.lib.pf_exchange_dedup(
                self.ctx.h, ns, C.c_void_p(recv[0]) if recv[1] else None, recv[1],
                unique_index.data_ptr() if unique_index.numel() else None, n_unique.data_ptr(), None,
                int(bool(keep_unique))))
            return
        self.ctx._check(self.ctx.lib.pf_exchange_dedup(
            self.ctx.h, ns, recv.data_ptr() if recv.numel() else None, recv.shape[0],
            unique_index.data_ptr() if unique_index.numel() else None, n_unique.data_ptr(), None,
            int(bool(keep_unique))))

    def unique_keys(self, ns):
        n = C.c_uint64()
        self.ctx._check(self.ctx.lib.pf_exchange_unique_count(self.ctx.h, ns, C.byref(n)))
        out = np.zeros((n.value, self.key_words(ns)), np.uint32)
        self.ctx._check(self.ctx.lib.pf_exchange_unique_export(self.ctx.h, ns, out.ctypes.data))
        return out

    def unpack(self, ns, returned, owner_base, local_to_global, writer):
        self.ctx._check(self.ctx.lib.pf_exchange_unpack(
            self.ctx.h, ns, returned.data_ptr() if returned.numel() else None,
            owner_base.data_ptr(), local_to_global.data_ptr() if local_to_global.numel() else None,
            writer.data_ptr() if writer is not None and writer.numel() else None))


class _NoStream:
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


class PatternExchange:
    """Global numbering of the patterns of all ranks.  `run()` returns, per
    namespace, the local->global id table, the writer flags and the counts."""

    def __init__(self, ctx, device, backend=None, group=None, peer_memory=None):
        import os
        self.backend = backend if backend is not None else DeviceBackend(ctx, device)
        self.device = device
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self._marks = None
        self.consider_missing = bool(getattr(ctx, "consider_missing", False)) if ctx is not None \
            else bool(getattr(backend, "consider_missing", False))
        # peer memory (ranks of one box, NVLink): the keys are written straight into the owners'
        # receive buffers; falls back to the NCCL all-to-all for good if a buffer cannot be mapped
        explicit = peer_memory is not None       # (tests drive the protocol with a host model)
        if peer_memory is None:
            peer_memory = os.environ.get("PF_EXCHANGE_PEER", "1") != "0"
        self.peer = bool(peer_memory) and self.world > 1 and hasattr(self.backend, "scatter") \
            and (explicit or getattr(device, "type", "cpu") == "cuda")
        self.recv_slack_rows = 1024                      # a receive buffer grows to need * 5/4 + this
        self._peer_maps = {KMER: {}, CLUSTER: {}}        # ns -> {rank: (handle, mapped pointer)}
        self._peer_seen = {KMER: False, CLUSTER: False}

    def close(self):
        """Unmap the peers' receive buffers; collective: every rank has unmapped before any rank
        goes on to destroy its context (and with it the buffer the others had mapped)."""
        opened = any(self._peer_seen.values())
        for maps in self._peer_maps.values():
            for _, mapped in maps.values():
                self.backend.close_peer(mapped)
            maps.clear()
        if opened and self.world > 1:
            if self.device.type == "cuda":
                torch.cuda.synchronize(self.device)
            self._host_all_ok(True)
        self._peer_seen = {KMER: False, CLUSTER: False}

    # -- collectives (world 1: plain copies, so that a single process runs the same path) --
    def _a2a(self, out, inp, out_split=None, in_split=None):
        if self.world == 1:
            out.copy_(inp)
        else:
            dist.all_to_all_single(out, inp, output_split_sizes=out_split, input_split_sizes=in_split,
                                   group=self.group)

    def _gather(self, out, inp):
        if self.world == 1:
            out.copy_(inp)
        else:
            dist.all_gather_into_tensor(out, inp, group=self.group)

    def _pack(self, ns, mask_remap):
        be, dev = self.backend, self.device
        n_local = be.n_local(ns)
        send = torch.empty((n_local, be.key_words(ns)), dtype=torch.int32, device=dev)
        return {"ns": ns, "n_local": n_local, "send": send, "bytes_sent": int(send.numel() * 4),
                "send_counts": be.pack(ns, self.world, mask_remap, send)}

    def _counts(self, packs):
        """Bucket sizes of every packed namespace to their owners: one small all-to-all."""
        world, dev = self.world, self.device
        sc = torch.tensor([p["send_counts"] for p in packs], dtype=torch.int64).t().contiguous().to(dev)
        rc = torch.empty_like(sc)                                    # [world, n_packs]
        self._a2a(rc, sc)
        rc = rc.cpu().tolist()
        for j, p in enumerate(packs):
            p["recv_counts"] = [int(rc[r][j]) for r in range(world)]

    def _finish(self, p, want_writer, want_unique=False):
        """Keys to the owners, owner-side dedup, ids back: all asynchronous on the stream."""
        be, world, dev, ns = self.backend, self.world, self.device, p["ns"]
        n_recv = sum(p["recv_counts"])
        recv = torch.empty((n_recv, p["send"].shape[1]), dtype=torch.int32, device=dev)
        self._a2a(recv, p["send"], p["recv_counts"], p["send_counts"])
        self._mark(f"keys all-to-all ns{ns}")
        return self._finish_owner(p, recv, n_recv, want_writer, want_unique)

    def _finish_owner(self, p, recv, n_recv, want_writer, want_unique):
        """Owner-side dedup of the received keys (tensor or (pointer, rows)), ids back."""
        be, world, dev, ns = self.backend, self.world, self.device, p["ns"]
        uniq_idx = torch.empty(n_recv, dtype=torch.int32, device=dev)
        nu = torch.zeros(1, dtype=torch.int32, device=dev)
        be.dedup(ns, recv, uniq_idx, nu, want_unique)
        self._mark(f"owner dedup ns{ns}")
        all_nu = torch.empty(world, dtype=torch.int32, device=dev)
        self._gather(all_nu, nu)
        owner_base = (torch.cumsum(all_nu, 0, dtype=torch.int32) - all_nu).contiguous()
        returned = torch.empty(p["n_local"], dtype=torch.int32, device=dev)
        self._a2a(returned, uniq_idx, p["send_counts"], p["recv_counts"])
        l2g = torch.empty(p["n_local"], dtype=torch.int32, device=dev)
        writer = torch.empty(p["n_local"], dtype=torch.uint8, device=dev) if want_writer else None
        be.unpack(ns, returned, owner_base, l2g, writer)
        self._mark(f"ids back + unpack ns{ns}")
        p.update(local_to_global=l2g, writer=writer, all_nu=all_nu, keep=(recv, uniq_idx, returned, owner_base))
        return p

    def _host_all_ok(self, ok):
        t = torch.tensor([1 if ok else 0], dtype=torch.int32, device=self.device)
        dist.all_reduce(t, op=dist.ReduceOp.MIN, group=self.group)
        return bool(t.item())

    def _exchange_peer(self, ns, mask_remap, want_writer, want_unique):
        """One namespace over peer memory.  Returns None (on every rank alike) if a receive buffer
        could not be mapped: the caller then takes the NCCL path, now and from then on."""
        be, world, dev, rank = self.backend, self.world, self.device, self.rank
        n_local = be.n_local(ns)
        counts = be.classify(ns, world, mask_remap)                     # one sync
        self._mark(f"classify ns{ns}")
        ptr, cap, handle = be.recv_buffer(ns, 1)
        # every rank's bucket sizes, receive capacity and handle: all ranks then know every
        # rank's row count and which buffers have to grow
        mine = torch.tensor(counts + [cap] + np.frombuffer(handle, np.int64).tolist(), dtype=torch.int64).to(dev)
        allv = torch.empty(world * (world + 9), dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(allv, mine, group=self.group)
        allv = allv.cpu().numpy().reshape(world, world + 9)             # sync
        M = allv[:, :world]                                             # M[src][dst]
        need = M.sum(axis=0)
        grow = need > allv[:, world]
        handles = [allv[r, world + 1:].tobytes() for r in range(world)]
        maps = self._peer_maps[ns]
        opening = bool(grow.any()) or not self._peer_seen[ns]
        if grow.any():
            # mappings of a buffer that is about to be freed go first; its owner waits for that
            for r in np.nonzero(grow)[0].tolist():
                if r in maps:
                    be.close_peer(maps.pop(r)[1])
            if dev.type == "cuda":
                torch.cuda.synchronize(dev)
            self._host_all_ok(True)                                     # barrier
            if grow[rank]:
                ptr, cap, handle = be.recv_buffer(ns, int(need[rank]) + int(need[rank]) // 4 + self.recv_slack_rows)
            mine = torch.from_numpy(np.frombuffer(handle, np.int64).copy()).to(dev)
            allh = torch.empty(world * 8, dtype=torch.int64, device=dev)
            dist.all_gather_into_tensor(allh, mine, group=self.group)
            allh = allh.cpu().numpy().reshape(world, 8)
            handles = [allh[r].tobytes() for r in range(world)]
        ok = True
        ptrs = [0] * world
        for r in range(world):
            if r == rank:
                ptrs[r] = ptr
                continue
            have = maps.get(r)
            if have is not None and have[0] == handles[r]:
                ptrs[r] = have[1]
                continue
            try:
                if have is not None:
                    be.close_peer(maps.pop(r)[1])
                ptrs[r] = be.open_peer(handles[r])
                maps[r] = (handles[r], ptrs[r])
            except Exception:
                ok = False
        if opening:
            self._peer_seen[ns] = True
            if not self._host_all_ok(ok):
                return None
        elif not ok:
            raise RuntimeError("pattern exchange: a cached peer mapping went away")
        self._mark(f"sizes + buffers ns{ns}")
        row0 = [int(M[:rank, r].sum()) for r in range(world)]
        be.scatter(ns, world, mask_remap, ptrs, row0)
        # every rank's scatter has completed before anyone reads its receive buffer
        flag = torch.zeros(1, dtype=torch.int32, device=dev)
        dist.all_reduce(flag, group=self.group)
        self._mark(f"keys to the owners ns{ns}")
        p = {"ns": ns, "n_local": n_local, "send_counts": counts, "recv_counts": [int(x) for x in M[:, rank]],
             "bytes_sent": n_local * be.key_words(ns) * 4, "flag": flag}
        return self._finish_owner(p, (ptr, int(need[rank])), int(need[rank]), want_writer, want_unique)

    def _mark(self, name):
        """PF_EXCHANGE_TIMING=1: an event on the exchange's stream at every stage boundary."""
        if self._marks is not None:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            self._marks.append((name, e))

    def run(self, want_unique=False, want_writer=False):
        import os
        import time
        t0 = time.perf_counter()
        be = self.backend
        use_stream = self.device.type == "cuda" and hasattr(be, "stream")
        self._marks = [] if (use_stream and os.environ.get("PF_EXCHANGE_TIMING")) else None
        with (torch.cuda.stream(be.stream()) if use_stream else _NoStream()):
            self._mark("start")
            cl = km = None
            if self.peer:
                cl = self._exchange_peer(CLUSTER, None, want_writer, want_unique)
                if cl is not None:
                    km = self._exchange_peer(KMER, cl["local_to_global"] if self.consider_missing else None,
                                             want_writer, want_unique)
                if cl is None or km is None:
                    self.peer = False            # (every rank took the same decision)
                    cl = km = None
            if cl is not None:
                pass
            elif self.consider_missing:
                cl = self._pack(CLUSTER, None)
                # k-mer keys end with the GLOBAL id of the cluster pattern giving their NaN plane:
                # the cluster namespace has to be numbered first
                self._counts([cl])
                self._finish(cl, want_writer, want_unique)
                self._mark("cluster namespace")
                km = self._pack(KMER, cl["local_to_global"])
                self._mark("pack kmer")
                self._counts([km])
                self._mark("counts")
            else:
                cl = self._pack(CLUSTER, None)
                km = self._pack(KMER, None)
                self._counts([cl, km])
                self._finish(cl, want_writer, want_unique)
            if "all_nu" not in km:
                self._finish(km, want_writer, want_unique)
            counts = torch.stack([cl["all_nu"], km["all_nu"]]).cpu().tolist()     # the final sync
        ms = (time.perf_counter() - t0) * 1e3
        stages = None
        if self._marks:
            stages = [(b[0], round(a[1].elapsed_time(b[1]), 3)) for a, b in zip(self._marks, self._marks[1:])]
        out = {}
        for name, p, c in (("cluster", cl, counts[0]), ("kmer", km, counts[1])):
            out[name] = {"local_to_global": p["local_to_global"], "writer": p["writer"],
                         "n_global": int(sum(c)), "n_owned": int(c[self.rank]),
                         "owned_base": int(sum(c[:self.rank])), "bytes_sent": p["bytes_sent"],
                         "ms": {"total_both_namespaces": ms, "stages": stages}}
            if want_unique:
                # (each namespace keeps its owner-side unique keys in its OWN scratch - PatternSpace::x_unique
                #  of ctx->cp / ctx->kp - so the k-mer exchange has not overwritten the cluster namespace's)
                out[name]["owned_keys"] = be.unique_keys(p["ns"])
        return out


class _DeviceBytes:
    """A device buffer of the library (raw address) as seen by torch: __cuda_array_interface__."""

    def __init__(self, ptr, n, typestr="|u1"):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2}


def _device_view(ptr, n, device, typestr="|u1", dtype=torch.uint8):
    if n == 0 or not ptr:
        return torch.empty(0, dtype=dtype, device=device)
    return torch.as_tensor(_DeviceBytes(ptr, n, typestr), device=device)


class NativePatternExchange:
    """The same global numbering as PatternExchange, in ONE library call (pf_exchange_run): the
    transport choice, the peer mappings and the agreement points are the library's; this class only
    hands it the collectives of torch.distributed (NCCL) as a pf_comm.  `run()` returns what
    PatternExchange.run returns."""

    def __init__(self, ctx, device, group=None):
        from . import capi
        self.ctx, self.device, self.group = ctx, device, group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
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

    def run(self, want_unique=False, want_writer=False, flags=0):
        import time
        from . import capi
        t0 = time.perf_counter()
        flags |= (capi.PF_EXCHANGE_WRITER if want_writer else 0) | (capi.PF_EXCHANGE_KEEP_UNIQUE if want_unique else 0)
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
        """Collective, like PatternExchange.close: the peers' buffers are unmapped on every rank
        before any rank goes on to destroy its context."""
        if self._ran:
            self.ctx.exchange_release(self.comm)
            self._ran = False
