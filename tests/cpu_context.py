"""TEST INFRASTRUCTURE ONLY — a stand-in for `capi.Context` that answers `submit` / `collect`
from the C oracle (oracle/oracle.c) instead of the GPU.

The `-m "not gpu"` tier has no device, yet the host side of the drop-in (CLI wiring, both
feeders, the packer, the native text formatters, gzip members, the id tables, batching and
`--multiple-files` resets) is most of the Python in the package.  With this class patched in
for `capi.Context` the whole CLI runs on the CPU and its three files are compared with the
unmodified reference's goldens (tests/test_cli_host.py).  What is checked there is the HOST
logic: the oracle supplies the rows the kernels would.  The CUDA path itself is checked by the
`-m gpu` tests; nothing under panfeed_b200/ imports this file.

The batch is decoded from the packed planes exactly as the device reads them (2-bit plane,
4-bit plane for sequences flagged PF_SEQ_AMBIGUOUS, 48-byte descriptors), so a packing mistake
shows up as wrong k-mers.
"""
import numpy as np

from oracle import oracle_c
from panfeed_b200 import capi
from panfeed_b200.panfeed import pattern_id

_ACGT = np.frombuffer(b"ACGT", np.uint8)
_AMB = np.frombuffer(capi.AMB_ALPHABET.encode(), np.uint8)
_SH2 = (62 - 2 * np.arange(32)).astype(np.uint64)
_SH4 = (60 - 4 * np.arange(16)).astype(np.uint64)
_CODE2 = np.full(256, 255, np.uint8)
_CODE2[_ACGT] = np.arange(4)
_CODE4 = np.full(256, 255, np.uint8)
_CODE4[_AMB] = np.arange(16)


def decode_batch(hb):
    """HostBatch -> (ASCII bases back to back, oracle SEQ array, presence matrix [clusters, S])."""
    n = len(hb.seqs)
    seqs = np.zeros(n, oracle_c.SEQ_DTYPE)
    chunks, off = [], 0
    code2 = ((hb.packed[:, None] >> _SH2[None, :]) & np.uint64(3)).astype(np.uint8).ravel() if hb.packed.size \
        else np.zeros(0, np.uint8)
    code4 = None
    if hb.amb is not None and hb.amb.size:
        code4 = ((hb.amb[:, None] >> _SH4[None, :]) & np.uint64(15)).astype(np.uint8).ravel()
    for i in range(n):
        q = hb.seqs[i]
        ln = int(q["len"])
        if q["flags"] & capi.PF_SEQ_AMBIGUOUS:
            a = int(q["amb_off"])
            text = _AMB[code4[a:a + ln]]
        else:
            a = int(q["base_off"])
            text = _ACGT[code2[a:a + ln]]
        chunks.append(text.tobytes())
        seqs[i] = (off, ln, q["cluster"], q["sample"], 1 if q["flags"] & capi.PF_SEQ_TARGET else 0,
                   q["start"], q["end"], q["offset"], q["strand"])
        off += ln
    return b"".join(chunks), seqs


def encode_kmers(strs, k):
    """S{k} array -> (narrow mask, uint64 codes of the narrow ones, [n, 2] (hi, lo) of the wide
    ones): the inverse of packer.kmers_to_str / packer.wide_kmers_to_str."""
    n = len(strs)
    if n == 0:
        return np.zeros(0, bool), np.zeros(0, np.uint64), np.zeros((0, 2), np.uint64)
    sym = np.frombuffer(np.ascontiguousarray(strs).tobytes(), np.uint8).reshape(n, k)
    c2 = _CODE2[sym]
    narrow = (c2 != 255).all(axis=1) & (k <= 32)
    codes = np.zeros(int(narrow.sum()), np.uint64)
    if narrow.any():
        sh = (2 * (k - 1 - np.arange(k))).astype(np.uint64)
        codes = (c2[narrow].astype(np.uint64) << sh[None, :]).sum(axis=1, dtype=np.uint64)
    wsym = sym[~narrow]
    wide = np.zeros((len(wsym), 2), np.uint64)
    for i in range(k):
        if k > 32:
            c, pos = _CODE2[wsym[:, i]].astype(np.uint64), 2 * (k - 1 - i)
        else:
            c, pos = _CODE4[wsym[:, i]].astype(np.uint64), 4 * (k - 1 - i)
        if pos < 64:
            wide[:, 1] |= c << np.uint64(pos)
        else:
            wide[:, 0] |= c << np.uint64(pos - 64)
    return narrow, codes, wide


class OracleContext:
    """The attributes and methods of capi.Context the host mirror uses."""

    instances = []          # every context created (tests look at what the CLI asked for)

    def __init__(self, k, n_samples, canonical=True, consider_missing=False, cluster_equal_filter=False,
                 emit_positions=False, maf=0.01, sort_bits=0, device=0, mode=0, debug_flags=0):
        self.k, self.S = k, n_samples
        self.W = (n_samples + 31) // 32
        self.consider_missing, self.canonical = bool(consider_missing), bool(canonical)
        self.Wk = self.W + 1 if self.consider_missing else self.W
        self.cluster_equal_filter = bool(cluster_equal_filter)
        self.emit_positions, self.maf = emit_positions, maf
        self.reset_patterns()
        self._hb = None
        self.n_batches = self.n_bases = self.n_rows = 0
        OracleContext.instances.append(self)

    # ---- pattern namespaces: insertion-ordered pools keyed on the full key, like K4 ----
    def reset_patterns(self):
        self._cp, self._kp = {}, {}           # key bytes -> pool index
        self._cp_rows, self._kp_rows = [], []

    @staticmethod
    def _intern(pool, rows, key_row):
        key = key_row.tobytes()
        at = pool.get(key)
        if at is None:
            at = pool[key] = len(rows)
            rows.append(key_row.copy())
        return at

    def submit(self, hb):
        if self._hb is not None:
            raise capi.PfError(-3, "pf_submit: a batch is already in flight")
        self._hb = hb

    def collect(self, copy=True):
        hb, self._hb = self._hb, None
        if hb is None:
            raise capi.PfError(-3, "pf_collect without pf_submit")
        k, W = self.k, self.W
        bases, seqs = decode_batch(hb)
        idx = np.arange(self.S)
        presab = ((hb.presence[:, idx >> 5] >> (idx & 31)) & 1).astype(np.uint8).reshape(len(hb.clusters), self.S)
        o = oracle_c.run_arrays(bases, seqs, presab, k, self.canonical, self.consider_missing,
                                self.cluster_equal_filter, self.maf)
        cp_base, kp_base = len(self._cp_rows), len(self._kp_rows)
        cl_map = np.array([self._intern(self._cp, self._cp_rows, row) for row in o["cluster_pattern_bits"]],
                          np.uint32).reshape(-1)
        km_map = np.zeros(len(o["kmer_pattern_bits"]), np.uint32)
        for j, row in enumerate(o["kmer_pattern_bits"]):
            if self.consider_missing:       # the key ends with the id of the cluster pattern giving the NaN plane
                row = np.concatenate([row, [cl_map[o["kmer_pattern_cluster"][j]]]]).astype(np.uint32)
            km_map[j] = self._intern(self._kp, self._kp_rows, row)
        narrow, codes, wide = encode_kmers(o["row_kmer"], k)
        row_pattern = km_map[o["row_pattern"]] if len(km_map) else np.zeros(0, np.uint32)
        out = {
            "row_cluster": o["row_cluster"][narrow], "row_kmer": codes, "row_count": o["row_count"][narrow],
            "row_pattern": row_pattern[narrow],
            "wide_row_cluster": o["row_cluster"][~narrow], "wide_row_kmer": wide,
            "wide_row_count": o["row_count"][~narrow], "wide_row_pattern": row_pattern[~narrow],
            "cluster_pattern": cl_map[o["cluster_pattern"]] if len(cl_map) else np.zeros(0, np.uint32),
            "kmer_pattern_base": kp_base,
            "new_kmer_patterns": (np.stack(self._kp_rows[kp_base:]) if len(self._kp_rows) > kp_base
                                  else np.zeros((0, self.Wk), np.uint32)),
            "cluster_pattern_base": cp_base,
            "new_cluster_patterns": (np.stack(self._cp_rows[cp_base:]) if len(self._cp_rows) > cp_base
                                     else np.zeros((0, W), np.uint32)),
            "pos_kmer": np.zeros(0, np.uint64), "pos_seq": np.zeros(0, np.uint32),
            "pos_contig_start": np.zeros(0, np.int32), "pos_gene_start": np.zeros(0, np.int32),
            "pos_flags": np.zeros(0, np.uint8), "pos_wide_kmer": np.zeros((0, 2), np.uint64),
            "n_pos": 0, "pos_strand_bits": np.zeros(0, np.uint32),
        }
        if self.emit_positions:
            # compact form: one bit per base position of the packed plane, set where the reverse
            # complement was the k-mer written (used_strand -1, panfeed.py:69-75)
            out["n_pos"] = len(o["pos_seq"])
            bits = np.zeros(hb.packed.size, np.uint32)
            if self.canonical and len(o["pos_seq"]):
                rc = o["pos_used_strand"] < 0
                at = hb.seqs["base_off"][o["pos_seq"][rc]].astype(np.int64) + o["pos_pos"][rc].astype(np.int64)
                np.bitwise_or.at(bits, at >> 5, (np.uint32(1) << (at & 31).astype(np.uint32)))
            out["pos_strand_bits"] = bits
        self.n_batches += 1
        self.n_bases += int(seqs["len"].sum())
        self.n_rows += len(o["row_cluster"])
        return out

    def pattern_ids(self, cluster_namespace, first, count):
        ids = np.zeros(count, "S24")
        idx = np.arange(self.S)
        for j in range(count):
            if cluster_namespace:
                row = self._cp_rows[first + j]
                vec = ((row[idx >> 5] >> (idx & 31)) & 1).astype(np.int64)
            else:
                row = self._kp_rows[first + j]
                vec = ((row[idx >> 5] >> (idx & 31)) & 1).astype(np.float64)
                if self.consider_missing:
                    pres = self._cp_rows[int(row[self.W])]
                    vec[((pres[idx >> 5] >> (idx & 31)) & 1) == 0] = np.nan
            ids[j] = pattern_id(vec).encode()
        return ids

    def export_patterns(self, cluster_namespace, first, count):
        rows = self._cp_rows if cluster_namespace else self._kp_rows
        w = self.W if cluster_namespace else self.Wk
        return np.stack(rows[first:first + count]) if count else np.zeros((0, w), np.uint32)

    def stats(self):
        return {"batches": self.n_batches, "bases": self.n_bases, "rows": self.n_rows,
                "kmer_patterns": len(self._kp_rows), "cluster_patterns": len(self._cp_rows)}

    def close(self):
        pass

    # ---- sharded runs: the pattern exchange over gloo on host arrays ----
    def exchange(self, device):
        return HostExchange(self)


class HostExchange:
    """The global numbering pf_exchange_run gives, on host arrays between CPU processes (gloo):
    every rank's keys go to every rank (all_gather_object); owner = a hash of the full key mod
    world; the first sender in rank order writes the pattern; global id = the owner's base + the
    pattern's order at its owner.  Lets `PatternStore.finish_sharded` run between CPU processes
    and returns what dist.PatternExchange.run returns."""

    def __init__(self, ctx):
        self.ctx = ctx

    def _number(self, keys, world, rank):
        import zlib
        import torch.distributed as dist
        every = [keys]
        if dist.is_initialized():
            every = [None] * world
            dist.all_gather_object(every, keys)
        at_owner = [{} for _ in range(world)]           # owner -> {key: (order, first sender)}
        for r, rk in enumerate(every):
            for k in rk:
                b = k.tobytes()
                d = at_owner[zlib.crc32(b) % world]
                d.setdefault(b, (len(d), r))
        n_owned = [len(d) for d in at_owner]
        base = np.concatenate([[0], np.cumsum(n_owned)]).astype(np.int64)
        l2g = np.zeros(len(keys), np.int32)
        writer = np.zeros(len(keys), np.uint8)
        for i, k in enumerate(keys):
            b = k.tobytes()
            o = zlib.crc32(b) % world
            order, first = at_owner[o][b]
            l2g[i] = base[o] + order
            writer[i] = first == rank
        owned = np.array([np.frombuffer(b, np.uint32) for b in at_owner[rank]], np.uint32).reshape(
            n_owned[rank], keys.shape[1])
        return l2g, writer, n_owned, int(base[rank]), owned

    def run(self, want_unique=False, want_writer=False):
        import torch
        import torch.distributed as dist
        world = dist.get_world_size() if dist.is_initialized() else 1
        rank = dist.get_rank() if dist.is_initialized() else 0
        out, cl_l2g = {}, None
        for name, rows, w in (("cluster", self.ctx._cp_rows, self.ctx.W), ("kmer", self.ctx._kp_rows, self.ctx.Wk)):
            keys = np.stack(rows).astype(np.uint32) if rows else np.zeros((0, w), np.uint32)
            if name == "kmer" and self.ctx.consider_missing and len(keys):
                keys[:, -1] = cl_l2g[keys[:, -1]]       # the NaN plane by its GLOBAL cluster-pattern id
            l2g, writer, n_owned, base, owned = self._number(keys, world, rank)
            if name == "cluster":
                cl_l2g = l2g.astype(np.uint32)
            out[name] = {"local_to_global": torch.from_numpy(l2g),
                         "writer": torch.from_numpy(writer) if want_writer else None,
                         "n_global": int(sum(n_owned)), "n_owned": n_owned[rank], "owned_base": base,
                         "bytes_sent": int(keys.nbytes), "ms": {"total_both_namespaces": 0.0, "stages": None}}
            if want_unique:
                out[name]["owned_keys"] = owned
        return out

    def close(self):
        pass
