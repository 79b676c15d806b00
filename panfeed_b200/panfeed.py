"""The reference's hot-path callables, re-hosted on the CUDA library.

Same names, argument meaning and output files as
`/root/reference/panfeed/panfeed.py`:

    cluster_cutter(cluster_gen, klength, stroi, multiple_files, canon,
                   consider_missing_cluster, output, compress)     panfeed.py:23
    pattern_hasher(cluster_dict_iter, kmer_stroi, hash_pat, kmer_hash, genepres,
                   patfilt, maf, output, patterns, consider_missing_cluster,
                   compress)                                        panfeed.py:132
    write_headers(hash_pat, kmer_hash, genepres)                    panfeed.py:116

What changes is where the work happens.  `cluster_cutter` only packs the
cluster (host); the k-mer extraction, sorting, presence-bitset reduction, MAF /
same-as-cluster filters and the global pattern dedup all run on the GPU inside
`pattern_hasher`, many clusters per launch.  The second element of the tuple
`cluster_cutter` returns is therefore a `PackedCluster`, not a dict, and
`patterns` is a `PatternStore` (the device-resident pattern table plus the id
strings handed out so far) instead of a Python set.  There is no CPU path.
"""
import binascii
import hashlib
import logging
import os

import numpy as np

from . import capi, packer
from .input import create_hash_files, create_kmer_stroi

logger = logging.getLogger("panfeed.panfeed")

# k-mer records per GPU batch (whole clusters are never split)
BATCH_RECORDS = 192 * 1024 * 1024

_COMP = bytes.maketrans(b"ACTGNYRWSKMDVHBX", b"TGACNRYWSMKHBDVX")


def pattern_id(vec):
    """base64(md5(raw little-endian bytes of the vector))[:24] (panfeed.py:175-176,
    206-207): int64 bytes for cluster rows, float64 bytes for k-mer rows.  Host-side
    definition of the id, kept for tools and tests; the product derives ids on the
    device (`Context.pattern_ids`, kernel K5)."""
    return binascii.b2a_base64(hashlib.md5(np.ascontiguousarray(vec).view(np.uint8)).digest()
                               ).decode()[:24]


def cluster_cutter(cluster_gen, klength, stroi, multiple_files, canon,
                   consider_missing_cluster, output, compress=False):
    """Pack one cluster for the GPU.  Returns the reference's 4-tuple shape
    (idx, <payload>, clusterpresab, memchunk); the positional rows the reference
    formats here (panfeed.py:90-107) come back from the device in
    `pattern_hasher`, so memchunk is always None."""
    cluster, idx, clusterpresab = cluster_gen
    logger.debug(f"Packing sequences of {idx}")
    pc = packer.PackedCluster(cluster, idx, clusterpresab, stroi)
    pc.k, pc.canonical, pc.consider_missing = klength, bool(canon), bool(consider_missing_cluster)
    return idx, pc, clusterpresab, None


def write_headers(hash_pat, kmer_hash, genepres):
    hash_pat.write("hashed_pattern" + "".join(f"\t{s}" for s in sorted(genepres.columns)) + "\n")
    hash_pat.flush()
    kmer_hash.write("cluster\tk-mer\thashed_pattern\n")
    kmer_hash.flush()


class _IdTable:
    """Growable numpy S24 array: the id strings of one pattern namespace, appended batch by
    batch (rebuilding an array from a Python list of every id issued so far would make a first
    pass quadratic in the number of patterns)."""

    def __init__(self):
        self.buf = np.zeros(1024, "S24")
        self.n = 0

    def append(self, ids):
        m = len(ids)
        if self.n + m > len(self.buf):
            grown = np.zeros(max(2 * len(self.buf), self.n + m), "S24")
            grown[:self.n] = self.buf[:self.n]
            self.buf = grown
        self.buf[self.n:self.n + m] = ids
        self.n += m

    def view(self):
        return self.buf[:self.n]


class PatternStore:
    """What `patterns` is in this build: the GPU context (pattern tables and
    pools live in HBM) and the ids of every pattern numbered so far.

    sharded=True (several ranks, `torchrun -m panfeed_b200`): this rank sees only its shard of
    the clusters, so whether a pattern is NEW is a global question: hashes_to_patterns rows are
    not written batch by batch but once, by `finish_sharded`, after the pattern exchange."""

    def __init__(self, sharded=False):
        self.ctx = None
        self.key = None
        self.sharded = bool(sharded)
        self.kmer_ids = _IdTable()       # pool index -> id (float64 namespace)
        self.cluster_ids = _IdTable()    # pool index -> id (int64 namespace)
        self.cluster_bits = []           # per batch: presence words of the new cluster patterns (NaN planes)
        self._cluster_bits_cat = None
        self.n_patterns = 0              # len() of the reference's `patterns` set

    def __len__(self):
        return self.n_patterns

    def context(self, k, S, canonical, consider_missing, cluster_equal_filter, maf,
                device=0, sort_bits=0):
        key = (k, S, canonical, consider_missing, cluster_equal_filter, maf, device)
        if self.ctx is None:
            # positional rows in the compact form: only the used_strand bits leave the device
            self.ctx = capi.Context(k, S, canonical, consider_missing, cluster_equal_filter,
                                    emit_positions=2, maf=maf, sort_bits=sort_bits,
                                    device=device)
            self.key = key
        elif key != self.key:
            raise ValueError("pattern_hasher was called with options that differ from the ones "
                             "its PatternStore was created with")
        return self.ctx

    def cluster_planes(self):
        """[n cluster patterns, W] presence words of every cluster pattern numbered so far."""
        if self.cluster_bits and (self._cluster_bits_cat is None or len(self.cluster_bits) > 1):
            self._cluster_bits_cat = np.concatenate(self.cluster_bits)
            self.cluster_bits = [self._cluster_bits_cat]
        return self._cluster_bits_cat

    def reset(self):
        """`patterns = set()` of --multiple-files (panfeed.py:165)."""
        if self.ctx is not None:
            self.ctx.reset_patterns()
        self.kmer_ids, self.cluster_ids = _IdTable(), _IdTable()
        self.cluster_bits, self._cluster_bits_cat = [], None
        self.n_patterns = 0

    def close(self):
        if self.ctx is not None:
            self.ctx.close()
            self.ctx = None

    def finish_sharded(self, hash_pat, k, S, canonical, consider_missing, cluster_equal_filter, maf,
                       device, chunk=1 << 16):
        """After the last batch of a sharded run: the global pattern exchange
        (dist.PatternExchange: pf_exchange_run over NCCL), then the hashes_to_patterns rows of the patterns THIS
        rank is the writer of (the owner of a pattern names the first rank that sent it), so
        that the ranks together write every pattern once - the job of the reference's single
        writer process and its `patterns` set (__main__.py:67-81, panfeed.py:210-212)."""
        import torch
        from . import dist as pfdist
        ctx = self.context(k, S, canonical, consider_missing, cluster_equal_filter, maf, device)
        # (a context may bring its own exchange: the CPU tests' stand-in does)
        if hasattr(ctx, "exchange"):
            exchange = ctx.exchange(device)
        else:
            exchange = pfdist.PatternExchange(ctx, torch.device("cuda", device))
        out = exchange.run(want_writer=True)
        exchange.close()
        W = (S + 31) // 32
        written = 0
        for ns, name, ids in ((True, "cluster", self.cluster_ids.view()), (False, "kmer", self.kmer_ids.view())):
            wr = out[name]["writer"].cpu().numpy().astype(bool)
            assert len(wr) == len(ids), "pattern ids out of step with the device pools"
            for c0 in range(0, len(wr), chunk):
                sel = wr[c0:c0 + chunk]
                if not sel.any():
                    continue
                bits = ctx.export_patterns(ns, c0, len(sel))[sel]
                present = None
                if consider_missing and not ns:
                    present = self.cluster_planes()[bits[:, W].astype(np.int64)]
                write_text(hash_pat, capi.format_patterns(bits, S, ids[c0:c0 + chunk][sel], present))
                written += int(sel.sum())
        self.n_patterns = out["cluster"]["n_global"] + out["kmer"]["n_global"]
        return {"written_here": written, "cluster_patterns_global": out["cluster"]["n_global"],
                "kmer_patterns_global": out["kmer"]["n_global"]}


def write_text(handle, data):
    """`data` (bytes or a uint8 array of UTF-8 text) to a handle opened in text mode, without a
    Python str in between: a batch's rows are hundreds of MB, and decode + join + the text layer's
    re-encode cost more than formatting them.  Plain files take the bytes through their binary
    buffer, GzipTextWriter takes bytes as they are, anything else (StringIO) gets a str."""
    if len(data) == 0:
        return
    raw = getattr(handle, "buffer", None)
    if raw is not None:
        handle.flush()
        raw.write(data)
    elif hasattr(handle, "parts"):                  # input.GzipTextWriter
        handle.write(bytes(data))
    else:
        handle.write(bytes(data).decode())


def _run_batch(store, ctx, hb, meta, idxs, S, k, canonical, consider_missing, annotate=None):
    """One GPU batch (`hb`: the capi.HostBatch; meta(i) -> (strain, feature id, contig) of its
    sequence i; idxs: the names of its clusters) -> (kmers.tsv text, list of hashes_to_patterns
    texts, kmers_to_hashes text) as bytes / uint8 arrays; the arrays are the formatters' reused
    buffers, to be written out before the next batch."""
    ctx.submit(hb)
    # views of the context's pinned result buffers (valid until the next collect): everything below
    # reads them before this function returns; what outlives the batch is copied explicitly
    r = ctx.collect(copy=False)

    # ---- new patterns -> ids (MD5 on the device, K5) + hashes_to_patterns rows.  The pattern
    #      tables are keyed on the full vector, so every new pattern is a new id: nothing is
    #      looked up per pattern on the host. ----
    pat_text = []
    new_cp = r["new_cluster_patterns"]
    if len(new_cp):
        new_ids = ctx.pattern_ids(True, r["cluster_pattern_base"], len(new_cp))
        store.cluster_ids.append(new_ids)
        store.cluster_bits.append(new_cp.copy())
        if not store.sharded:
            pat_text.append(capi.format_patterns(new_cp, S, new_ids, raw=True, scratch="cluster_patterns"))
            store.n_patterns += len(new_cp)
    new_kp = r["new_kmer_patterns"]
    if len(new_kp):
        W = (S + 31) // 32
        new_ids = ctx.pattern_ids(False, r["kmer_pattern_base"], len(new_kp))
        store.kmer_ids.append(new_ids)
        if not store.sharded:
            present = None
            if consider_missing:      # NaN cells = samples whose cluster is absent (the key's last word
                present = store.cluster_planes()[new_kp[:, W].astype(np.int64)]   # names that cluster pattern)
            pat_text.append(capi.format_patterns(new_kp, S, new_ids, present, raw=True, scratch="kmer_patterns"))
            store.n_patterns += len(new_kp)

    # ---- kmers_to_hashes rows, cluster by cluster: formatted by the library's host threads
    #      (pf_format_kmer_rows; inside a cluster the plain k-mers in alphabetical order, then the
    #      rows holding N/IUPAC symbols - the reference's order is arbitrary too) --------------
    hash_text, _ = capi.format_kmer_rows(r, k, [str(idx).encode() for idx in idxs], store.kmer_ids.view(),
                                         store.cluster_ids.view(), raw=True)

    # ---- kmers.tsv rows from the positional records: formatted by the library's host
    #      threads (pf_format_positions_compact: the device only returns the used_strand bit
    #      of every window, the rest of a row follows from the batch itself), 1e8 rows are too
    #      many for Python.  Only the target sequences need their leading fields (and with them
    #      their lazily built metadata). ----
    pos_text = b""
    if annotate is not None:
        # --associations: the get-kmers lines instead of kmers.tsv, joined on the device (assoc.py)
        annotate.batch(hb, r, ctx.assoc_collect(), k, canonical, idxs, meta)
    elif r["n_pos"]:
        leads = [b""] * len(hb.seqs)
        cl, strand = hb.seqs["cluster"], hb.seqs["strand"]
        for i in np.nonzero(hb.seqs["flags"] & capi.PF_SEQ_TARGET)[0].tolist():
            m = meta(i)
            leads[i] = f"{idxs[cl[i]]}\t{m[0]}\t{m[1]}\t{m[2]}\t{strand[i]}\t".encode()
        pos_text = capi.format_positions_compact(hb, r["pos_strand_bits"], k, canonical, leads, raw=True)
    return pos_text, pat_text, hash_text

def pattern_hasher(cluster_dict_iter, kmer_stroi, hash_pat, kmer_hash, genepres, patfilt, maf,
                   output, patterns=None, consider_missing_cluster=False, compress=False,
                   device=0, sort_bits=0, annotate=None):
    """Consumes `cluster_cutter` results, runs K1..K4 on the GPU in batches of
    whole clusters and writes the three files exactly as the reference does
    (panfeed.py:152-233).  Returns the updated `patterns` (a PatternStore).
    annotate (an assoc.AnnotatedWriter, --associations): the positional rows are joined to the
    passing associations on the device and written there instead of to kmer_stroi."""
    multiple_files = hash_pat is None or kmer_hash is None
    if patterns is None or isinstance(patterns, set):
        patterns = PatternStore()
    S = len(genepres.columns)

    pending, pending_records = [], 0

    def flush(ready=None):
        """Runs the pending clusters as one batch, or `ready`: a batch the native feeder cut and
        packed as a whole (feeder.NativePackedBatch)."""
        nonlocal pending, pending_records, hash_pat, kmer_hash
        if ready is not None:
            first, hb, meta, idxs = ready, ready.hb, ready.meta, ready.idxs
        elif pending:
            pcs = [p[1] for p in pending]
            idxs = [p[0] for p in pending]
            first = pcs[0]
            hb, seq_meta, _ = packer.pack_batch(pcs, list(range(len(pcs))))
            meta = seq_meta.__getitem__
        else:
            return
        ctx = patterns.context(first.k, S, first.canonical, bool(consider_missing_cluster),
                               patfilt == False, maf, device, sort_bits)  # noqa: E712
        if annotate is not None and not annotate.loaded:
            ctx.assoc_load(annotate.digests)
            annotate.loaded = True
        pos_text, pat_texts, hash_text = _run_batch(patterns, ctx, hb, meta, idxs, S, first.k,
                                                    first.canonical, bool(consider_missing_cluster), annotate)
        if multiple_files:
            path = os.path.join(output, idxs[0])
            if not os.path.exists(path):
                os.mkdir(path)
            ks = create_kmer_stroi(path, compress)
            write_text(ks, pos_text)
            ks.close()
            hp, kh = create_hash_files(path, compress)
            write_headers(hp, kh, genepres)
            for t in pat_texts:
                write_text(hp, t)
            write_text(kh, hash_text)
            hp.close()
            kh.close()
        else:
            if kmer_stroi is not None:
                write_text(kmer_stroi, pos_text)
            for t in pat_texts:
                write_text(hash_pat, t)
            write_text(kmer_hash, hash_text)
        if ready is None:
            pending, pending_records = [], 0

    for idx, pc, clusterpresab, memchunk in cluster_dict_iter:
        if hasattr(pc, "hb"):               # a whole batch from the native feeder (never with --multiple-files)
            flush()
            flush(pc)
            continue
        if multiple_files:
            flush()
            patterns.reset()
        n = pc.n_records(pc.k, pc.canonical)
        if pending and pending_records + n > BATCH_RECORDS:
            flush()
        pending.append((idx, pc))
        pending_records += n
        if multiple_files:
            flush()
    flush()
    if not multiple_files:
        hash_pat.flush()
        kmer_hash.flush()
    return patterns
