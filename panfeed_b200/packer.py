"""Host packer: cluster items -> 2-bit / 4-bit planes + descriptors.

Re-expresses what the reference hands from `iter_gene_clusters` to
`cluster_cutter` (`/root/reference/panfeed/input.py:455-468`,
`panfeed/panfeed.py:31,47-49`): per cluster a dict strain -> [Seqinfo] and the
int presence vector.  Only `Seqinfo.sequence` is packed; the complement string
the reference carries (`input.py:448-452`) is implied (the kernel derives the
reverse complement from the 2-bit codes, with pyfaidx's table for IUPAC codes).
"""
import numpy as np

from . import capi

_LUT2 = np.full(256, 255, np.uint8)
for _i, _c in enumerate("ACGT"):
    _LUT2[ord(_c)] = _i
_LUT4 = np.full(256, 255, np.uint8)
for _i, _c in enumerate(capi.AMB_ALPHABET):
    _LUT4[ord(_c)] = _i
_SHIFT2 = (62 - 2 * np.arange(32)).astype(np.uint64)
_SHIFT4 = (60 - 4 * np.arange(16)).astype(np.uint64)


class PackedCluster:
    """One cluster, packed and ordered by sample rank (what `cluster_cutter`
    returns in place of its k-mer dict)."""
    __slots__ = ("idx", "clusterpresab", "seq_bytes", "sample", "target",
                 "start", "end", "offset", "strand", "meta", "k", "canonical",
                 "consider_missing")

    def __init__(self, cluster, idx, clusterpresab, stroi):
        self.idx = idx
        self.clusterpresab = np.asarray(clusterpresab)
        rank = {s: i for i, s in enumerate(sorted(cluster.keys()))}
        rows = []
        for strain in cluster.keys():
            for q in cluster[strain]:
                rows.append((rank[strain], strain, q))
        rows.sort(key=lambda r: r[0])      # stable: paralog order is kept
        self.seq_bytes = [r[2].sequence.encode("ascii") for r in rows]
        self.sample = np.array([r[0] for r in rows], np.uint32)
        self.target = np.array([r[1] in stroi for r in rows], bool)
        self.start = np.array([r[2].start for r in rows], np.int32)
        self.end = np.array([r[2].end for r in rows], np.int32)
        self.offset = np.array([r[2].offset for r in rows], np.int32)
        self.strand = np.array([r[2].strand for r in rows], np.int32)
        self.meta = [(r[1], r[2].id, r[2].chromosome) for r in rows]

    def n_records(self, k, canonical):
        n = sum(max(0, len(b) - k + 1) for b in self.seq_bytes)
        return n if canonical else 2 * n


def presence_words(presab):
    """int vector [S] -> uint32 words, bit (s & 31) of word (s >> 5)."""
    presab = np.asarray(presab)
    S = presab.shape[0]
    W = (S + 31) // 32
    bits = np.zeros(W * 32, np.uint8)
    bits[:S] = presab != 0
    return (bits.reshape(W, 32).astype(np.uint32) <<
            np.arange(32, dtype=np.uint32)).sum(axis=1, dtype=np.uint64).astype(np.uint32)


def pack_planes_numpy(seq_bytes):
    """Reference implementation of the plane packing with numpy look-up tables (the product
    uses the library's native packer, `capi.pack_sequences`; the tests compare the two).
    -> (packed, base_off, amb_seq, amb_plane or None, amb_off)."""
    n_seqs = len(seq_bytes)
    lens = np.array([len(b) for b in seq_bytes], np.int64)
    padded = (lens + 63) // 64 * 64
    offs = np.zeros(n_seqs + 1, np.int64)
    np.cumsum(padded, out=offs[1:])
    total = int(offs[-1])
    ascii_plane = np.full(total, ord("A"), np.uint8)
    for b, o in zip(seq_bytes, offs[:-1]):
        ascii_plane[o:o + len(b)] = np.frombuffer(b, np.uint8)
    code2 = _LUT2[ascii_plane]
    bad = code2 == 255
    amb_seq = np.zeros(n_seqs, bool)
    amb_plane = None
    amb_off = np.zeros(n_seqs, np.uint64)
    if bad.any():
        which = np.searchsorted(offs, np.nonzero(bad)[0], side="right") - 1
        amb_seq[np.unique(which)] = True
        chunks, cur = [], 0
        for i in np.nonzero(amb_seq)[0]:
            seg = ascii_plane[offs[i]:offs[i] + padded[i]]
            c4 = _LUT4[seg]
            if (c4 == 255).any():
                sym = chr(int(seg[np.nonzero(c4 == 255)[0][0]]))
                raise ValueError(f"unsupported sequence symbol {sym!r}: only "
                                 f"{capi.AMB_ALPHABET} (IUPAC, upper case) are accepted")
            amb_off[i] = cur
            chunks.append(c4)
            cur += len(c4)
        c4 = np.concatenate(chunks)
        amb_plane = (c4.reshape(-1, 16).astype(np.uint64) << _SHIFT4).sum(
            axis=1, dtype=np.uint64)
        code2[bad] = 0
    packed = (code2.reshape(-1, 32).astype(np.uint64) << _SHIFT2).sum(
        axis=1, dtype=np.uint64)
    return packed, offs[:-1].astype(np.uint64), amb_seq, amb_plane, amb_off


class SeqMeta:
    """(strain, feature id, contig) of every sequence of a batch, cluster after cluster; the
    per-cluster lists are only built when an entry is read (clusters cut by the native feeder
    make theirs on demand, and only the positional rows of a second pass need them)."""

    def __init__(self, clusters, counts):
        self.clusters = clusters
        self.first = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)

    def __len__(self):
        return int(self.first[-1])

    def __getitem__(self, i):
        if i < 0:
            i += len(self)
        c = int(np.searchsorted(self.first, i, side="right")) - 1
        return self.clusters[c].meta[i - int(self.first[c])]

    def __iter__(self):
        for pc in self.clusters:
            yield from pc.meta


def pack_batch(packed_clusters, cluster_ids=None):
    """-> (capi.HostBatch, seq_meta (SeqMeta), cluster idx list).  Clusters are
    `PackedCluster`s (Python cutting) or `feeder.NativePackedCluster`s (slices of the planes the
    library packed when it cut them)."""
    # planes: clusters the native feeder packed at cutting time bring their word ranges; runs of
    # clusters that still hold ASCII sequences are packed here; the pieces are then laid end to end
    # (every sequence starts on a 64-base boundary, so that equals packing everything at once)
    parts, lens, run = [], [], []

    def flush_run():
        if run:
            n = len(run)
            off = np.zeros(n + 1, np.uint64)
            np.cumsum(np.fromiter((len(b) for b in run), np.uint64, n), out=off[1:])
            parts.append(capi.pack_blob(b"".join(run), off))
            run.clear()

    for pc in packed_clusters:
        if hasattr(pc, "packed_words"):
            flush_run()
            parts.append((pc.packed_words, pc.base_rel, pc.is_amb, pc.amb_words if pc.is_amb.any() else None,
                          pc.amb_rel))
            lens.append(pc.seq_len)
        else:
            run.extend(pc.seq_bytes)
            lens.append(np.fromiter((len(b) for b in pc.seq_bytes), np.int64, len(pc.seq_bytes)))
    flush_run()
    lens = np.concatenate(lens).astype(np.int64) if lens else np.zeros(0, np.int64)
    n_seqs = len(lens)
    words, amb_words = 0, 0
    base_off, amb_seq, amb_off, amb_planes = [], [], [], []
    for pk, bo, ia, ap, ao in parts:
        ia = np.asarray(ia, bool)
        base_off.append(np.asarray(bo, np.uint64) + np.uint64(words * 32))
        amb_seq.append(ia)
        amb_off.append(np.where(ia, np.asarray(ao, np.uint64) + np.uint64(amb_words * 16), np.uint64(0)).astype(np.uint64))
        words += len(pk)
        if ap is not None and len(ap):
            amb_planes.append(ap)
            amb_words += len(ap)
    packed = np.concatenate([p[0] for p in parts]) if parts else np.zeros(0, np.uint64)
    base_off = np.concatenate(base_off) if base_off else np.zeros(0, np.uint64)
    amb_seq = np.concatenate(amb_seq) if amb_seq else np.zeros(0, bool)
    amb_off = np.concatenate(amb_off) if amb_off else np.zeros(0, np.uint64)
    amb_plane = np.concatenate(amb_planes) if amb_planes else None

    seqs = np.zeros(n_seqs, capi.SEQ_DTYPE)
    clusters = np.zeros(len(packed_clusters), capi.CLUSTER_DTYPE)
    S = len(packed_clusters[0].clusterpresab) if packed_clusters else 0
    W = (S + 31) // 32
    presence = np.zeros((len(packed_clusters), W), np.uint32)
    ids, counts = [], []
    i = 0
    for ci, pc in enumerate(packed_clusters):
        n = len(pc.sample)
        sl = slice(i, i + n)
        seqs["cluster"][sl] = ci
        seqs["sample"][sl] = pc.sample
        seqs["flags"][sl] = pc.target.astype(np.uint32) * capi.PF_SEQ_TARGET
        seqs["start"][sl] = pc.start
        seqs["end"][sl] = pc.end
        seqs["offset"][sl] = pc.offset
        seqs["strand"][sl] = pc.strand
        clusters["id"][ci] = ci if cluster_ids is None else cluster_ids[ci]
        presence[ci] = presence_words(pc.clusterpresab)
        counts.append(n)
        ids.append(pc.idx)
        i += n
    seqs["base_off"] = base_off
    seqs["len"] = lens.astype(np.uint32)
    seqs["flags"] |= amb_seq.astype(np.uint32) * capi.PF_SEQ_AMBIGUOUS
    seqs["amb_off"] = amb_off
    return capi.HostBatch(packed, seqs, clusters, presence, amb_plane), SeqMeta(list(packed_clusters), counts), ids


_ACGT = np.frombuffer(b"ACGT", np.uint8)
_AMB = np.frombuffer(capi.AMB_ALPHABET.encode(), np.uint8)


def kmers_to_str(kmers, k):
    """uint64 2-bit k-mers -> numpy bytes array S{k}."""
    kmers = np.asarray(kmers, np.uint64)
    if kmers.size == 0:
        return np.zeros(0, f"S{k}")
    sh = (2 * (k - 1 - np.arange(k))).astype(np.uint64)
    codes = ((kmers[:, None] >> sh[None, :]) & np.uint64(3)).astype(np.uint8)
    return np.ascontiguousarray(_ACGT[codes]).view(f"S{k}").ravel()


def wide_kmers_to_str(kmers, k, n_words=2):
    """[n, n_words] uint64 k-mers (most significant word first) -> numpy bytes array S{k}: 4 bits
    per symbol (codes of AMB_ALPHABET) when k symbols fit that way - N/IUPAC k-mers of k <= 32 in
    two words, of k <= 64 in four (xwide rows) - else 2 bits per base (two words, k > 32)."""
    kmers = np.asarray(kmers, np.uint64).reshape(-1, n_words)
    if kmers.shape[0] == 0:
        return np.zeros(0, f"S{k}")
    bits = 4 if k <= 16 * n_words else 2
    alphabet = _AMB if bits == 4 else _ACGT
    out = np.zeros((kmers.shape[0], k), np.uint8)
    for i in range(k):
        pos = bits * (k - 1 - i)           # bit offset from the bottom of the last word
        word = kmers[:, n_words - 1 - pos // 64] >> np.uint64(pos % 64)
        out[:, i] = alphabet[(word & np.uint64((1 << bits) - 1)).astype(np.uint8)]
    return np.ascontiguousarray(out).view(f"S{k}").ravel()
