"""--associations: a second pass that writes panfeed-get-kmers' table itself.

The reference closes the GWAS loop with two steps: a second pass writes kmers.tsv (one text row
per k-mer instance of every target strain), then `panfeed-get-kmers` reads it back with
kmers_to_hashes.tsv and joins both to the passing associations in pandas (get_kmers.py:88-145).
Here the join runs on the device while the batch is there (pf_assoc_collect, kernels K6): the
passing patterns are a table of MD5 digests in device memory, every pattern is looked up by the
digest K5 computes, every target window finds its row by (cluster, k-mer).  Only the lines of the
answer are formatted (pf_format_annotated), into <out>/annotated_kmers.tsv.

The association columns are printed as pandas prints them after the reference's join: each passing
association is formatted once, by pandas, with the dtypes the joined frame would give it.  Two
facts of that frame are global and only known at the end of the run; batches whose text depends
on them are held back until they are known:
  - default (right join): a window whose k-mer does not pass has empty association fields, which
    makes pandas print integer / boolean association columns as floats / objects;
  - --only-passing (left join): a passing k-mer without a target window, or a passing cluster-row
    hash, has empty positional fields, which makes pandas print all integer positional columns as
    floats ("361.0").
Each fact is an OR over the batches, so a sharded run (torchrun, whole clusters per rank) ORs the
ranks' facts once after their last batch; every rank writes a piece, rank 0 merges them.
"""
import io
import logging
import os

import numpy as np

from . import capi
from .input import GzipTextWriter, part_path

logger = logging.getLogger("panfeed.assoc")

POSITIONAL = ["strain", "feature_id", "contig", "feature_strand", "contig_start", "contig_end", "gene_start",
              "gene_end", "strand"]


def load_passing(path, column, threshold):
    """The passing associations (postgwas.passing_associations) whose id names a pattern, indexed by
    id, and their digests ([n, 16] uint8, row i = association row i)."""
    from .postgwas import passing_associations
    a = passing_associations(path, column, threshold)
    digests, keep = capi.id_digests(list(a.index))
    skipped = len(a) - len(keep)
    if skipped:
        logger.warning(f"{skipped} passing association ids are not pattern ids (24 characters of base64): skipped")
    a = a.iloc[keep]
    if a.index.duplicated().any():
        raise ValueError("the associations file lists a pattern id more than once")
    a.index.name = "hashed_pattern"
    return a, digests


def snippets(a, upcast):
    """One text per association row: the hashed_pattern and association fields, as pandas' to_csv prints
    them.  upcast: with the dtypes a frame in which some rows lack them has (int -> float, bool -> object)."""
    if len(a) == 0:
        return []
    if upcast:
        a = a.reset_index().reindex(range(len(a) + 1)).iloc[:len(a)].set_index("hashed_pattern")
    buf = io.StringIO()
    a.to_csv(buf, sep="\t", header=False, lineterminator="\n")
    lines = buf.getvalue().split("\n")[:-1]
    if len(lines) != len(a):
        raise ValueError("association fields that hold line breaks are not supported")
    return [x.encode() for x in lines]


class AnnotatedWriter:
    """<out>/annotated_kmers.tsv(.gz): the header, then the lines of every batch.

    rank (a sharded run, one process per GPU): this rank's header-less piece of that file under
    <out>/.parts/ instead; rank 0 merges the pieces after `header`.  The upcast fact is then the OR
    over the ranks: a rank holds both variants of its batches until `finish` has learnt it."""

    NAME = "annotated_kmers.tsv"

    def __init__(self, output, a, digests, only_passing, compress, rank=None):
        self.only_passing = bool(only_passing)
        if rank is None:
            path = os.path.join(output, self.NAME + (".gz" if compress else ""))
        else:
            path = part_path(output, self.NAME, rank, compress)
        self.handle = GzipTextWriter(path) if compress else open(path, "wb")
        self.digests = digests
        self.loaded = False              # pf_assoc_load on the run's context (pattern_hasher, first batch)
        self.fields = 1 + len(a.columns)
        self.snips = {False: snippets(a, False), True: snippets(a, True)}
        # the text of a batch depends on the global fact only where the two variants differ
        self.same = (not self.only_passing) and self.snips[False] == self.snips[True]
        self.upcast = False
        self.pending = []
        self.bytes = 0
        self.header = "\t".join(["cluster", "k-mer", "hashed_pattern"] + [str(c) for c in a.columns] + POSITIONAL) + "\n"
        if rank is None:
            self._write(self.header.encode())

    def _write(self, data):
        if len(data):
            self.handle.write(bytes(data))
            self.bytes += len(data)

    def _format(self, job, upcast):
        hb, r, assoc, k, canonical, tags, leads = job
        flags = capi.PF_ANNOT_ONLY_PASSING if self.only_passing else 0
        snips = self.snips[False]
        if self.only_passing:
            flags |= capi.PF_ANNOT_FLOAT_POSITIONS if upcast else 0
        else:
            snips = self.snips[upcast]
        return capi.format_annotated(hb, r["pos_strand_bits"], k, canonical, r, assoc, tags, leads, snips,
                                     self.fields, flags)

    def batch(self, hb, r, assoc, k, canonical, idxs, meta):
        """One batch: hb its HostBatch, r its collect() (views are fine: used before returning), assoc its
        assoc_collect(), idxs the names of its clusters, meta(i) -> (strain, feature id, contig)."""
        seqs = hb.seqs
        target = (seqs["flags"] & capi.PF_SEQ_TARGET) != 0
        live = target & (assoc["cluster_pass"][seqs["cluster"]] != 0) & (seqs["len"] >= k)
        if self.only_passing:
            flag = bool((assoc["row_seen"] == 0).any() or (assoc["cluster_assoc"] != capi.PF_ASSOC_NONE).any())
        else:
            rows = int(((seqs["len"][live].astype(np.int64) - k + 1).sum()) * (1 if canonical else 2))
            flag = rows > len(assoc["window"])
        leads = [b""] * len(seqs)
        for i in np.nonzero(live)[0].tolist():
            m = meta(i)
            leads[i] = f"{m[0]}\t{m[1]}\t{m[2]}\t".encode()
        job = (hb, r, assoc, k, canonical, [str(x).encode() for x in idxs], leads)
        if flag and not self.upcast:
            self.upcast = True
            for _, up in self.pending:
                self._write(up)
            self.pending = []
        if self.upcast or self.same:
            self._write(self._format(job, self.upcast))
        else:
            self.pending.append((bytes(self._format(job, False)), bytes(self._format(job, True))))

    def finish(self, any_rank=bool):
        """After the last batch: any_rank(local fact) -> the fact over all ranks (a collective in a
        sharded run, which every rank must call exactly once, batches or not), then the held
        batches in the variant it selects, and the file is closed."""
        upcast = any_rank(self.upcast)
        for text, up in self.pending:
            self._write(up if upcast else text)
        self.pending = []
        self.handle.close()
