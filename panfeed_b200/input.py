"""Feeder: input discovery, GFF3/FASTA reading, panaroo table, per-cluster
sequence cutting.  Same function names, arguments and yield shapes as the
reference's `panfeed/input.py`, so that the reference's `__main__` wiring
(`__main__.py:244-276`) works against this module unchanged.

Behavioural spec: SURVEY.md App. A1.  Differences from the reference, on purpose:
  * no pyfaidx: contigs are read once into memory (upper-cased, like
    `Fasta(..., sequence_always_upper=True)`, input.py:262-266); no
    `<out>/fastas/*.fasta(.fai)` scratch files are written, so `clean_up_fasta`
    has nothing to remove;
  * a strain that is in the panaroo table but has no GFF raises instead of
    silently producing misaligned presence vectors (reference defect,
    SURVEY.md App. A1.4).
"""
import logging
import os
import sys

import numpy as np
import pandas as pd

from .classes import Feature, Seqinfo

logger = logging.getLogger("panfeed.input")

# pyfaidx's complement table (third party, un-vendored in the reference)
_COMPLEMENT = str.maketrans("ACTGNactgnYRWSKMDVHBXyrwskmdvhbx",
                            "TGACNtgacnRYWSMKHBDVXrywsmkhbdvx")


def _genome_name(path):
    return ".".join(os.path.split(path)[-1].split(".")[:-1])


def _listing(arg):
    """A directory listing or the lines of a file of files (input.py:20-27)."""
    if os.path.isfile(arg):
        return [line.rstrip() for line in open(arg)], True
    return os.listdir(arg), False


def what_are_my_inputfiles(gffdir, fastadir=None):
    """-> (sorted genome names with a .gff, sorted genome names that also have
    a .fasta/.fna).  input.py:16-65."""
    gffs = {_genome_name(f) for f in _listing(gffdir)[0] if f.endswith(".gff")}
    fastas = set()
    if fastadir is not None:
        for f in _listing(fastadir)[0]:
            if f.endswith(".fasta") or f.endswith(".fna"):
                g = _genome_name(f)
                if g in gffs:
                    fastas.add(g)
    if not gffs:
        logger.error(f"No GFF files found in the inputs provided ({gffdir})")
        sys.exit(1)
    return sorted(gffs), sorted(fastas)


def read_fasta_text(lines):
    """FASTA lines -> {record name (up to first blank): upper-case sequence}."""
    contigs, name, parts = {}, None, []
    for line in lines:
        line = line.rstrip("\r\n")
        if line.startswith(">"):
            if name is not None:
                contigs[name] = "".join(parts).upper()
            fields = line[1:].split()
            name, parts = (fields[0] if fields else ""), []
        elif name is not None:
            parts.append(line.strip())
    if name is not None:
        contigs[name] = "".join(parts).upper()
    return contigs


def parse_gff(file_name, feature_types=None):
    """CDS features with an ID attribute -> {ID: Feature}.  input.py:274-332."""
    wanted = {"CDS"} if feature_types is None else feature_types
    features = {}
    with open(file_name) as handle:
        for line in handle:
            head = line.lstrip()
            if head.startswith("##FASTA"):
                break
            if head.startswith("#"):
                continue
            cols = line.split("\t")
            try:
                if cols[2] not in wanted:
                    continue
                start, end = int(cols[3]), int(cols[4])
                strand = 1 if cols[6] == "+" else -1
                ident = None
                for field in cols[8].split(";"):
                    if field.startswith("ID") and "=" in field:
                        ident = field.split("=")[1]
                if ident is None:
                    continue
                features[ident] = Feature(ident, cols[0], start, end, strand)
            except Exception as exc:            # same tolerance as the reference
                logger.warning(f'{exc}, skipping line "{line.rstrip()}" from {file_name}')
    return features


def prep_data_n_fasta(filelist, fastalist, gffdir, fastadir, output):
    """-> {genome: (contigs dict, features dict)}.  input.py:68-138, with the
    nucleotides kept in memory instead of behind a faidx file."""
    gff_files, gff_is_list = _listing(gffdir)
    if gff_is_list:
        gff_path = {_genome_name(f): f for f in gff_files if f.endswith(".gff")}
    else:
        gff_path = {g: os.path.join(gffdir, f"{g}.gff") for g in filelist}
    fasta_path = {}
    if fastadir is not None:
        files, is_list = _listing(fastadir)
        for f in files:
            if f.endswith(".fna") or f.endswith(".fasta"):
                fasta_path[_genome_name(f)] = f if is_list else os.path.join(fastadir, f)
    data = {}
    for genome in filelist:
        logger.debug(f"Handling {genome}")
        if genome in fastalist:
            if genome not in fasta_path:
                logger.error(f"Neither {genome}.fna not {genome}.fasta found in {fastadir}")
                sys.exit(1)
            with open(fasta_path[genome]) as fh:
                contigs = read_fasta_text(fh)
        else:
            text = open(gff_path[genome]).read().split("##FASTA")[1]
            contigs = read_fasta_text(text.split("\n"))
        data[genome] = (contigs, parse_gff(gff_path[genome]))
    return data


def clean_up_fasta(filelist, fastalist, output, fastadir):
    """Nothing to remove: no scratch FASTA/faidx files are created (input.py:141-180)."""
    return None


class GzipTextWriter:
    """Text handle over a .gz file, like gzip.open(path, "wt", compresslevel=9) (input.py:235-259),
    but the deflate runs on the library's host threads: text is collected and written as a run of
    complete gzip members (pf_gzip_members) whenever `flush_bytes` have accumulated.  Any gzip
    reader sees one stream; unlike the reference's handles this one is also safe to fill from the
    single writer of a multi-core run."""

    def __init__(self, path, level=9, flush_bytes=64 << 20):
        self.f = open(path, "wb")
        self.level = level
        self.flush_bytes = flush_bytes
        self.parts = []
        self.size = 0
        self.wrote = False

    def write(self, text):
        if not text:
            return 0
        data = text.encode() if isinstance(text, str) else bytes(text)
        self.parts.append(data)
        self.size += len(data)
        if self.size >= self.flush_bytes:
            self._emit()
        return len(text)

    def _emit(self):
        if self.size == 0:
            return
        from . import capi
        self.f.write(capi.gzip_members(b"".join(self.parts), self.level))
        self.parts, self.size, self.wrote = [], 0, True

    def flush(self):
        """Keeps the text buffered (a gzip member per flush() would bloat the file); the file on
        disk is complete after close()."""
        self.f.flush()

    def close(self):
        if self.f.closed:
            return
        self._emit()
        if not self.wrote:                      # nothing was written: still a valid (empty) gzip file
            from . import capi
            self.f.write(capi.gzip_members(b"", self.level))
        self.f.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


KMERS_TSV_HEADER = ("cluster\tstrain\tfeature_id\tcontig\tfeature_strand\tcontig_start\t"
                    "contig_end\tgene_start\tgene_end\tstrand\tk-mer\n")


def create_kmer_stroi(output, compress=False):
    """kmers.tsv(.gz) with its header.  input.py:235-246."""
    if compress:
        handle = GzipTextWriter(os.path.join(output, "kmers.tsv.gz"))
    else:
        handle = open(os.path.join(output, "kmers.tsv"), "w")
    handle.write(KMERS_TSV_HEADER)
    handle.flush()
    return handle


OUTPUT_NAMES = ("kmers.tsv", "hashes_to_patterns.tsv", "kmers_to_hashes.tsv")


def part_path(output, name, rank, compress=False):
    """<output>/.parts/<name>[.gz].<rank>: a rank's header-less piece of output file `name`."""
    return os.path.join(output, ".parts", f"{name}{'.gz' if compress else ''}.{rank}")


def create_part_files(output, rank, compress=False, names=OUTPUT_NAMES):
    """Sharded run: this rank's header-less pieces of the outputs `names` (by default kmers.tsv,
    hashes_to_patterns, kmers_to_hashes) under <output>/.parts/.  With --compress every piece is
    a complete gzip stream, so the merged file is a run of gzip members."""
    os.makedirs(os.path.join(output, ".parts"), exist_ok=True)
    handles = []
    for name in names:
        path = part_path(output, name, rank, compress)
        handles.append(GzipTextWriter(path) if compress else open(path, "w"))
    return tuple(handles)


def merge_part_files(output, world, headers, compress=False, names=OUTPUT_NAMES):
    """Rank 0, after every rank closed its pieces: header + the pieces in rank order -> the
    output files `names`; the pieces are removed."""
    import shutil
    from . import capi
    for name, header in zip(names, headers, strict=True):
        final = os.path.join(output, name + (".gz" if compress else ""))
        with open(final, "wb") as out:
            out.write(capi.gzip_members(header.encode(), 9) if compress else header.encode())
            for r in range(world):
                with open(part_path(output, name, r, compress), "rb") as piece:
                    shutil.copyfileobj(piece, out, 16 << 20)
    shutil.rmtree(os.path.join(output, ".parts"))


def create_hash_files(output, compress=False):
    """(hashes_to_patterns, kmers_to_hashes) handles.  input.py:249-259."""
    if compress:
        return (GzipTextWriter(os.path.join(output, "hashes_to_patterns.tsv.gz")),
                GzipTextWriter(os.path.join(output, "kmers_to_hashes.tsv.gz")))
    return (open(os.path.join(output, "hashes_to_patterns.tsv"), "w"),
            open(os.path.join(output, "kmers_to_hashes.tsv"), "w"))


def set_input_output(stroi_in, genes_in, presence_absence, output,
                     single_file=True, compress=False, make_outputs=True, native_table=False):
    """-> (stroi, genes, kmer_stroi, hash_pat, kmer_hash, genepres).  input.py:183-232.
    make_outputs=False (ranks of a sharded run: the output directory and the three files
    belong to rank 0) only reads the inputs.  native_table: `genepres` is a feeder.PanarooTable
    (same columns / index / rows, read by the library) instead of a DataFrame."""
    if native_table:        # the library's reader (feeder.PanarooTable): no Python object per cell
        from .feeder import PanarooTable
        genepres = PanarooTable(presence_absence)
    else:
        genepres = pd.read_csv(presence_absence, sep=",", index_col=0, low_memory=False).drop(
            columns=["Non-unique Gene name", "Annotation"])
    if stroi_in is not None:
        stroi = {line.rstrip("\n") for line in open(stroi_in)}
    else:
        logger.warning("No target strains provided")
        stroi = ""
    genes = None
    if genes_in is not None:
        genes = {line.rstrip("\n") for line in open(genes_in)}
    kmer_stroi = hash_pat = kmer_hash = None
    if not make_outputs:
        return stroi, genes, kmer_stroi, hash_pat, kmer_hash, genepres
    if os.path.exists(output):
        logger.error(f"Output directory {output} exists! Please remove it and restart")
        sys.exit(1)
    os.mkdir(output)
    if single_file:
        kmer_stroi = create_kmer_stroi(output, compress)
        hash_pat, kmer_hash = create_hash_files(output, compress)
    return stroi, genes, kmer_stroi, hash_pat, kmer_hash, genepres


def cut_window(feat, up, down, down_start_codon):
    """Contig slice [a, b) (python semantics), Seqinfo.start/end and the true
    upstream offset of one feature.  SURVEY.md App. A1.6-7, input.py:413-446."""
    over_up = feat.strand > 0 and feat.start - 1 - up < 0
    over_down = feat.strand < 0 and feat.start - 1 - down < 0
    offset = feat.start - 1 if over_up else up
    offset_d = feat.start - 1 if over_down else down
    if feat.strand > 0:
        a = feat.start - 1 - offset
        seq_start = feat.start - offset
        b = seq_end = (feat.start if down_start_codon else feat.end) + offset_d
    else:
        b = seq_end = feat.end + offset
        if down_start_codon:
            a = feat.end - 1 - offset_d
            seq_start = feat.end - offset_d
        else:
            a = feat.start - 1 - offset_d
            seq_start = feat.start - offset_d
    return a, b, seq_start, seq_end, offset


def iter_gene_clusters(panaroo, genome_data, up, down, down_start_codon, patfilt,
                       gene_list=None, raise_missing=False):
    """Yields (dict strain -> [Seqinfo], cluster id, int presence vector) per
    panaroo row, as input.py:335-468.  `patfilt` is accepted and unused, as in
    the reference."""
    missing = set(panaroo.columns).difference(genome_data.keys())
    if missing:
        raise KeyError(f"{len(missing)} strains of the pangenome table have no GFF "
                       f"(e.g. {sorted(missing)[0]}); the reference would emit misaligned "
                       "presence vectors here, this build refuses")
    n_rows = panaroo.shape[0]
    order = sorted(panaroo.columns)
    rank = {s: i for i, s in enumerate(order)}
    for i, (idx, row) in enumerate(panaroo.iterrows()):
        if gene_list is not None and idx not in gene_list:
            logger.debug(f"Skipping {idx} ({i + 1}/{n_rows})")
            continue
        logger.debug(f"Extracting sequences from {idx} ({i + 1}/{n_rows})")
        present = row.dropna()
        clusterpresab = np.zeros(len(row.index), dtype=int)
        for strain in present.index:
            clusterpresab[rank[strain]] = 1
        gene_sequences = {}
        for strain, cell in present.items():
            strain = str(strain)
            contigs, features = genome_data[strain]
            cuts = gene_sequences[strain] = []
            for gene in cell.split(";"):
                feat = features.get(gene)
                if feat is None:
                    logger.warning(f"Could not find gene {gene} from {idx} in {strain}")
                    if raise_missing:
                        raise KeyError(f"Could not find gene {gene} from {idx} in {strain}")
                    continue
                contig = contigs.get(feat.chromosome)
                if contig is None:
                    logger.warning(f"Could not find chromosome {feat.chromosome} in {strain}")
                    if raise_missing:
                        raise KeyError(f"Could not find chromosome {feat.chromosome} in {strain}")
                    continue
                a, b, seq_start, seq_end, offset = cut_window(feat, up, down, down_start_codon)
                piece = contig[a:b]
                if feat.strand < 0:
                    piece = piece.translate(_COMPLEMENT)[::-1]
                cuts.append(Seqinfo(piece, piece.translate(_COMPLEMENT), feat.id,
                                    feat.chromosome, seq_start, seq_end, feat.strand, offset))
        for strain in row.index.difference(present.index):
            gene_sequences[strain] = []
        yield gene_sequences, idx, clusterpresab
