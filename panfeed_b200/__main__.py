"""`panfeed` command line of the B200 build: the reference's options
(`/root/reference/panfeed/__main__.py:84-223`) and wiring (`:226-369`), with the
two hot callables running on the GPU.  `--cores` and `-ql` are accepted for
compatibility; clusters are batched to the device instead of forked workers, so
row order is deterministic and `--compress` output is always valid gzip.

Several GPUs: `torchrun --nproc-per-node N -m panfeed_b200 <same options>` (one process per
GPU).  The reference's parallel mode is a reader, N-2 `cluster_cutter` workers and ONE writer
that owns the `patterns` set (`__main__.py:299-344`, `:70`); here whole clusters are sharded
over the ranks (greedy by number of genes), every rank writes header-less pieces of
kmers.tsv / kmers_to_hashes for its clusters, one exchange (dist.PatternExchange, the library's
pf_exchange_run over NCCL) decides
which rank writes each pattern's hashes_to_patterns row, and rank 0 joins the pieces into the
same three files a single process writes.  With --associations every rank writes a piece of
annotated_kmers.tsv instead of kmers.tsv (assoc.AnnotatedWriter: the ranks OR their upcast facts
once, just before the exchange)."""
import argparse
import logging
import os
import sys
from functools import partial

import numpy as np

from . import __version__
from .input import (KMERS_TSV_HEADER, OUTPUT_NAMES, clean_up_fasta, create_part_files, iter_gene_clusters,
                    merge_part_files, prep_data_n_fasta, set_input_output, what_are_my_inputfiles)
from .panfeed import PatternStore, cluster_cutter, pattern_hasher, write_headers

logger = logging.getLogger("panfeed")


def set_logging(v):
    logger.propagate = True
    logger.setLevel(logging.DEBUG)
    ch = logging.StreamHandler()
    ch.setLevel(logging.DEBUG if v >= 1 else logging.INFO)
    ch.setFormatter(logging.Formatter("%(asctime)s - %(name)s - %(message)s", "%H:%M:%S"))
    logger.addHandler(ch)


def get_options(argv=None):
    p = argparse.ArgumentParser(
        prog="panfeed",
        description="Get gene cluster specific k-mers from a set of bacterial genomes "
                    "(B200-native build)")
    p.add_argument("-g", "--gff", required=True,
                   help="Directory with all samples' GFF files, or a file listing them")
    p.add_argument("-p", "--presence-absence", required=True,
                   help="Gene clusters presence absence table as output by panaroo")
    p.add_argument("--targets", default=None,
                   help="File with the samples whose k-mer positions are logged")
    p.add_argument("--genes", default=None,
                   help="File with the gene clusters to process (default: all)")
    p.add_argument("-o", "--output", default="panfeed",
                   help="Output directory (must not exist)")
    p.add_argument("-f", "--fasta", help="Directory or file of files with nucleotide fastas")
    p.add_argument("-k", "--kmer-length", type=int, default=31,
                   help="K-mer length, 1..64 (a k-mer is packed into one or two 64-bit words; the "
                        "reference accepts longer k-mers, this build exits with an error).  33..64 run on "
                        "the 128-bit record engine, several times slower than 1..32; their k-mers holding "
                        "N/IUPAC symbols take 256-bit records")
    p.add_argument("--maf", type=float, default=0.01, help="Minor allele frequency threshold")
    p.add_argument("--upstream", type=int, default=0)
    p.add_argument("--downstream", type=int, default=0)
    p.add_argument("--downstream-start-codon", action="store_true", default=False)
    p.add_argument("--non-canonical", action="store_true", default=False)
    p.add_argument("--no-filter", action="store_true", default=False)
    p.add_argument("--consider-missing", action="store_true", default=False)
    p.add_argument("--multiple-files", action="store_true", default=False)
    p.add_argument("--compress", action="store_true", default=False)
    p.add_argument("--python-feeder", action="store_true", default=False,
                   help="parse GFF/FASTA and cut the cluster sequences with the Python loops that mirror the "
                        "reference's input.py instead of the library's native feeder (pf_feeder_*, the "
                        "default: same outputs, an order of magnitude faster)")
    p.add_argument("--native-feeder", action="store_true", default=False,
                   help="accepted for compatibility: the native feeder is the default")
    p.add_argument("--cores", type=int, default=1, help="accepted for compatibility (GPU build)")
    p.add_argument("-ql", "--queue-limit", type=int, default=3,
                   help="accepted for compatibility (GPU build)")
    p.add_argument("--stop-on-missing", action="store_true", default=False)
    # (the association options exist in the parsed namespace only when given: without them a run is
    #  the reference's, option for option)
    assoc = p.add_argument_group("post-GWAS annotation (panfeed-get-kmers in the same run)")
    assoc.add_argument("--associations", default=argparse.SUPPRESS,
                       help="pyseer-style associations table (tab-separated, a header, the pattern id in the first "
                            "column): write <output>/annotated_kmers.tsv, the table panfeed-get-kmers would print "
                            "for this run's kmers_to_hashes.tsv and kmers.tsv, instead of kmers.tsv.  The join runs "
                            "on the GPU (under torchrun every rank joins its own clusters and rank 0 writes the one "
                            "file); kmers_to_hashes.tsv and hashes_to_patterns.tsv are written as usual.  Not with "
                            "--multiple-files")
    assoc.add_argument("--association-threshold", type=float, default=argparse.SUPPRESS,
                       help="p-value threshold (get-kmers -t, default 1)")
    assoc.add_argument("--association-column", default=argparse.SUPPRESS,
                       help="p-value column (get-kmers -c, default lrt-pvalue)")
    assoc.add_argument("--only-passing", action="store_true", default=argparse.SUPPRESS,
                       help="only the passing k-mers (get-kmers --only-passing)")
    p.add_argument("--device", type=int, default=0, help="CUDA device")
    p.add_argument("-v", action="count", default=0)
    p.add_argument("--version", action="version", version="%(prog)s " + __version__)
    return p.parse_args(argv)


def main(argv=None):
    args = get_options(argv)
    for name, default in (("associations", None), ("association_threshold", 1.0),
                          ("association_column", "lrt-pvalue"), ("only_passing", False)):
        if not hasattr(args, name):
            setattr(args, name, default)
    set_logging(args.v)
    klength = args.kmer_length
    if args.downstream_start_codon and args.upstream + args.downstream < klength:
        logger.warning("Query sequence is shorter than k-mer length"
                       "Decrease k-mer size or increase query sequence length")
        sys.exit(1)
    if args.maf > 0.5:
        logger.warning("--maf should be below 0.5")
        sys.exit(1)
    if klength < 1 or klength > 64:
        logger.error("this build supports k-mer lengths 1..64 (2 bits per base in one or two 64-bit words)")
        sys.exit(1)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    sharded = world > 1
    if args.associations is not None and args.multiple_files:
        logger.error("--associations writes one file: it cannot be combined with --multiple-files")
        sys.exit(1)
    if sharded:
        import torch
        import torch.distributed as tdist
        args.device = int(os.environ.get("LOCAL_RANK", "0"))
        os.environ.setdefault("PF_HOST_THREADS", str(max(2, (os.cpu_count() or 16) // world)))
        if os.environ.get("PF_DIST_BACKEND", "nccl") == "nccl":
            torch.cuda.set_device(args.device)
            tdist.init_process_group("nccl", device_id=torch.device("cuda", args.device))
        else:       # the CPU tests of the sharded wiring rendezvous over gloo (the GPU context is a stand-in there)
            tdist.init_process_group(os.environ["PF_DIST_BACKEND"])
        if os.path.exists(args.output):          # every rank sees the same answer: no rank is left waiting
            logger.error(f"Output directory {args.output} exists! Please remove it and restart")
            tdist.barrier()
            sys.exit(1)
        tdist.barrier()

    logger.info("Looking at input GFF files")
    filelist, fastalist = what_are_my_inputfiles(args.gff, args.fasta)
    logger.info(f"Found {len(filelist)} input genomes")
    logger.info("Preparing output files")
    (stroi, genes, kmer_stroi, hash_pat, kmer_hash, genepres) = set_input_output(
        args.targets, args.genes, args.presence_absence, args.output,
        not args.multiple_files, args.compress, make_outputs=not sharded,
        native_table=not args.python_feeder)
    all_columns = genepres
    annotate = None
    if args.associations is not None:
        from .assoc import AnnotatedWriter, load_passing
        a, digests = load_passing(args.associations, args.association_column, args.association_threshold)
        logger.info(f"{len(a)} patterns pass the association threshold {args.association_threshold}")
        if not sharded:
            # annotated_kmers.tsv takes the place of kmers.tsv
            kmer_stroi.close()
            os.remove(os.path.join(args.output, "kmers.tsv.gz" if args.compress else "kmers.tsv"))
            kmer_stroi = None
            annotate = AnnotatedWriter(args.output, a, digests, args.only_passing, args.compress)
    if sharded:
        if rank == 0:
            os.mkdir(args.output)
        tdist.barrier()
        if args.associations is not None:          # a piece of annotated_kmers.tsv in place of kmers.tsv's
            hash_pat, kmer_hash = create_part_files(args.output, rank, args.compress, OUTPUT_NAMES[1:])
            annotate = AnnotatedWriter(args.output, a, digests, args.only_passing, args.compress, rank=rank)
        elif not args.multiple_files:
            kmer_stroi, hash_pat, kmer_hash = create_part_files(args.output, rank, args.compress)
        # whole clusters to ranks, greedy by the number of genes (cells) of the rows that will be cut
        from .dist import shard_clusters
        native_table = hasattr(genepres, "n_present")
        weights = genepres.n_present() if native_table else genepres.notna().sum(axis=1).to_numpy()
        if genes is not None:
            weights = weights * np.isin(np.array(list(genepres.index), dtype=object), list(genes))
        mine = shard_clusters(weights, world)[rank]
        genepres = genepres.take(mine) if native_table else genepres.iloc[mine]
        logger.info(f"rank {rank}/{world}: {len(mine)} of {len(weights)} clusters")
    logger.info("Preparing inputs")
    if not args.multiple_files and not sharded:
        write_headers(hash_pat, kmer_hash, genepres)
    logger.info("Extracting k-mers")
    if not args.python_feeder:
        from .feeder import iter_packed_batches, iter_packed_clusters, prefetch, prep_feeder
        native, genome_index = prep_feeder(filelist, fastalist, args.gff, args.fasta, args.output)
        # whole GPU batches straight from the library; --multiple-files runs cluster by cluster
        cut = iter_packed_clusters if args.multiple_files else iter_packed_batches
        cut_clusters = cut(genepres, native, genome_index, args.upstream, args.downstream,
                           args.downstream_start_codon, stroi, klength, not args.non_canonical,
                           args.consider_missing, genes, args.stop_on_missing)
        if not args.multiple_files:
            cut_clusters = prefetch(cut_clusters)      # the next batch is cut while this one runs
    else:
        data = prep_data_n_fasta(filelist, fastalist, args.gff, args.fasta, args.output)
        iter_i = iter_gene_clusters(genepres, data, args.upstream, args.downstream,
                                    args.downstream_start_codon, not args.no_filter, genes,
                                    args.stop_on_missing)
        iter_o = partial(cluster_cutter, klength=klength, stroi=stroi,
                         multiple_files=args.multiple_files, canon=not args.non_canonical,
                         consider_missing_cluster=args.consider_missing, output=args.output,
                         compress=args.compress)
        cut_clusters = (iter_o(x) for x in iter_i)
    patterns = PatternStore(sharded=sharded and not args.multiple_files)
    func_w = partial(pattern_hasher, kmer_stroi=kmer_stroi, hash_pat=hash_pat,
                     kmer_hash=kmer_hash, genepres=all_columns, patfilt=not args.no_filter,
                     maf=args.maf, consider_missing_cluster=args.consider_missing,
                     output=args.output, compress=args.compress, device=args.device, annotate=annotate)
    # one streaming call: the generator packs clusters while the GPU batches them
    patterns = func_w(cut_clusters, patterns=patterns)
    if annotate is not None:
        # the upcast facts over every rank (one process: its own).  Sharded, a collective: every rank
        # calls it exactly once, here, after its last batch and before the pattern exchange,
        # whether it had clusters or not
        any_rank = bool
        if sharded:
            from .dist import any_rank as or_over_ranks
            dev = torch.device("cuda", args.device) if tdist.get_backend() == "nccl" else torch.device("cpu")
            any_rank = partial(or_over_ranks, device=dev)
        annotate.finish(any_rank)
    if patterns.sharded:
        info = patterns.finish_sharded(hash_pat, klength, len(all_columns.columns), not args.non_canonical,
                                       args.consider_missing, args.no_filter, args.maf, args.device)
        logger.info(f"rank {rank}: wrote {info['written_here']} of {info['cluster_patterns_global']} + "
                    f"{info['kmer_patterns_global']} patterns")
    patterns.close()

    for handle in (kmer_stroi, hash_pat, kmer_hash):
        if handle is not None:
            handle.close()
    if sharded:
        tdist.barrier()
        if rank == 0 and not args.multiple_files:
            import io
            import time
            hp, kh = io.StringIO(), io.StringIO()
            write_headers(hp, kh, all_columns)
            first = (KMERS_TSV_HEADER, OUTPUT_NAMES[0]) if annotate is None else (annotate.header, annotate.NAME)
            t0 = time.perf_counter()
            merge_part_files(args.output, world, (first[0], hp.getvalue(), kh.getvalue()), args.compress,
                             (first[1],) + OUTPUT_NAMES[1:])
            logger.info(f"rank 0: merged the pieces of {world} ranks in {time.perf_counter() - t0:.2f} s")
        tdist.barrier()
        tdist.destroy_process_group()
    logger.info("Removing temporary fasta files and faidx indices")
    clean_up_fasta(filelist, fastalist, args.output, args.fasta)


if __name__ == "__main__":
    main()
