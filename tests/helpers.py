"""Shared helpers for the parity tests."""
import argparse
import gzip
import json
import os

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")
EXPECTED = os.path.join(GOLDEN, "expected")
FILES = ["kmers.tsv", "kmers_to_hashes.tsv", "hashes_to_patterns.tsv"]


def modes():
    with open(os.path.join(EXPECTED, "modes.json")) as fh:
        return json.load(fh)


def golden(mode, name):
    return gzip.open(os.path.join(EXPECTED, mode, name + ".gz"),
                     "rt").read()


def hot_kats():
    with open(os.path.join(EXPECTED, "hot_kats.json")) as fh:
        return json.load(fh)


def cli_options():
    """The reference's parsed command line for a minimal argument list: {"argv", "options"}."""
    with open(os.path.join(EXPECTED, "cli_options.json")) as fh:
        return json.load(fh)


def cli_kwargs(args):
    """Translate a reference-style argument list into keyword arguments
    (options of /root/reference/panfeed/__main__.py:84-223)."""
    p = argparse.ArgumentParser()
    p.add_argument("-g", "--gff")
    p.add_argument("-p", "--presence-absence")
    p.add_argument("--targets")
    p.add_argument("--genes")
    p.add_argument("-f", "--fasta")
    p.add_argument("-k", "--kmer-length", type=int, default=31)
    p.add_argument("--maf", type=float, default=0.01)
    p.add_argument("--upstream", type=int, default=0)
    p.add_argument("--downstream", type=int, default=0)
    p.add_argument("--downstream-start-codon", action="store_true")
    p.add_argument("--non-canonical", action="store_true")
    p.add_argument("--no-filter", action="store_true")
    p.add_argument("--consider-missing", action="store_true")
    p.add_argument("--compress", action="store_true")
    p.add_argument("--cores", type=int, default=1)
    a = p.parse_args(args)

    def path(x):
        return None if x is None else os.path.join(GOLDEN, x)
    return dict(gff=path(a.gff), presence_absence=path(a.presence_absence),
                targets=path(a.targets), genes=path(a.genes),
                fasta=path(a.fasta), k=a.kmer_length, maf=a.maf,
                upstream=a.upstream, downstream=a.downstream,
                downstream_start_codon=a.downstream_start_codon,
                non_canonical=a.non_canonical, no_filter=a.no_filter,
                consider_missing=a.consider_missing)


def sorted_lines(text):
    return sorted(text.split("\n"))
