#!/usr/bin/env python
"""Generate golden outputs by running the UNMODIFIED reference.

Runs `python -m panfeed` from /root/reference (read-only, never copied) with the
test-only pyfaidx stand-in on PYTHONPATH, once per argument combination of
`/root/reference/tests/unit_test.sh:18-52` plus a few extra modes, on the toy
pangenome written by make_fixture.py, and stores the three output files
gzip-compressed under tests/golden/expected/<mode>/.  Also writes
hot_kats.json: known answers obtained by calling the reference's
`cluster_cutter` / `pattern_hasher` directly (panfeed.py:23-235), and
cli_options.json: the reference's parsed command line with every default.

This only works in the build container (needs /root/reference).  The outputs
are committed; the GPU box and the tests read the committed files only.
"""
import gzip
import io
import json
import os
import shutil
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"
STANDIN = os.path.join(HERE, "pyfaidx_standin")

BASE = ["--gff", "fixture/gffs/", "--presence-absence",
        "fixture/gene_presence_absence.csv"]
T = ["--targets", "fixture/stroi.txt"]
MODES = {
    # the 12 combinations of unit_test.sh
    "basic": BASE + T,
    "cores": BASE + T + ["--cores", "4"],
    "nolog": BASE,
    "upstream": BASE + T + ["--upstream", "100", "--downstream", "0"],
    "downstream": BASE + T + ["--upstream", "0", "--downstream", "100"],
    "updownstream": BASE + T + ["--upstream", "100", "--downstream", "100"],
    "downstart": BASE + T + ["--upstream", "100", "--downstream", "100",
                             "--downstream-start-codon"],
    "noncanonical": BASE + T + ["--non-canonical"],
    "nofilter": BASE + T + ["--no-filter"],
    "highmaf": BASE + T + ["--maf", "0.1"],
    "considermissing": BASE + T + ["--consider-missing"],
    "fileoffiles": ["--gff", "fixture/input_gffs.txt", "--fasta",
                    "fixture/input_fastas.txt", "--presence-absence",
                    "fixture/gene_presence_absence.csv"] + T,
    # extras named by BASELINE.json north_star
    "secondpass": BASE + T + ["--genes", "fixture/genes.txt", "--upstream",
                              "100", "--downstream", "100"],
    "k15": BASE + T + ["-k", "15", "--upstream", "30", "--downstream", "30"],
    "k32": BASE + T + ["-k", "32"],
    # k > 32 (two-word k-mers here; the clusters without N/IUPAC symbols)
    "k40": BASE + T + ["-k", "40", "--upstream", "30", "--downstream", "30", "--genes", "fixture/genes_acgt.txt"],
    "k64_nc": BASE + T + ["-k", "64", "--non-canonical", "--upstream", "60", "--downstream", "60",
                          "--maf", "0.1", "--genes", "fixture/genes_acgt.txt"],
    "cm_nofilter_up": BASE + T + ["--consider-missing", "--no-filter",
                                  "--upstream", "100", "--downstream", "100",
                                  "--maf", "0.2"],
    "nc_updown": BASE + T + ["--non-canonical", "--upstream", "50",
                             "--downstream", "50"],
    "compress": BASE + T + ["--compress", "--genes", "fixture/genes.txt"],
}
FILES = ["kmers.tsv", "kmers_to_hashes.tsv", "hashes_to_patterns.tsv"]


def run_modes():
    env = dict(os.environ)
    env["PYTHONPATH"] = STANDIN + os.pathsep + REF
    exp = os.path.join(HERE, "expected")
    shutil.rmtree(exp, ignore_errors=True)
    os.makedirs(exp)
    with open(os.path.join(exp, "modes.json"), "w") as fh:
        json.dump(MODES, fh, indent=1, sort_keys=True)
    for mode, args in MODES.items():
        tmp = tempfile.mkdtemp(prefix="pfgold_")
        out = os.path.join(tmp, "out")
        r = subprocess.run([sys.executable, "-m", "panfeed"] + args +
                           ["--output", out], cwd=HERE, env=env,
                           capture_output=True, text=True)
        if r.returncode != 0:
            raise SystemExit(f"{mode} failed:\n{r.stderr[-2000:]}")
        os.makedirs(os.path.join(exp, mode))
        for f in FILES:
            src = os.path.join(out, f)
            if os.path.exists(src + ".gz"):
                data = gzip.open(src + ".gz", "rb").read()
            else:
                data = open(src, "rb").read()
            if mode == "cores":   # row order is nondeterministic (SURVEY §3.2)
                lines = data.split(b"\n")
                data = b"\n".join(sorted(lines))
            with gzip.GzipFile(os.path.join(exp, mode, f + ".gz"), "wb",
                               mtime=0) as fh:
                fh.write(data)
        shutil.rmtree(tmp)
        print(mode, "ok")


def hot_kats():
    """Known answers from the reference's hot functions called directly."""
    sys.path.insert(0, STANDIN)
    sys.path.insert(0, REF)
    import hashlib, binascii
    import numpy as np
    from panfeed.panfeed import cluster_cutter, pattern_hasher
    from panfeed.classes import Seqinfo
    import random

    kats = {"md5_ids": [], "maf_windows": [], "clusters": []}

    def pid(v):
        return binascii.b2a_base64(hashlib.md5(v.view(np.uint8)).digest()
                                   ).decode()[:24]
    for desc, v in [
        ("int64 all-ones S=12", np.ones(12, dtype=int)),
        ("float64 e0 S=12", np.eye(1, 12, 0, dtype=np.float64)[0]),
        ("float64 all-ones S=12", np.ones(12, dtype=np.float64)),
        ("float64 nan-mix S=12", np.array([1, np.nan, 0, np.nan, 0, 0, 0,
                                           np.nan, 0, 0, 0, 0], dtype=float)),
        ("int64 mix S=12", np.array([1, 0, 1, 0, 1, 1, 1, 0, 1, 1, 1, 1])),
    ]:
        kats["md5_ids"].append({"desc": desc, "dtype": str(v.dtype),
                                "values": [None if x != x else float(x)
                                           for x in v.tolist()],
                                "id": pid(v)})

    # MAF windows via the reference's float expression (panfeed.py:190-200)
    for n, maf in [(500, 0.01), (10000, 0.01), (50000, 0.01), (12, 0.01),
                   (500, 0.1), (8, 0.01), (8, 0.2), (7, 0.3), (3, 0.5),
                   (1, 0.01), (2, 0.0), (1000, 0.05), (333, 0.123)]:
        keep = []
        for c in range(n + 1):
            vec = np.zeros(n, dtype=np.float64)
            vec[:c] = 1
            af = vec.sum() / vec.shape[0]
            if af >= 0.5:
                af = 1 - af
            if not (af < maf):
                keep.append(c)
        kats["maf_windows"].append({"n": n, "maf": maf,
                                    "lo": keep[0] if keep else None,
                                    "hi": keep[-1] if keep else None,
                                    "contiguous": keep == list(range(
                                        keep[0], keep[-1] + 1)) if keep else True})

    # direct hot-function runs on hand-built Seqinfo clusters
    comp = str.maketrans("ACGTN", "TGCAN")
    rng = random.Random(7)
    for case, (S, L, k, canon, cm, patfilt, maf) in enumerate([
            (6, 60, 11, True, False, True, 0.01),
            (9, 80, 31, True, True, True, 0.2),
            (5, 50, 8, False, False, False, 0.01),   # even k: palindromes
            (40, 120, 31, True, False, False, 0.05),
            (33, 70, 32, True, True, False, 0.01),
    ]):
        names = [f"g{i:03d}" for i in range(S)]
        order = names[:]
        rng.shuffle(order)
        anc = "".join(rng.choice("ACGT") for _ in range(L))
        presab = np.zeros(S, dtype=int)
        cluster = {}
        seqs_json = {}
        absent = []
        for s in order:
            if rng.random() < 0.25:
                absent.append(s)
                continue
            presab[sorted(names).index(s)] = 1
            lst = []
            for _ in range(2 if rng.random() < 0.2 else 1):
                q = "".join(c if rng.random() > 0.03 else rng.choice("ACGT")
                            for c in anc)
                strand = rng.choice([1, -1])
                lst.append(Seqinfo(q, q.translate(comp), f"{s}_id", "ctg",
                                   101, 100 + L, strand, rng.choice([0, 7])))
            cluster[s] = lst
            seqs_json[s] = [list(x) for x in lst]
        for s in absent:
            cluster[s] = []
            seqs_json[s] = []
        stroi = set(order[:2])
        ret = cluster_cutter((cluster, f"case{case}", presab), k, stroi, False,
                             canon, cm, None)
        k2h, h2p, kst = io.StringIO(), io.StringIO(), io.StringIO()
        pats = pattern_hasher((ret,), kst, h2p, k2h, None, patfilt, maf, None,
                              patterns=set(), consider_missing_cluster=cm)
        kats["clusters"].append({
            "S": S, "k": k, "canon": canon, "consider_missing": cm,
            "patfilt": patfilt, "maf": maf, "idx": f"case{case}",
            "strain_order": list(cluster.keys()), "stroi": sorted(stroi),
            "clusterpresab": presab.tolist(), "seqs": seqs_json,
            "kmers_tsv": kst.getvalue(), "kmers_to_hashes": k2h.getvalue(),
            "hashes_to_patterns": h2p.getvalue(), "n_patterns": len(pats)})
    with open(os.path.join(HERE, "expected", "hot_kats.json"), "w") as fh:
        json.dump(kats, fh, indent=0)
    print("hot_kats ok")


def cli_options():
    """The reference's parsed command line (vars(get_options()), __main__.py:84-223) for the
    two required options only: every destination with its default."""
    argv = ["-g", "x", "-p", "y"]
    code = ("import sys, json; sys.argv = ['panfeed'] + json.loads(sys.argv[1]); "
            "from panfeed.__main__ import get_options; print(json.dumps(vars(get_options())))")
    env = dict(os.environ, PYTHONPATH=STANDIN + os.pathsep + REF)
    r = subprocess.run([sys.executable, "-c", code, json.dumps(argv)], env=env,
                       capture_output=True, text=True, check=True)
    options = json.loads(r.stdout.strip().splitlines()[-1])
    doc = {"argv": argv,
           "source": "vars(get_options()) of the unmodified reference's panfeed/__main__.py "
                     "for `panfeed -g x -p y`",
           "options": dict(sorted(options.items()))}
    with open(os.path.join(HERE, "expected", "cli_options.json"), "w") as fh:
        json.dump(doc, fh, indent=1)
        fh.write("\n")
    print("cli_options ok")


if __name__ == "__main__":
    if not os.path.isdir(os.path.join(HERE, "fixture")):
        sys.path.insert(0, HERE)
        import make_fixture
        make_fixture.build(os.path.join(HERE, "fixture"))
    run_modes()
    hot_kats()
    cli_options()
