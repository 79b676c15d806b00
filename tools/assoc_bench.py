"""Second pass with the post-GWAS annotation: (a) `python -m panfeed_b200` writing kmers.tsv, then
`panfeed-get-kmers` (postgwas.get_kmers_main) on its files, against (b) the same second pass with
--associations, on a synthetic pangenome (the generator of tools/cli_bench.py) in which every
genome is a target.  The associations table names every pattern of the run; ~5 % pass.
Prints both wall times, the bytes each path wrote and whether the two tables hold the same lines.
usage: python tools/assoc_bench.py [genomes] [clusters] [gene_len] [--no-host]   (config #3: 500 200 1000)
--no-host: skip get-kmers (a pandas join whose time grows faster than the number of rows: at config #3's
1.2e8 rows it does not finish in a practical time) and the comparison."""
import contextlib
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, ".")
HOST = "--no-host" not in sys.argv
argv = [a for a in sys.argv[1:] if a != "--no-host"]
G = int(argv[0]) if len(argv) > 0 else 500
N = int(argv[1]) if len(argv) > 1 else 200
L = int(argv[2]) if len(argv) > 2 else 1000
rng = np.random.default_rng(1)
tmp = tempfile.mkdtemp(prefix="pf_assoc_bench_")
gffdir = os.path.join(tmp, "gffs")
os.mkdir(gffdir)
anc = rng.integers(0, 4, (N, L))
founders = [np.where(rng.random((N, L)) < 0.01, (anc + rng.integers(1, 4, (N, L))) & 3, anc) for _ in range(8)]
lut = np.frombuffer(b"ACGT", np.uint8)
names = [f"s{g:04d}" for g in range(G)]
cols = {}
for name in names:
    rows, parts, col, pos = [], [], [], 1
    for c in range(N):
        if rng.random() < 0.1:
            col.append("")
            continue
        q = founders[int(rng.integers(8))][c].copy()
        m = rng.random(L) < 0.001
        q[m] = (q[m] + rng.integers(1, 4, int(m.sum()))) & 3
        strand = "+" if rng.random() < 0.5 else "-"
        rows.append(f"{name}_c1\tsynth\tCDS\t{pos + 150}\t{pos + 149 + L}\t.\t{strand}\t0\tID={name}_{c:05d};x=1")
        parts.append(lut[rng.integers(0, 4, 150)].tobytes().decode() + lut[q].tobytes().decode())
        pos += 150 + L
        col.append(f"{name}_{c:05d}")
    cols[name] = col
    text = "".join(parts)
    with open(os.path.join(gffdir, name + ".gff"), "w") as fh:
        fh.write("##gff-version 3\n" + "\n".join(rows) + "\n##FASTA\n>" + name + "_c1\n")
        fh.write("\n".join(text[i:i + 60] for i in range(0, len(text), 60)) + "\n")
csv = os.path.join(tmp, "gpa.csv")
with open(csv, "w") as fh:
    fh.write("Gene,Non-unique Gene name,Annotation," + ",".join(names) + "\n")
    for c in range(N):
        fh.write(f"cl{c},,x," + ",".join(cols[n][c] for n in names) + "\n")
targets = os.path.join(tmp, "targets.txt")
open(targets, "w").write("\n".join(names) + "\n")
base = ["-g", gffdir, "-p", csv, "--targets", targets, "--upstream", "100", "--downstream", "100"]
print(f"pangenome: {G} genomes x {N} clusters of {L} bp, every genome a target")

from panfeed_b200 import postgwas  # noqa: E402
from panfeed_b200.__main__ import main  # noqa: E402


def size(d):
    return sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d) if os.path.isfile(os.path.join(d, f)))


# warm-up (CUDA context, module load) on a few clusters, not timed
open(os.path.join(tmp, "genes.txt"), "w").write("cl0\n")
main(base + ["--genes", os.path.join(tmp, "genes.txt"), "-o", os.path.join(tmp, "warm")])

# (a) second pass, then get-kmers on its files
out_a = os.path.join(tmp, "a")
t0 = time.perf_counter()
main(base + ["-o", out_a])
t1 = time.perf_counter()
print(f"(a) second pass: {t1 - t0:.2f} s", flush=True)
ids = np.loadtxt(os.path.join(out_a, "hashes_to_patterns.tsv"), dtype=str, usecols=0, skiprows=1, comments=None)
pv = np.where(rng.random(len(ids)) < 0.05, rng.random(len(ids)) * 0.05, 0.05 + rng.random(len(ids)) * 0.95)
assoc = os.path.join(tmp, "assoc.tsv")
with open(assoc, "w") as fh:
    fh.write("variant\taf\tfilter-pvalue\tlrt-pvalue\tbeta\n")
    fh.write("".join(f"{h}\t{a:.3f}\t{p:.4g}\t{p:.4g}\t{b:.5f}\n"
                     for h, a, p, b in zip(ids, rng.random(len(ids)), pv, rng.normal(size=len(ids)))))
table_a = os.path.join(tmp, "annotated_a.tsv")
t2 = t3 = time.perf_counter()
if HOST:
    with open(table_a, "w") as fh, contextlib.redirect_stdout(fh):
        postgwas.get_kmers_main(["-a", assoc, "-p", os.path.join(out_a, "kmers_to_hashes.tsv"),
                                 "-k", os.path.join(out_a, "kmers.tsv"), "-t", "0.05"])
    t3 = time.perf_counter()
    print(f"(a) get-kmers: {t3 - t2:.2f} s", flush=True)
bytes_a = size(out_a) + (os.path.getsize(table_a) if HOST else 0)

# (b) the second pass with --associations
out_b = os.path.join(tmp, "b")
t4 = time.perf_counter()
main(base + ["-o", out_b, "--associations", assoc, "--association-threshold", "0.05"])
t5 = time.perf_counter()
bytes_b = size(out_b)
table_b = os.path.join(out_b, "annotated_kmers.tsv")

lines = sum(1 for _ in open(table_b)) - 1
print(f"passing patterns: {(pv <= 0.05).sum()} of {len(ids)}; annotated lines: {lines}")
kmers_mb = os.path.getsize(os.path.join(out_a, 'kmers.tsv')) / 1e6
if HOST:
    same = subprocess.run(f"cmp <(LC_ALL=C sort {table_a}) <(LC_ALL=C sort {table_b})", shell=True,
                          executable="/bin/bash").returncode == 0
    print(f"(a) second pass {t1 - t0:.2f} s + get-kmers {t3 - t2:.2f} s = {t1 - t0 + t3 - t2:.2f} s wall, "
          f"{bytes_a / 1e6:.0f} MB written (kmers.tsv {kmers_mb:.0f} MB)")
else:
    print(f"(a) second pass {t1 - t0:.2f} s wall, {bytes_a / 1e6:.0f} MB written (kmers.tsv {kmers_mb:.0f} MB); "
          f"get-kmers not run")
print(f"(b) second pass with --associations {t5 - t4:.2f} s wall, {bytes_b / 1e6:.0f} MB written")
if HOST:
    print(f"same lines: {same}")
shutil.rmtree(tmp)
