"""Second pass with the post-GWAS annotation: (a) `python -m panfeed_b200` writing kmers.tsv, then
`panfeed-get-kmers` (postgwas.get_kmers_main) on its files, against (b) the same second pass with
--associations, on a synthetic pangenome (the generator of tools/cli_bench.py) in which every
genome is a target.  The associations table names every pattern of the run; ~5 % pass.
Prints both wall times, the bytes each path wrote and whether the two tables hold the same lines.
usage: python tools/assoc_bench.py [genomes] [clusters] [gene_len] [--no-host] [--ranks=1,2,4,8]
(config #3: 500 200 1000)
--no-host: skip get-kmers (a pandas join whose time grows faster than the number of rows: at config #3's
1.2e8 rows it does not finish in a practical time) and the comparison.
--ranks=N,...: instead of (a) and (b), (c): the second pass with --associations as a fresh
`python -m panfeed_b200` (1) or `torchrun --nproc-per-node N -m panfeed_b200` (one GPU per rank) for
each N.  Prints each launch's wall time (process start-up included), the bytes it wrote, the time of
rank 0's merge of the pieces, and whether its table holds the lines of the one-process table.  Where
the box has fewer than N GPUs, only rank 0's merge is timed: the one-process table cut into N pieces
and merged by input.merge_part_files."""
import contextlib
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, ".")
RANKS = [int(x) for a in sys.argv[1:] if a.startswith("--ranks=") for x in a.split("=", 1)[1].split(",")]
HOST = "--no-host" not in sys.argv and not RANKS
argv = [a for a in sys.argv[1:] if not a.startswith("--")]
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


def write_assoc(h2p):
    """The associations table over every pattern of a run's hashes_to_patterns.tsv, ~5 % passing at 0.05."""
    ids = np.loadtxt(h2p, dtype=str, usecols=0, skiprows=1, comments=None)
    pv = np.where(rng.random(len(ids)) < 0.05, rng.random(len(ids)) * 0.05, 0.05 + rng.random(len(ids)) * 0.95)
    with open(assoc, "w") as fh:
        fh.write("variant\taf\tfilter-pvalue\tlrt-pvalue\tbeta\n")
        fh.write("".join(f"{h}\t{a:.3f}\t{p:.4g}\t{p:.4g}\t{b:.5f}\n"
                         for h, a, p, b in zip(ids, rng.random(len(ids)), pv, rng.normal(size=len(ids)))))
    return ids, pv


assoc = os.path.join(tmp, "assoc.tsv")
ENV = dict(os.environ, PYTHONPATH=os.getcwd() + os.pathsep + os.environ.get("PYTHONPATH", ""))


def launch(n, out):
    """(c): one launch on n ranks -> (wall s, rank 0's merge s or None)."""
    cmd = [sys.executable, "-m", "panfeed_b200"]
    if n > 1:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n),
               "--master-addr", "127.0.0.1", "--master-port", str(29590 + n), "-m", "panfeed_b200"]
    t = time.perf_counter()
    r = subprocess.run(cmd + base + ["-o", out, "--associations", assoc, "--association-threshold", "0.05"],
                       capture_output=True, text=True, env=ENV)
    wall = time.perf_counter() - t
    if r.returncode != 0:
        sys.exit(r.stdout[-2000:] + r.stderr[-4000:])
    merge = [float(x.split(" in ")[-1].split()[0]) for x in r.stderr.splitlines() if "merged the pieces" in x]
    return wall, (merge[0] if merge else None)


def sorted_md5(path):
    """md5 of the table's lines after sorting (GNU sort, all cores, in memory where it fits)."""
    r = subprocess.run(f"LC_ALL=C sort -S 40% --parallel={os.cpu_count()} -T {tmp} {path} | md5sum",
                       shell=True, capture_output=True, text=True, check=True)
    return r.stdout.split()[0]


if RANKS:
    # every launch is a fresh process and this one never touches the GPU, so each rank has its device
    # to itself.  The pattern ids come from a first pass without --targets: the same patterns as the
    # second pass, without writing its kmers.tsv
    from panfeed_b200.input import merge_part_files, part_path
    first = base[:4] + base[6:]
    subprocess.run([sys.executable, "-m", "panfeed_b200"] + first + ["-o", os.path.join(tmp, "ids")],
                   check=True, capture_output=True, env=ENV)
    ids, pv = write_assoc(os.path.join(tmp, "ids", "hashes_to_patterns.tsv"))
    n_gpus = len(subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True).stdout.splitlines())
    print(f"passing patterns: {(pv <= 0.05).sum()} of {len(ids)}; {n_gpus} GPU(s)", flush=True)
    ref = None
    for n in RANKS:
        if n > n_gpus:
            print(f"(c) {n} ranks: not run, {n_gpus} GPU(s)", end="")
            if ref is None:
                print()
                continue
            # rank 0's merge alone: the 1-rank table cut into n pieces at line boundaries, then merged
            table, d = os.path.join(tmp, f"c{ref[0]}", "annotated_kmers.tsv"), os.path.join(tmp, f"m{n}")
            os.makedirs(os.path.join(d, ".parts"))
            with open(table, "rb") as src:
                header = src.readline().decode()
                per = (os.path.getsize(table) - len(header)) // n + 1
                for r in range(n):
                    with open(part_path(d, "annotated_kmers.tsv", r), "wb") as piece:
                        left = per if r < n - 1 else os.path.getsize(table)
                        while left > 0 and (chunk := src.read(min(left, 64 << 20))):
                            piece.write(chunk)
                            left -= len(chunk)
                        piece.write(src.readline())
            t = time.perf_counter()
            merge_part_files(d, n, (header,), names=("annotated_kmers.tsv",))
            merged = os.path.join(d, "annotated_kmers.tsv")
            print(f"; rank 0's merge alone of {n} pieces of the 1-rank table: {time.perf_counter() - t:.2f} s "
                  f"({os.path.getsize(merged) / 1e6:.0f} MB, same bytes: "
                  f"{subprocess.run(['cmp', '-s', merged, table]).returncode == 0})", flush=True)
            shutil.rmtree(d)
            continue
        out_c = os.path.join(tmp, f"c{n}")
        wall, merge = launch(n, out_c)
        table = os.path.join(out_c, "annotated_kmers.tsv")
        lines = sum(1 for _ in open(table, "rb")) - 1
        digest = sorted_md5(table)
        ref = ref or (n, digest)
        merged = f", rank 0's merge {merge:.2f} s" if merge is not None else ""
        print(f"(c) {n} rank(s): {wall:.2f} s wall{merged}, {size(out_c) / 1e6:.0f} MB written, {lines} annotated "
              f"lines, same sorted lines as {ref[0]} rank(s): {digest == ref[1]}", flush=True)
        if n != ref[0]:
            shutil.rmtree(out_c)
    shutil.rmtree(tmp)
    sys.exit(0)

# warm-up (CUDA context, module load) on a few clusters, not timed
open(os.path.join(tmp, "genes.txt"), "w").write("cl0\n")
main(base + ["--genes", os.path.join(tmp, "genes.txt"), "-o", os.path.join(tmp, "warm")])

# (a) second pass, then get-kmers on its files
out_a = os.path.join(tmp, "a")
t0 = time.perf_counter()
main(base + ["-o", out_a])
t1 = time.perf_counter()
print(f"(a) second pass: {t1 - t0:.2f} s", flush=True)
ids, pv = write_assoc(os.path.join(out_a, "hashes_to_patterns.tsv"))
table_a = os.path.join(tmp, "annotated_a.tsv")
t2 = t3 = time.perf_counter()
if HOST:
    with open(table_a, "w") as fh, contextlib.redirect_stdout(fh):
        postgwas.get_kmers_main(["-a", assoc, "-p", os.path.join(out_a, "kmers_to_hashes.tsv"),
                                 "-k", os.path.join(out_a, "kmers.tsv"), "-t", "0.05"])
    t3 = time.perf_counter()
    print(f"(a) get-kmers: {t3 - t2:.2f} s", flush=True)
bytes_a = size(out_a) + (os.path.getsize(table_a) if HOST else 0)
kmers_mb = os.path.getsize(os.path.join(out_a, 'kmers.tsv')) / 1e6


# (b) the second pass with --associations
out_b = os.path.join(tmp, "b")
t4 = time.perf_counter()
main(base + ["-o", out_b, "--associations", assoc, "--association-threshold", "0.05"])
t5 = time.perf_counter()
bytes_b = size(out_b)
table_b = os.path.join(out_b, "annotated_kmers.tsv")

lines = sum(1 for _ in open(table_b)) - 1
print(f"passing patterns: {(pv <= 0.05).sum()} of {len(ids)}; annotated lines: {lines}")
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
