"""--associations: the second pass writes panfeed-get-kmers' table itself, the join on the device.
Against the unmodified get_kmers.py's stdout on the fixture (tests/golden/expected/postgwas), and
against the host path - the same run without --associations followed by postgwas.get_kmers_main on
its files - for other k-mer lengths, option sets and association tables, N/IUPAC windows included."""
import contextlib
import gzip
import io
import os

import numpy as np
import pytest

import helpers
from panfeed_b200 import postgwas
from panfeed_b200.panfeed import pattern_id

pytestmark = pytest.mark.gpu

POST = os.path.join(helpers.EXPECTED, "postgwas")
ASSOC = os.path.join(POST, "associations.tsv")
UPDOWN = helpers.modes()["updownstream"]
WHOLE = ["--gff", "fixture/gffs/", "--presence-absence", "fixture/gene_presence_absence.csv",
         "--targets", "fixture/stroi.txt", "--upstream", "100", "--downstream", "100"]


def _read(path):
    if os.path.exists(path + ".gz"):
        return gzip.open(path + ".gz", "rt").read()
    return open(path).read()


def _cli(args, out):
    from panfeed_b200.__main__ import main
    cwd = os.getcwd()
    os.chdir(helpers.GOLDEN)
    try:
        main(args + ["--output", str(out)])
    finally:
        os.chdir(cwd)


def _lines(text):
    return sorted(x for x in text.split("\n") if x)


def _host_join(out, assoc, extra):
    """postgwas.get_kmers_main on a run's own kmers_to_hashes.tsv / kmers.tsv."""
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        postgwas.get_kmers_main(["-a", str(assoc), "-p", os.path.join(out, "kmers_to_hashes.tsv"),
                                 "-k", os.path.join(out, "kmers.tsv"), "--clusters-per-iteration", "100000"] + extra)
    return buf.getvalue()


@pytest.mark.parametrize("variant", ["native", "compress", "python-feeder"])
@pytest.mark.parametrize("case, extra", [("kmers_t0.3", ["--association-threshold", "0.3"]),
                                         ("kmers_t0.3_passing", ["--association-threshold", "0.3", "--only-passing"]),
                                         ("kmers_t0.1_iter2", ["--association-threshold", "0.1"])])
def test_matches_reference_get_kmers(case, extra, variant, tmp_path):
    args = UPDOWN + ["--associations", ASSOC] + extra
    if variant == "compress":
        args.append("--compress")
    if variant == "python-feeder":
        args.append("--python-feeder")
    _cli(args, tmp_path / "out")
    got = _read(str(tmp_path / "out" / "annotated_kmers.tsv"))
    want = gzip.open(os.path.join(POST, case + ".txt.gz"), "rt").read()
    assert got.split("\n")[0] == want.split("\n")[0]
    assert _lines(got) == _lines(want)
    assert not os.path.exists(tmp_path / "out" / "kmers.tsv")
    assert os.path.exists(str(tmp_path / "out" / "kmers_to_hashes.tsv") + (".gz" if variant == "compress" else ""))
    if variant == "compress":
        assert os.path.exists(tmp_path / "out" / "annotated_kmers.tsv.gz")
    if "--only-passing" in extra:       # the float-formatted positions and the cluster-row line
        assert "\t1.0\t361.0\t392.0\t" in got
        assert any(x.startswith("group_core\t\t") for x in got.split("\n"))


def _random_assoc(out, path, rng, frac, int_column=False, extra_ids=()):
    """An associations table over the run's own hashes: a random `frac` passes at 0.5."""
    ids = [x.split("\t")[0] for x in _read(os.path.join(out, "hashes_to_patterns.tsv")).split("\n")[1:] if x]
    p = np.where(rng.random(len(ids)) < frac, rng.random(len(ids)) * 0.5, 0.6 + rng.random(len(ids)) * 0.4)
    rows = ["variant\taf\tlrt-pvalue\tbeta" + ("\tcount" if int_column else "")]
    for i, (h, v) in enumerate(zip(ids, p)):
        rows.append(f"{h}\t{rng.random():.3f}\t{v:.4f}\t{rng.normal():.5f}" + (f"\t{i}" if int_column else ""))
    for h in extra_ids:
        rows.append(f"{h}\t0.5\t0.01\t1.0" + ("\t7" if int_column else ""))
    path.write_text("\n".join(rows) + "\n")


CASES = {
    "k31": ["-k", "31"],
    "k15": ["-k", "15"],
    "k40": ["-k", "40"],
    "k64_nc": ["-k", "64", "--non-canonical"],
    "k31_nc": ["-k", "31", "--non-canonical"],
    "k31_cm": ["-k", "31", "--consider-missing"],
    "k31_nofilter": ["-k", "31", "--no-filter"],
    "k33_cm": ["-k", "33", "--consider-missing"],
}


@pytest.mark.parametrize("only_passing", [False, True])
@pytest.mark.parametrize("case", sorted(CASES))
def test_matches_host_join(case, only_passing, tmp_path):
    """The whole fixture (its N run and IUPAC codes included) against the host path."""
    rng = np.random.default_rng(sum(case.encode()) * 2 + only_passing)
    args = WHOLE + CASES[case]
    _cli(args, tmp_path / "plain")
    assoc = tmp_path / "assoc.tsv"
    _random_assoc(tmp_path / "plain", assoc, rng, 0.2, int_column=(case == "k31"))
    extra = ["--only-passing"] if only_passing else []
    want = _host_join(str(tmp_path / "plain"), assoc, ["-t", "0.5"] + extra)
    _cli(args + ["--associations", str(assoc), "--association-threshold", "0.5"] + extra, tmp_path / "joined")
    got = _read(str(tmp_path / "joined" / "annotated_kmers.tsv"))
    assert got.split("\n")[0] == want.split("\n")[0]
    assert _lines(got) == _lines(want)
    assert len(_lines(got)) > 1
    for name in ("kmers_to_hashes.tsv", "hashes_to_patterns.tsv"):
        assert _lines(_read(str(tmp_path / "joined" / name))) == _lines(_read(str(tmp_path / "plain" / name)))


def test_edge_cases(tmp_path):
    """A cluster whose only passing hash is its cluster row, a passing k-mer without a target window,
    one pattern in two clusters, ids that are unknown or not ids at all."""
    _cli(UPDOWN, tmp_path / "plain")
    k2h = [x.split("\t") for x in _read(str(tmp_path / "plain" / "kmers_to_hashes.tsv")).split("\n")[1:] if x]
    kmers = _read(str(tmp_path / "plain" / "kmers.tsv"))
    seen = {(x.split("\t")[0], x.split("\t")[-1]) for x in kmers.split("\n")[1:] if x}
    cluster_rows = [r for r in k2h if r[1] == ""]
    by_hash = {}
    for r in k2h:
        if r[1]:
            by_hash.setdefault(r[2], []).append(r)
    shared = [h for h, rs in by_hash.items() if len({r[0] for r in rs}) > 1]
    unseen = [r for r in k2h if r[1] and (r[0], r[1]) not in seen]
    assert cluster_rows and shared and unseen
    # a cluster row of a cluster none of whose k-mers pass
    lone = cluster_rows[0]
    chosen = {lone[2], shared[0], unseen[0][2]}
    chosen -= {r[2] for r in k2h if r[0] == lone[0] and r[1] and r[2] in chosen}
    chosen.add(lone[2])
    junk = ["notanid", "x" * 24, pattern_id(np.arange(7, dtype=np.int64)), "QUJD" * 6]
    lines = ["variant\taf\tlrt-pvalue"] + [f"{h}\t0.5\t0.01" for h in sorted(chosen)] + [f"{h}\t0.5\t0.01" for h in junk]
    assoc = tmp_path / "assoc.tsv"
    assoc.write_text("\n".join(lines) + "\n")
    for extra in ([], ["--only-passing"]):
        want = _host_join(str(tmp_path / "plain"), assoc, ["-t", "0.05"] + extra)
        out = tmp_path / ("joined" + "".join(extra))
        _cli(UPDOWN + ["--associations", str(assoc), "--association-threshold", "0.05"] + extra, out)
        got = _read(str(out / "annotated_kmers.tsv"))
        assert _lines(got) == _lines(want), extra
        if extra:                      # the cluster-row line of the cluster none of whose k-mers pass
            assert lone[0] + "\t\t" + lone[2] + "\t0.5\t0.01" + "\t" * 9 in got.split("\n")
    # nothing passes: the header alone
    _cli(UPDOWN + ["--associations", str(assoc), "--association-threshold", "0.001"], tmp_path / "none")
    got = _read(str(tmp_path / "none" / "annotated_kmers.tsv"))
    assert got == ("cluster\tk-mer\thashed_pattern\taf\tlrt-pvalue\tstrain\tfeature_id\tcontig\tfeature_strand\t"
                   "contig_start\tcontig_end\tgene_start\tgene_end\tstrand\n")

