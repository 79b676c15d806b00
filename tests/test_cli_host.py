"""Host logic of the drop-in CLI on the CPU: `python -m panfeed_b200` with the GPU context
replaced by the oracle-backed stand-in (tests/cpu_context.py).  Everything around the kernels
runs for real — option handling, file discovery, both feeders, the packer, batching, the id
tables, the library's native text formatters and gzip members — and the three files must equal
the UNMODIFIED reference's goldens (tests/golden/expected, /root/reference/tests/unit_test.sh
modes + extras) after sorting, like tests/test_gpu_cli.py demands of the CUDA path."""
import gzip
import os

import pytest

import helpers
from cpu_context import OracleContext
from panfeed_b200 import capi


def _read(path):
    if os.path.exists(path + ".gz"):
        return gzip.open(path + ".gz", "rt").read()
    return open(path).read()


def _run_cli(args, out, monkeypatch):
    from panfeed_b200.__main__ import main
    monkeypatch.setattr(capi, "Context", OracleContext)
    OracleContext.instances.clear()
    cwd = os.getcwd()
    os.chdir(helpers.GOLDEN)
    try:
        main(args + ["--output", out])
    finally:
        os.chdir(cwd)


@pytest.mark.parametrize("feeder", ["python", "native"])
@pytest.mark.parametrize("mode", sorted(helpers.modes()))
def test_cli_host_logic_matches_reference(mode, feeder, tmp_path, monkeypatch):
    args = list(helpers.modes()[mode]) + (["--native-feeder"] if feeder == "native" else ["--python-feeder"])
    out = str(tmp_path / "out")
    _run_cli(args, out, monkeypatch)
    for name in helpers.FILES:
        got = _read(os.path.join(out, name))
        want = helpers.golden(mode, name)
        assert got.split("\n")[0] == [x for x in want.split("\n") if x.startswith(
            ("cluster\t", "hashed_pattern"))][0]
        assert helpers.sorted_lines(got) == helpers.sorted_lines(want), (mode, name)
    assert len(OracleContext.instances) == 1          # one context per run, whatever the batching
    if mode == "compress":
        assert os.path.exists(os.path.join(out, "kmers.tsv.gz"))


def test_cli_host_logic_small_batches(tmp_path, monkeypatch):
    """Several GPU batches per run (BATCH_RECORDS forced down): pattern bases, id tables and the
    cluster-absent NaN planes carry over from batch to batch."""
    from panfeed_b200 import panfeed
    monkeypatch.setattr(panfeed, "BATCH_RECORDS", 2000)
    for mode in ("considermissing", "secondpass"):
        out = str(tmp_path / mode)
        _run_cli(list(helpers.modes()[mode]) + ["--python-feeder"], out, monkeypatch)
        assert OracleContext.instances[0].n_batches > 1
        for name in helpers.FILES:
            assert helpers.sorted_lines(_read(os.path.join(out, name))) == \
                helpers.sorted_lines(helpers.golden(mode, name)), (mode, name)


@pytest.mark.parametrize("feeder", [[], ["--python-feeder"]])
def test_cli_host_logic_multiple_files(feeder, tmp_path, monkeypatch):
    """--multiple-files: one directory per cluster, the pattern set reset per cluster
    (panfeed.py:35-43,153-167); against the reference's restatement per cluster."""
    import pandas as pd
    from oracle import ref_port
    out = str(tmp_path / "out")
    _run_cli(["--gff", "fixture/gffs/", "--presence-absence", "fixture/gene_presence_absence.csv",
              "--targets", "fixture/stroi.txt", "--multiple-files"] + feeder, out, monkeypatch)
    cwd = os.getcwd()
    os.chdir(helpers.GOLDEN)
    try:
        table = pd.read_csv("fixture/gene_presence_absence.csv", sep=",", index_col=0,
                            low_memory=False).drop(columns=["Non-unique Gene name", "Annotation"])
        genomes = ref_port.load_inputs("fixture/gffs/")
        stroi = {x.rstrip("\n") for x in open("fixture/stroi.txt")}
        h2p_head, k2h_head = ref_port.headers(table.columns)
        n = 0
        for item in ref_port.feed_clusters(table, genomes, 0, 0, False):
            res = ref_port.kmer_stage(item, 31, stroi, True, False)
            a, b, c = ref_port.pattern_stage((res,), True, 0.01, False, set())
            d = os.path.join(out, item[1])
            assert helpers.sorted_lines(open(os.path.join(d, "kmers.tsv")).read()) == \
                helpers.sorted_lines(ref_port.KMERS_HEADER + a)
            assert helpers.sorted_lines(open(os.path.join(d, "hashes_to_patterns.tsv")).read()) == \
                helpers.sorted_lines(h2p_head + b)
            assert helpers.sorted_lines(open(os.path.join(d, "kmers_to_hashes.tsv")).read()) == \
                helpers.sorted_lines(k2h_head + c)
            n += 1
        assert n > 1
    finally:
        os.chdir(cwd)


def test_cli_host_logic_native_feeder_many_batches(tmp_path, monkeypatch):
    """--native-feeder with the library's whole-batch cuts forced down to a few clusters each."""
    import functools
    from panfeed_b200 import feeder
    monkeypatch.setattr(feeder, "iter_packed_batches",
                        functools.partial(feeder.iter_packed_batches, first_cells=9, target_bases=5000))
    for mode in ("considermissing", "secondpass", "nc_updown"):
        out = str(tmp_path / mode)
        _run_cli(list(helpers.modes()[mode]) + ["--native-feeder"], out, monkeypatch)
        assert OracleContext.instances[0].n_batches > 2
        for name in helpers.FILES:
            assert helpers.sorted_lines(_read(os.path.join(out, name))) == \
                helpers.sorted_lines(helpers.golden(mode, name)), (mode, name)


@pytest.mark.parametrize("feeder", [[], ["--python-feeder"]])
def test_cli_stop_on_missing_raises(feeder, tmp_path, monkeypatch):
    """--stop-on-missing: a feature id of the table that no GFF holds ends the run with the
    reference's KeyError (input.py:396-400) - also when the cut runs on the feeder's thread."""
    genes = tmp_path / "genes.txt"
    genes.write_text("group_acc1\n")                          # names s07_refound_1, which no GFF has
    with pytest.raises(KeyError, match="Could not find gene s07_refound_1 from group_acc1 in s07"):
        _run_cli(["--gff", "fixture/gffs/", "--presence-absence", "fixture/gene_presence_absence.csv",
                  "--genes", str(genes), "--stop-on-missing"] + feeder, str(tmp_path / "out"), monkeypatch)
    # without the flag the gene is skipped with a warning and the run completes
    _run_cli(["--gff", "fixture/gffs/", "--presence-absence", "fixture/gene_presence_absence.csv",
              "--genes", str(genes)] + feeder, str(tmp_path / "out2"), monkeypatch)
    assert os.path.getsize(os.path.join(str(tmp_path / "out2"), "kmers_to_hashes.tsv")) > 100


def test_cli_options_and_defaults_are_the_references():
    """Every option of the reference's command line (`panfeed/__main__.py:84-223`) exists here
    with the same destination and default; only --device and the feeder switches are new.  The
    reference's parsed options are stored in tests/golden/expected/cli_options.json
    (tests/golden/make_golden.py)."""
    gold = helpers.cli_options()
    ref = gold["options"]
    from panfeed_b200.__main__ import get_options
    ours = vars(get_options(gold["argv"]))
    assert len(ref) >= 20
    for name, default in ref.items():
        assert name in ours, name
        assert ours[name] == default, (name, ours[name], default)
    assert set(ours) - set(ref) == {"device", "native_feeder", "python_feeder"}
