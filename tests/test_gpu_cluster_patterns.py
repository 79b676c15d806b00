"""kB3_cluster_emit writes a cluster's rows from one CTA and hands K4 one candidate per bitset
that is distinct within the cluster; K4 numbers the candidates and every row takes its
candidate's id.  Against the C oracle, row for row, with the pattern sets compared through
their bitsets and the number of new patterns equal to the oracle's distinct patterns."""
import numpy as np
import pytest

from test_gpu_parity import _compare_with_oracle, _random_items

pytestmark = pytest.mark.gpu


def _check_patterns(out, want, cm):
    """The new patterns are the oracle's distinct patterns, each once."""
    got = out["kmer_pattern_bits"]
    assert len(got) == len(want["kmer_pattern_bits"])
    if cm:
        got_set = {(r.tobytes(), c) for r, c in zip(got, out["kmer_pattern_cluster"].tolist())}
        assert len(got_set) == len(got)
    else:
        got_set = {r.tobytes() for r in got}
        assert len(got_set) == len(got)
        assert got_set == {r.tobytes() for r in want["kmer_pattern_bits"]}
    assert np.array_equal(np.unique(out["row_pattern"]), np.arange(len(got)))


def _run(items, stroi, S, canon=True, cm=False, nf=False, maf=0.01, **kw):
    out, want = _compare_with_oracle(items, stroi, S, 31, canon, cm, nf, maf, **kw)
    assert out["stats"]["engine"] == 2
    _check_patterns(out, want, cm)
    return out, want


@pytest.mark.parametrize("S,canon", [(40, True), (129, False), (500, True)])
def test_shared_patterns_match_oracle(S, canon):
    """Three founders per cluster and few private mutations: most rows share their bitset with
    other rows of their cluster."""
    rng = np.random.default_rng(3100 + S)
    items, stroi = _random_items(rng, S, 31, 6 if S < 200 else 3, 400, div=0.01)
    out, _ = _run(items, stroi, S, canon, batch_clusters=3)
    assert len(out["row_pattern"]) > 2 * len(out["kmer_pattern_bits"])


@pytest.mark.parametrize("S,nf", [(40, False), (129, True), (500, True)])
def test_consider_missing_and_no_filter(S, nf):
    """--consider-missing: K4's key is the bitset plus the cluster pattern word, which is the
    same for every row of a cluster, so the cluster-local dedup on the bitset stays exact."""
    rng = np.random.default_rng(3200 + S)
    items, stroi = _random_items(rng, S, 31, 5 if S < 200 else 3, 350, div=0.01)
    _run(items, stroi, S, True, True, nf, 0.02, batch_clusters=5)


@pytest.mark.parametrize("S,canon", [(40, True), (129, False), (500, True)])
def test_maf0_one_sample_rows(S, canon):
    """maf 0: one-sample survivors have no bitset in slab_rows; they are compared and written
    through their one-hot form, against rows of the same pattern that do have one."""
    rng = np.random.default_rng(3300 + S)
    items, stroi = _random_items(rng, S, 31, 4 if S < 200 else 2, 300)
    _run(items, stroi, S, canon, False, False, 0.0, batch_clusters=2)


@pytest.mark.parametrize("smem_kb", ["0", "1"])
def test_tiny_pattern_table(smem_kb, monkeypatch):
    """PF_PATTERN_SMEM_KB 0: every row is its own candidate; 1 KB: clusters of up to 63 survivors
    use the table, larger ones fall back to a candidate per row.  K4 merges them all."""
    monkeypatch.setenv("PF_PATTERN_SMEM_KB", smem_kb)
    rng = np.random.default_rng(3400)
    items, stroi = _random_items(rng, 90, 31, 8, 300, div=0.01)
    tiny = _random_items(rng, 90, 31, 4, 50, div=0.0)[0]           # clusters with few survivors
    _run(items + tiny, stroi, 90, True, True, False, 0.01, batch_clusters=4)


def test_clusters_merged_in_global_table(monkeypatch):
    """PF_MERGE_SMEM_KB 0: every cluster's partial rows are merged by kB1_insert (dirty owners
    whose bitsets were written by folds) before the per-cluster emit."""
    monkeypatch.setenv("PF_MERGE_SMEM_KB", "0")
    rng = np.random.default_rng(3500)
    items, stroi = _random_items(rng, 90, 31, 6, 300, div=0.01)
    _run(items, stroi, 90, True, False, False, 0.0, batch_clusters=3)


def test_pipelined_submit(monkeypatch):
    """Pipelined sub-batches: the row -> candidate -> pattern gather runs before each
    sub-batch's rows are copied back."""
    monkeypatch.setenv("PF_PIPELINE_SEQS", "1024")
    rng = np.random.default_rng(3600)
    items, stroi = _random_items(rng, 60, 31, 60, 260, div=0.01)
    out, _ = _run(items, stroi, 60, True, True, False, 0.02, batch_clusters=len(items))
    assert out["stats"]["sub_batches"] >= 2


@pytest.mark.parametrize("batch_clusters", [4, 2])
def test_pattern_shared_across_clusters(batch_clusters):
    """Two clusters with the same sequences in the same samples have the same patterns: each
    pattern is a candidate of both clusters (in one batch, or in two), and K4 gives it one id."""
    rng = np.random.default_rng(3700)
    items, stroi = _random_items(rng, 40, 31, 2, 300, div=0.01)
    twins = [(cluster, name + "_twin", presab.copy()) for cluster, name, presab in items]
    out, want = _run(items + twins, stroi, 40, True, False, False, 0.01, batch_clusters=batch_clusters)
    n = len(out["row_pattern"]) // 2
    assert n > 0
    # each pattern id is used by rows of both copies
    cl = out["row_cluster"]
    first = set(out["row_pattern"][cl < 2].tolist())
    second = set(out["row_pattern"][cl >= 2].tolist())
    assert first == second
