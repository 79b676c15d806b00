"""bench.py --dump-outputs: the arrays written for comparing two builds output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

S, C, N = 70, 50, 20000
ID0 = 1000                   # cluster ids (pf_cluster_desc.id) are not batch indices
W = (S + 31) // 32


class _Batch:
    def __init__(self, ids):
        self.clusters = np.zeros(len(ids), [("id", "<u4"), ("reserved", "<u4")])
        self.clusters["id"] = ids


class _Ctx:
    """export_patterns of a context whose tables hold `kmer` / `cluster` patterns."""

    def __init__(self, kmer, cluster):
        self.tables = (kmer, cluster)

    def export_patterns(self, ns, first, count):
        return self.tables[ns][first:first + count]


@pytest.fixture(scope="module")
def step():
    """Rows of one step over C clusters; the k-mer patterns of the first 25 are 0..149."""
    rng = np.random.default_rng(0)
    cl = np.sort(rng.integers(ID0, ID0 + C, N)).astype(np.uint32)
    km = rng.integers(0, 2 ** 62, N, dtype=np.uint64)
    kpat = rng.integers(0, 2 ** 32, (300, W + 1), dtype=np.uint64).astype(np.uint32)
    cpat = rng.integers(0, 2 ** 32, (C, W), dtype=np.uint64).astype(np.uint32)
    pid = rng.integers(0, 300, N).astype(np.uint32)
    pid = np.where(cl < ID0 + 25, pid % 150, pid).astype(np.uint32)
    cnt = np.unpackbits(kpat[:, :W].view(np.uint8), axis=1).sum(axis=1)[pid].astype(np.uint32)
    return dict(cl=cl, km=km, kpat=kpat, cpat=cpat, pid=pid, cnt=cnt)


def _dump(step, tmp_path, bounds, shuffle=False):
    """The step fed as batches [bounds[i], bounds[i+1]) of clusters, as pf_collect returns them."""
    rng = np.random.default_rng(1)
    d = bench.OutputDump(S, C)
    ctx = _Ctx(step["kpat"], step["cpat"])
    kbase = 0
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        rows = np.flatnonzero((step["cl"] >= ID0 + lo) & (step["cl"] < ID0 + hi))
        if shuffle:
            rows = rng.permutation(rows)
        new_k = 150 if hi <= 25 else 300 - kbase
        r = {"row_cluster": step["cl"][rows], "row_kmer": step["km"][rows],
             "row_count": step["cnt"][rows], "row_pattern": step["pid"][rows],
             "wide_row_cluster": np.zeros(0, np.uint32), "wide_row_kmer": np.zeros((0, 2), np.uint64),
             "wide_row_count": np.zeros(0, np.uint32), "wide_row_pattern": np.zeros(0, np.uint32),
             "cluster_pattern": np.arange(lo, hi, dtype=np.uint32),
             "kmer_pattern_base": kbase, "new_kmer_patterns": step["kpat"][kbase:kbase + new_k],
             "cluster_pattern_base": lo, "new_cluster_patterns": step["cpat"][lo:hi], "n_pos": 0}
        d.add(r, _Batch(np.arange(ID0 + lo, ID0 + hi)), ctx)
        kbase += new_k
    info = d.write(str(tmp_path))
    return info, {n: np.load(os.path.join(str(tmp_path), n + ".npy")) for n in info["arrays"]}


def test_every_row_when_the_step_fits(step, tmp_path):
    info, a = _dump(step, tmp_path, [0, C])
    assert not info["rows_sampled"] and info["bytes"] <= 64 * 10 ** 6
    assert all(x.dtype == np.float64 for x in a.values())
    o = np.lexsort((step["km"], step["cl"]))
    assert np.array_equal(a["row_cluster"], step["cl"][o])
    k = a["row_kmer"].astype(np.uint64)
    assert not k[:, :2].any()
    assert np.array_equal((k[:, 2] << np.uint64(32)) | k[:, 3], step["km"][o])
    assert np.array_equal(a["row_count"], step["cnt"][o])
    assert np.array_equal(a["row_pattern_bits"], step["kpat"][step["pid"][o], :W])
    assert np.array_equal(a["cluster_id"], ID0 + np.arange(C))
    assert np.array_equal(a["cluster_rows"], np.bincount(step["cl"] - ID0, minlength=C))
    assert np.array_equal(a["cluster_count_sum"], np.bincount(step["cl"] - ID0, weights=step["cnt"], minlength=C))
    assert np.array_equal(a["cluster_samples"], np.unpackbits(step["cpat"].view(np.uint8), axis=1).sum(axis=1))
    assert np.array_equal(a["totals"], [N, 300, C, 0])


def test_sample_depends_on_neither_row_order_nor_batches(step, tmp_path, monkeypatch):
    """Over the budget: the same rows whether the step came in one batch or in two (the second
    naming patterns of the first), in order or shuffled."""
    monkeypatch.setattr(bench, "DUMP_BYTES", 8 * (4 * C + 4) + 4096 + 8 * (6 + W) * 1000)
    info1, a = _dump(step, tmp_path / "one", [0, C])
    info2, b = _dump(step, tmp_path / "two", [0, 25, C], shuffle=True)
    assert info1["rows_sampled"] and info1["arrays"]["row_cluster"] == [1000]
    assert info1["arrays"] == info2["arrays"]
    for name in a:
        assert np.array_equal(a[name], b[name]), name
    full = set(zip(step["cl"].tolist(), step["km"].tolist()))
    k = a["row_kmer"].astype(np.uint64)
    assert set(zip(a["row_cluster"].astype(np.int64).tolist(),
                   ((k[:, 2] << np.uint64(32)) | k[:, 3]).tolist())) <= full


@pytest.mark.gpu
def test_bench_dumps_the_same_outputs_twice(tmp_path):
    """Two runs of the timed path with the same arguments write the same arrays, and so does the
    streamed path over the same clusters in four batches (later batches name patterns found by
    earlier ones)."""
    out = []
    for run, extra in (("a", []), ("b", []), ("streamed", ["--batch-clusters", "10"])):
        d = str(tmp_path / run)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--clusters", "40", "--steps", "2",
                            "--warmup", "1", "--no-extra", "--no-e2e", "--no-cpu-baseline", "--dump-outputs", d]
                           + extra, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-4000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == 2 and line["dump_outputs"]["dir"] == d
        out.append({n: np.load(os.path.join(d, n + ".npy")) for n in line["dump_outputs"]["arrays"]})
    a = out[0]
    for b in out[1:]:
        assert a.keys() == b.keys()
        for name in a:
            assert np.array_equal(a[name], b[name]), name
    assert a["totals"][0] == len(a["row_cluster"]) > 1000
    pc = np.unpackbits(a["row_pattern_bits"].astype(np.uint32).view(np.uint8), axis=1).sum(axis=1)
    assert np.array_equal(pc, a["row_count"])
    assert a["cluster_rows"].sum() == a["totals"][0]
