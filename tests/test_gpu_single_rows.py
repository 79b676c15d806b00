"""kA writes a partial row carried by ONE sample as its key and a one-sample code only, with no
bitset; kB1 writes such a row's bitset out when another row of its k-mer is folded into it, and
kB3 / kB4 / kB6 read the code where they used to read the row.  These inputs make one-sample rows
pass the MAF window (maf 0) and fold into each other in every combination, against the C oracle."""
from collections import defaultdict

import numpy as np
import pytest

from oracle import ref_port
from test_gpu_ka_segments import _cluster as _overflow_cluster
from test_gpu_parity import _compare_with_oracle, _random_items

pytestmark = pytest.mark.gpu

_COMP = str.maketrans("ACGT", "TGCA")
# frame shifts of a sample's copy behind an indel near its start: not multiples of 16, so the
# same k-mer starts in different runs of 16 windows in different samples
SHIFTS = (0, -5, 3, -11, -21, 9, -37)


def _names(S):
    return [f"g{i:05d}" for i in range(S)]


def _shifted_cluster(rng, names, L, name, n_sites, max_carriers=4, private=0.0, p_absent=0.1):
    """One ancestor; `n_sites` variant sites behind position 60, each carried by 1..max_carriers
    random samples; every copy gets one of SHIFTS by an indel at position 20 and, at rate
    `private`, bases of its own.  A k-mer over a variant site then has one partial row per run
    its carriers' copies put it in: one-sample rows next to one-sample and many-sample rows."""
    anc = rng.choice(list("ACGT"), L)
    present = [s for s in names if rng.random() >= p_absent]
    copies = {s: anc.copy() for s in present}
    for pos in rng.choice(np.arange(60, L), size=min(n_sites, L - 60), replace=False):
        alt = rng.choice([b for b in "ACGT" if b != anc[pos]])
        for s in rng.choice(present, size=min(len(present), int(rng.integers(1, max_carriers + 1))),
                            replace=False):
            copies[s][pos] = alt
    cluster = {s: [] for s in names}
    presab = np.zeros(len(names), dtype=int)
    rank = {s: i for i, s in enumerate(names)}
    for s in present:
        q = copies[s]
        if private:
            m = rng.random(L) < private
            q[m] = rng.choice(list("ACGT"), int(m.sum()))
        shift = int(rng.choice(SHIFTS))
        if shift < 0:
            q = np.concatenate([q[:20], q[20 - shift:]])
        elif shift > 0:
            q = np.concatenate([q[:20], rng.choice(list("ACGT"), shift), q[20:]])
        q = "".join(q)
        cluster[s] = [ref_port.CutSeq(q, q.translate(_COMP), s + "_f", "ctg", 101, 100 + len(q), 1, 0)]
        presab[rank[s]] = 1
    return (cluster, name, presab)


def _fold_kinds(items, k):
    """Per k-mer (canonical), the sample count of each partial row kA writes for it (one row per
    run of 16 windows that holds it): how many k-mers have two one-sample rows only, one-sample
    next to many-sample rows, and three or more one-sample rows."""
    kinds = {"single+single": 0, "single+multi": 0, "3+ singles": 0}
    for cluster, _, _ in items:
        rows = defaultdict(lambda: defaultdict(set))
        for s, lst in cluster.items():
            for cs in lst:
                q = cs.sequence
                for p in range(len(q) - k + 1):
                    f = q[p:p + k]
                    rows[min(f, f.translate(_COMP)[::-1])][p // 16].add(s)
        for by_run in rows.values():
            if len(by_run) < 2:
                continue
            sizes = [len(v) for v in by_run.values()]
            singles = sizes.count(1)
            if singles == len(sizes) == 2:
                kinds["single+single"] += 1
            if singles and singles < len(sizes):
                kinds["single+multi"] += 1
            if singles >= 3:
                kinds["3+ singles"] += 1
    return kinds


@pytest.mark.parametrize("S,canon,cm", [(40, True, False), (40, False, True), (500, True, True),
                                        (500, False, False)])
def test_one_sample_rows_pass_the_window(S, canon, cm):
    """maf 0: every k-mer passes, so kB3 writes the one-hot bitsets of one-sample rows."""
    rng = np.random.default_rng(900 + S + 2 * canon + cm)
    items, stroi = _random_items(rng, S, 31, 4 if S < 100 else 2, 300)
    out, _ = _compare_with_oracle(items, stroi, S, 31, canon, cm, False, 0.0, batch_clusters=2)
    assert out["stats"]["engine"] == 2


def _fold_items(seed, S=40, n_clusters=3):
    rng = np.random.default_rng(seed)
    names = _names(S)
    items = [_shifted_cluster(rng, names, 420, f"f{c}", n_sites=30) for c in range(n_clusters)]
    kinds = _fold_kinds(items, 31)
    assert all(v > 0 for v in kinds.values()), kinds
    return items


@pytest.mark.parametrize("seed,canon,maf", [(71, True, 0.0), (72, False, 0.0), (73, True, 0.05),
                                            (74, False, 0.05)])
def test_folds_of_one_sample_rows(seed, canon, maf):
    """single -> single (count 2; at maf 0.05 and 40 samples exactly the lower bound), single ->
    many, many -> single and several singles into one single owner, in the shared-memory merge
    (kB1_local); the seeds change which row of a k-mer becomes its owner."""
    items = _fold_items(seed)
    out, _ = _compare_with_oracle(items, set(), 40, 31, canon, False, False, maf, batch_clusters=3)
    assert out["stats"]["engine"] == 2
    assert out["stats"]["partial_rows"] > out["stats"]["unique_kmers"]


@pytest.mark.parametrize("seed", [75, 76])
def test_folds_of_one_sample_rows_global_table(seed, monkeypatch):
    """The same folds in the global-memory merge (kB1_insert): no shared-memory table."""
    monkeypatch.setenv("PF_MERGE_SMEM_KB", "0")
    items = _fold_items(seed)
    out, _ = _compare_with_oracle(items, set(), 40, 31, True, True, False, 0.0, batch_clusters=3)
    assert out["stats"]["engine"] == 2
    assert out["stats"]["partial_rows"] > out["stats"]["unique_kmers"]


@pytest.mark.parametrize("seed", [77, 78])
def test_folds_of_one_sample_rows_weak_fingerprints(seed, monkeypatch):
    """The same folds with a 1-bit fingerprint: nearly every probe of an occupied slot compares
    full keys, so rows of other k-mers are met on the way to the owner."""
    monkeypatch.setenv("PF_MERGE_FP_BITS", "1")
    items = _fold_items(seed)
    out, _ = _compare_with_oracle(items, set(), 40, 31, False, False, False, 0.05, batch_clusters=3)
    assert out["stats"]["engine"] == 2
    assert out["stats"]["partial_rows"] > out["stats"]["unique_kmers"]


@pytest.mark.parametrize("S,maf", [(1300, 0.0), (1300, 0.01), (10000, 0.0), (10000, 0.01)])
def test_sample_slices(S, maf):
    """S > 1024: kB4 counts a one-sample row as 1 and kB6 writes its single word into the k-mer's
    row; the frame shifts fold rows inside a slice first."""
    rng = np.random.default_rng(80 + S // 1000 + int(maf * 100))
    names = _names(S)
    L = 200 if S < 5000 else 90
    items = [_shifted_cluster(rng, names, L, f"s{c}", n_sites=20, private=0.0002 if S > 5000 else 0.001)
             for c in range(2)]
    out, _ = _compare_with_oracle(items, set(), S, 31, True, maf > 0, False, maf, batch_clusters=2)
    assert out["stats"]["engine"] == 2


@pytest.mark.parametrize("cm", [False, True])
def test_rescue_launches(cm):
    """Runs over 40 bases of every sample's own overflow kA's table and are rerun with larger
    tables: those rows are nearly all one-sample rows, and at maf 0 they are all emitted.
    (Canonical only: with both strands the runs exceed the largest table and the batch goes to
    the record engine.)"""
    rng = np.random.default_rng(62)
    names = [f"g{i:04d}" for i in range(150)]
    items = [_overflow_cluster(rng, names, 640, f"o{c}", middle=40) for c in range(3)]
    out, _ = _compare_with_oracle(items, set(), 150, 31, True, cm, False, 0.0, batch_clusters=3)
    assert out["stats"]["engine"] == 2
