"""kA puts every sequence's run into the chunk table, ragged tails and windows over N / IUPAC
symbols included (a live-window mask in the chunk key), and builds each k-mer row from the list
of (chunk, window) pairs that carry it: a one-chunk row of a one-sample chunk is a one-sample
row, other rows OR their chunks' bitsets.  A full chunk table overflows the run like a full
k-mer table does.  These inputs stress each of those, against the C oracle."""
import numpy as np
import pytest

from oracle import ref_port
from test_gpu_ka_segments import _cluster
from test_gpu_parity import _compare_with_oracle, _random_items

pytestmark = pytest.mark.gpu

_COMP = str.maketrans("ACGTNRYK", "TGCANRYK")


def _names(S):
    return [f"g{i:04d}" for i in range(S)]


def _cut(q, s, i=0):
    q = "".join(q)
    return ref_port.CutSeq(q, q.translate(_COMP), f"{s}_{i}", "ctg", 101, 100 + len(q), 1, 0)


def _items_from(clusters, names):
    return [({s: lst for s, lst in zip(names, seqs)}, f"c{i}", np.array([int(bool(x)) for x in seqs]))
            for i, seqs in enumerate(clusters)]


@pytest.mark.parametrize("seg_runs", ["1", "16"])
@pytest.mark.parametrize("S", [32, 500, 1024])
def test_ragged_tails(S, seg_runs, monkeypatch):
    """Every copy cut to its own length: runs end with 1..15 live windows, and equal tails of
    one haplotype meet in one chunk."""
    monkeypatch.setenv("PF_KA_SEG_RUNS", seg_runs)
    rng = np.random.default_rng(3100 + S)
    names = _names(S)
    items = [_cluster(rng, names, 260, f"r{c}", min_len=120) for c in range(2)]
    lens = {len(cs.sequence) for cl, _, _ in items for lst in cl.values() for cs in lst}
    assert {(n - 31 + 1) % 16 for n in lens} >= set(range(1, 16))
    out, _ = _compare_with_oracle(items, set(), S, 31, True, False, False, 0.0, batch_clusters=2)
    assert out["stats"]["engine"] == 2


@pytest.mark.parametrize("canon", [True, False])
def test_ambiguous_runs(canon):
    """N runs at the start, middle and end of runs of 16 windows, IUPAC codes, and one sequence
    that is all N: only the windows that touch no such symbol are counted."""
    rng = np.random.default_rng(3200 + canon)
    S, L = 60, 300
    names = _names(S)
    clusters = []
    for c in range(2):
        anc = rng.choice(list("ACGT"), L)
        seqs = []
        for i in range(S):
            q = anc.copy()
            m = rng.random(L) < 0.003
            q[m] = rng.choice(list("ACGT"), int(m.sum()))
            if i % 3 == 0:
                at = int(rng.choice([32, 40, 47, 64 + 15, 128 + 8]))   # start / middle / end of a run
                q[at:at + int(rng.integers(1, 6))] = "N"
            if i % 7 == 1:
                q[int(rng.integers(0, L))] = rng.choice(list("RYK"))
            if c == 0 and i == 5:
                q[:] = "N"
            seqs.append([_cut(q, names[i])])
        clusters.append(seqs)
    out, _ = _compare_with_oracle(_items_from(clusters, names), set(), S, 31, canon, False, False, 0.0,
                                  batch_clusters=2)
    assert out["stats"]["engine"] == 2


@pytest.mark.parametrize("canon", [True, False])
def test_paralogs(canon):
    """Identical copies of one sample meet in one chunk whose popcount stays 1; copies that
    differ by a private SNP give k-mers carried by two chunks of one sample only, which must
    still come out as one-sample rows."""
    rng = np.random.default_rng(3300 + canon)
    S, L = 40, 280
    names = _names(S)
    anc = rng.choice(list("ACGT"), L)
    seqs = []
    for i in range(S):
        q = anc.copy()
        m = rng.random(L) < 0.01
        q[m] = rng.choice(list("ACGT"), int(m.sum()))
        lst = [_cut(q, names[i], 0)]
        if i % 2 == 0:
            lst.append(_cut(q, names[i], 1))                     # identical paralog
        if i % 5 == 0:
            p = q.copy()
            pos = int(rng.integers(40, L - 40))
            p[pos] = "A" if p[pos] != "A" else "C"
            lst.append(_cut(p, names[i], 2))                     # paralog with its own SNP
        seqs.append(lst)
    out, _ = _compare_with_oracle(_items_from([seqs], names), set(), S, 31, canon, False, False, 0.0,
                                  batch_clusters=1)
    assert out["stats"]["engine"] == 2


@pytest.mark.parametrize("S,L,snps", [(500, 220, 2), (1024, 2000, 1), (1024, 220, 2)])
def test_every_sequence_its_own_haplotype(S, L, snps):
    """Every sequence carries private SNPs: many distinct chunks per run, most k-mer rows of
    one sample; the batch stays on the block engine.  (1024, 220, 2) holds ~3,000 distinct
    k-mers per run: more than rows with bitsets took in shared memory, which sent such a batch
    to the record engine before rows became lists."""
    rng = np.random.default_rng(3400 + S + L)
    names = _names(S)
    anc = rng.choice(list("ACGT"), L)
    seqs = []
    for i in range(S):
        q = anc.copy()
        for pos in rng.choice(L, size=snps, replace=False):
            q[pos] = rng.choice([b for b in "ACGT" if b != q[pos]])
        seqs.append([_cut(q, names[i])])
    out, _ = _compare_with_oracle(_items_from([seqs], names), set(), S, 31, True, False, False, 0.0,
                                  batch_clusters=1)
    assert out["stats"]["engine"] == 2


@pytest.mark.parametrize("slots,cslots", [("64", "32"), ("128", "32"), ("8192", "32")])
def test_table_overflow_and_rescue(slots, cslots, monkeypatch):
    """Chunk tables of 24 chunks and small k-mer tables: runs overflow and are rerun with the
    rescue tables."""
    monkeypatch.setenv("PF_BLOCK_SLOTS", slots)
    monkeypatch.setenv("PF_BLOCK_CSLOTS", cslots)
    rng = np.random.default_rng(3500 + int(slots))
    names = _names(200)
    items = [_cluster(rng, names, 300, f"o{c}", min_len=200, amb_rate=0.002 * c) for c in range(3)]
    out, _ = _compare_with_oracle(items, set(), 200, 31, True, False, False, 0.0, batch_clusters=3)
    assert out["stats"]["engine"] == 2


@pytest.mark.parametrize("S,k,canon", [(60, 31, False), (5, 4, True), (40, 16, True), (1300, 31, True)])
def test_modes_and_slices(S, k, canon):
    """--non-canonical k = 31 (a node per strand), canonical even k (palindromes list one pair
    twice) and sample slices of 512."""
    rng = np.random.default_rng(3600 + S + k)
    items, _ = _random_items(rng, S, k, 3 if S < 1000 else 2, 200 if S < 1000 else 150)
    out, _ = _compare_with_oracle(items, set(), S, k, canon, False, False, 0.0, batch_clusters=3)
    assert out["stats"]["engine"] == 2
