"""kA walks segments of consecutive runs of one (cluster, slice) per CTA: sequences stay in
registers from run to run and the shared tables are reset lazily between runs.  These inputs
stress what that changes, at fixed segment lengths (PF_KA_SEG_RUNS; a batch this small would
otherwise get one-run segments) and at the length the library picks, against the C oracle."""
import numpy as np
import pytest

from oracle import ref_port
from test_gpu_parity import _compare_with_oracle, _random_items

pytestmark = pytest.mark.gpu

# 3: segments start at odd runs too (a run in the middle of a 64-bit word); 64: segments span
# several clusters; None: the library's choice
SEG_RUNS = ["3", "16", "64", None]

_COMP = str.maketrans("ACGTN", "TGCAN")


def _cluster(rng, names, L, name, copies=1, min_len=None, middle=0, amb_rate=0.0):
    """Copies of three founders of length L.  min_len: every copy is cut to a random length in
    [min_len, L], so sequences end in different runs; middle: that many random bases of each
    copy's own are put in the middle (a stretch of runs whose distinct k-mers overflow kA's
    table, between runs that fit); amb_rate: N / IUPAC bases."""
    anc = rng.choice(list("ACGT"), L)
    founders = []
    for _ in range(3):
        f = anc.copy()
        m = rng.random(L) < 0.03
        f[m] = rng.choice(list("ACGT"), int(m.sum()))
        founders.append(f)
    cluster = {}
    for s in names:
        lst = []
        for _ in range(copies):
            q = founders[int(rng.integers(3))].copy()
            m = rng.random(L) < 0.004
            q[m] = rng.choice(list("ACGT"), int(m.sum()))
            if middle:
                q = np.concatenate([q[:L // 2], rng.choice(list("ACGT"), middle), q[L // 2:]])
            if min_len is not None:
                q = q[:int(rng.integers(min_len, L + 1))]
            if amb_rate:
                m = rng.random(len(q)) < amb_rate
                q[m] = rng.choice(list("NRYK"), int(m.sum()))
            q = "".join(q)
            lst.append(ref_port.CutSeq(q, q.translate(_COMP), s + "_f", "ctg", 101, 100 + len(q),
                                       int(rng.choice([1, -1])), int(rng.choice([0, 5]))))
        cluster[s] = lst
    return (cluster, name, np.ones(len(names), dtype=int))


def _names(S):
    return [f"g{i:04d}" for i in range(S)]


@pytest.mark.parametrize("seg_runs", SEG_RUNS)
def test_more_sequences_than_registers_hold(seg_runs, monkeypatch):
    """300 samples x 3 paralogs: 900 sequences of one cluster, more than the 2 x 256 that the
    threads of a CTA hold; the rest are read from global memory at every run."""
    if seg_runs:
        monkeypatch.setenv("PF_KA_SEG_RUNS", seg_runs)
    rng = np.random.default_rng(61)
    names = _names(300)
    items = [_cluster(rng, names, 900, f"p{c}", copies=3) for c in range(2)]
    out, _ = _compare_with_oracle(items, set(names[:4]), 300, 31, True, False, False, 0.01,
                                  batch_clusters=2)
    assert out["stats"]["engine"] == 2


@pytest.mark.parametrize("seg_runs", SEG_RUNS)
def test_overflow_in_the_middle_of_a_segment(seg_runs, monkeypatch):
    """A stretch of 40 bases of every sample's own makes the runs over it overflow kA's table
    (they are rerun as single items with larger tables); the runs after them in the same
    segment must start from clean tables."""
    if seg_runs:
        monkeypatch.setenv("PF_KA_SEG_RUNS", seg_runs)
    rng = np.random.default_rng(62)
    names = _names(150)
    items = [_cluster(rng, names, 640, f"o{c}", middle=40) for c in range(3)]
    out, _ = _compare_with_oracle(items, set(), 150, 31, True, False, False, 0.0, batch_clusters=3)
    assert out["stats"]["engine"] == 2


@pytest.mark.parametrize("seg_runs", SEG_RUNS)
def test_ragged_ambiguous_sequences(seg_runs, monkeypatch):
    """Lengths from 40 to 700 bases: sequences end in different runs of a segment (and some
    before it starts); N / IUPAC bases send runs down the per-window path."""
    if seg_runs:
        monkeypatch.setenv("PF_KA_SEG_RUNS", seg_runs)
    rng = np.random.default_rng(63)
    names = _names(90)
    items = [_cluster(rng, names, 700, f"r{c}", copies=1 + c % 2, min_len=40,
                      amb_rate=0.002 if c % 2 else 0.0) for c in range(4)]
    out, _ = _compare_with_oracle(items, set(names[:3]), 90, 31, False, True, False, 0.02,
                                  batch_clusters=4)
    assert out["stats"]["engine"] == 2


@pytest.mark.parametrize("seg_runs", SEG_RUNS)
def test_sample_slices(seg_runs, monkeypatch):
    """S > 1024: segments are runs of one slice of 512 samples."""
    if seg_runs:
        monkeypatch.setenv("PF_KA_SEG_RUNS", seg_runs)
    rng = np.random.default_rng(64)
    items, stroi = _random_items(rng, 1300, 31, 3, 400, amb_rate=0.001)
    out, _ = _compare_with_oracle(items, stroi, 1300, 31, True, True, False, 0.01, batch_clusters=3)
    assert out["stats"]["engine"] == 2
