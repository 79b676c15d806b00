"""Parity of the CUDA path (through the C-ABI) against the reference goldens
and the C oracle.  Bit-exact after canonical sorting; pattern ids are compared
through their full vectors (rendered to the reference's MD5 ids)."""
import os

import numpy as np
import pytest

import gpu_util
import helpers
import render
from oracle import oracle_c, ref_port
from test_oracle_c import _items

pytestmark = pytest.mark.gpu

# engines of the library (pf_stats.engine): block aggregation (default for S <= 1024),
# records + partition mode, records + full sort
ENGINES = {"block": dict(mode=0, debug_flags=0),
           "records": dict(mode=0, debug_flags=2),
           "fullsort": dict(mode=1, debug_flags=2)}


def _render_gpu(out, S, k, consider_missing, canonical):
    res = dict(out)
    res["row_kmer"] = [x.decode() for x in out["row_kmer"]]
    res["pos_seq"] = res["pos_pos"] = res["pos_used_strand"] = res["pos_kmer"] = []
    got = render.render(res, out["ids"], out["seq_meta"], out["seqs"], S, k,
                        consider_missing, canonical)
    got["kmers.tsv"] = gpu_util.kmers_tsv_lines(out, k, canonical)
    return got


@pytest.mark.parametrize("engine", sorted(ENGINES))
@pytest.mark.parametrize("mode", sorted(helpers.modes()))
def test_fixture_modes_match_reference_goldens(mode, engine):
    kw = helpers.cli_kwargs(helpers.modes()[mode])
    cwd = os.getcwd()
    os.chdir(helpers.GOLDEN)
    try:
        items, stroi, S = _items(kw)
    finally:
        os.chdir(cwd)
    out = gpu_util.run_gpu(items, stroi, S, kw["k"], not kw["non_canonical"],
                           kw["consider_missing"], kw["no_filter"], kw["maf"],
                           batch_clusters=3, **ENGINES[engine])
    got = _render_gpu(out, S, kw["k"], kw["consider_missing"],
                      not kw["non_canonical"])
    for name in helpers.FILES:
        assert sorted(got[name]) == render.golden_body(
            helpers.golden(mode, name)), (mode, name)


def _random_items(rng, S, k, n_clusters, L, amb_rate=0.0, div=0.03):
    comp = str.maketrans("ACGTN", "TGCAN")
    names = [f"g{i:0{max(4, len(str(S - 1)))}d}" for i in range(S)]     # sorted order == rank order
    rank = {s: i for i, s in enumerate(names)}
    order = list(rng.permutation(names))
    items = []
    for c in range(n_clusters):
        Lc = int(rng.integers(max(1, L // 2), L + 1))
        anc = rng.choice(list("ACGT"), Lc)
        founders = []
        for _ in range(3):
            f = anc.copy()
            m = rng.random(Lc) < div
            f[m] = rng.choice(list("ACGT"), int(m.sum()))
            founders.append(f)
        presab = np.zeros(S, dtype=int)
        cluster, absent = {}, []
        p_present = rng.uniform(0.2, 1.0)
        for s in order:
            if rng.random() > p_present:
                absent.append(s)
                continue
            presab[rank[s]] = 1
            lst = []
            for _ in range(2 if rng.random() < 0.1 else 1):
                q = founders[int(rng.integers(3))].copy()
                m = rng.random(Lc) < 0.004
                q[m] = rng.choice(list("ACGT"), int(m.sum()))
                if amb_rate:
                    m = rng.random(Lc) < amb_rate
                    q[m] = rng.choice(list("NRYK"), int(m.sum()))
                q = "".join(q)
                lst.append(ref_port.CutSeq(q, q.translate(comp), s + "_f", "ctg",
                                           101, 100 + Lc,
                                           int(rng.choice([1, -1])),
                                           int(rng.choice([0, 5]))))
            cluster[s] = lst
        for s in absent:
            cluster[s] = []
        items.append((cluster, f"cl{c}", presab))
    return items, set(order[:max(1, S // 10)])


def _compare_with_oracle(items, stroi, S, k, canon, cm, nf, maf, **gpu_kw):
    want = oracle_c.run(items, stroi, k, canon, cm, nf, maf, n_threads=4)
    w = dict(want)
    w["row_kmer"] = [x.decode() for x in want["row_kmer"]]
    w["pos_kmer"] = [x.decode() for x in want["pos_kmer"]]
    want_lines = render.render(w, want["ids"], want["seq_meta"], want["seqs"],
                               S, k, cm, canon)
    out = gpu_util.run_gpu(items, stroi, S, k, canon, cm, nf, maf, **gpu_kw)
    got = _render_gpu(out, S, k, cm, canon)
    for name in helpers.FILES:
        assert sorted(got[name]) == sorted(want_lines[name]), name
    return out, want


CASES = [
    # S,   k, clusters, L,  canon, cm,    nf,    maf,  amb,  sort_bits, batch
    (40,  31, 5, 300, True,  False, False, 0.01, 0.0,  0, 2),
    (40,  31, 5, 300, True,  False, False, 0.01, 0.0,  8, 5),    # heavy prefix sharing
    (70,  15, 4, 200, False, False, True,  0.05, 0.0,  16, 4),
    (33,  32, 4, 250, True,  True,  False, 0.10, 0.0,  0, 1),
    (33,  32, 4, 250, False, True,  True,  0.02, 0.002, 8, 2),   # k=32 non-canonical + IUPAC
    (129, 21, 3, 400, True,  True,  True,  0.01, 0.001, 0, 3),
    (5,   4,  3, 60,  True,  False, False, 0.0,  0.0,  8, 3),    # tiny even k: palindromes
    (1,   31, 2, 100, True,  False, False, 0.01, 0.0,  0, 2),    # single sample
    (600, 31, 2, 700, True,  False, False, 0.01, 0.0,  0, 1),    # multi-tile segments
    # k > 32: two-word k-mers through the 128-bit record pipeline
    (40,  33, 4, 300, True,  False, False, 0.01, 0.0,  0, 2),
    (70,  48, 3, 250, False, True,  True,  0.05, 0.0,  16, 3),
    (33,  64, 3, 200, True,  True,  False, 0.02, 0.0,  0, 1),
]


@pytest.mark.parametrize("engine", sorted(ENGINES))
@pytest.mark.parametrize("case", CASES, ids=[str(i) for i in range(len(CASES))])
def test_random_clusters_match_oracle(case, engine):
    S, k, nc, L, canon, cm, nf, maf, amb, sb, bc = case
    rng = np.random.default_rng(1000 + S * 7 + k)
    items, stroi = _random_items(rng, S, k, nc, L, amb)
    out, _ = _compare_with_oracle(items, stroi, S, k, canon, cm, nf, maf,
                                  batch_clusters=bc, sort_bits=sb, **ENGINES[engine])
    if engine == "block" and k <= 32 and not (k == 32 and not canon):
        assert out["stats"]["engine"] == 2
    else:
        assert out["stats"]["engine"] == (1 if engine == "fullsort" else 0)
    if k > 32:
        assert len(out["row_kmer"]) > 0 and all(len(x) == k for x in out["row_kmer"][:50])


@pytest.mark.parametrize("case", CASES[:6], ids=[str(i) for i in range(6)])
def test_unfused_partition_path(case):
    """debug_flags=1: K1 writes records, separate histogram and first pass."""
    S, k, nc, L, canon, cm, nf, maf, amb, sb, bc = case
    rng = np.random.default_rng(1000 + S * 7 + k)
    items, stroi = _random_items(rng, S, k, nc, L, amb)
    _compare_with_oracle(items, stroi, S, k, canon, cm, nf, maf,
                         batch_clusters=bc, sort_bits=sb, mode=0, debug_flags=3)


def test_partition_direct_rescue_launch():
    """Tiles with more distinct k-mers than the direct variant holds (768) are
    re-run one prefix-run per CTA; result must stay exact with one sorted byte."""
    rng = np.random.default_rng(78)
    comp = str.maketrans("ACGT", "TGCA")
    S = 6
    names = [f"g{i}" for i in range(S)]
    cluster = {}
    for s in names:
        q = "".join(rng.choice(list("ACGT"), 20000))
        cluster[s] = [ref_port.CutSeq(q, q.translate(comp), s + "_f", "c", 1, 20000, 1, 0)]
    items = [(cluster, "mid", np.ones(S, dtype=int))]
    out, want = _compare_with_oracle(items, set(), S, 31, True, False, False, 0.0,
                                     batch_clusters=1, mode=0, debug_flags=2)
    assert out["stats"]["sort_passes"] == 1


def test_partition_general_variant_large_S():
    """S > 1024 takes the general k3_local variant (pair set + rounds of bitsets)."""
    rng = np.random.default_rng(5)
    items, stroi = _random_items(rng, 1500, 31, 2, 260)
    out, want = _compare_with_oracle(items, stroi, 1500, 31, True, True, False, 0.01,
                                     batch_clusters=2, mode=0)


def test_partition_mode_escalates_on_table_overflow():
    """One sorted byte, > 3072 distinct k-mers under a prefix: the CTA table
    overflows, the library must add sorted bits and still be exact."""
    rng = np.random.default_rng(77)
    comp = str.maketrans("ACGT", "TGCA")
    S = 4
    names = [f"g{i}" for i in range(S)]
    cluster = {}
    for s in names:   # unrelated random sequences: every k-mer is unique
        q = "".join(rng.choice(list("ACGT"), 300000))
        cluster[s] = [ref_port.CutSeq(q, q.translate(comp), s + "_f", "c", 1, 300000, 1, 0)]
    items = [(cluster, "big", np.ones(S, dtype=int))]
    out, want = _compare_with_oracle(items, set(), S, 31, True, False, False, 0.0,
                                     batch_clusters=1, sort_bits=8, mode=0, debug_flags=2)
    assert out["stats"]["sort_passes"] >= 2


def _unrelated_cluster(rng, S, L, name="u"):
    """Every sequence is independent random DNA: no k-mer is shared, so a position
    block holds 16 * S distinct k-mers."""
    comp = str.maketrans("ACGT", "TGCA")
    names = [f"g{i:04d}" for i in range(S)]
    cluster = {}
    for s in names:
        q = "".join(rng.choice(list("ACGT"), L))
        cluster[s] = [ref_port.CutSeq(q, q.translate(comp), s + "_f", "c", 1, L, 1, 0)]
    return (cluster, name, np.ones(S, dtype=int))


def test_block_engine_grows_its_table():
    """16 * 150 = 2400 distinct k-mers per block: the first table (256 slots) overflows,
    the overflowing blocks are rerun with tables of 512 ... 4096 slots until they fit, and
    the batch stays on the block engine."""
    rng = np.random.default_rng(11)
    items = [_unrelated_cluster(rng, 150, 120)]
    out, want = _compare_with_oracle(items, set(), 150, 31, True, False, False, 0.0,
                                     batch_clusters=1)
    assert out["stats"]["engine"] == 2
    assert out["stats"]["block_slots"] >= 512     # every block overflowed: next batch starts larger


def test_block_engine_falls_back_to_records():
    """16 * 700 distinct k-mers per block exceed the largest table: the batch is rerun
    through the record path and is still exact."""
    rng = np.random.default_rng(12)
    items = [_unrelated_cluster(rng, 700, 80)]
    out, want = _compare_with_oracle(items, set(), 700, 31, True, False, False, 0.0,
                                     batch_clusters=1)
    assert out["stats"]["engine"] == 0


def test_block_engine_merges_misaligned_copies():
    """Indels, shifted starts and paralogs put the same k-mer into different position
    blocks of different sequences: kB must merge the partial bitsets by key."""
    rng = np.random.default_rng(13)
    comp = str.maketrans("ACGT", "TGCA")
    S, k = 90, 31
    names = [f"g{i:04d}" for i in range(S)]
    items = []
    for c in range(4):
        anc = rng.choice(list("ACGT"), 700)
        presab = np.zeros(S, dtype=int)
        cluster = {}
        for i, s in enumerate(names):
            if rng.random() < 0.15:
                cluster[s] = []
                continue
            presab[i] = 1
            lst = []
            for _ in range(3 if rng.random() < 0.1 else 1):
                q = list(anc[int(rng.integers(0, 40)):700 - int(rng.integers(0, 40))])
                for _ in range(int(rng.integers(0, 4))):        # indels
                    p = int(rng.integers(0, len(q)))
                    if rng.random() < 0.5:
                        del q[p:p + int(rng.integers(1, 9))]
                    else:
                        q[p:p] = list(rng.choice(list("ACGT"), int(rng.integers(1, 9))))
                m = rng.random(len(q)) < 0.003
                q = np.array(q)
                q[m] = rng.choice(list("ACGT"), int(m.sum()))
                q = "".join(q)
                lst.append(ref_port.CutSeq(q, q.translate(comp), s + "_f", "ctg", 11,
                                           10 + len(q), int(rng.choice([1, -1])), 3))
            cluster[s] = lst
        items.append((cluster, f"mis{c}", presab))
    stroi = set(names[:5])
    for canon in (True, False):
        out, want = _compare_with_oracle(items, stroi, S, k, canon, True, False, 0.02,
                                         batch_clusters=3)
        assert out["stats"]["engine"] == 2


@pytest.mark.parametrize("canon,cm", [(True, True), (False, False)])
def test_block_engine_sample_slices(canon, cm):
    """S > 1024: kA works per slice of 512 samples, kB4/kB5 link the slices of a k-mer, sum the
    counts for the MAF window and assemble the full-width bitsets."""
    rng = np.random.default_rng(31)
    S = 1300
    items, stroi = _random_items(rng, S, 31, 3, 220)
    out, want = _compare_with_oracle(items, stroi, S, 31, canon, cm, False, 0.01, batch_clusters=2)
    assert out["stats"]["engine"] == 2


def test_block_engine_sample_slices_10k():
    """BASELINE config #4's sample count on short clusters (the oracle's limit)."""
    rng = np.random.default_rng(32)
    S = 10000
    items, stroi = _random_items(rng, S, 31, 2, 90)
    out, want = _compare_with_oracle(items, set(), S, 31, True, False, False, 0.01, batch_clusters=2)
    assert out["stats"]["engine"] == 2


def test_block_engine_sample_slices_50k_consider_missing():
    """BASELINE config #5's sample count with the cluster-absent encoding (NaN plane, MAF over
    the present samples only) on short clusters (the oracle's limit), against the C oracle."""
    rng = np.random.default_rng(33)
    S = 50000
    items, stroi = _random_items(rng, S, 31, 2, 80)
    out, want = _compare_with_oracle(items, set(), S, 31, True, True, False, 0.01, batch_clusters=2)
    assert out["stats"]["engine"] == 2


@pytest.mark.parametrize("smem_kb,S", [("0", 90), ("2", 90), ("2", 1300)])
def test_block_engine_merge_spills_to_global_table(smem_kb, S, monkeypatch):
    """kB1_local merges a cluster's partial rows in shared memory; a cluster with more rows than
    its table holds goes through the global-memory table instead (kB1_insert).  With the table cut
    to 0 / 2 KB every / the larger (cluster, slice) takes that path; results must not change
    (paralogs and the 0 / 5 base offsets of the random clusters put k-mers into several runs)."""
    monkeypatch.setenv("PF_MERGE_SMEM_KB", smem_kb)
    rng = np.random.default_rng(41)
    items, stroi = _random_items(rng, S, 31, 6, 300 if S < 1000 else 200)
    out, want = _compare_with_oracle(items, stroi, S, 31, True, False, False, 0.01, batch_clusters=3)
    assert out["stats"]["engine"] == 2


@pytest.mark.parametrize("fp_bits,S", [("0", 90), ("2", 90), ("1", 1300)])
def test_block_engine_merge_fingerprint_mismatches(fp_bits, S, monkeypatch):
    """kB1_local stores a 15-bit fingerprint per table entry and confirms a match on the full key;
    a match between different k-mers must keep probing.  With a 0..2-bit fingerprint nearly every
    probe of an occupied slot is such a match; results must not change."""
    monkeypatch.setenv("PF_MERGE_FP_BITS", fp_bits)
    rng = np.random.default_rng(43)
    items, stroi = _random_items(rng, S, 31, 5, 300 if S < 1000 else 200)
    out, want = _compare_with_oracle(items, stroi, S, 31, True, False, False, 0.01, batch_clusters=3)
    assert out["stats"]["engine"] == 2


@pytest.mark.parametrize("engine", ["block", "records"])
def test_pipelined_submit_matches_oracle(engine, monkeypatch):
    """pf_submit of a batch above the split threshold: sub-batches of whole clusters through
    two device slots (H2D / kernels / D2H overlapped); rows, pattern ids, cluster rows and
    positional records must be those of the one big batch."""
    monkeypatch.setenv("PF_PIPELINE_SEQS", "1024")       # sub-batches of ~1024 sequences
    rng = np.random.default_rng(21)
    S, k = 60, 31
    items, stroi = _random_items(rng, S, k, 70, 260)
    names = sorted(items[0][0].keys())
    empty = ({s: [] for s in names}, "cl_empty", np.zeros(S, dtype=int))
    items = items[:20] + [empty] + items[20:50] + [empty, empty] + items[50:] + [empty]
    out, want = _compare_with_oracle(items, stroi, S, k, True, True, False, 0.02,
                                     batch_clusters=len(items), **ENGINES[engine])
    assert out["stats"]["sub_batches"] >= 3


def test_pipelined_and_plain_submits_share_one_context(monkeypatch):
    """Batches above and below the split threshold alternate on one context: pattern numbering
    continues across pipelined and plain submits, results are those of the oracle."""
    monkeypatch.setenv("PF_PIPELINE_SEQS", "600")
    rng = np.random.default_rng(22)
    S, k = 50, 21
    items, stroi = _random_items(rng, S, k, 90, 200)
    out, want = _compare_with_oracle(items, stroi, S, k, False, False, True, 0.04,
                                     batch_clusters=[40, 3, 35, 12])


def test_pipelined_submit_with_sample_slices(monkeypatch):
    """Pipelined sub-batches through the sample-sliced block engine (S > 1024)."""
    monkeypatch.setenv("PF_PIPELINE_SEQS", "2000")
    rng = np.random.default_rng(23)
    S = 1100
    items, stroi = _random_items(rng, S, 31, 8, 150)
    out, want = _compare_with_oracle(items, stroi, S, 31, True, True, False, 0.01,
                                     batch_clusters=len(items))
    assert out["stats"]["engine"] == 2 and out["stats"]["sub_batches"] >= 2


def test_empty_and_ragged_batches():
    rng = np.random.default_rng(3)
    items, stroi = _random_items(rng, 12, 31, 3, 120)
    # a cluster with no sequences at all, one whose sequences are all shorter than k
    names = sorted(items[0][0].keys())
    empty = ({s: [] for s in names}, "cl_empty", np.zeros(12, dtype=int))
    short_seq = ref_port.CutSeq("ACGTACGTAC", "TGCATGCATG", "x", "c", 1, 10, 1, 0)
    presab = np.zeros(12, dtype=int)
    presab[0] = 1
    short = ({s: ([short_seq] if s == names[0] else []) for s in names},
             "cl_short", presab)
    items = [empty] + items[:1] + [short] + items[1:] + [empty]
    _compare_with_oracle(items, stroi, 12, 31, True, False, False, 0.01,
                         batch_clusters=2)


def test_synthetic_device_batch_matches_oracle():
    """pf_synth_fill batch: CUDA path vs C oracle on the unpacked bases."""
    from panfeed_b200 import capi, packer
    S, C, L, k = 96, 6, 420, 31
    hb = capi.synth_batch(0, 20261018, S, C, total_clusters=C, gene_len=L,
                          all_targets=False)
    # unpack to ASCII for the oracle
    sh = (62 - 2 * np.arange(32)).astype(np.uint64)
    codes = ((hb.packed[:, None] >> sh[None, :]) & np.uint64(3)).astype(np.uint8).ravel()
    ascii_plane = np.frombuffer(b"ACGT", np.uint8)[codes]
    seqs = np.zeros(len(hb.seqs), oracle_c.SEQ_DTYPE)
    for f in ("len", "cluster", "sample", "start", "end", "offset", "strand"):
        seqs[f] = hb.seqs[f]
    seqs["off"] = hb.seqs["base_off"]
    idx = np.arange(S)
    presab = ((hb.presence[:, idx >> 5] >> (idx & 31)) & 1).astype(np.uint8)
    want = oracle_c.run_arrays(ascii_plane, seqs, presab, k, True, False, False,
                               0.01, n_threads=4)
    ctx = capi.Context(k, S, maf=0.01)
    try:
        ctx.submit(hb)
        r = ctx.collect()
        st = ctx.stats()
    finally:
        ctx.close()
    assert st["instances"] == want["n_instances"]
    got_rows = sorted(zip(r["row_cluster"].tolist(),
                          packer.kmers_to_str(r["row_kmer"], k).tolist(),
                          r["row_count"].tolist(),
                          [r["new_kmer_patterns"][p].tobytes() for p in r["row_pattern"]]))
    want_rows = sorted(zip(want["row_cluster"].tolist(), want["row_kmer"].tolist(),
                           want["row_count"].tolist(),
                           [want["kmer_pattern_bits"][p].tobytes() for p in want["row_pattern"]]))
    assert len(got_rows) > 100
    assert got_rows == want_rows
    assert len(r["new_kmer_patterns"]) == len(want["kmer_pattern_bits"])
    assert st["unique_kmers"] == want["n_unique"]


@pytest.mark.parametrize("engine", ["block", "records"])
def test_malformed_batches_are_refused_with_the_same_message(engine):
    """Descriptor validation runs on the device (plan_from_raw), whether the context plans for the
    block engine or plans record offsets at upload (debug_flags=2): a malformed batch is refused
    with one message naming the first bad sequence, and the context stays usable."""
    from panfeed_b200 import capi
    S, C, L, k = 40, 3, 200, 31
    good = capi.synth_batch(0, 5, S, C, total_clusters=C, gene_len=L)
    ctx = capi.Context(k, S, maf=0.01, debug_flags=ENGINES[engine]["debug_flags"])
    try:
        cases = []
        bad = capi.HostBatch(good.packed, good.seqs.copy(), good.clusters, good.presence.copy())
        s = int(bad.seqs["sample"][7])
        c = int(bad.seqs["cluster"][7])
        bad.presence[c, s >> 5] &= ~np.uint32(1 << (s & 31))
        cases.append((bad, f"seq 7: sample {s} is not marked present in cluster {c}"))
        bad = capi.HostBatch(good.packed, good.seqs.copy(), good.clusters, good.presence)
        bad.seqs["strand"][11] = 0
        cases.append((bad, "seq 11: strand must be +1/-1"))
        bad = capi.HostBatch(good.packed, good.seqs.copy(), good.clusters, good.presence)
        bad.seqs["base_off"][5] += 32
        cases.append((bad, "seq 5: base_off must be a multiple of 64"))
        bad = capi.HostBatch(good.packed, good.seqs.copy(), good.clusters, good.presence)
        bad.seqs["len"][len(bad.seqs) - 1] += 4096
        cases.append((bad, f"seq {len(bad.seqs) - 1}: bases run past the packed plane"))
        bad = capi.HostBatch(good.packed, good.seqs.copy(), good.clusters, good.presence)
        j = int(np.nonzero(bad.seqs["cluster"] == 1)[0][3])       # a sequence inside cluster 1 claims cluster 0
        bad.seqs["cluster"][j] = 0
        cases.append((bad, f"seq {j}: clusters must be non-decreasing"))
        # sequence 9 flagged as holding N/IUPAC symbols, against a 4-bit plane that covers it
        n_sym = int(good.seqs["len"][9] + 63) // 64 * 64
        for amb_off, amb_words, msg in ((16, n_sym // 16, "seq 9: amb_off must be a multiple of 32"),
                                        (0, 1, "seq 9: symbols run past the 4-bit plane"),
                                        (0, 0, "seq 9 is ambiguous but amb_codes is NULL")):
            seqs = good.seqs.copy()
            seqs["flags"][9] |= 2
            seqs["amb_off"][9] = amb_off
            amb = np.zeros(amb_words, np.uint64) if amb_words else None
            cases.append((capi.HostBatch(good.packed, seqs, good.clusters, good.presence, amb), msg))
        for hb, msg in cases:
            with pytest.raises(capi.PfError) as e:
                ctx.submit(hb)
            assert str(e.value).split(": ", 1)[1] == msg, (msg, str(e.value))
        ctx.submit(good)
        r = ctx.collect()
        assert len(r["row_cluster"]) > 0
    finally:
        ctx.close()


def _related_cluster(rng, S, L, name):
    """Every sample carries one copy of one of three close founders: a position block holds a
    few dozen distinct k-mers."""
    comp = str.maketrans("ACGT", "TGCA")
    anc = rng.choice(list("ACGT"), L)
    founders = []
    for _ in range(3):
        f = anc.copy()
        m = rng.random(L) < 0.02
        f[m] = rng.choice(list("ACGT"), int(m.sum()))
        founders.append("".join(f))
    cluster = {}
    for i in range(S):
        q = founders[int(rng.integers(3))]
        cluster[f"g{i:04d}"] = [ref_port.CutSeq(q, q.translate(comp), f"g{i:04d}_f", "c", 1, L, 1, 0)]
    return (cluster, name, np.ones(S, dtype=int))


def test_pipelined_submit_with_two_consecutive_fallbacks(monkeypatch):
    """Sub-batches 1 and 2 fall back from the block engine to the records; the second fall-back
    turns the block engine off for the context while sub-batch 3 has already been uploaded with a
    block plan only.  That sub-batch must still run through the record engine, exactly."""
    monkeypatch.setenv("PF_PIPELINE_SEQS", "1024")       # one 700-sequence cluster per sub-batch
    rng = np.random.default_rng(24)
    S, k = 700, 31
    items = ([_related_cluster(rng, S, 200, "r0")]
             + [_unrelated_cluster(rng, S, 80, f"u{i}") for i in range(2)]
             + [_related_cluster(rng, S, 200, f"r{i}") for i in range(1, 4)])
    out, want = _compare_with_oracle(items, set(), S, k, True, False, False, 0.0,
                                     batch_clusters=len(items))
    assert out["stats"]["sub_batches"] >= 4


@pytest.mark.parametrize("canon", [True, False])
def test_pipelined_submit_compact_positions(canon, monkeypatch):
    """The compact positional form (emit_positions = 2: one used_strand bit per window) through a
    pipelined submit (device-planned sub-batches, the bit plane copied slice by slice) against the
    21-byte record form of the same batch (host-planned, plain): every record's strand bit, and
    the kmers.tsv text both forms format, must agree."""
    from panfeed_b200 import capi
    monkeypatch.setenv("PF_PIPELINE_SEQS", "1500")
    S, C, L, k = 48, 120, 260, 21
    hb = capi.synth_batch(0, 77, S, C, total_clusters=C, gene_len=L, all_targets=True)
    hb.seqs["flags"][::3] = 0                      # a third of the sequences are not targets
    res = {}
    for mode in (2, 1):
        ctx = capi.Context(k, S, canonical=canon, emit_positions=mode, maf=0.02)
        try:
            ctx.submit(hb)
            res[mode] = (ctx.collect(), ctx.stats())
        finally:
            ctx.close()
    (rc, stc), (rr, st) = res[2], res[1]
    assert stc["sub_batches"] >= 3
    nwin = np.maximum(hb.seqs["len"].astype(np.int64) - k + 1, 0)
    n_target = int(nwin[(hb.seqs["flags"] & 1) != 0].sum())
    assert rc["n_pos"] == rr["n_pos"] == n_target
    leads = [f"c{int(q['cluster'])}\ts{int(q['sample'])}\tg{i}\tctg\t{int(q['strand'])}\t".encode()
             for i, q in enumerate(hb.seqs)]
    a = capi.format_positions_compact(hb, rc["pos_strand_bits"], k, canon, leads)
    b = capi.format_positions(rr, k, canon, leads, hb.seqs["strand"])
    assert len(a) > 0 and sorted(a.split(b"\n")) == sorted(b.split(b"\n"))
    assert np.array_equal(np.sort(rc["row_kmer"]), np.sort(rr["row_kmer"]))
