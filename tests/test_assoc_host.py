"""Host side of --associations, no GPU: pattern ids back to the MD5 digests the device looks up,
and pf_format_annotated against pandas' own join (get_kmers.py:108-145) of the same rows."""
import io

import numpy as np
import pandas as pd
import pytest

from panfeed_b200 import assoc, capi
from panfeed_b200.__main__ import main
from panfeed_b200.panfeed import pattern_id

import helpers


def test_id_digest_round_trip():
    rng = np.random.default_rng(11)
    vecs = [rng.integers(0, 2, rng.integers(1, 90)).astype(dt) for dt in (np.int64, np.float64) for _ in range(40)]
    ids = [pattern_id(v) for v in vecs]
    bad = ["", "abc", "x" * 24, ids[0][:23], ids[1] + "A", "!" * 22 + "=="]
    digests, keep = capi.id_digests(ids + bad)
    assert keep.tolist() == list(range(len(ids)))
    assert capi.base64_ids(digests).astype(str).tolist() == ids
    import hashlib
    assert digests[0].tobytes() == hashlib.md5(vecs[0].view(np.uint8)).digest()


def test_associations_refused_with_multiple_files(tmp_path):
    with pytest.raises(SystemExit) as e:
        main(helpers.modes()["updownstream"] + ["--associations", "x.tsv", "--multiple-files",
                                                 "--output", str(tmp_path / "o")])
    assert e.value.code == 1


ACGT = np.frombuffer(b"ACGT", np.uint8)


def _batch(rng, k, canonical):
    """A small random batch of target (and non-target) sequences, its rows, strand bits and the
    kmers.tsv frame of its target windows."""
    n_clusters, L = 4, 40
    seqs = np.zeros(10, capi.SEQ_DTYPE)
    texts = []
    for i in range(len(seqs)):
        n = int(rng.integers(k, L))
        texts.append(ACGT[rng.integers(0, 4, n)].tobytes())
    seq_off = np.zeros(len(texts) + 1, np.uint64)
    np.cumsum([len(t) for t in texts], out=seq_off[1:])
    packed, base_off, _, _, _ = capi.pack_blob(b"".join(texts), seq_off)
    seqs["base_off"] = base_off
    seqs["len"] = [len(t) for t in texts]
    seqs["cluster"] = np.arange(len(seqs)) % n_clusters
    seqs["flags"] = np.where(np.arange(len(seqs)) % 5 == 4, 0, capi.PF_SEQ_TARGET)
    seqs["start"] = rng.integers(1, 500, len(seqs))
    seqs["end"] = seqs["start"] + seqs["len"] - 1
    seqs["offset"] = rng.integers(0, 30, len(seqs))
    seqs["strand"] = np.where(rng.random(len(seqs)) < 0.5, 1, -1)
    hb = capi.HostBatch(packed, seqs, np.zeros(n_clusters, capi.CLUSTER_DTYPE), np.zeros((n_clusters, 1), np.uint32))
    comp = bytes.maketrans(b"ACGT", b"TGCA")
    bits = np.zeros(max(1, packed.size), np.uint32)
    kmers = {}                     # (cluster, k-mer) -> row
    pos = []
    for i, t in enumerate(texts):
        c = int(seqs["cluster"][i])
        for p in range(len(t) - k + 1):
            f = t[p:p + k]
            r = f.translate(comp)[::-1]
            outs = []
            if canonical:
                use_rc = r < f
                if use_rc:
                    j = int(base_off[i]) + p
                    bits[j >> 5] |= np.uint32(1 << (j & 31))
                outs.append((r if use_rc else f, -1 if use_rc else 1, 0))
            else:
                outs += [(f, int(seqs["strand"][i]), 0), (r, -int(seqs["strand"][i]), 1)]
            for km, used, o in outs:
                kmers.setdefault((c, km), len(kmers))
                if seqs["flags"][i] & capi.PF_SEQ_TARGET:
                    s = int(seqs["strand"][i])
                    c0 = int(seqs["start"][i]) + p if s > 0 else int(seqs["end"][i]) - p - k
                    g0 = p - int(seqs["offset"][i])
                    pos.append((c, km, i, p, o, s, c0, g0, used))
    extra = [(int(c), ACGT[rng.integers(0, 4, k)].tobytes()) for c in rng.integers(0, n_clusters, 5)]
    for key in extra:                          # rows that no target window carries
        kmers.setdefault(key, len(kmers))
    keys = list(kmers)
    enc = lambda s: int("".join("%d" % b"ACGT".index(x) for x in s), 4)   # noqa: E731
    r = {"row_cluster": np.array([c for c, _ in keys], np.uint32),
         "row_kmer": np.array([enc(km) for _, km in keys], np.uint64),
         "wide_row_cluster": np.zeros(0, np.uint32), "wide_row_kmer": np.zeros((0, 2), np.uint64),
         "xwide_row_cluster": np.zeros(0, np.uint32), "xwide_row_kmer": np.zeros((0, 4), np.uint64),
         "pos_strand_bits": bits}
    return hb, r, kmers, pos


@pytest.mark.parametrize("only_passing", [False, True])
@pytest.mark.parametrize("k, canonical", [(7, True), (5, False), (31, True)])
def test_format_annotated_matches_pandas_join(k, canonical, only_passing):
    rng = np.random.default_rng(k * 10 + canonical + 2 * only_passing)
    hb, r, kmers, pos = _batch(rng, k, canonical)
    n_clusters = len(hb.clusters)
    keys = list(kmers)
    # patterns: each row a random pattern id; cluster rows their own; ~30 % of both pass
    n_assoc = 12
    ids = ["%022d==" % i for i in range(40)]
    row_hash = [ids[int(x)] for x in rng.integers(0, 40, len(keys))]
    cluster_hash = [ids[int(x)] for x in rng.integers(0, 40, n_clusters)]
    passing = sorted(set(rng.choice(40, n_assoc, replace=False).tolist()))
    a = pd.DataFrame({"af": rng.random(len(passing)).round(3), "count": rng.integers(0, 9, len(passing)),
                      "note": ["n%d" % i for i in range(len(passing))]}, index=[ids[i] for i in passing])
    a.index.name = "hashed_pattern"
    arow = {h: j for j, h in enumerate(a.index)}
    tags = [b"cl%d" % c for c in range(n_clusters)]
    # what the device returns
    window, window_assoc, seen = [], [], set()
    for c, km, i, p, o, *_ in pos:
        h = row_hash[kmers[(c, km)]]
        if h in arow:
            window.append(((int(hb.seqs["base_off"][i]) + p) << 1 | o))
            window_assoc.append(arow[h])
            seen.add(kmers[(c, km)])
    cl_assoc = np.array([arow.get(h, capi.PF_ASSOC_NONE) for h in cluster_hash], np.uint32)
    prow = [j for j in range(len(keys)) if row_hash[j] in arow]
    cl_pass = np.array([cl_assoc[c] != capi.PF_ASSOC_NONE or any(keys[j][0] == c for j in prow)
                        for c in range(n_clusters)], np.uint8)
    res = {"window": np.array(window, np.uint64), "window_assoc": np.array(window_assoc, np.uint32),
           "cluster_pass": cl_pass, "cluster_assoc": cl_assoc, "row": np.array(prow, np.uint32),
           "row_assoc": np.array([arow[row_hash[j]] for j in prow], np.uint32),
           "row_seen": np.array([j in seen for j in prow], np.uint8)}
    leads = [b"s%d\tf%d\tctg%d\t" % (i, i, i) for i in range(len(hb.seqs))]
    # pandas: the reference's join over the same three tables
    h = pd.DataFrame({"cluster": [tags[c].decode() for c, _ in keys] + [t.decode() for t in tags],
                      "k-mer": [km.decode() for _, km in keys] + [np.nan] * n_clusters,
                      "hashed_pattern": row_hash + cluster_hash})
    h = h[h["hashed_pattern"].isin(arow)].set_index("hashed_pattern")
    kt = pd.DataFrame([(tags[c].decode(), km.decode(), "s%d" % i, "f%d" % i, "ctg%d" % i, s, c0, c0 + k, g0, g0 + k, u)
                       for c, km, i, p, o, s, c0, g0, u in pos if cl_pass[c]],
                      columns=["cluster", "k-mer", "strain", "feature_id", "contig", "feature_strand", "contig_start",
                               "contig_end", "gene_start", "gene_end", "strand"]).set_index(["cluster", "k-mer"])
    b = a.join(h, how="inner").reset_index().set_index(["cluster", "k-mer"])
    b = b.join(kt, how="left" if only_passing else "right")
    buf = io.StringIO()
    b.to_csv(buf, sep="\t")
    want = buf.getvalue()
    # the native formatter with the upcast pandas applied (known from the frame here)
    if only_passing:
        upcast = bool(b["strain"].isna().any())
        flags = capi.PF_ANNOT_ONLY_PASSING | (capi.PF_ANNOT_FLOAT_POSITIONS if upcast else 0)
        snips = assoc.snippets(a, False)
    else:
        upcast = bool(b["af"].isna().any())
        flags = 0
        snips = assoc.snippets(a, upcast)
    got = capi.format_annotated(hb, r["pos_strand_bits"], k, canonical, r, res, tags, leads, snips,
                                1 + len(a.columns), flags).decode()
    head = want.split("\n")[0]
    assert head == "\t".join(["cluster", "k-mer", "hashed_pattern"] + list(a.columns) + assoc.POSITIONAL)
    assert sorted(got.split("\n")[:-1]) == sorted(want.split("\n")[1:-1])
    if only_passing:
        assert upcast and ".0\t" in got
    else:
        assert upcast and "\t\t\t\t" in got
