"""The host side of k = 33..64 with N/IUPAC symbols: 4-word k-mers (4 bits per symbol) in the
row formatter (xwide rows after a cluster's wide rows), in the positional formatter (pos_flags
bit 2 -> pos_xwide_kmer) and in packer's decoder, against plain Python renderings.  No GPU."""
import numpy as np
import pytest

from panfeed_b200 import capi, packer

_COMP = bytes.maketrans(b"ACTGNYRWSKMDVHBX", b"TGACNRYWSMKHBDVX")


def _pack4_words(s, n_words):
    v = 0
    for ch in s:
        v = (v << 4) | capi.AMB_ALPHABET.index(ch)
    return [(v >> (64 * (n_words - 1 - i))) & ((1 << 64) - 1) for i in range(n_words)]


def _pack2_words(s):
    v = 0
    for ch in s:
        v = (v << 2) | "ACGT".index(ch)
    return [v >> 64, v & ((1 << 64) - 1)]


@pytest.mark.parametrize("k", [1, 17, 33, 48, 63, 64])
def test_four_word_decoder_matches_python(k):
    rng = np.random.default_rng(k)
    texts = ["".join(rng.choice(list(capi.AMB_ALPHABET), k)) for _ in range(200)]
    words = np.array([_pack4_words(t, 4) for t in texts], np.uint64)
    got = packer.wide_kmers_to_str(words, k, 4)
    assert [x.decode() for x in got] == texts


@pytest.mark.parametrize("k", [5, 32, 33, 64])
def test_two_word_decoder_is_unchanged(k):
    """n_words defaults to 2: 4 bits per symbol up to k = 32, 2 bits per base above."""
    rng = np.random.default_rng(100 + k)
    alphabet = list(capi.AMB_ALPHABET) if k <= 32 else list("ACGT")
    texts = ["".join(rng.choice(alphabet, k)) for _ in range(100)]
    words = np.array([_pack4_words(t, 2) if k <= 32 else _pack2_words(t) for t in texts], np.uint64)
    assert [x.decode() for x in packer.wide_kmers_to_str(words, k)] == texts
    assert packer.wide_kmers_to_str(np.zeros((0, 2), np.uint64), k).shape == (0,)


@pytest.mark.parametrize("k", [33, 40, 64])
@pytest.mark.parametrize("threads", [1, 4])
def test_kmer_rows_with_xwide_rows_match_python(k, threads):
    """Per cluster: header, (no narrow rows at k > 32), wide rows sorted by k-mer, then xwide rows
    sorted by k-mer (the reference's rows of a cluster, in an order of our own)."""
    rng = np.random.default_rng(k * 10 + threads)
    nc, nw, nx = 17, 3000 if threads > 1 else 400, 900 if threads > 1 else 120
    ids = np.array([("%022d==" % i).encode() for i in range(600)], "S24")
    cids = np.array([("c%021d==" % i).encode() for i in range(30)], "S24")
    tags = [str(int(x)).encode() for x in rng.integers(0, 100000, nc)]
    wtext = ["".join(rng.choice(list("ACGT"), k)) for _ in range(nw)]
    xtext = ["".join(rng.choice(list("ACGTNRYK"), k)) for _ in range(nx)]
    r = {"cluster_pattern": rng.integers(0, 30, nc).astype(np.uint32),
         "row_cluster": np.zeros(0, np.uint32), "row_kmer": np.zeros(0, np.uint64),
         "row_pattern": np.zeros(0, np.uint32),
         "wide_row_cluster": rng.integers(0, nc, nw).astype(np.uint32),
         "wide_row_kmer": np.array([_pack2_words(t) for t in wtext], np.uint64),
         "wide_row_pattern": rng.integers(0, 600, nw).astype(np.uint32),
         "xwide_row_cluster": rng.integers(0, nc - 1, nx).astype(np.uint32),    # the last cluster has none
         "xwide_row_kmer": np.array([_pack4_words(t, 4) for t in xtext], np.uint64),
         "xwide_row_pattern": rng.integers(0, 600, nx).astype(np.uint32)}
    got, off = capi.format_kmer_rows(r, k, tags, ids, cids, n_threads=threads)
    want = []
    for c, tag in enumerate(tags):
        want.append(tag + b"\t\t" + cids[r["cluster_pattern"][c]] + b"\n")
        for cl, text, pat in (("wide_row_cluster", wtext, "wide_row_pattern"),
                              ("xwide_row_cluster", xtext, "xwide_row_pattern")):
            sel = sorted(np.flatnonzero(r[cl] == c).tolist(), key=lambda i: (text[i], i))
            want += [tag + b"\t" + text[i].encode() + b"\t" + ids[r[pat][i]] + b"\n" for i in sel]
    assert got == b"".join(want)
    assert int(off[-1]) == len(got)
    # a bad pattern index of an xwide row is refused like one of any other row
    r["xwide_row_pattern"] = r["xwide_row_pattern"].copy()
    r["xwide_row_pattern"][0] = 600
    with pytest.raises(capi.PfError):
        capi.format_kmer_rows(r, k, tags, ids, cids)


@pytest.mark.parametrize("k", [33, 48, 64])
@pytest.mark.parametrize("canonical", [True, False])
def test_position_rows_with_flag_bit_2_match_python(k, canonical):
    """pos_flags bit 1: pos_kmer indexes pos_wide_kmer (2 bits per base); bit 2: it indexes
    pos_xwide_kmer (4 bits per symbol)."""
    rng = np.random.default_rng(7 * k + canonical)
    n, n_seqs = 5000, 23
    leads = [f"cl{i % 4}\tstrain_{i}\tgene{i}\tctg{i % 3}\t{s}\t".encode()
             for i, s in enumerate(rng.choice([1, -1], n_seqs))]
    strand = np.array([int(x.split(b"\t")[4]) for x in leads], np.int32)
    kmers, flags, wide, xwide, texts = [], [], [], [], []
    for _ in range(n):
        used = int(rng.integers(0, 2))
        if rng.random() < 0.1:
            t = "".join(rng.choice(list("ACGTNRYKMSWBDHVX"), k))
            kmers.append(len(xwide))
            xwide.append(_pack4_words(t, 4))
            flags.append(4 | used)
        else:
            t = "".join(rng.choice(list("ACGT"), k))
            kmers.append(len(wide))
            wide.append(_pack2_words(t))
            flags.append(2 | used)
        texts.append(t)
    r = {"pos_kmer": np.array(kmers, np.uint64), "pos_seq": rng.integers(0, n_seqs, n).astype(np.uint32),
         "pos_contig_start": rng.integers(-50, 5_000_000, n).astype(np.int32),
         "pos_gene_start": rng.integers(-300, 3000, n).astype(np.int32),
         "pos_flags": np.array(flags, np.uint8),
         "pos_wide_kmer": np.array(wide, np.uint64).reshape(-1, 2),
         "pos_xwide_kmer": np.array(xwide, np.uint64).reshape(-1, 4)}
    got = capi.format_positions(r, k, canonical, leads, strand, n_threads=3)
    want = []
    for i in range(n):
        s = int(r["pos_seq"][i])
        c0, g0 = int(r["pos_contig_start"][i]), int(r["pos_gene_start"][i])
        head = leads[s].decode() + f"{c0}\t{c0 + k}\t{g0}\t{g0 + k}\t"
        if canonical:
            want.append(f"{head}{-1 if r['pos_flags'][i] & 1 else 1}\t{texts[i]}\n")
        else:
            st = int(strand[s])
            rc = texts[i].encode().translate(_COMP)[::-1].decode()
            want.append(f"{head}{st}\t{texts[i]}\n{head}{-st}\t{rc}\n")
    assert got.decode() == "".join(want)
