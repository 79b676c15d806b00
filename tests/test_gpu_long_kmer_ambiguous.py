"""k-mers of 33..64 bases on sequences holding N/IUPAC symbols: the windows that touch a non-ACGT
symbol go through 256-bit records (4 bits per symbol), the others through the 128-bit ones.
Everything is checked against the C oracle (random clusters, edge cases) or the reference port
(the CLI on the whole fixture, ambiguous clusters included)."""
import gzip
import os

import numpy as np
import pytest

import helpers
import render
from oracle import oracle_c, ref_port
from panfeed_b200 import capi, packer
from test_gpu_parity import _random_items, _render_gpu

pytestmark = pytest.mark.gpu

_COMP = str.maketrans("ACGTNRYKMSWBDHVX", "TGCANYRMKSWVHDBX")
ENGINES = {"records": dict(mode=0, debug_flags=2), "fullsort": dict(mode=1, debug_flags=2)}


def _run_gpu(items, stroi, S, k, canonical, consider_missing, cluster_equal_filter, maf,
             batch_clusters, mode, debug_flags):
    """items -> the dict gpu_util.run_gpu returns (the layout gpu_util.kmers_tsv_lines and
    test_gpu_parity._render_gpu read), with every row section of a k > 32 batch: the wide rows
    (2 bits per base) and the xwide rows (k-mers holding N/IUPAC symbols, 4 words of 4-bit
    symbols), and positional k-mers taken from pos_wide_kmer (flag bit 1) or pos_xwide_kmer
    (flag bit 2)."""
    ctx = capi.Context(k, S, canonical, consider_missing, cluster_equal_filter,
                       emit_positions=bool(stroi), maf=maf, mode=mode, debug_flags=debug_flags)
    cols = {n: [] for n in ("row_cluster", "row_kmer", "row_count", "row_pattern", "cluster_pattern",
                            "kp", "cp", "pos", "ids", "seq_meta", "seqs", "seq_cluster_idx")}
    seq_base = 0
    try:
        for b0 in range(0, len(items), batch_clusters):
            chunk = items[b0:b0 + batch_clusters]
            pcs = [packer.PackedCluster(c, idx, pa, stroi) for c, idx, pa in chunk]
            hb, meta, ids = packer.pack_batch(pcs, list(range(b0, b0 + len(chunk))))
            ctx.submit(hb)
            r = ctx.collect()
            assert r["kmer_pattern_base"] == sum(len(x) for x in cols["kp"])
            for sec, words in (("wide_", 2), ("xwide_", 4)):
                cols["row_cluster"].append(r[sec + "row_cluster"])
                cols["row_kmer"].append(packer.wide_kmers_to_str(r[sec + "row_kmer"], k, words))
                cols["row_count"].append(r[sec + "row_count"])
                cols["row_pattern"].append(r[sec + "row_pattern"])
            assert len(r["row_cluster"]) == 0                     # no one-word k-mers above 32 bases
            cols["cluster_pattern"].append(r["cluster_pattern"])
            cols["kp"].append(r["new_kmer_patterns"])
            cols["cp"].append(r["new_cluster_patterns"])
            fl = r["pos_flags"]
            kmer_s = np.zeros(len(fl), f"S{k}")
            for bit, arr, words in ((2, "pos_wide_kmer", 2), (4, "pos_xwide_kmer", 4)):
                sel = (fl & bit) != 0
                if sel.any():
                    kmer_s[sel] = packer.wide_kmers_to_str(r[arr], k, words)[r["pos_kmer"][sel].astype(np.int64)]
            assert (((fl & 2) != 0) ^ ((fl & 4) != 0)).all()       # every record names exactly one array
            cols["pos"].append((r["pos_seq"].astype(np.int64) + seq_base, kmer_s, r["pos_contig_start"],
                                r["pos_gene_start"], fl))
            cols["ids"] += ids
            cols["seq_cluster_idx"] += [ids[c] for c in hb.seqs["cluster"]]
            cols["seq_meta"] += meta
            cols["seqs"].append(hb.seqs)
            seq_base += len(hb.seqs)
        stats = ctx.stats()
    finally:
        ctx.close()
    W = (S + 31) // 32
    kp = np.concatenate(cols["kp"])
    return {"row_cluster": np.concatenate(cols["row_cluster"]), "row_kmer": np.concatenate(cols["row_kmer"]),
            "row_count": np.concatenate(cols["row_count"]), "row_pattern": np.concatenate(cols["row_pattern"]),
            "cluster_pattern": np.concatenate(cols["cluster_pattern"]), "ids": cols["ids"],
            "seq_meta": cols["seq_meta"], "seqs": np.concatenate(cols["seqs"]), "stats": stats,
            "seq_cluster_idx": cols["seq_cluster_idx"], "kmer_pattern_bits": kp[:, :W],
            "kmer_pattern_cluster": kp[:, W] if consider_missing else np.full(len(kp), 0xffffffff, np.uint32),
            "cluster_pattern_bits": np.concatenate(cols["cp"]), "pos": cols["pos"]}


def _compare_with_oracle(items, stroi, S, k, canon, cm, nf, maf, batch_clusters, mode, debug_flags):
    """All three files of the GPU path against the C oracle's, after sorting."""
    want = oracle_c.run(items, stroi, k, canon, cm, nf, maf, n_threads=4)
    w = dict(want)
    w["row_kmer"] = [x.decode() for x in want["row_kmer"]]
    w["pos_kmer"] = [x.decode() for x in want["pos_kmer"]]
    want_lines = render.render(w, want["ids"], want["seq_meta"], want["seqs"], S, k, cm, canon)
    out = _run_gpu(items, stroi, S, k, canon, cm, nf, maf, batch_clusters, mode, debug_flags)
    got = _render_gpu(out, S, k, cm, canon)
    for name in helpers.FILES:
        assert sorted(got[name]) == sorted(want_lines[name]), name
    return out, want


def _has_ambiguous_row(out):
    return any(set(x.decode()) - set("ACGT") for x in out["row_kmer"])


def _shared_sites(items, rng, n_sites=2, frac=0.5):
    """A random N/IUPAC symbol is carried by one sample and rarely passes the MAF filter: put a few
    symbols at the same positions of about half the sequences of every cluster as well."""
    comp = str.maketrans("ACGTN", "TGCAN")              # (the convention of _random_items)
    out = []
    for cluster, idx, presab in items:
        L = min((len(cs.sequence) for lst in cluster.values() for cs in lst), default=0)
        sites = rng.integers(0, L, n_sites).tolist() if L else []
        syms = rng.choice(list("NRYK"), n_sites).tolist()
        new = {}
        for s, lst in cluster.items():
            new[s] = []
            for cs in lst:
                q = list(cs.sequence)
                if rng.random() < frac:
                    for p, c in zip(sites, syms):
                        q[p] = c
                q = "".join(q)
                new[s].append(cs._replace(sequence=q, compsequence=q.translate(comp)))
        out.append((new, idx, presab))
    return out


CASES = [
    # S,    k, clusters, L,  canon, cm,    nf,    maf,  amb,   batch, engine
    (40,   33, 4, 300, True,  False, False, 0.01, 0.01,  2, "records"),
    (40,   40, 4, 300, False, False, False, 0.01, 0.01,  2, "fullsort"),
    (129,  48, 3, 300, True,  True,  False, 0.05, 0.006, 3, "records"),
    (129,  63, 3, 260, False, True,  True,  0.02, 0.006, 1, "fullsort"),
    (40,   64, 3, 260, True,  False, True,  0.01, 0.01,  3, "fullsort"),
    (40,   64, 3, 260, False, True,  False, 0.0,  0.01,  3, "records"),
    # W > 32 (maf 0 keeps the k-mers over the random, one-sample symbols too)
    (1500, 48, 2, 160, True,  True,  False, 0.01, 0.003, 2, "records"),
    (1500, 40, 2, 140, False, False, True,  0.0,  0.003, 1, "fullsort"),
]


@pytest.mark.parametrize("case", CASES, ids=[str(i) for i in range(len(CASES))])
def test_random_ambiguous_clusters_match_oracle(case):
    """Random clusters whose sequences carry N/R/Y/K symbols, with target sequences, against the C
    oracle: all three files, and the number of distinct (cluster, k-mer) pairs."""
    S, k, nc, L, canon, cm, nf, maf, amb, bc, engine = case
    rng = np.random.default_rng(4000 + S * 7 + k)
    items, stroi = _random_items(rng, S, k, nc, L, amb)
    items = _shared_sites(items, rng)
    out, want = _compare_with_oracle(items, stroi, S, k, canon, cm, nf, maf,
                                     batch_clusters=bc, **ENGINES[engine])
    assert out["stats"]["engine"] == (1 if engine == "fullsort" else 0)
    assert _has_ambiguous_row(out)
    assert out["stats"]["unique_kmers"] == want["n_unique"]


def _cluster(seqs_by_sample, S, name):
    names = [f"g{i:04d}" for i in range(S)]
    cluster, presab = {}, np.zeros(S, dtype=int)
    for i, s in enumerate(names):
        lst = []
        for j, q in enumerate(seqs_by_sample.get(i, [])):
            lst.append(ref_port.CutSeq(q, q.translate(_COMP), f"{s}_f{j}", "ctg", 11, 10 + len(q),
                                       1 if (i + j) % 2 else -1, 3))
        cluster[s] = lst
        presab[i] = 1 if i in seqs_by_sample else 0
    return (cluster, name, presab), set(names)


def _edge_items(k, rng):
    S = 6
    acgt = lambda n: "".join(rng.choice(list("ACGT"), n))                                   # noqa: E731
    half = acgt(k // 2 - 3) + "NRY"
    pal = half + half.translate(_COMP)[::-1]                                                # fwd == rc
    assert pal == pal.translate(_COMP)[::-1] and len(pal) == k - (k % 2)
    base = acgt(3 * k)
    items, stroi = [], set()
    cases = [
        {0: ["N" * (2 * k)], 1: [base], 2: [base]},                                         # all N
        {0: [base[:k] + "N" * (k + 7) + base[k:]], 1: [base], 3: [base[:k] + "N" * (k + 7) + base[k:]]},
        {1: ["N" + base[1:]], 2: [base[:-1] + "Y"], 4: ["K" + base[1:-1] + "R"]},          # first / last base
        {0: [base[:k // 2] + "N" + base[k // 2 + 1:k]], 5: [base[:k]]},                     # exactly k symbols
        {2: [base[:k] + "RYKM" + base[k:]], 3: [base], 4: [base], 5: [base]},              # one sample only
        {0: [acgt(5) + pal + acgt(9)], 1: [acgt(3) + pal + acgt(20)], 2: ["N" * k]},       # palindromes
    ]
    for c, spec in enumerate(cases):
        item, names = _cluster(spec, S, f"edge{c}")
        items.append(item)
        stroi |= names
    return items, stroi, S


@pytest.mark.parametrize("k", [40, 64])
@pytest.mark.parametrize("canon", [True, False])
def test_edge_cases_match_oracle(k, canon):
    """All-N sequence, an N run longer than k, ambiguous first / last base, a sequence of exactly k
    symbols with one N, an ambiguous k-mer of one sample, ambiguous palindromes (fwd == rc)."""
    rng = np.random.default_rng(k + 2 * canon)
    items, stroi, S = _edge_items(k, rng)
    out, want = _compare_with_oracle(items, stroi, S, k, canon, False, False, 0.0,
                                     batch_clusters=2, mode=0, debug_flags=2)
    assert _has_ambiguous_row(out)
    assert out["stats"]["unique_kmers"] == want["n_unique"]


def test_pattern_shared_by_both_sections_has_one_id():
    """Samples 0 and 1 carry the same sequence with an N in it, samples 2 and 3 other sequences:
    the ACGT k-mers and the N k-mers of samples {0, 1} have one presence pattern, which must get
    one pattern id whether its rows sit in the 128-bit or the 256-bit section."""
    rng = np.random.default_rng(9)
    k, S = 40, 4
    a = "".join(rng.choice(list("ACGT"), 200))
    shared = a[:100] + "N" + a[101:]
    item, _ = _cluster({0: [shared], 1: [shared], 2: ["".join(rng.choice(list("ACGT"), 200))],
                        3: ["".join(rng.choice(list("ACGT"), 200))]}, S, "mix")
    pcs = [packer.PackedCluster(item[0], item[1], item[2], set())]
    hb, _, _ = packer.pack_batch(pcs, [0])
    ctx = capi.Context(k, S, maf=0.0)
    try:
        ctx.submit(hb)
        r = ctx.collect()
    finally:
        ctx.close()
    kp = r["new_kmer_patterns"][:, 0]
    assert len(np.unique(kp)) == len(kp)                       # patterns are numbered once each
    ids_w = set(r["wide_row_pattern"][kp[r["wide_row_pattern"]] == 0b11].tolist())
    ids_x = set(r["xwide_row_pattern"][kp[r["xwide_row_pattern"]] == 0b11].tolist())
    assert len(r["xwide_row_cluster"]) == k                    # the k windows over the N
    assert len(ids_w) == 1 and ids_w == ids_x


@pytest.mark.parametrize("canon", [True, False])
def test_positional_forms_agree_on_ambiguous_windows(canon):
    """emit_positions 1 (records; k-mers of ambiguous windows in pos_xwide_kmer, flag bit 2) and 2
    (the used_strand bit plane, corrected for ambiguous windows behind the 2-bit kernel) must give
    the same kmers.tsv text for every window, including the strand of ambiguous ones."""
    rng = np.random.default_rng(17 + canon)
    S, k = 30, 48
    items, _ = _random_items(rng, S, k, 5, 300, amb_rate=0.02)
    names = sorted(items[0][0].keys())
    pcs = [packer.PackedCluster(c, idx, pa, set(names)) for c, idx, pa in items]
    hb, _, _ = packer.pack_batch(pcs, list(range(len(items))))
    res = {}
    for mode in (1, 2):
        ctx = capi.Context(k, S, canonical=canon, emit_positions=mode, maf=0.02)
        try:
            ctx.submit(hb)
            res[mode] = ctx.collect()
        finally:
            ctx.close()
    rr, rc = res[1], res[2]
    assert len(rr["pos_xwide_kmer"]) > 0 and ((rr["pos_flags"] & 4) != 0).any()
    assert not ((rr["pos_flags"] & 6) == 6).any()
    leads = [f"c{int(q['cluster'])}\ts{int(q['sample'])}\tg{i}\tctg\t{int(q['strand'])}\t".encode()
             for i, q in enumerate(hb.seqs)]
    a = capi.format_positions_compact(hb, rc["pos_strand_bits"], k, canon, leads)
    b = capi.format_positions(rr, k, canon, leads, hb.seqs["strand"])
    assert len(a) > 0 and sorted(a.split(b"\n")) == sorted(b.split(b"\n"))
    assert any(set(x.rsplit("\t", 1)[1]) - set("ACGT") for x in b.decode().split("\n")[:-1])


def _read(path):
    if os.path.exists(path + ".gz"):
        return gzip.open(path + ".gz", "rt").read()
    return open(path).read()


CLI_MODES = {
    "k40_all": [a for a in helpers.modes()["k40"] if a not in ("--genes", "fixture/genes_acgt.txt")],
    "k64_nc_all": [a for a in helpers.modes()["k64_nc"] if a not in ("--genes", "fixture/genes_acgt.txt")],
    "k33_cm_updown": ["--gff", "fixture/gffs/", "--presence-absence", "fixture/gene_presence_absence.csv",
                      "--targets", "fixture/stroi.txt", "-k", "33", "--consider-missing",
                      "--upstream", "100", "--downstream", "100"],
}


@pytest.mark.parametrize("feeder", ["python", "native"])
@pytest.mark.parametrize("mode", sorted(CLI_MODES))
def test_cli_long_kmers_on_whole_fixture(mode, feeder, tmp_path):
    """The CLI at k > 32 on every fixture cluster (the N run and the IUPAC codes included) against
    the reference port, after sorting."""
    from panfeed_b200.__main__ import main
    args = CLI_MODES[mode]
    assert "--genes" not in args
    out = str(tmp_path / "out")
    cwd = os.getcwd()
    os.chdir(helpers.GOLDEN)
    try:
        main(args + ["--native-feeder" if feeder == "native" else "--python-feeder", "--output", out])
        want = ref_port.run(**helpers.cli_kwargs(args))
    finally:
        os.chdir(cwd)
    k = int(args[args.index("-k") + 1])
    for name in helpers.FILES:
        got = _read(os.path.join(out, name))
        assert helpers.sorted_lines(got) == helpers.sorted_lines(want[name]), (mode, name)
    k2h = _read(os.path.join(out, "kmers_to_hashes.tsv")).split("\n")[1:]
    kmers = [x.split("\t")[1] for x in k2h if x.count("\t") == 2 and x.split("\t")[1]]
    assert kmers and all(len(x) == k for x in kmers)
    assert any("N" in x for x in kmers)
