"""--associations in a sharded run (`torchrun -m panfeed_b200`, one process per GPU) on the CPU: two
or three processes over gloo, each with an oracle-backed stand-in for its GPU context that also
answers pf_assoc_load / pf_assoc_collect.  Every rank joins its own clusters and writes a piece of
annotated_kmers.tsv, the ranks OR their upcast facts, rank 0 merges; the merged table must equal
the unmodified get-kmers' goldens.  The writer's piece mode is also checked on its own: a rank
whose own batches never needed the upcast must print them upcast when another rank's did."""
import gzip
import io
import os

import numpy as np
import pandas as pd
import pytest

import helpers
from cpu_context import OracleContext, decode_batch, encode_kmers
from oracle import oracle_c
from panfeed_b200 import assoc, capi
from panfeed_b200.panfeed import _COMP
from test_assoc_host import _batch
from torchrun_util import torchrun

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
POST = os.path.join(helpers.EXPECTED, "postgwas")
ASSOC = os.path.join(POST, "associations.tsv")
UPDOWN = helpers.modes()["updownstream"]


class AssocOracleContext(OracleContext):
    """OracleContext plus the --associations calls: the K6 result contract of pf_assoc_collect
    (include/panfeed_b200.h) computed on the host from the oracle's rows and positional records."""

    def assoc_load(self, digests):
        self._assoc = {x: i for i, x in enumerate(capi.base64_ids(digests).astype(str).tolist())}
        self._ids = {}

    def _id(self, cluster_namespace, p):
        key = (cluster_namespace, int(p))
        if key not in self._ids:
            self._ids[key] = self.pattern_ids(cluster_namespace, int(p), 1)[0].decode()
        return self._ids[key]

    def collect(self, copy=True):
        hb = self._hb
        out = super().collect(copy)
        out.setdefault("xwide_row_cluster", np.zeros(0, np.uint32))
        out.setdefault("xwide_row_kmer", np.zeros((0, 4), np.uint64))
        bases, seqs = decode_batch(hb)
        idx = np.arange(self.S)
        presab = ((hb.presence[:, idx >> 5] >> (idx & 31)) & 1).astype(np.uint8).reshape(len(hb.clusters), self.S)
        o = oracle_c.run_arrays(bases, seqs, presab, self.k, self.canonical, self.consider_missing,
                                self.cluster_equal_filter, self.maf)
        self._last = (hb, out, o)
        return out

    def assoc_collect(self):
        hb, out, o = self._last
        none = capi.PF_ASSOC_NONE
        narrow = encode_kmers(o["row_kmer"], self.k)[0]
        order = np.concatenate([np.nonzero(narrow)[0], np.nonzero(~narrow)[0]])   # result row -> oracle row
        pats = np.concatenate([out["row_pattern"], out["wide_row_pattern"]])
        row_a = [self._assoc.get(self._id(False, p), none) for p in pats]
        at = {(int(o["row_cluster"][i]), o["row_kmer"][i]): j for j, i in enumerate(order.tolist())}
        cl_assoc = np.array([self._assoc.get(self._id(True, p), none) for p in out["cluster_pattern"]], np.uint32)
        window, window_assoc, seen = [], [], set()
        for si, p, km in zip(o["pos_seq"].tolist(), o["pos_pos"].tolist(), o["pos_kmer"]):
            strands = [km] if self.canonical else [km, km.translate(_COMP)[::-1]]
            for bit, x in enumerate(strands):
                j = at.get((int(hb.seqs["cluster"][si]), x))
                if j is not None and row_a[j] != none:
                    window.append((int(hb.seqs["base_off"][si]) + p) << 1 | bit)
                    window_assoc.append(row_a[j])
                    seen.add(j)
        rows = [j for j in range(len(order)) if row_a[j] != none]
        cl_pass = cl_assoc != none
        for j in rows:
            cl_pass[int(o["row_cluster"][order[j]])] = True
        return {"window": np.array(window, np.uint64), "window_assoc": np.array(window_assoc, np.uint32),
                "cluster_pass": cl_pass.astype(np.uint8), "cluster_assoc": cl_assoc,
                "row": np.array(rows, np.uint32), "row_assoc": np.array([row_a[j] for j in rows], np.uint32),
                "row_seen": np.array([j in seen for j in rows], np.uint8)}


WORKER = r'''
import os, sys
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, os.path.join(sys.argv[1], "tests"))
from test_assoc_sharded_host import AssocOracleContext
from panfeed_b200 import capi
capi.Context = AssocOracleContext
from panfeed_b200.__main__ import main
main(sys.argv[2:])
'''


def _read(path):
    if os.path.exists(path + ".gz"):
        return gzip.open(path + ".gz", "rt").read()
    return open(path).read()


def _lines(text):
    return sorted(x for x in text.split("\n") if x)


def _sharded(args, world, out, port, tmp_path):
    """The CLI as `world` processes over gloo, bounded by a timeout: a rank left waiting in a
    collective fails the test, and torchrun stops every rank (tests/torchrun_util.py)."""
    worker = tmp_path / "worker.py"
    worker.write_text(WORKER)
    env = dict(os.environ, PF_DIST_BACKEND="gloo")
    r = torchrun([str(worker), ROOT] + args + ["--output", str(out)], world, port, helpers.GOLDEN, 300, env)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert not os.path.exists(os.path.join(out, ".parts"))
    assert not os.path.exists(os.path.join(out, "kmers.tsv")) and not os.path.exists(os.path.join(out, "kmers.tsv.gz"))
    return _read(os.path.join(out, "annotated_kmers.tsv"))


CASES = [("kmers_t0.3", ["--association-threshold", "0.3"]),
         ("kmers_t0.3_passing", ["--association-threshold", "0.3", "--only-passing"]),
         ("kmers_t0.1_iter2", ["--association-threshold", "0.1"])]


@pytest.mark.parametrize("world, compress", [(2, False), (3, True)])
@pytest.mark.parametrize("case, extra", CASES)
def test_sharded_matches_reference_get_kmers(case, extra, world, compress, tmp_path):
    out = tmp_path / "out"
    port = 29730 + 2 * [c[0] for c in CASES].index(case) + compress
    got = _sharded(UPDOWN + ["--associations", ASSOC] + extra + (["--compress"] if compress else []),
                   world, out, port, tmp_path)
    want = gzip.open(os.path.join(POST, case + ".txt.gz"), "rt").read()
    assert got.split("\n")[0] == want.split("\n")[0]
    assert _lines(got) == _lines(want)
    if compress:
        assert os.path.exists(out / "annotated_kmers.tsv.gz")
    # kmers_to_hashes / hashes_to_patterns: those of any run of these options (the reference's)
    for name in ("kmers_to_hashes.tsv", "hashes_to_patterns.tsv"):
        got_t, want_t = _read(str(out / name)), helpers.golden("updownstream", name)
        assert got_t.split("\n")[0] == want_t.split("\n")[0]
        assert helpers.sorted_lines(got_t) == helpers.sorted_lines(want_t), name


def _one_process(args, out, monkeypatch):
    from panfeed_b200.__main__ import main
    with monkeypatch.context() as m:
        m.setattr(capi, "Context", AssocOracleContext)
        m.chdir(helpers.GOLDEN)
        main(args + ["--output", str(out)])
    return {name: _read(str(out / name)) for name in
            ("annotated_kmers.tsv", "kmers_to_hashes.tsv", "hashes_to_patterns.tsv")}


def test_ranks_without_clusters_and_nothing_passing(tmp_path, monkeypatch):
    """--genes lists one cluster and three ranks run: two ranks cut no batch and create no context
    before the exchange, yet take part in the OR; the run ends with the one-process run's files.
    A threshold nothing passes: the merged table is the header alone, as in one process."""
    k2h = helpers.golden("updownstream", "kmers_to_hashes.tsv").split("\n")
    genes = tmp_path / "genes.txt"
    genes.write_text(k2h[1].split("\t")[0] + "\n")
    for i, (extra, world) in enumerate([(["--genes", str(genes), "--association-threshold", "0.3"], 3),
                                        (["--genes", str(genes), "--association-threshold", "0.3",
                                          "--only-passing"], 3),
                                        (["--association-threshold", "0.001"], 2)]):
        args = UPDOWN + ["--associations", ASSOC] + extra
        want = _one_process(args, tmp_path / f"one{i}", monkeypatch)
        out = tmp_path / f"sharded{i}"
        got = _sharded(args, world, out, 29740 + i, tmp_path)
        assert got.split("\n")[0] == want["annotated_kmers.tsv"].split("\n")[0]
        assert _lines(got) == _lines(want["annotated_kmers.tsv"])
        for name in ("kmers_to_hashes.tsv", "hashes_to_patterns.tsv"):
            assert _lines(_read(str(out / name))) == _lines(want[name]), name
        if i < 2:
            assert len(_lines(got)) > 1
        else:
            assert got == want["annotated_kmers.tsv"] == want["annotated_kmers.tsv"].split("\n")[0] + "\n"


@pytest.mark.parametrize("only_passing", [False, True])
def test_held_batches_follow_the_global_fact(only_passing, tmp_path):
    """A piece writer whose own batch does not need the upcast (every target window passes, every
    passing row has a window, no cluster-row hash passes) holds it, and prints it in the variant
    that any_rank returns: pandas' join of the same rows, alone or with a line that another rank
    holds (empty association fields in the right join, empty positions in the left join)."""
    rng = np.random.default_rng(21 + only_passing)
    k, canonical = 7, True
    hb, r, kmers, pos = _batch(rng, k, canonical)
    n_clusters = len(hb.clusters)
    keys = list(kmers)
    row_hash = ["%022d==" % j for j in range(len(keys))]
    cluster_hash = ["c%021d==" % c for c in range(n_clusters)]
    seen = sorted({kmers[(c, km)] for c, km, *_ in pos})
    a = pd.DataFrame({"af": rng.random(len(seen)).round(3), "count": rng.integers(0, 9, len(seen)),
                      "hit": rng.random(len(seen)) < 0.5}, index=[row_hash[j] for j in seen])
    a.index.name = "hashed_pattern"
    arow = {h: i for i, h in enumerate(a.index)}
    tags = [b"cl%d" % c for c in range(n_clusters)]
    window = [(int(hb.seqs["base_off"][i]) + p) << 1 | o for c, km, i, p, o, *_ in pos]
    res = {"window": np.array(window, np.uint64),
           "window_assoc": np.array([arow[row_hash[kmers[(c, km)]]] for c, km, *_ in pos], np.uint32),
           "cluster_pass": np.array([any(keys[j][0] == c for j in seen) for c in range(n_clusters)], np.uint8),
           "cluster_assoc": np.full(n_clusters, capi.PF_ASSOC_NONE, np.uint32),
           "row": np.array(seen, np.uint32), "row_assoc": np.array([arow[row_hash[j]] for j in seen], np.uint32),
           "row_seen": np.ones(len(seen), np.uint8)}
    # pandas: the reference's join over the same tables
    h = pd.DataFrame({"cluster": [tags[c].decode() for c, _ in keys] + [t.decode() for t in tags],
                      "k-mer": [km.decode() for _, km in keys] + [np.nan] * n_clusters,
                      "hashed_pattern": row_hash + cluster_hash})
    h = h[h["hashed_pattern"].isin(arow)].set_index("hashed_pattern")
    kt = pd.DataFrame([(tags[c].decode(), km.decode(), "s%d" % i, "f%d" % i, "ctg%d" % i, s, c0, c0 + k, g0, g0 + k, u)
                       for c, km, i, p, o, s, c0, g0, u in pos],
                      columns=["cluster", "k-mer"] + assoc.POSITIONAL).set_index(["cluster", "k-mer"])
    b = a.join(h, how="inner").reset_index().set_index(["cluster", "k-mer"])
    b = b.join(kt, how="left" if only_passing else "right")
    assert not b.isna().any().any()
    other = b.iloc[:1].copy()              # the line of another rank that makes the fact true
    for col in (assoc.POSITIONAL if only_passing else ["hashed_pattern"] + list(a.columns)):
        other[col] = np.nan
    os.makedirs(tmp_path / ".parts")
    texts = []
    for rank, upcast in enumerate([False, True]):
        w = assoc.AnnotatedWriter(str(tmp_path), a, None, only_passing, False, rank=rank)
        w.batch(hb, r, res, k, canonical, [t.decode() for t in tags], lambda i: ("s%d" % i, "f%d" % i, "ctg%d" % i))
        assert w.pending and not w.upcast
        asked = []
        w.finish(lambda flag: asked.append(flag) or upcast)
        assert asked == [False]
        buf = io.StringIO()
        (pd.concat([b, other]) if upcast else b).to_csv(buf, sep="\t")
        want = buf.getvalue().split("\n")[1:-1]
        if upcast:
            want = want[:-1]
        got = open(os.path.join(tmp_path, ".parts", f"annotated_kmers.tsv.{rank}")).read()
        assert w.header == buf.getvalue().split("\n")[0] + "\n"
        assert sorted(got.split("\n")[:-1]) == sorted(want)
        texts.append(got)
    assert texts[0] != texts[1]
