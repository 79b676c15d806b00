"""The multi-GPU product path on real hardware, two ranks over NCCL
(`torchrun --nproc-per-node 2`; skipped on a box with one GPU):

  * `torchrun -m panfeed_b200 ...` shards the clusters, runs the pattern exchange and writes ONE
    set of three files: they must equal the unmodified reference's goldens after sorting, like
    the single-process CLI (the reference's own parallel mode, `__main__.py:299-344`, is held to
    the same sorted comparison: its row order is nondeterministic);
  * `selfcheck.check_exchange`: local keys == the owners' keys under the returned global ids, no
    duplicate in the global tables, and the same pattern sets as ONE context over all clusters,
    with and without the cluster-absent encoding.
"""
import gzip
import os
import subprocess
import sys

import pytest

import helpers

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


# ranks of the torchrun launches (PF_TEST_RANKS=8 on an 8-GPU box: some ranks then own no cluster
# of the five-cluster fixture at all, which the product path must survive)
RANKS = max(2, int(os.environ.get("PF_TEST_RANKS", "2")))
needs_two = pytest.mark.skipif(_n_gpus() < RANKS, reason=f"needs {RANKS} GPUs")


def _torchrun(args, port, cwd, timeout=900, extra_env=None):
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    env.update(extra_env or {})
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(RANKS),
                        "--master-addr", "127.0.0.1", "--master-port", str(port)] + args,
                       capture_output=True, text=True, timeout=timeout, env=env, cwd=cwd)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    return r


def _read(path):
    if os.path.exists(path + ".gz"):
        return gzip.open(path + ".gz", "rt").read()
    return open(path).read()


CASES = [("basic", ["--python-feeder"]), ("considermissing", []), ("cm_nofilter_up", []), ("noncanonical", []),
         ("compress", []), ("secondpass", ["--native-feeder"])]


@needs_two
@pytest.mark.parametrize("mode,extra", CASES)
def test_cli_two_ranks_match_reference(mode, extra, tmp_path):
    out = str(tmp_path / "out")
    args = ["-m", "panfeed_b200"] + list(helpers.modes()[mode]) + extra + ["--output", out]
    _torchrun(args, 29610 + [c[0] for c in CASES].index(mode), helpers.GOLDEN)
    assert not os.path.exists(os.path.join(out, ".parts"))
    for name in helpers.FILES:
        got = _read(os.path.join(out, name))
        want = helpers.golden(mode, name)
        assert got.split("\n")[0] == [x for x in want.split("\n") if x.startswith(
            ("cluster\t", "hashed_pattern"))][0]
        assert helpers.sorted_lines(got) == helpers.sorted_lines(want), (mode, name)
    if mode == "compress":
        assert os.path.exists(os.path.join(out, "hashes_to_patterns.tsv.gz"))


@needs_two
def test_cli_two_ranks_multiple_files(tmp_path):
    """--multiple-files under torchrun: every rank writes the directories of its own clusters (the
    pattern set is per cluster there, panfeed.py:165: no exchange); checked per cluster against
    the oracle port like the single-process test."""
    import pandas as pd
    from oracle import ref_port
    out = str(tmp_path / "out")
    _torchrun(["-m", "panfeed_b200", "--gff", "fixture/gffs/", "--presence-absence",
               "fixture/gene_presence_absence.csv", "--targets", "fixture/stroi.txt", "--multiple-files",
               "--output", out], 29640, helpers.GOLDEN)
    cwd = os.getcwd()
    os.chdir(helpers.GOLDEN)
    try:
        table = pd.read_csv("fixture/gene_presence_absence.csv", sep=",", index_col=0,
                            low_memory=False).drop(columns=["Non-unique Gene name", "Annotation"])
        genomes = ref_port.load_inputs("fixture/gffs/")
        stroi = {x.rstrip("\n") for x in open("fixture/stroi.txt")}
        h2p_head, k2h_head = ref_port.headers(table.columns)
        n = 0
        for item in ref_port.feed_clusters(table, genomes, 0, 0, False):
            res = ref_port.kmer_stage(item, 31, stroi, True, False)
            a, b, c = ref_port.pattern_stage((res,), True, 0.01, False, set())
            d = os.path.join(out, item[1])
            assert helpers.sorted_lines(open(os.path.join(d, "kmers.tsv")).read()) == \
                helpers.sorted_lines(ref_port.KMERS_HEADER + a)
            assert helpers.sorted_lines(open(os.path.join(d, "hashes_to_patterns.tsv")).read()) == \
                helpers.sorted_lines(h2p_head + b)
            assert helpers.sorted_lines(open(os.path.join(d, "kmers_to_hashes.tsv")).read()) == \
                helpers.sorted_lines(k2h_head + c)
            n += 1
        assert n >= 5
    finally:
        os.chdir(cwd)


WORKER = r'''
import os, sys, json
import torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from panfeed_b200 import selfcheck
local = int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
res = [selfcheck.check_exchange(local, cm, n_samples=int(sys.argv[2]), clusters_per_rank=int(sys.argv[3]),
                                gene_len=int(sys.argv[4])) for cm in (False, True)]
if dist.get_rank() == 0:
    print("SELFCHECK " + json.dumps(res))
dist.barrier()
dist.destroy_process_group()
'''


@needs_two
@pytest.mark.parametrize("samples,clusters,gene_len,peer", [(256, 6, 400, "1"), (1500, 3, 300, "1"), (256, 6, 400, "0")])
def test_exchange_two_ranks_nccl(samples, clusters, gene_len, peer, tmp_path):
    """(1500 samples: sample slices of the block engine, 47-word keys.)  peer = 1: the keys go
    straight into the owners' receive buffers (CUDA IPC mappings, NVLink stores); 0: the NCCL
    all-to-all of the keys, which is also what a box without peer access falls back to."""
    path = tmp_path / "worker.py"
    path.write_text(WORKER)
    r = _torchrun([str(path), ROOT, str(samples), str(clusters), str(gene_len)],
                  29650 + samples % 7 + 3 * int(peer), ROOT, extra_env={"PF_EXCHANGE_PEER": peer})
    assert "SELFCHECK" in r.stdout, r.stdout[-2000:]
    line = [x for x in r.stdout.splitlines() if x.startswith("SELFCHECK")][0]
    print(line)
    if peer == "0":
        assert "nccl all-to-all" in line


def test_exchange_selfcheck_single_rank():
    """World size 1 goes through the same pack / dedup / unpack kernels (plain copies for the
    collectives): runs on any GPU box."""
    from panfeed_b200 import selfcheck
    for cm in (False, True):
        res = selfcheck.check_exchange(0, cm, n_samples=300, clusters_per_rank=5, gene_len=350)
        assert res["ok"] and res["kmer_patterns_global"] == res["kmer_patterns_local"] > 0
