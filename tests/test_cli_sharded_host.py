"""The sharded CLI (`torchrun -m panfeed_b200`, one process per GPU) on the CPU: two processes
over gloo, each with the oracle-backed stand-in for its GPU context (tests/cpu_context.py) and
a host model of the pattern exchange (its `exchange`, in place of dist.PatternExchange).
Everything else is the product's own code: cluster sharding, per-rank piece files,
`PatternStore.finish_sharded` (the writer flags, the hashes_to_patterns rows), the merge on rank 0.  The three files must equal
the unmodified reference's goldens, as tests/test_gpu_multirank.py demands on real ranks."""
import gzip
import os
import subprocess
import sys

import pytest

import helpers

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = r'''
import os, sys
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, os.path.join(sys.argv[1], "tests"))
from cpu_context import OracleContext
from panfeed_b200 import capi
capi.Context = OracleContext
from panfeed_b200.__main__ import main
main(sys.argv[2:])
'''


def _read(path):
    if os.path.exists(path + ".gz"):
        return gzip.open(path + ".gz", "rt").read()
    return open(path).read()


@pytest.mark.parametrize("mode,extra,world", [("basic", [], 2), ("considermissing", ["--python-feeder"], 2),
                                              ("secondpass", [], 3), ("compress", [], 2), ("cm_nofilter_up", [], 2)])
def test_sharded_cli_host_logic_matches_reference(mode, extra, world, tmp_path):
    worker = tmp_path / "worker.py"
    worker.write_text(WORKER)
    out = str(tmp_path / "out")
    port = 29700 + sorted(helpers.modes()).index(mode)
    env = dict(os.environ, PF_DIST_BACKEND="gloo")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
                        "--master-addr", "127.0.0.1", "--master-port", str(port), str(worker), ROOT] +
                       list(helpers.modes()[mode]) + extra + ["--output", out],
                       capture_output=True, text=True, timeout=600, env=env, cwd=helpers.GOLDEN)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert not os.path.exists(os.path.join(out, ".parts"))
    for name in helpers.FILES:
        got = _read(os.path.join(out, name))
        want = helpers.golden(mode, name)
        assert got.split("\n")[0] == [x for x in want.split("\n") if x.startswith(("cluster\t", "hashed_pattern"))][0]
        assert helpers.sorted_lines(got) == helpers.sorted_lines(want), (mode, name)
