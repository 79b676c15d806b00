"""--associations under `torchrun --nproc-per-node N -m panfeed_b200`, real NCCL ranks (N = 2 and 4;
skipped on a box with fewer GPUs): every rank joins its own clusters on its GPU, the ranks OR their
upcast facts, rank 0 merges the pieces into one annotated_kmers.tsv.  It must equal the unmodified
get-kmers' goldens, and the one-GPU --associations run of the same options on the whole fixture."""
import gzip
import os

import numpy as np
import pytest

import helpers
from torchrun_util import torchrun
from test_gpu_associations import ASSOC, CASES, POST, UPDOWN, WHOLE, _cli, _lines, _random_assoc, _read

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


RANKS = [pytest.param(n, marks=pytest.mark.skipif(_n_gpus() < n, reason=f"needs {n} GPUs")) for n in (2, 4)]


def _torchrun(args, ranks, out, port):
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = torchrun(["-m", "panfeed_b200"] + args + ["--output", str(out)], ranks, port, helpers.GOLDEN, 600, env)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert not os.path.exists(os.path.join(out, ".parts"))
    assert not os.path.exists(os.path.join(out, "kmers.tsv")) and not os.path.exists(os.path.join(out, "kmers.tsv.gz"))
    return _read(os.path.join(out, "annotated_kmers.tsv"))


GOLDEN_CASES = [("kmers_t0.3", ["--association-threshold", "0.3"]),
                ("kmers_t0.3_passing", ["--association-threshold", "0.3", "--only-passing"]),
                ("kmers_t0.1_iter2", ["--association-threshold", "0.1", "--compress"])]


@pytest.mark.parametrize("ranks", RANKS)
@pytest.mark.parametrize("case, extra", GOLDEN_CASES)
def test_ranks_match_reference_get_kmers(case, extra, ranks, tmp_path):
    got = _torchrun(UPDOWN + ["--associations", ASSOC] + extra, ranks, tmp_path / "out",
                    29760 + 4 * [c[0] for c in GOLDEN_CASES].index(case) + ranks // 2)
    want = gzip.open(os.path.join(POST, case + ".txt.gz"), "rt").read()
    assert got.split("\n")[0] == want.split("\n")[0]
    assert _lines(got) == _lines(want)
    for name in ("kmers_to_hashes.tsv", "hashes_to_patterns.tsv"):
        got_t, want_t = _read(str(tmp_path / "out" / name)), helpers.golden("updownstream", name)
        assert got_t.split("\n")[0] == want_t.split("\n")[0]
        assert helpers.sorted_lines(got_t) == helpers.sorted_lines(want_t), name


@pytest.mark.parametrize("ranks", RANKS)
@pytest.mark.parametrize("case", ["k31", "k40", "k64_nc", "k31_cm"])
def test_ranks_match_one_gpu(case, ranks, tmp_path):
    """The whole fixture (its N run and IUPAC codes included), both join modes, against one GPU."""
    rng = np.random.default_rng(sum(case.encode()) + ranks)
    args = WHOLE + CASES[case]
    _cli(args, tmp_path / "plain")
    assoc = tmp_path / "assoc.tsv"
    _random_assoc(tmp_path / "plain", assoc, rng, 0.2, int_column=True)
    for i, extra in enumerate([[], ["--only-passing"]]):
        joined = args + ["--associations", str(assoc), "--association-threshold", "0.5"] + extra
        one = tmp_path / f"one{i}"
        _cli(joined, one)
        want = _read(str(one / "annotated_kmers.tsv"))
        out = tmp_path / f"ranks{i}"
        got = _torchrun(joined, ranks, out, 29780 + 8 * ["k31", "k40", "k64_nc", "k31_cm"].index(case) + 2 * i + ranks // 2)
        assert got.split("\n")[0] == want.split("\n")[0]
        assert _lines(got) == _lines(want)
        assert len(_lines(got)) > 1
        for name in ("kmers_to_hashes.tsv", "hashes_to_patterns.tsv"):
            assert _lines(_read(str(out / name))) == _lines(_read(str(one / name))), name
