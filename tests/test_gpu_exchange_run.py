"""pf_exchange_run: the global pattern dedup of a sharded run in one library call.

Contexts own disjoint cluster shards and run the exchange from one host thread each over the
in-process communicator (capi.LocalComm), on one GPU or on several; the invariants are those of
selfcheck.check_exchange:
  * local key == the owner's unique key at the returned global id;
  * the global pattern sets equal those of ONE context that saw every cluster;
  * exactly one writer per distinct pattern across ranks;
  * n_global, n_owned and owned_base agree on every rank.
Also: a C program driving the call from pthreads.  Real ranks over NCCL: tests/test_gpu_multirank.py."""
import os
import subprocess
import threading

import numpy as np
import pytest
import torch

import gpu_util  # noqa: F401  (path setup)
from panfeed_b200 import capi, dist as pfdist, packer
from test_gpu_parity import _random_items

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
S, K = 48, 21
FLAGS = capi.PF_EXCHANGE_WRITER | capi.PF_EXCHANGE_KEEP_UNIQUE


def _submit(ctx, items, stroi, base):
    pcs = [packer.PackedCluster(c, idx, pa, stroi) for c, idx, pa in items]
    hb, _, _ = packer.pack_batch(pcs, list(range(base, base + len(items))))
    ctx.submit(hb)
    return ctx.collect()


def _threads(world, fn, comm=None, timeout=600):
    """fn(rank, pf_comm) on one thread per rank; a rank that raises aborts the communicator so that
    no other rank waits for it.  -> (results, errors) per rank."""
    own = comm is None
    comm = comm or capi.LocalComm(world)
    res, err = [None] * world, [None] * world

    def body(r):
        try:
            res[r] = fn(r, comm.get(r))
        except BaseException as e:       # noqa: BLE001
            err[r] = e
            comm.abort()
    ths = [threading.Thread(target=body, args=(r,)) for r in range(world)]
    for t in ths:
        t.start()
    for t in ths:
        t.join(timeout)
    assert not any(t.is_alive() for t in ths), "a rank hangs"
    if own:
        comm.close()
    return res, err


def _host(ptr, n, dtype, device):
    if n == 0:
        return np.zeros(0, dtype)
    if dtype is np.uint32:
        return pfdist._device_view(ptr, n, device, "<i4", torch.int32).cpu().numpy().view(np.uint32)
    return pfdist._device_view(ptr, n, device).cpu().numpy()


def _outcome(ctx, out, device):
    """Host copies of one rank's result (the library's tables are reused by its next call)."""
    got = {}
    for name, ns in (("cluster", True), ("kmer", False)):
        r = out[name]
        n = int(r["n_local"])
        got[name] = dict(r, l2g=_host(r["local_to_global"], n, np.uint32, device),
                         writer=_host(r["writer"], n, np.uint8, device), owned_keys=ctx.exchange_unique_keys(ns),
                         keys=ctx.export_patterns(ns, 0, n) if n else np.zeros((0, ctx.W if ns else ctx.Wk), np.uint32))
    return got


def _check(outs, ctxs, items, cm):
    """The invariants against one context over every cluster."""
    world = len(outs)
    W = (S + 31) // 32
    for name in ("cluster", "kmer"):
        ng = {o[name]["n_global"] for o in outs}
        assert len(ng) == 1, (name, ng)
        owned = [o[name]["n_owned"] for o in outs]
        assert sum(owned) == outs[0][name]["n_global"]
        assert [o[name]["owned_base"] for o in outs] == [sum(owned[:r]) for r in range(world)]
        table = np.concatenate([o[name]["owned_keys"] for o in outs]) if world else None
        assert len(table) == outs[0][name]["n_global"]
        for r, o in enumerate(outs):
            keys = o[name]["keys"].copy()
            if name == "kmer" and cm and len(keys):
                keys[:, W] = outs[r]["cluster"]["l2g"][keys[:, W]]
            assert np.array_equal(table[o[name]["l2g"]], keys), (name, r)
        written = np.concatenate([o[name]["l2g"][o[name]["writer"] != 0] for o in outs])
        assert sorted(written.tolist()) == list(range(outs[0][name]["n_global"])), name
    one = capi.Context(K, S, True, cm, False, False, 0.02)
    r_all = _submit(one, items, set(), 0)
    one.close()
    assert outs[0]["cluster"]["n_global"] == len(r_all["new_cluster_patterns"])
    assert outs[0]["kmer"]["n_global"] == len(r_all["new_kmer_patterns"])
    seen = {}
    for r, o in enumerate(outs):
        cp = o["cluster"]["keys"]
        for row, gid in zip(o["kmer"]["keys"], o["kmer"]["l2g"]):
            key = row[:W].tobytes() + (cp[row[W]].tobytes() if cm else b"")
            assert seen.setdefault(key, int(gid)) == int(gid)
    cp_all = r_all["new_cluster_patterns"]
    want = {row[:W].tobytes() + (cp_all[row[W]].tobytes() if cm else b"") for row in r_all["new_kmer_patterns"]}
    assert set(seen) == want


def _shards(items, world, empty_rank):
    owners = world - 1 if (empty_rank and world > 1) else world
    return [items[r::owners] if r < owners else [] for r in range(world)]


def _contexts(shards, cm, devices):
    ctxs = []
    for r, sh in enumerate(shards):
        ctx = capi.Context(K, S, True, cm, False, False, 0.02, device=devices[r])
        if sh:
            _submit(ctx, sh, set(), 1000 * r)
        ctxs.append(ctx)
    return ctxs


def _exchange(ctxs, devices, flags, comm=None):
    res, err = _threads(len(ctxs), lambda r, c: _outcome(ctxs[r], ctxs[r].exchange_run(c, flags),
                                                         torch.device("cuda", devices[r])), comm)
    assert not any(err), err
    return res


@pytest.mark.parametrize("world", [1, 2, 3, 4])
@pytest.mark.parametrize("cm", [False, True])
@pytest.mark.parametrize("no_peer", [False, True])
def test_exchange_run_threads_one_gpu(world, cm, no_peer):
    rng = np.random.default_rng(100 + world)
    items, _ = _random_items(rng, S, K, 7, 260)
    devices = [0] * world
    shards = _shards(items, world, empty_rank=world >= 3)        # world 3, 4: the last rank owns no cluster
    ctxs = _contexts(shards, cm, devices)
    flags = FLAGS | (capi.PF_EXCHANGE_NO_PEER if no_peer else 0)
    outs = _exchange(ctxs, devices, flags)
    _check(outs, ctxs, items, cm)
    _threads(world, lambda r, c: ctxs[r].exchange_release(c))
    for c in ctxs:
        c.close()


@pytest.mark.parametrize("no_peer", [False, True])
def test_exchange_run_twice_grows_and_reuses(no_peer):
    """A second call on the same contexts after more batches: the receive buffers grow (and the
    peers' mappings are replaced), the tables are numbered afresh over everything seen so far."""
    world, cm = 3, True
    rng = np.random.default_rng(7)
    first, _ = _random_items(rng, S, K, 3, 200)
    more, _ = _random_items(rng, S, K, 80, 1200)
    devices = [0] * world
    comm = capi.LocalComm(world)
    ctxs = _contexts(_shards(first, world, False), cm, devices)
    flags = FLAGS | (capi.PF_EXCHANGE_NO_PEER if no_peer else 0)
    outs = _exchange(ctxs, devices, flags, comm)
    _check(outs, ctxs, first, cm)
    for r, sh in enumerate(_shards(more, world, False)):
        _submit(ctxs[r], sh, set(), 5000 + 1000 * r)
    outs2 = _exchange(ctxs, devices, flags, comm)
    # (one context over all clusters, in the order the shards saw them)
    order = [it for r in range(world) for it in _shards(first, world, False)[r] + _shards(more, world, False)[r]]
    _check(outs2, ctxs, order, cm)
    # (the receive buffers had to grow: every owner now receives more than the first call's need
    #  * 5/4 + 1024 rows, on average)
    sent1 = sum(o["kmer"]["n_local"] for o in outs)
    sent2 = sum(o["kmer"]["n_local"] for o in outs2)
    assert sent2 / world > 1.25 * sent1 / world + 1024, (sent1, sent2)
    _, err = _threads(world, lambda r, c: ctxs[r].exchange_release(c), comm)
    assert not any(err), err
    for c in ctxs:
        c.close()
    comm.close()


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("delta", [1, -1])
def test_exchange_run_ranks_agree_on_a_bad_world(world, delta):
    """One rank is handed a pf_comm with the wrong world: every rank returns PF_ERR_INVALID from the
    record exchange (nobody hangs, nothing reaches the device beyond the local classify)."""
    rng = np.random.default_rng(5)
    items, _ = _random_items(rng, S, K, 4, 200)
    devices = [0] * world
    ctxs = _contexts(_shards(items, world, False), False, devices)

    def rank(r, c):
        if r == 0:
            c.world = c.world + delta
        return ctxs[r].exchange_run(c, FLAGS)
    res, err = _threads(world, rank)
    assert all(isinstance(e, capi.PfError) for e in err), err
    assert [e.code for e in err] == [-1] * world, [str(e) for e in err]
    # the contexts are still usable: a correct exchange afterwards
    outs = _exchange(ctxs, devices, FLAGS)
    _check(outs, ctxs, [it for sh in _shards(items, world, False) for it in sh], False)
    for c in ctxs:
        c.close()


def test_exchange_run_without_all_to_all_refuses_no_peer_on_every_rank():
    """PF_EXCHANGE_NO_PEER with a communicator that has no all_to_all_v: PF_ERR_UNSUPPORTED on every
    rank, none of them waits."""
    world = 2
    rng = np.random.default_rng(9)
    items, _ = _random_items(rng, S, K, 4, 200)
    ctxs = _contexts(_shards(items, world, False), False, [0] * world)

    def rank(r, c):
        c.all_to_all_v = capi.ALL_TO_ALL_V_FN()
        return ctxs[r].exchange_run(c, FLAGS | capi.PF_EXCHANGE_NO_PEER)
    _, err = _threads(world, rank)
    assert [getattr(e, "code", None) for e in err] == [-4] * world, err

    def peer_only(r, c):
        c.all_to_all_v = capi.ALL_TO_ALL_V_FN()
        return _outcome(ctxs[r], ctxs[r].exchange_run(c, FLAGS), torch.device("cuda", 0))
    outs, err = _threads(world, peer_only)
    assert not any(err), err
    _check(outs, ctxs, [it for sh in _shards(items, world, False) for it in sh], False)
    for c in ctxs:
        c.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("cm", [False, True])
@pytest.mark.parametrize("no_peer", [False, True])
def test_exchange_run_threads_several_gpus(cm, no_peer):
    world = min(torch.cuda.device_count(), 4)
    rng = np.random.default_rng(200)
    items, _ = _random_items(rng, S, K, 9, 260)
    devices = list(range(world))
    ctxs = _contexts(_shards(items, world, False), cm, devices)
    outs = _exchange(ctxs, devices, FLAGS | (capi.PF_EXCHANGE_NO_PEER if no_peer else 0))
    _check(outs, ctxs, items, cm)
    _threads(world, lambda r, c: ctxs[r].exchange_release(c))
    for c in ctxs:
        c.close()


def _synth_counts(world, n_samples, clusters, seed, spread):
    """The C program's run, from Python: the same synthetic batches and parameters."""
    n_dev = torch.cuda.device_count()
    ctxs = []
    for r in range(world):
        dev = r % n_dev if spread else 0
        hb = capi.synth_batch(dev, seed, n_samples, clusters, first_cluster=r * clusters,
                              total_clusters=world * clusters, gene_len=600)
        ctx = capi.Context(31, n_samples, maf=0.01, device=dev)
        ctx.submit(hb)
        ctx.collect()
        ctxs.append(ctx)
    res, err = _threads(world, lambda r, c: ctxs[r].exchange_run(c, capi.PF_EXCHANGE_WRITER))
    assert not any(err), err
    for c in ctxs:
        c.close()
    return res[0]["kmer"]["n_global"], res[0]["cluster"]["n_global"]


@pytest.mark.parametrize("world,spread", [(1, 0), (3, 0), (4, 1)])
def test_c_program_runs_the_exchange_from_threads(tmp_path, world, spread):
    cc = os.environ.get("CC", "cc")
    exe = str(tmp_path / "exchange_threads")
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    libdir = os.path.join(ROOT, "panfeed_b200", "csrc")
    subprocess.run([cc, "-O2", "-Wall", "-std=c11", "-pthread", "-I", os.path.join(ROOT, "include"),
                    "-I", os.path.join(cuda, "include"), os.path.join(ROOT, "tests", "c", "exchange_threads.c"),
                    "-o", exe, "-L", libdir, "-lpanfeed_b200", "-L", os.path.join(cuda, "lib64"), "-lcudart",
                    f"-Wl,-rpath,{libdir}:{os.path.join(cuda, 'lib64')}"], check=True)
    n_samples, clusters, seed = 64, 6, 20261020
    r = subprocess.run([exe, str(world), str(n_samples), str(clusters), str(seed), str(spread)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    got = dict(kv.split("=") for kv in r.stdout.split())
    assert int(got["world"]) == world
    assert got["kmer_writers"] == got["kmer_global"] and got["cluster_writers"] == got["cluster_global"]
    km, cl = _synth_counts(world, n_samples, clusters, seed, spread)
    assert (int(got["kmer_global"]), int(got["cluster_global"])) == (km, cl)
    assert km > 0 and cl > 0

