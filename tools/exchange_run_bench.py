"""Time pf_exchange_run (one library call per rank, one host thread per rank, in-process
communicator) at world 1..N in ONE process, for both transports of the keys.

Every rank holds the patterns of config 2's shape (bench.py --config 2: 500 genomes, 4,000 gene
clusters per rank of a 4,000*N-cluster synthetic pangenome, pf_synth batches).  Ranks go round-robin
over the visible GPUs (--devices 1: all on cuda:0).  Prints one JSON line per measurement.

    python tools/exchange_run_bench.py --max-world 4 [--clusters 4000] [--reps 3] [--devices N]
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from panfeed_b200 import capi  # noqa: E402

SEED = 20261018 + 2          # bench.py config 2


def _ranks(world, fn):
    comm = capi.LocalComm(world)
    out, err = [None] * world, [None] * world

    def body(r):
        try:
            out[r] = fn(r, comm.get(r))
        except BaseException as e:       # noqa: BLE001
            err[r] = e
            comm.abort()
    ths = [threading.Thread(target=body, args=(r,)) for r in range(world)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    comm.close()
    if any(err):
        raise RuntimeError(err)
    return out


def main():
    p = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    p.add_argument("--max-world", type=int, default=4)
    p.add_argument("--clusters", type=int, default=4000, help="clusters per rank (config 2: 4,000)")
    p.add_argument("--samples", type=int, default=500)
    p.add_argument("--reps", type=int, default=3)
    p.add_argument("--devices", type=int, default=0, help="GPUs to spread the ranks over (0: all visible)")
    a = p.parse_args()
    n_dev = a.devices or torch.cuda.device_count()
    dev_name = torch.cuda.get_device_name(0)
    try:                                 # the number belongs with the card's power limit
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        power = "unknown"
    arena = capi.SynthArena()
    ctxs = []
    for r in range(a.max_world):
        d = r % n_dev
        hb = capi.synth_batch(d, SEED, a.samples, a.clusters, first_cluster=r * a.clusters,
                              total_clusters=a.max_world * a.clusters, arena=arena)
        ctx = capi.Context(31, a.samples, maf=0.01, device=d)
        ctx.submit(hb)
        ctx.collect(copy=False)
        ctxs.append(ctx)
    st = ctxs[0].stats()
    base = {"gpu": dev_name, "power_limit": power, "gpus_used": min(n_dev, a.max_world), "samples": a.samples,
            "clusters_per_rank": a.clusters, "kmer_patterns_rank0": int(st["kmer_patterns"]),
            "cluster_patterns_rank0": int(st["cluster_patterns"])}

    def timed(world, flags):
        times = []
        for _ in range(a.reps + 1):                     # the first call maps and sizes the buffers
            def one(r, c):
                torch.cuda.synchronize(r % n_dev)
                t0 = time.perf_counter()
                res = ctxs[r].exchange_run(c, flags)
                return time.perf_counter() - t0, res["kmer"]["n_global"]
            out = _ranks(world, one)
            times.append(max(t for t, _ in out) * 1e3)
        return sorted(times[1:])[len(times[1:]) // 2], out[0][1]

    for world in range(1, a.max_world + 1):
        for name, flags in (("native_peer", capi.PF_EXCHANGE_WRITER),
                            ("native_all_to_all", capi.PF_EXCHANGE_WRITER | capi.PF_EXCHANGE_NO_PEER)):
            ms, n_global = timed(world, flags)
            print(json.dumps(dict(base, impl=name, world=world, ms_median=round(ms, 2),
                                  kmer_global=int(n_global))), flush=True)
    for c in ctxs:
        c.close()


if __name__ == "__main__":
    main()
