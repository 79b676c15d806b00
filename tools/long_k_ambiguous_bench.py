"""k = 48 on a synthetic batch shaped like BASELINE config #2 (500 samples, 1.2-kb clusters),
ACGT-only and with 1 % / 10 % of the sequences carrying a 5-symbol N run (those sequences get a
4-bit plane built from their 2-bit codes and PF_SEQ_AMBIGUOUS, so their windows over the run go
through the 256-bit records).  One resident batch per step: pipelined submits are switched off
(PF_PIPELINE_SEQS=0; batches with N/IUPAC symbols are never pipelined), so all variants take the
same path.  400 clusters are 157,106 sequences, 1.9e8 windows.

Reports the resident time per step from the library's CUDA events (pf_stats.ms_total), the
per-stage times and a host wall clock around submit + collect (upload and planning included),
variants alternated --repeats times after a warm-up, the card's name and power limit read in the
same run; then compares sampled clusters of the 10 % variant with the C oracle
(at maf 0, where the rows of the one-sample N windows survive).

    python tools/long_k_ambiguous_bench.py [--clusters 400] [--steps 5] [--repeats 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

from panfeed_b200 import capi  # noqa: E402

STAGES = ["ms_extract", "ms_hist", "ms_sort", "ms_mark", "ms_count", "ms_reduce", "ms_dedup", "ms_total"]
_CODE4 = np.array([0, 2, 4, 11], np.uint64)        # A C G T in PF_AMB_ALPHABET
_N4 = 8


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split("\n")[0]
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                       # the numbers are still measured; say what is missing
        return {"name": None, "error": str(e)}


def codes2(packed, off, n):
    """2-bit codes of bases [off, off + n) of the packed plane."""
    idx = off + np.arange(n, dtype=np.uint64)
    return ((packed[(idx >> np.uint64(5)).astype(np.int64)] >> (np.uint64(62) - np.uint64(2) * (idx & np.uint64(31))))
            & np.uint64(3)).astype(np.uint8)


def with_n_runs(hb, frac, seed, run=5):
    """A copy of `hb` in which a fraction `frac` of the sequences carry an N run of `run` symbols
    at a random position: 4-bit plane of those sequences, PF_SEQ_AMBIGUOUS, 2-bit code 0 (A) under
    the N symbols as the packer writes it."""
    if frac == 0:
        return hb, np.zeros(0, np.int64)
    rng = np.random.default_rng(seed)
    seqs = hb.seqs.copy()
    packed = hb.packed.copy()
    n = len(seqs)
    pick = np.sort(rng.choice(n, max(1, int(round(frac * n))), replace=False))
    pick = pick[seqs["len"][pick] >= run]
    amb_off = np.zeros(n, np.uint64)
    total = 0
    for i in pick:
        amb_off[i] = total
        total += (int(seqs["len"][i]) + 31) // 32 * 32
    plane = np.zeros((total + 15) // 16, np.uint64)
    for i in pick:
        L = int(seqs["len"][i])
        c = _CODE4[codes2(packed, int(seqs["base_off"][i]), L)]
        p = int(rng.integers(0, L - run + 1))
        c[p:p + run] = _N4
        for j in range(p, p + run):                          # 2-bit plane: code 0 under the N symbols
            b = int(seqs["base_off"][i]) + j
            packed[b >> 5] &= ~np.uint64(3 << (62 - 2 * (b & 31)))
        a = int(amb_off[i])
        pad = np.zeros((L + 15) // 16 * 16, np.uint64)
        pad[:L] = c
        words = np.zeros(len(pad) // 16, np.uint64)
        for q in range(16):
            words |= pad[q::16] << np.uint64(60 - 4 * q)
        plane[a // 16:a // 16 + len(words)] = words
    seqs["amb_off"] = amb_off
    seqs["flags"][pick] |= capi.PF_SEQ_AMBIGUOUS
    return capi.HostBatch(packed, seqs, hb.clusters, hb.presence, plane), pick


def timed(ctx, hb, steps):
    rows = []
    for _ in range(steps):
        ctx.reset_patterns()
        t0 = time.perf_counter()
        ctx.submit(hb)
        r = ctx.collect(copy=False)
        wall_ms = (time.perf_counter() - t0) * 1e3          # host side included: upload, planning, D2H
        st = ctx.stats()
        rows.append({s: float(st[s]) for s in STAGES} | {"wall_ms": wall_ms} |
                    {"rows": int(len(r["row_cluster"]) + len(r["wide_row_cluster"]) + len(r["xwide_row_cluster"])),
                     "xwide_rows": int(len(r["xwide_row_cluster"]))})
    return rows


def ascii_of(hb, i):
    q = hb.seqs[i]
    L = int(q["len"])
    if q["flags"] & capi.PF_SEQ_AMBIGUOUS:
        idx = int(q["amb_off"]) + np.arange(L)
        c = (hb.amb[idx >> 4] >> (np.uint64(60) - np.uint64(4) * (idx & 15).astype(np.uint64))) & np.uint64(15)
        return np.frombuffer(capi.AMB_ALPHABET.encode(), np.uint8)[c.astype(np.int64)]
    return np.frombuffer(b"ACGT", np.uint8)[codes2(hb.packed, int(q["base_off"]), L)]


def check_with_oracle(hb, k, S, n_clusters, seed):
    """Rows of `n_clusters` sampled clusters (the whole batch on the device) against the C oracle on
    those clusters: (cluster, k-mer, count, pattern bits) of every surviving row.  maf 0: an N run
    is carried by one sample, which the timed runs' 1 % filter drops; here its rows must show."""
    from oracle import oracle_c
    from panfeed_b200 import packer
    ctx = capi.Context(k, S, maf=0.0)
    try:
        ctx.submit(hb)
        r = ctx.collect()
    finally:
        ctx.close()
    kp = r["new_kmer_patterns"]
    got_all = []
    for cl, km, cnt, pid in ((r["wide_row_cluster"], packer.wide_kmers_to_str(r["wide_row_kmer"], k),
                              r["wide_row_count"], r["wide_row_pattern"]),
                             (r["xwide_row_cluster"], packer.wide_kmers_to_str(r["xwide_row_kmer"], k, 4),
                              r["xwide_row_count"], r["xwide_row_pattern"])):
        got_all += list(zip(cl.tolist(), km.tolist(), cnt.tolist(), [kp[p].tobytes() for p in pid]))
    rng = np.random.default_rng(seed)
    amb_clusters = np.unique(hb.seqs["cluster"][(hb.seqs["flags"] & capi.PF_SEQ_AMBIGUOUS) != 0])
    pick = sorted(rng.choice(amb_clusters, min(n_clusters, len(amb_clusters)), replace=False).tolist())
    ids = hb.clusters["id"]
    sel = np.flatnonzero(np.isin(hb.seqs["cluster"], pick))
    chunks, off = [], 0
    seqs = np.zeros(len(sel), oracle_c.SEQ_DTYPE)
    for j, i in enumerate(sel):
        a = ascii_of(hb, i)
        seqs[j]["off"] = off
        chunks.append(a.tobytes())
        off += len(a)
        for f in ("len", "sample", "start", "end", "offset", "strand"):
            seqs[j][f] = hb.seqs[i][f]
        seqs[j]["cluster"] = pick.index(int(hb.seqs[i]["cluster"]))
    idx = np.arange(S)
    presab = ((hb.presence[pick][:, idx >> 5] >> (idx & 31)) & 1).astype(np.uint8)
    want = oracle_c.run_arrays(b"".join(chunks), seqs, presab, k, True, False, False, 0.0, n_threads=8)
    want_rows = sorted(zip([int(ids[pick[c]]) for c in want["row_cluster"]], want["row_kmer"].tolist(),
                           want["row_count"].tolist(), [want["kmer_pattern_bits"][p].tobytes() for p in want["row_pattern"]]))
    picked_ids = {int(ids[c]) for c in pick}
    got_rows = sorted(x for x in got_all if x[0] in picked_ids)
    n_amb = sum(1 for x in want_rows if set(x[1].decode()) - set("ACGT"))
    return {"clusters": len(pick), "maf": 0.0, "rows": len(want_rows), "rows_with_N": n_amb,
            "match": got_rows == want_rows and n_amb > 0}


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--clusters", type=int, default=400)
    p.add_argument("--samples", type=int, default=500)
    p.add_argument("--gene-len", type=int, default=1200)
    p.add_argument("--k", type=int, default=48)
    p.add_argument("--steps", type=int, default=5)
    p.add_argument("--warmup", type=int, default=2)
    p.add_argument("--repeats", type=int, default=3)
    p.add_argument("--check-clusters", type=int, default=4)
    p.add_argument("--out", default=None)
    a = p.parse_args()
    os.environ["PF_PIPELINE_SEQS"] = "0"      # one resident batch per step for every variant
    S, k = a.samples, a.k
    out = {"gpu": gpu_info(), "k": k, "samples": S, "clusters": a.clusters, "gene_len": a.gene_len,
           "steps": a.steps, "repeats": a.repeats}
    base = capi.synth_batch(0, 20261020, S, a.clusters, total_clusters=a.clusters, gene_len=a.gene_len)
    variants = {"acgt": with_n_runs(base, 0.0, 1)[0], "amb1": with_n_runs(base, 0.01, 2)[0],
                "amb10": with_n_runs(base, 0.10, 3)[0]}
    out["sequences"] = int(len(base.seqs))
    out["ambiguous_sequences"] = {v: int(((hb.seqs["flags"] & capi.PF_SEQ_AMBIGUOUS) != 0).sum())
                                  for v, hb in variants.items()}
    ctx = capi.Context(k, S, maf=0.01)
    res = {v: [] for v in variants}
    try:
        for v, hb in variants.items():                     # warm-up: every variant's buffers and modules
            timed(ctx, hb, a.warmup)
        t0 = time.time()
        for rep in range(a.repeats):
            for v, hb in variants.items():
                res[v].append(timed(ctx, hb, a.steps))
        out["wall_s"] = time.time() - t0
    finally:
        ctx.close()
    out["results"] = {}
    for v, reps in res.items():
        per_rep = [float(np.median([x["ms_total"] for x in rr])) for rr in reps]
        out["results"][v] = {
            "ms_total_median_per_repeat": per_rep,
            "ms_total_median": float(np.median([x["ms_total"] for rr in reps for x in rr])),
            "stages_median": {s: float(np.median([x[s] for rr in reps for x in rr])) for s in STAGES},
            "wall_ms_median": float(np.median([x["wall_ms"] for rr in reps for x in rr])),
            "wall_ms_median_per_repeat": [float(np.median([x["wall_ms"] for x in rr])) for rr in reps],
            "rows": reps[0][0]["rows"], "xwide_rows": reps[0][0]["xwide_rows"]}
    acgt = out["results"]["acgt"]["ms_total_median"]
    for v in ("amb1", "amb10"):
        out["results"][v]["vs_acgt"] = out["results"][v]["ms_total_median"] / acgt
    out["oracle_check"] = check_with_oracle(variants["amb10"], k, S, a.check_clusters, 5)
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(text + "\n")
    return 0 if out["oracle_check"]["match"] else 1


if __name__ == "__main__":
    sys.exit(main())
