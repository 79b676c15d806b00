#!/usr/bin/env python
"""Benchmark of the per-gene-cluster k-mer streaming hot path (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
                    [--config 2|3|4|5] [--extra 3,4,5 | --no-extra] [--dump-outputs DIR]

Headline (default `--config 2`): a step = one pass of K1..K4 over the whole synthetic
pangenome of BASELINE.json configs[1] (500 genomes x 4,000 gene clusters, 1.2 kb cut sequences,
k=31, first pass).  `value` = input bases/s with the batch already resident in HBM (CUDA events
on the context's stream); `e2e` = the same through pf_submit/pf_collect from pinned HOST
buffers (H2D + kernels + D2H inside the timed region) - the number to compare with the CPU
arm.  N > 1: every rank runs its own 4,000 clusters of a 4,000*N-cluster pangenome (weak
scaling) and a step ends with the global pattern dedup exchange (NCCL all-to-all).

`extra_configs` in the same JSON line: the other BASELINE configs at FULL size, streamed batch
by batch (the inputs of configs 4 / 5 are 15 GB per GPU): #3 second pass (200 clusters, every
sample a --targets strain), #4 10,000 genomes x 5,000 clusters sharded over the N ranks
(strong scaling), #5 50,000 genomes x 8,000 clusters with the cluster-absent encoding,
1,000 clusters per rank (the full config at N = 8), each with ONE global pattern exchange at
the end of the run, as a real run does.

`--steps K` is the number of timed steps of the headline: K executions of the resident batch,
or K passes over all batches when the headline config is streamed.  `--dump-outputs DIR` then
writes what the last of them computed (rows, pattern bits, per-cluster sums) to DIR as .npy
files (class OutputDump); the inputs are seeded, so two builds can be compared on them.

`--impl reference` times the UNMODIFIED reference's own hot functions (cluster_cutter +
pattern_hasher of oracle/_ref/panfeed/panfeed.py, installed from /root/reference by
oracle/make_ref.sh) on all host cores, on clusters unpacked from the same pf_synth_fill
generator the GPU arm uses.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED0 = 20261018             # SURVEY.md 8(d): seed = 20261018 + config_id
R_BYTES = 12                 # declared record of SURVEY 8(d): 8-byte key + 4-byte sample rank

# BASELINE.json configs[1..4] (config_id 2..5).  clusters = of the whole pangenome;
# "strong": the same clusters sharded over the ranks, "weak": `clusters` per rank.
CONFIGS = {
    2: dict(samples=500, clusters=4000, cm=False, targets=False, batch=4000, scaling="weak",
            name="BASELINE.json configs[1]: synthetic 500 genomes x 4,000 gene clusters "
                 "(~1 kb + 100 bp flanks), first pass"),
    3: dict(samples=500, clusters=200, cm=False, targets=True, batch=200, scaling="strong",
            name="BASELINE.json configs[2]: same pangenome, second pass over 200 clusters, every "
                 "sample a --targets strain (positional kmers.tsv records)"),
    4: dict(samples=10000, clusters=5000, cm=False, targets=False, batch=240, scaling="strong",
            name="BASELINE.json configs[3]: synthetic 10,000 genomes x 5,000 clusters "
                 "(10k-bit presence patterns), clusters sharded over the ranks"),
    5: dict(samples=50000, clusters=1000, cm=True, targets=False, batch=60, scaling="weak",
            name="BASELINE.json configs[4]: synthetic 50,000 genomes x 8,000 clusters, cluster-absent "
                 "encoding, global pattern dedup over NCCL; 1,000 clusters per rank (= the full "
                 "8,000 at N = 8)"),
}


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS),
                   help="BASELINE config (2..5) the headline line is measured on")
    p.add_argument("--extra", default=None,
                   help="comma-separated configs measured at full size into extra_configs "
                        "(default with --config 2: 3,4,5)")
    p.add_argument("--no-extra", action="store_true")
    p.add_argument("--samples", type=int, default=None)
    p.add_argument("--clusters", type=int, default=None)
    p.add_argument("--batch-clusters", type=int, default=None)
    p.add_argument("--gene-len", type=int, default=1200)
    p.add_argument("-k", type=int, default=31)
    p.add_argument("--maf", type=float, default=0.01)
    p.add_argument("--consider-missing", action="store_true")
    p.add_argument("--targets-all", action="store_true",
                   help="second pass: every sample is a --targets strain (same as --config 3 shape)")
    p.add_argument("--sort-bits", type=int, default=0)
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-selfcheck", action="store_true")
    p.add_argument("--cpu-seconds", type=float, default=15.0)
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write what the last step computed to DIR/<name>.npy "
                        "(float64, at most 64 MB in all; see OutputDump)")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    return args


def config_of(args, cid):
    c = dict(CONFIGS[cid])
    c["id"] = cid
    if cid == args.config:
        if args.samples:
            c["samples"] = args.samples
        if args.clusters:
            c["clusters"] = args.clusters
        if args.batch_clusters:
            c["batch"] = args.batch_clusters
        if args.consider_missing:
            c["cm"] = True
        if args.targets_all:
            c["targets"] = True
    c["gene_len"], c["k"], c["maf"] = args.gene_len, args.k, args.maf
    c["seed"] = SEED0 + cid
    return c


# --------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------
class ClockSampler:
    """SM clock and clock-event reasons of one GPU, sampled every `period` s (default 5 ms; 50 ms
    for the streamed configs, whose timed regions last seconds: NVML queries take driver locks
    that CUDA calls of the measured thread also need) through NVML from a thread of this process
    while the timed region runs (the timed region is tens of ms: an
    `nvidia-smi -lms` child would not have printed its first line by the time it ends).
    Falls back to `nvidia-smi -lms 20` when NVML cannot be loaded."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device, period=0.005):
        self.device = device
        self.period = period
        self.p = None
        self.f = None
        self.thread = None
        self.stop_flag = False
        self.samples = []        # (sm_mhz, reasons bitmask)
        self.max_mhz = None
        self.nvml = None
        self.handle = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(device).uuid)
                if not uuid.startswith("GPU-"):
                    uuid = "GPU-" + uuid
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
                idx = device
                if vis:
                    ent = vis.split(",")[device].strip()
                    idx = int(ent) if ent.isdigit() else device
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None

    def _loop(self):
        nv = self.nvml
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)
                try:
                    why = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:
                    why = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.samples.append((float(mhz), int(why)))
            except Exception:
                pass
            time.sleep(self.period)

    def start(self):
        if self.nvml is not None:
            import threading
            self.stop_flag = False
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
            return
        try:
            self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.p = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "20", "-i", str(self.device)], stdout=self.f,
                stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.thread is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
            nv = self.nvml
            if not self.samples:
                return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["no samples"]}
            names = (("hw_slowdown", nv.nvmlClocksThrottleReasonHwSlowdown),
                     ("hw_thermal_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown),
                     ("sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwThermalSlowdown),
                     ("sw_power_cap", nv.nvmlClocksThrottleReasonSwPowerCap),
                     ("hw_power_brake_slowdown", nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown))
            reasons = sorted({n for _, why in self.samples for n, bit in names if why & bit})
            sm = [m for m, _ in self.samples]
            return {"sm_mhz": float(np.median(sm)), "sm_min_mhz": float(min(sm)), "sm_max_mhz": self.max_mhz,
                    "reasons": reasons, "samples": len(sm),
                    "source": f"nvml, {self.period * 1e3:.0f} ms period, timed region only"}
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.split(",") for r in open(self.f.name).read().strip().split("\n") if r]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for n, v in zip(names, r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(n)
            except (ValueError, IndexError):
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)),
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi -lms 20"}


# --------------------------------------------------------------------------
# CPU legs (oracle = test infrastructure; allowed here as the measured baseline)
# --------------------------------------------------------------------------
def unpack_ascii(hb, seq_slice):
    """ASCII bases + oracle seq array for a slice of a HostBatch's sequences."""
    from oracle import oracle_c
    seqs = hb.seqs[seq_slice]
    w0 = int(seqs["base_off"][0]) // 32
    w1 = int(seqs["base_off"][-1] + (seqs["len"][-1] + 63) // 64 * 64) // 32
    sh = (62 - 2 * np.arange(32)).astype(np.uint64)
    codes = ((hb.packed[w0:w1, None] >> sh[None, :]) & np.uint64(3)).astype(np.uint8).ravel()
    ascii_plane = np.frombuffer(b"ACGT", np.uint8)[codes]
    out = np.zeros(len(seqs), oracle_c.SEQ_DTYPE)
    for f in ("len", "sample", "start", "end", "offset", "strand"):
        out[f] = seqs[f]
    out["cluster"] = seqs["cluster"] - seqs["cluster"][0]
    out["off"] = seqs["base_off"] - np.uint64(w0 * 32)
    return ascii_plane, out


def cpu_baseline_c(hb, S, k, maf, consider_missing, budget_s):
    """C oracle, all host cores, on the first n clusters of the workload."""
    from oracle import oracle_c
    oracle_c.build()
    cores = os.cpu_count() or 1
    first = np.searchsorted(hb.seqs["cluster"], np.arange(len(hb.clusters) + 1))
    idx = np.arange(S)
    n = min(len(hb.clusters), max(cores, 8))
    best = None
    while True:
        sl = slice(int(first[0]), int(first[n]))
        ascii_plane, seqs = unpack_ascii(hb, sl)
        presab = ((hb.presence[:n, idx >> 5] >> (idx & 31)) & 1).astype(np.uint8)
        t0 = time.perf_counter()
        res = oracle_c.run_arrays(ascii_plane, seqs, presab, k, True, consider_missing,
                                  False, maf, n_threads=cores)
        dt = time.perf_counter() - t0
        bases = int(seqs["len"].sum())
        best = {"value": bases / dt, "unit": "bases/s", "cores": cores, "kind": "port",
                "sample": f"oracle/oracle.c (C restatement, {cores} threads) on the first {n} "
                          f"clusters of the workload: {bases} bases in {dt:.2f} s",
                "unique_kmers_per_s": res["n_unique"] / dt}
        if dt >= budget_s / 3 or n >= len(hb.clusters):
            return best
        n = min(len(hb.clusters), max(n + 1, int(n * min(8.0, budget_s / max(dt, 1e-3)) * 0.7)))


_REF = {}


def load_reference():
    """The unmodified reference package from oracle/_ref (oracle/make_ref.sh) -> its hot
    functions and Seqinfo.  None if it has not been installed."""
    if "mod" in _REF:
        return _REF["mod"]
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    mod = None
    if os.path.exists(os.path.join(ref_dir, "panfeed", "panfeed.py")):
        sys.path.insert(0, ref_dir)          # panfeed + the pyfaidx stand-in its input.py imports
        import logging
        logging.getLogger("panfeed").setLevel(logging.ERROR)
        from panfeed import panfeed as ref_panfeed      # noqa: E402
        from panfeed.classes import Seqinfo             # noqa: E402
        mod = (ref_panfeed, Seqinfo)
    _REF["mod"] = mod
    return mod


def reference_items(hb, S, Seqinfo):
    """Clusters of a HostBatch as the reference's feeder yields them (input.py:468):
    (dict strain -> [Seqinfo], cluster id, int64 presence vector)."""
    comp = bytes.maketrans(b"ACGT", b"TGCA")
    names = [f"g{i:05d}" for i in range(S)]
    first = np.searchsorted(hb.seqs["cluster"], np.arange(len(hb.clusters) + 1))
    sh = (62 - 2 * np.arange(32)).astype(np.uint64)
    lut = np.frombuffer(b"ACGT", np.uint8)
    idx = np.arange(S)
    items = []
    for c in range(len(hb.clusters)):
        presab = ((hb.presence[c, idx >> 5] >> (idx & 31)) & 1).astype(int)
        cluster = {}
        for q in hb.seqs[first[c]:first[c + 1]]:
            w0 = int(q["base_off"]) // 32
            w1 = w0 + (int(q["len"]) + 31) // 32
            codes = ((hb.packed[w0:w1, None] >> sh[None, :]) & np.uint64(3)).astype(np.uint8).ravel()
            seq = lut[codes[:int(q["len"])]].tobytes()
            cluster.setdefault(names[int(q["sample"])], []).append(
                Seqinfo(seq.decode(), seq.translate(comp).decode(), f"{names[int(q['sample'])]}_1", "ctg",
                        int(q["start"]), int(q["end"]), int(q["strand"]), int(q["offset"])))
        for i, s in enumerate(names):          # absent strains: empty lists (input.py:464-466)
            if not presab[i]:
                cluster[s] = []
        items.append((cluster, f"group_{int(hb.clusters['id'][c])}", presab))
    return items, names


def _ref_worker(job):
    """One cluster through the reference's cluster_cutter + pattern_hasher (panfeed.py:23-235),
    StringIO sinks instead of files."""
    import io
    import pandas as pd
    item, names, k, maf, cm, kind = job
    bases = sum(len(q.sequence) for v in item[0].values() for q in v)
    if kind == "reference":
        ref_panfeed, _ = load_reference()
        ret = ref_panfeed.cluster_cutter(item, k, "", False, True, cm, None)
        hp, kh = io.StringIO(), io.StringIO()
        genepres = pd.DataFrame(columns=names)
        pats = ref_panfeed.pattern_hasher((ret,), io.StringIO(), hp, kh, genepres, True, maf, None, patterns=set(),
                                          consider_missing_cluster=cm)
        return bases, len(ret[1]), len(pats)
    from oracle import ref_port
    res = ref_port.kmer_stage(item, k, "", True, cm)
    a, b, c = ref_port.pattern_stage((res,), True, maf, cm, set())
    return bases, len(res[1]), len(b) + len(c)


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path on all host
    cores (one worker process per core, each running cluster_cutter + pattern_hasher of the
    unmodified package: the arrangement of `panfeed --cores N`, __main__.py:299-344, without
    its single-writer pickle stream), on a bounded sample per step of the same synthetic
    workload the GPU arm runs (same generator, same seed, the first clusters)."""
    import multiprocessing as mp
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = config_of(args, args.config)
    cores = os.cpu_count() or 1
    S, L = cfg["samples"], cfg["gene_len"]
    per_step = cores                      # one cluster per core per step
    if S >= 5000:                         # the reference needs 8*S bytes per unique k-mer and hours per
        L = 200                           # 1.2-kb cluster at S >= 10,000 (SURVEY 8(d)): shortened clusters
    steps = args.warmup + args.steps
    n_sets = min(steps, 2)
    ref = load_reference()
    kind = "reference" if ref is not None else "port"
    generator = "pf_synth_fill (the GPU arm's generator, same seed)"
    try:
        from panfeed_b200 import capi
        hb = capi.synth_batch(0, cfg["seed"], S, per_step * n_sets, first_cluster=0,
                              total_clusters=cfg["clusters"], gene_len=L)
        if ref is not None:
            items, names = reference_items(hb, S, ref[1])
        else:
            from oracle.ref_port import CutSeq
            items, names = reference_items(hb, S, CutSeq)
    except Exception as e:                # no CUDA device: a numpy generator of the same model
        generator = f"numpy model of SURVEY 8(d) (pf_synth_fill unavailable: {type(e).__name__})"
        rng = np.random.default_rng(cfg["seed"])
        items = [numpy_cluster(rng, S, L, i, cfg["clusters"], ref[1] if ref else None)
                 for i in range(per_step * n_sets)]
        names = [f"g{i:05d}" for i in range(S)]
    sets = [items[i * per_step:(i + 1) * per_step] for i in range(n_sets)]
    ctx = mp.get_context("fork")
    times, bases_l, uniq_l = [], [], []
    with ctx.Pool(cores) as pool:
        for s in range(steps):
            jobs = [(it, names, cfg["k"], cfg["maf"], cfg["cm"], kind) for it in sets[s % len(sets)]]
            t0 = time.perf_counter()
            out = pool.map(_ref_worker, jobs, chunksize=1)
            dt = time.perf_counter() - t0
            if s >= args.warmup:
                times.append(dt)
                bases_l.append(sum(o[0] for o in out))
                uniq_l.append(sum(o[1] for o in out))
    total_t = sum(times)
    value = sum(bases_l) / total_t
    what = ("the UNMODIFIED reference package (oracle/_ref/panfeed/panfeed.py: cluster_cutter + pattern_hasher)"
            if kind == "reference" else
            "oracle/ref_port.py (Python restatement; oracle/_ref is not installed: run oracle/make_ref.sh)")
    line = {
        "impl": "reference", "metric": "input_bases_per_s", "value": value, "unit": "bases/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total_t / max(1, len(times)), "higher_is_better": True,
        "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": workload_config(cfg, 1),
        "unique_kmers_per_s": sum(uniq_l) / total_t,
        "cpu_baseline": {"value": value, "unit": "bases/s", "cores": cores, "kind": kind,
                         "sample": f"{what}, {cores} worker processes, {per_step} clusters of the workload "
                                   f"per step (clusters 0..{per_step * n_sets - 1}, gene_len {L}), inputs from "
                                   f"{generator}"},
        "e2e": {"value": value, "unit": "bases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def numpy_cluster(rng, S, L, cluster_index, total_clusters, Seqinfo=None):
    """One synthetic cluster as reference-style Seqinfo lists (numpy model of SURVEY 8(d));
    only used when no CUDA device is there for pf_synth_fill."""
    if Seqinfo is None:
        from oracle.ref_port import CutSeq as Seqinfo
    comp = str.maketrans("ACGT", "TGCA")
    anc = rng.integers(0, 4, L)
    founders = []
    for _ in range(8):
        f = anc.copy()
        m = rng.random(L) < 0.01
        f[m] = (f[m] + rng.integers(1, 4, int(m.sum()))) & 3
        founders.append(f)
    core = cluster_index < int(0.6 * total_clusters)
    p = 0.99 if core else rng.uniform(0.05, 0.95)
    names = [f"g{i:05d}" for i in range(S)]
    cluster, presab, absent = {}, np.zeros(S, dtype=int), []
    lut = np.frombuffer(b"ACGT", np.uint8)
    for i, s in enumerate(names):
        if rng.random() >= p:
            absent.append(s)
            continue
        presab[i] = 1
        lst = []
        for _ in range(2 if rng.random() < 0.01 else 1):
            q = founders[int(rng.integers(8))].copy()
            m = rng.random(L) < 0.001
            q[m] = (q[m] + rng.integers(1, 4, int(m.sum()))) & 3
            seq = lut[q].tobytes().decode()
            lst.append(Seqinfo(seq, seq.translate(comp), s + "_1", "ctg", 1001, 1000 + L,
                               int(rng.choice([1, -1])), 100))
        cluster[s] = lst
    for s in absent:
        cluster[s] = []
    return cluster, f"group_{cluster_index}", presab


def workload_config(cfg, world):
    per_rank = cfg["clusters"] if cfg["scaling"] == "weak" else -(-cfg["clusters"] // world)
    return {"workload": f"{cfg['name']}, k={cfg['k']}, {cfg['gene_len']} bp cut sequences",
            "baseline_config_id": cfg["id"], "samples": cfg["samples"],
            "clusters_total": cfg["clusters"] * (world if cfg["scaling"] == "weak" else 1),
            "clusters_per_gpu": per_rank, "gene_len": cfg["gene_len"], "k": cfg["k"], "maf": cfg["maf"],
            "consider_missing": bool(cfg["cm"]), "all_samples_targets": bool(cfg["targets"]),
            "l2": "inputs larger than L2: every step reads its whole packed plane (0.6 GB at 500 x 4000) and "
                  "writes / re-reads GBs of partial rows, far beyond the 126 MB L2; nothing survives between steps"}


# --------------------------------------------------------------------------
# --dump-outputs
# --------------------------------------------------------------------------
DUMP_BYTES = 64 * 10 ** 6
DUMP_SEED = 0x5EED5EED


def _mix64(x):
    """splitmix64 finaliser of a uint64 array."""
    with np.errstate(over="ignore"):
        x = x + np.uint64(0x9E3779B97F4A7C15)
        x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return x ^ (x >> np.uint64(31))


def _halves(x):
    """uint64 -> (high, low) 32-bit halves, each exact in float64."""
    return x >> np.uint64(32), x & np.uint64(0xFFFFFFFF)


class OutputDump:
    """What the timed path computed in its last step, as pf_collect hands it to a caller, written
    so that two builds can be compared array for array.  All arrays are float64 holding exact
    integers.  Pattern ids are numbered in discovery order, so each row carries the bits of its
    pattern instead, and rows are sorted by (cluster, k-mer).

      row_cluster [m]         global cluster id of the row
      row_kmer [m, 4]         the k-mer as 32-bit words (k <= 32: the first two are 0)
      row_count [m]           samples that carry the k-mer
      row_pattern_bits [m, W] its presence bitset, 32 samples a word
      cluster_id, cluster_rows, cluster_count_sum, cluster_samples [clusters]
                              every cluster: its rows, the sum of their counts, the popcount of
                              its cluster pattern
      totals [4]              rows, new k-mer patterns, new cluster patterns, positional records

    m is every row when they fit DUMP_BYTES; otherwise a fixed sample: the rows with the smallest
    seeded hash of (cluster, k-mer).  That sample depends on neither the row order nor on how the
    step was split into batches."""

    def __init__(self, n_samples, n_clusters):
        self.W = (n_samples + 31) // 32
        per_row = 8 * (1 + 4 + 1 + self.W)
        self.m = max(1, (DUMP_BYTES - 8 * (4 * n_clusters + 4) - 4096) // per_row)
        self.rows = None
        self.clusters = []
        self.totals = np.zeros(4, np.float64)

    @staticmethod
    def _bits(ctx, r, ns, ids, width):
        """Bits of pattern ids: this batch's new patterns from the result, older ones exported
        from the context's table."""
        key = "new_cluster_patterns" if ns else "new_kmer_patterns"
        base = r["cluster_pattern_base" if ns else "kmer_pattern_base"]
        ids = ids.astype(np.int64)
        out = np.zeros((len(ids), width), np.uint32)
        new = ids >= base
        out[new] = r[key][ids[new] - base][:, :width]
        if not new.all():
            old, inv = np.unique(ids[~new], return_inverse=True)
            table = np.stack([ctx.export_patterns(ns, i, 1)[0, :width] for i in old.tolist()])
            out[~new] = table[inv]
        return out

    def add(self, r, hb, ctx):
        """One collected batch (the result views are read here, not kept)."""
        narrow, wide = len(r["row_cluster"]), len(r["wide_row_cluster"])
        cl = np.concatenate([r["row_cluster"], r["wide_row_cluster"]]).astype(np.uint64)    # cluster ids
        k0 = np.concatenate([np.zeros(narrow, np.uint64), r["wide_row_kmer"][:, 0]])
        k1 = np.concatenate([r["row_kmer"], r["wide_row_kmer"][:, 1]])
        count = np.concatenate([r["row_count"], r["wide_row_count"]])
        pid = np.concatenate([r["row_pattern"], r["wide_row_pattern"]])
        cid = hb.clusters["id"].astype(np.uint64)      # cluster_pattern is in this (batch) order
        nc = len(cid)
        by_id = np.argsort(cid, kind="stable")
        local = by_id[np.searchsorted(cid[by_id], cl)]

        cbits = self._bits(ctx, r, 1, r["cluster_pattern"], self.W)
        self.clusters.append(np.stack([
            cid.astype(np.float64),
            np.bincount(local, minlength=nc).astype(np.float64),
            np.bincount(local, weights=count.astype(np.float64), minlength=nc),
            np.unpackbits(cbits.view(np.uint8), axis=1).sum(axis=1).astype(np.float64)], axis=1))
        self.totals += [narrow + wide, len(r["new_kmer_patterns"]), len(r["new_cluster_patterns"]), r["n_pos"]]

        h = _mix64(_mix64(_mix64(cl ^ np.uint64(DUMP_SEED)) ^ k0) ^ k1)
        if self.rows is not None and len(self.rows["h"]) >= self.m:
            sel = np.flatnonzero(h <= self.rows["h"].max())
        else:
            sel = np.arange(len(h))
        if len(sel) > self.m:
            sel = sel[np.argpartition(h[sel], self.m - 1)[:self.m]]
        batch = {"h": h[sel], "cl": cl[sel], "k0": k0[sel], "k1": k1[sel], "count": count[sel],
                 "bits": self._bits(ctx, r, 0, pid[sel], self.W)}
        if self.rows is not None:
            batch = {n: np.concatenate([self.rows[n], batch[n]]) for n in batch}
        if len(batch["h"]) > self.m:
            keep = batch["h"] <= np.partition(batch["h"], self.m - 1)[self.m - 1]
            batch = {n: a[keep] for n, a in batch.items()}
        self.rows = batch

    def write(self, out_dir):
        """DIR/<name>.npy for every array; returns {name: shape} and the bytes written."""
        rows = self.rows
        if len(rows["h"]) > self.m:            # hash ties at the cut: keep the smallest keys
            o = np.lexsort((rows["k1"], rows["k0"], rows["cl"], rows["h"]))[:self.m]
            rows = {n: a[o] for n, a in rows.items()}
        o = np.lexsort((rows["k1"], rows["k0"], rows["cl"]))
        clusters = np.concatenate(self.clusters)
        clusters = clusters[np.argsort(clusters[:, 0], kind="stable")]
        arrays = {
            "row_cluster": rows["cl"][o],
            "row_kmer": np.stack(_halves(rows["k0"][o]) + _halves(rows["k1"][o]), axis=1),
            "row_count": rows["count"][o],
            "row_pattern_bits": rows["bits"][o],
            "cluster_id": clusters[:, 0], "cluster_rows": clusters[:, 1],
            "cluster_count_sum": clusters[:, 2], "cluster_samples": clusters[:, 3],
            "totals": self.totals,
        }
        os.makedirs(out_dir, exist_ok=True)
        shapes, nbytes = {}, 0
        for name, a in arrays.items():
            a = np.ascontiguousarray(a, dtype=np.float64)
            np.save(os.path.join(out_dir, name + ".npy"), a)
            shapes[name] = list(a.shape)
            nbytes += a.nbytes
        assert nbytes <= DUMP_BYTES, nbytes
        return {"dir": out_dir, "arrays": shapes, "bytes": nbytes,
                "rows_sampled": bool(len(o) < self.totals[0])}


# --------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------
class Env:
    """Process-wide state of the B200 arm: ranks, device, collectives."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.affinity = pin_to_gpu_numa(self.local, self.world)
        if self.world > 1:
            # the ranks share the host: split its cores between their planning threads
            os.environ.setdefault("PF_HOST_THREADS", str(max(2, (os.cpu_count() or 16) // self.world)))
            # rank 0 prints ONE JSON line on stdout: NCCL's version banner / warnings go to stderr
            os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def reduce(self, x, op="max", dtype=None):
        """max / sum over ranks of a python number."""
        if self.world == 1:
            return x
        torch, dist = self.torch, self.dist
        t = torch.tensor([x], device=self.dev, dtype=dtype or (torch.float64 if isinstance(x, float) else torch.int64))
        dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
        return t.item()

    def gather(self, x):
        if self.world == 1:
            return [x]
        out = [None] * self.world
        self.dist.all_gather_object(out, x)
        return out


def pin_to_gpu_numa(local, world):
    """Bind this rank (its planning threads and the pinned buffers it allocates next) to the
    host cores NVML lists as local to its GPU, split between the ranks that share them.
    Returns a description for the bench line; any failure leaves the affinity alone."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        idx = local
        if vis:
            ent = vis.split(",")[local].strip()
            idx = int(ent) if ent.isdigit() else local
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        cpus = [i for i in range(n_cpu) if (words[i // 64] >> (i % 64)) & 1]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return {"pinned": False, "why": "no overlap between the GPU's cores and the allowed set"}
        if world > 1:
            # ranks whose GPUs share this core set take disjoint slices of it
            peers = []
            for r in range(world):
                try:
                    hr = pynvml.nvmlDeviceGetHandleByIndex(r if not vis else int(vis.split(",")[r]))
                    wr = pynvml.nvmlDeviceGetCpuAffinity(hr, (n_cpu + 63) // 64)
                    if list(wr) == list(words):
                        peers.append(r)
                except Exception:
                    pass
            if local in peers and len(peers) > 1:
                per = max(1, len(allowed) // len(peers))
                j = peers.index(local)
                mine = allowed[j * per:(j + 1) * per] or allowed
                allowed = mine
        os.sched_setaffinity(0, allowed)
        return {"pinned": True, "cores": len(allowed), "first_core": allowed[0], "last_core": allowed[-1]}
    except Exception as e:
        return {"pinned": False, "why": f"{type(e).__name__}: {e}"}


def rank_clusters(cfg, env):
    """(first global cluster, number of clusters, total clusters) of this rank."""
    if cfg["scaling"] == "weak":
        return env.rank * cfg["clusters"], cfg["clusters"], cfg["clusters"] * env.world
    per = -(-cfg["clusters"] // env.world)
    first = min(cfg["clusters"], env.rank * per)
    return first, min(per, cfg["clusters"] - first), cfg["clusters"]


def make_context(cfg, env, args):
    from panfeed_b200 import capi
    return capi.Context(cfg["k"], cfg["samples"], canonical=True, consider_missing=cfg["cm"],
                        cluster_equal_filter=False, emit_positions=2 if cfg["targets"] else 0, maf=cfg["maf"],
                        sort_bits=args.sort_bits, device=env.local)


def h2d_bytes(hb):
    return int(hb.packed.nbytes + hb.seqs.nbytes + hb.clusters.nbytes + hb.presence.nbytes)


STAGE_KEYS = ("ms_extract", "ms_hist", "ms_sort", "ms_mark", "ms_count", "ms_reduce", "ms_dedup", "ms_total")


def run_streamed(cfg, env, args, passes=1, warm_passes=1, dump=None):
    """One BASELINE config at FULL size, batch after batch (the inputs of configs 4 / 5 do not
    fit the host comfortably and a run of the product streams batches anyway).  Per pass:
      resident  pf_upload (untimed) + pf_execute timed with the library's CUDA events on the
                context's stream, summed over the batches;
      e2e       pinned host buffers -> pf_submit -> pf_collect (H2D + kernels + D2H), wall
                clock, summed over the batches;
    both followed by ONE global pattern exchange (N > 1), as in a real run.  The batches come
    from pf_synth_fill (bases generated on the device, copied to reused pinned host buffers)
    outside the timed regions.  `dump` (an OutputDump) is given the results of every batch of
    the last resident pass."""
    from panfeed_b200 import capi
    torch = env.torch
    first, n_cl, total = rank_clusters(cfg, env)
    S, L = cfg["samples"], cfg["gene_len"]
    ctx = make_context(cfg, env, args)
    exch = None
    if env.world > 1:
        from panfeed_b200 import dist as pfdist
        exch = pfdist.PatternExchange(ctx, env.dev)
    arena = capi.SynthArena()
    bounds = list(range(0, n_cl, cfg["batch"])) + [n_cl]

    def batch(b):
        return capi.synth_batch(env.local, cfg["seed"], S, bounds[b + 1] - bounds[b],
                                first_cluster=first + bounds[b], total_clusters=total, gene_len=L,
                                all_targets=cfg["targets"], arena=arena)

    n_b = len(bounds) - 1
    # warm-up: the first batches through both paths (buffers of the context grow to their size)
    for b in range(min(2, n_b)):
        hb = batch(b)
        ctx.upload(hb)
        ctx.execute()
        ctx.collect(copy=False)
        ctx.submit(hb)
        ctx.collect(copy=False)
    res = {}
    for mode in ("resident", "e2e"):
        if mode == "e2e" and args.no_e2e:
            continue
        def fresh():
            return {"ms": 0.0, "bases": 0, "instances": 0, "unique": 0, "rows": 0, "h2d": 0, "d2h": 0,
                    "launches": 0, "exchange_ms": 0.0, "stages": {k_: 0.0 for k_ in STAGE_KEYS}}
        tot = fresh()
        cold_ms = None
        exchange_ms_all = []
        # pass 0 is the cold pass of this mode (pools, tables and result buffers of the context grow
        # to the size of the workload: one-time allocations); it is reported as first_pass_ms and,
        # like the other warm-up passes, not averaged into the figures
        for pass_i in range(warm_passes + passes):
            if pass_i == 1:
                cold_ms = tot["ms"] + tot["exchange_ms"]
            if pass_i == warm_passes:
                tot = fresh()
            ctx.reset_patterns()
            env.barrier()
            for b in range(n_b):
                hb = batch(b)
                st0 = ctx.stats()
                if mode == "resident":
                    ctx.upload(hb)
                    ctx.execute()
                    st = ctx.stats()                # synchronises the stream, reads the stage events
                    tot["ms"] += st["ms_total"]
                    for k_ in STAGE_KEYS:
                        tot["stages"][k_] += st[k_]
                    r = ctx.collect(copy=False)
                    if dump is not None and pass_i == warm_passes + passes - 1:
                        dump.add(r, hb, ctx)
                else:
                    t0 = time.perf_counter()
                    ctx.submit(hb)
                    r = ctx.collect(copy=False)
                    tot["ms"] += (time.perf_counter() - t0) * 1e3
                    tot["h2d"] += h2d_bytes(hb)
                    tot["d2h"] += r["d2h_bytes"]
                st1 = ctx.stats()
                tot["bases"] += st1["bases"] - st0["bases"]
                tot["instances"] += st1["instances"] - st0["instances"]
                tot["unique"] += st1["unique_kmers"] - st0["unique_kmers"]
                tot["rows"] += st1["rows"] - st0["rows"]
                tot["launches"] += st1["total_launches"] - st0["total_launches"]
            tot["patterns_local"] = ctx.stats()["kmer_patterns"]
            tot["patterns_global"] = tot["patterns_local"]
            if exch is not None:
                env.barrier()
                t0 = time.perf_counter()
                out = exch.run()
                torch.cuda.synchronize(env.dev)
                tot["exchange_ms"] += (time.perf_counter() - t0) * 1e3
                exchange_ms_all.append(round((time.perf_counter() - t0) * 1e3, 2))
                tot["patterns_global"] = out["kmer"]["n_global"]
                tot["exchange_bytes_sent"] = out["kmer"]["bytes_sent"] + out["cluster"]["bytes_sent"]
                if out["kmer"]["ms"].get("stages"):
                    exchange_ms_all.append(out["kmer"]["ms"]["stages"])
        tot["cold_ms"] = cold_ms
        tot["exchange_ms_all"] = exchange_ms_all
        res[mode] = tot
    engine = ctx.stats()["engine"]
    if exch is not None:
        exch.close()
    ctx.close()
    del arena, exch
    torch.cuda.empty_cache()        # the exchange buffers of this config (torch's caching allocator)
    out = {"workload": workload_config(cfg, env.world), "n_gpus": env.world, "scaling": cfg["scaling"],
           "batches_per_gpu": n_b, "clusters_per_batch": cfg["batch"], "passes": passes, "warmup_passes": warm_passes,
           "engine": {0: "records (partition mode)", 1: "records (full sort)", 2: "block aggregation"}[engine]}
    for mode, tot in res.items():
        ms = env.reduce(tot["ms"] + tot["exchange_ms"], "max") / passes
        cold = env.reduce(tot["cold_ms"], "max")
        bases = env.reduce(tot["bases"], "sum") // passes
        uniq = env.reduce(tot["unique"], "sum") // passes
        d = {"ms": ms, "bases_per_s": bases / (ms * 1e-3), "unique_kmers_per_s": uniq / (ms * 1e-3),
             "bases": bases, "kmer_instances": env.reduce(tot["instances"], "sum") // passes,
             "unique_kmers": uniq, "rows": env.reduce(tot["rows"], "sum") // passes,
             "kmer_patterns_global": tot["patterns_global"],
             "kmer_patterns_sum_of_local": env.reduce(tot["patterns_local"], "sum"),
             "exchange_ms_once_per_run": env.reduce(tot["exchange_ms"], "max") / passes,
             "gpu_launches": env.reduce(tot["launches"], "sum") // passes,
             "first_pass_ms": cold, "exchange_ms_every_pass_this_rank": tot["exchange_ms_all"]}
        if mode == "resident":
            d["stages_ms"] = {k_: round(v_ / passes, 3) for k_, v_ in tot["stages"].items()}
            d["timing"] = "CUDA events of the library on the context's stream, per batch, summed; max over ranks"
        else:
            d["h2d_bytes"] = env.reduce(tot["h2d"], "sum") // passes
            d["d2h_bytes"] = env.reduce(tot["d2h"], "sum") // passes
            d["timing"] = "wall clock around pf_submit + pf_collect per batch, summed; max over ranks"
        out[mode] = d
    return out


def measure_pcie(env, nbytes=512 << 20):
    """Achieved H2D / D2H GB/s of every rank with all ranks copying at once: names the limiter
    of e2e at N > 1 by measurement (host DRAM / PCIe switch sharing), not by guess."""
    torch = env.torch
    host = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    devb = torch.empty(nbytes, dtype=torch.uint8, device=env.dev)
    out = {}
    for name, (dst, src) in (("h2d", (devb, host)), ("d2h", (host, devb))):
        dst.copy_(src, non_blocking=True)
        env.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(4):
            dst.copy_(src, non_blocking=True)
        e1.record()
        torch.cuda.synchronize(env.dev)
        out[name] = 4 * nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9
    # both directions at once, as the pipelined submit drives them
    s1, s2 = torch.cuda.Stream(env.dev), torch.cuda.Stream(env.dev)
    host2 = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    dev2 = torch.empty(nbytes, dtype=torch.uint8, device=env.dev)
    env.barrier()
    t0 = time.perf_counter()
    with torch.cuda.stream(s1):
        for _ in range(4):
            devb.copy_(host, non_blocking=True)
    with torch.cuda.stream(s2):
        for _ in range(4):
            host2.copy_(dev2, non_blocking=True)
    torch.cuda.synchronize(env.dev)
    dt = time.perf_counter() - t0
    out["bidir_each"] = 4 * nbytes / dt / 1e9
    g = env.gather({k_: round(v_, 1) for k_, v_ in out.items()})
    return {"GBps_per_rank_all_ranks_copying": g, "bytes_per_copy": nbytes}


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    # stdout carries ONE JSON line: everything libraries print there (NCCL's version banner comes
    # from C code, whatever NCCL_DEBUG_FILE says) goes to stderr until the line is printed
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line, default=str), flush=True)     # (a stray non-JSON value must not cost the line)
        os.dup2(2, 1)

    env = Env()
    torch, dist = env.torch, env.dist
    from panfeed_b200 import capi
    world, rank, local, dev = env.world, env.rank, env.local, env.dev
    cfg = config_of(args, args.config)

    # ---- on-hardware correctness of the exchange on THIS communicator, before any timing ----
    selfcheck = None
    if world > 1 and not args.no_selfcheck:
        from panfeed_b200 import selfcheck as sc
        selfcheck = [sc.check_exchange(local, cm) for cm in (False, True)]

    extra_ids = []
    if not args.no_extra:
        if args.extra is not None:
            extra_ids = [int(x) for x in args.extra.split(",") if x]
        elif args.config == 2:
            extra_ids = [3, 4, 5]

    if cfg["id"] != 2 or cfg["batch"] < cfg["clusters"]:
        # a streamed config as the headline: K = --steps passes over all its batches
        dump = None
        if args.dump_outputs and rank == 0:
            dump = OutputDump(cfg["samples"], rank_clusters(cfg, env)[1])
        sampler = ClockSampler(local, period=0.05)
        sampler.start()
        r = run_streamed(cfg, env, args, passes=args.steps, warm_passes=max(1, min(args.warmup, 3)), dump=dump)
        clocks = sampler.stop()
        if rank == 0:
            e2e = r.get("e2e")
            line = {"metric": "input_bases_per_s", "value": r["resident"]["bases_per_s"], "unit": "bases/s",
                    "n_gpus": world, "steps": r["passes"], "warmup": r["warmup_passes"], "ms_per_step": r["resident"]["ms"],
                    "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "u64",
                    "data": "synthetic", "config": r["workload"],
                    "unique_kmers_per_s": r["resident"]["unique_kmers_per_s"], "engine": r["engine"],
                    "streamed": r, "clocks": clocks, "gpu_launches": r["resident"]["gpu_launches"],
                    "e2e": None if e2e is None else {
                        "value": e2e["bases_per_s"], "unit": "bases/s", "ms_per_step": e2e["ms"],
                        "h2d_bytes_per_step": e2e["h2d_bytes"], "d2h_bytes_per_step": e2e["d2h_bytes"]},
                    "roofline": None, "exchange_selfcheck": selfcheck, "affinity": env.affinity}
            if dump is not None:
                line["dump_outputs"] = dump.write(args.dump_outputs)
            emit(line)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    S, C, L, k = cfg["samples"], cfg["clusters"], cfg["gene_len"], cfg["k"]
    total_clusters = C * world
    head_arena = capi.SynthArena()       # all four arrays of the batch in pinned host memory
    hb = capi.synth_batch(local, cfg["seed"], S, C, first_cluster=rank * C, total_clusters=total_clusters,
                          gene_len=L, all_targets=cfg["targets"], arena=head_arena)
    n_bases = hb.n_bases
    ctx = make_context(cfg, env, args)
    stream = torch.cuda.ExternalStream(ctx.stream_handle(), device=dev)
    exch = None
    if world > 1:
        from panfeed_b200 import dist as pfdist
        exch = pfdist.PatternExchange(ctx, dev)
    barrier = env.barrier
    exch_ms = {}
    exch_out = {}

    def step_resident():
        ctx.reset_patterns()
        ctx.execute()
        if exch is not None:
            out = exch.run()
            exch_out["last"] = out
            for ns in ("cluster", "kmer"):
                for k_, v_ in out[ns]["ms"].items():
                    if isinstance(v_, (int, float)):
                        exch_ms[ns + "_" + k_] = v_
                    elif v_:
                        exch_ms[ns + "_" + k_] = v_          # PF_EXCHANGE_TIMING: list of (stage, ms)

    # ---- value: batch resident in HBM -------------------------------------
    ctx.upload(hb)
    sampler = ClockSampler(local)
    for _ in range(max(3, args.warmup)):
        step_resident()
    launches0 = ctx.stats()["total_launches"]
    barrier()
    sampler.start()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    stage_ms = {}
    for _ in range(args.steps):
        step_resident()
        st = ctx.stats()
        for key in STAGE_KEYS:
            stage_ms[key] = stage_ms.get(key, 0.0) + st[key]
    e1.record(stream)
    barrier()
    clocks = sampler.stop()
    ms_total = env.reduce(float(e0.elapsed_time(e1)), "max")
    st = ctx.stats()
    launches = st["total_launches"] - launches0
    ms_step = ms_total / args.steps
    total_bases = env.reduce(n_bases, "sum")
    value = total_bases / (ms_step * 1e-3)
    # sizes of one step: read from a collect of the last execution
    r = ctx.collect(copy=False)
    dumped = None
    if args.dump_outputs and rank == 0:
        dump = OutputDump(S, C)
        dump.add(r, hb, ctx)
        dumped = dump.write(args.dump_outputs)
    st = ctx.stats()
    M = st["instances"]             # exactly one collected batch so far
    U = st["unique_kmers"]
    U_total = env.reduce(U, "sum")
    rows = st["rows"]
    passes = st["sort_passes"]
    for key in stage_ms:
        stage_ms[key] /= args.steps
    n_global = exch_out["last"]["kmer"]["n_global"] if exch_out else st["kmer_patterns"]

    # ---- e2e: pinned host buffers -> pf_submit -> pf_collect -----------------
    e2e = None
    if not args.no_e2e:
        for _ in range(2):
            ctx.reset_patterns()
            ctx.submit(hb)
            ctx.collect(copy=False)
        barrier()
        t0 = time.perf_counter()
        d2h = 0
        for _ in range(args.steps):
            ctx.reset_patterns()
            ctx.submit(hb)
            r = ctx.collect(copy=False)
            if exch is not None:
                exch.run()
            d2h = r["d2h_bytes"]
        torch.cuda.synchronize(dev)
        dt_rank = time.perf_counter() - t0
        dt = env.reduce(dt_rank, "max")
        h2d = h2d_bytes(hb)
        pst = ctx.stats()         # device times of the LAST pipelined submit, summed over its sub-batches
        e2e = {"value": total_bases * args.steps / dt, "unit": "bases/s",
               "stages_ms_pipelined_last_step": {k_: round(pst[k_], 3) for k_ in STAGE_KEYS + ("ms_h2d", "ms_d2h")},
               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "ms_per_step": 1e3 * dt / args.steps, "sub_batches": ctx.stats()["sub_batches"],
               "unique_kmers_per_s": U_total * args.steps / dt,
               "timing": "wall clock around K x (pf_submit + pf_collect [+ exchange]), max over ranks"}
        if world > 1:
            e2e["ms_per_step_per_rank"] = [round(1e3 * x / args.steps, 2) for x in env.gather(dt_rank)]
            e2e["achieved_GBps_per_rank_h2d_plus_d2h"] = [
                round((h2d + d2h) * args.steps / x / 1e9, 1) for x in env.gather(dt_rank)]
            e2e["pcie"] = measure_pcie(env)
            e2e["affinity_per_rank"] = env.gather(env.affinity)
    if exch is not None:
        exch.close()
    ctx.close()
    ctx = None

    # ---- the other BASELINE configs at full size --------------------------------
    extra = {}
    for cid in extra_ids:
        ecfg = config_of(args, cid)
        t0 = time.perf_counter()
        try:
            extra[f"config{cid}"] = run_streamed(ecfg, env, args)
            extra[f"config{cid}"]["bench_wall_s"] = round(time.perf_counter() - t0, 1)
        except Exception as e:          # an extra config must not take the headline down
            extra[f"config{cid}"] = {"error": f"{type(e).__name__}: {e}"}
            if world > 1:
                raise

    if rank == 0:
        line = headline_line(args, cfg, env, hb, st, stage_ms, ms_step, value, U, U_total, M, rows, passes,
                             n_bases, n_global, clocks, e2e, launches, exch_ms)
        if selfcheck is not None:
            line["exchange_selfcheck"] = selfcheck
        line["affinity"] = env.affinity
        if extra:
            line["extra_configs"] = extra
        if dumped is not None:
            line["dump_outputs"] = dumped
        if not args.no_cpu_baseline and world == 1:      # reported at N = 1 only
            line["cpu_baseline"] = cpu_baseline_c(hb, S, k, cfg["maf"], cfg["cm"], args.cpu_seconds)
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def headline_line(args, cfg, env, hb, st, stage_ms, ms_step, value, U, U_total, M, rows, passes, n_bases,
                  n_global, clocks, e2e, launches, exch_ms):
    """The JSON line of the headline config (one resident batch per step)."""
    S = cfg["samples"]
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    fused = stage_ms["ms_extract"] < 0.2          # K1 ran inside the histogram / first pass
    block = st["engine"] == 2                     # block aggregation: no records at all
    pass_ms = stage_ms["ms_sort"] / max(1, passes)
    k1_bytes = n_bases / 4 + 32 * len(hb.seqs) + R_BYTES * M          # SURVEY 8(d) K1
    pass_bytes = 2 * R_BYTES * M                                       # SURVEY 8(d) one K2 pass
    W4 = 4 * ((S + 31) // 32)
    tr = {}
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        pass
    n_launch = passes
    declared = None
    if block:
        kernel = ("kA_block_aggregate<canonical> (K1 extraction + all of K2 + the grouping of K3 in one "
                  "kernel: sequence chunks and k-mers are grouped in shared memory, no record reaches HBM)")
        pass_ms = stage_ms["ms_sort"]
        n_launch = 1
        wp = 16 if S > 1024 else (W4 // 4 + 3) // 4 * 4      # S > 1024: 512-sample slices, 16-word rows
        partial_bytes = st["partial_rows"] * (8 + 4 + 4 * wp)
        # what the kernel actually has to move: packed bases + 16-byte descriptors in,
        # partial rows (key, popcount, bitset) out
        alg_bytes = n_bases / 4 + 16 * len(hb.seqs) + partial_bytes
        per_rec = tr.get("kA_block_aggregate_dram_bytes_per_window")
        declared = {"what": "SURVEY 8(d) K1 figure (N/4 + 32*seqs + 12*M): the cheapest DECLARED stage this kernel "
                            "replaces; it never writes those 12-byte records, so this is not a bandwidth utilisation",
                    "bytes_per_launch": k1_bytes, "GBps": k1_bytes / (pass_ms * 1e-3) / 1e9,
                    "frac_of_peak": k1_bytes / (pass_ms * 1e-3) / 1e9 / peak}
        note = ("achieved = compulsory bytes of what the kernel does (packed bases + 16-B descriptors in, partial "
                "(k-mer, popcount, bitset) rows out) / its launch time.  The kernel is NOT HBM-bound: it replaces "
                "the declared K1 record write, the 8 declared radix passes of K2 and the record read of K3 "
                "(~220 B/base in SURVEY 8(d)) by grouping in shared memory, and is limited by instruction issue "
                "and shared-memory bandwidth (`limiter`, from the ncu capture in profiles/); launch_ms includes "
                "the rescue launches and their host syncs")
    elif fused:
        kernel = "k2_extract_scatter<canonical> (K1 extraction fused into the first radix pass)"
        alg_bytes = n_bases / 4 + R_BYTES * M
        per_rec = tr.get("k2_extract_scatter_dram_bytes_per_record")
        note = ("compulsory DRAM traffic of the fused kernel: packed bases in, 12-byte records out once "
                "(N/4 + R*M); it is instruction-bound")
    else:
        kernel = "k2_onesweep_pass<u64>"
        alg_bytes = pass_bytes
        per_rec = tr.get("k2_onesweep_pass_dram_bytes_per_record")
        note = "one radix pass reads and writes every 12-byte record once (2*R*M)"
    achieved = alg_bytes / (pass_ms * 1e-3) / 1e9
    traffic = per_rec * M if per_rec else None     # dram read+write per launch, scaled from the ncu capture
    roofline = {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes, "launch_ms": pass_ms, "launches_per_step": n_launch,
                "share_of_step": pass_ms / ms_step, "note": note}
    if block:
        roofline["limiter"] = tr.get("kA_limiter", "instruction issue / shared memory (see profiles/)")
        roofline["declared_model_side_figure"] = declared
    # whole-step DRAM rate from the summed ncu bytes of every kernel of a step
    step_bpw = tr.get("step_dram_bytes_per_window")
    whole_step = None
    if step_bpw and block:
        whole_step = {"dram_bytes_per_step": step_bpw * M, "dram_GBps": step_bpw * M / (ms_step * 1e-3) / 1e9,
                      "frac_of_peak": step_bpw * M / (ms_step * 1e-3) / 1e9 / peak,
                      "source": tr.get("step_source", "profiles/traffic.json")}
    k3_ms = stage_ms["ms_mark"] + stage_ms["ms_count"] + stage_ms["ms_reduce"]
    k4_stage = {"ms": stage_ms["ms_dedup"],
                "alg_GBps": (rows * W4 + st["kmer_patterns"] * W4 + 4 * rows) / max(stage_ms["ms_dedup"], 1e-6) / 1e6}
    if block:
        stages = {
            "kA_block_aggregate(+rescue launches, host syncs)": {
                "ms": stage_ms["ms_sort"], "reads_GB": n_bases / 4 / 1e9,
                "partial_rows": st["partial_rows"], "writes_GB": partial_bytes / 1e9},
            "kB_merge(kB1 merge + emit, incl. host sync)": {
                "ms": k3_ms, "alg_bytes": 2 * partial_bytes + 12 * U + rows * W4,
                "alg_GBps": (2 * partial_bytes + 12 * U + rows * W4) / max(k3_ms, 1e-6) / 1e6},
            "k4_dedup": k4_stage,
            "raw_ms": {k_: round(v_, 3) for k_, v_ in stage_ms.items()},
        }
    else:
        stages = {
            "k1_histogram(+extract)": {"ms": stage_ms["ms_extract"] + stage_ms["ms_hist"],
                                       "reads_GB": n_bases / 4 / 1e9},
            "k2_radix_passes": {"ms": stage_ms["ms_sort"], "passes": passes, "first_pass_fused_with_k1": fused},
            "k3_reduce(mark+local+rescue, incl. host sync)": {"ms": k3_ms},
            "k4_dedup": k4_stage,
            "raw_ms": {k_: round(v_, 3) for k_, v_ in stage_ms.items()},
        }
    line = {
        "metric": "input_bases_per_s", "value": value, "unit": "bases/s", "n_gpus": env.world,
        "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "u64",
        "data": "synthetic", "config": workload_config(cfg, env.world),
        "value_definition": "batch resident in HBM (contract); BASELINE's metric incl. H2D/D2H is `e2e`",
        "unique_kmers_per_s": U_total / (ms_step * 1e-3),
        "bases_per_step_per_gpu": n_bases, "kmer_instances_per_step_per_gpu": M,
        "unique_kmers_per_step_per_gpu": U, "rows_per_step_per_gpu": rows,
        "patterns_per_gpu": st["kmer_patterns"], "kmer_patterns_global": n_global,
        "engine": {0: "records (partition mode)", 1: "records (full sort)", 2: "block aggregation"}[st["engine"]],
        "roofline": roofline, "whole_step": whole_step, "stages": stages,
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
    }
    if cfg["targets"]:
        line["positional_records_per_s"] = env.world * M / (ms_step * 1e-3)
    if exch_ms:
        line["exchange_ms_last_step_rank0"] = {k_: round(v_, 3) if isinstance(v_, (int, float)) else v_
                                               for k_, v_ in exch_ms.items()}
    return line


if __name__ == "__main__":
    main()
