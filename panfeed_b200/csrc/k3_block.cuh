// Block aggregation: K1 + K2 + K3 without ever materialising a record.
//
// The sequences of one gene cluster are near-identical copies of one gene, so the windows
// that START inside the same run of 16 positions of every sequence of the cluster hold only
// a few hundred distinct k-mers between them (one per haplotype and position), however many
// samples there are.
//
//   kA_block_aggregate  work item: (cluster, run of 16 window positions[, slice of 512 samples]).
//                       A CTA walks a SEGMENT of consecutive runs of one (cluster, slice): it
//                       keeps its sequences' descriptors and words in registers from run to
//                       run (one new 64-bit word per sequence every second run) and undoes
//                       only what a run touched in its tables.
//                       Level 1: every sequence contributes the R = k + 15 bases its 16
//                       windows cover as ONE 128-bit chunk; identical chunks (same haplotype)
//                       meet in a shared-memory chunk table and only OR one sample bit there:
//                       ~25 instructions per sequence and run instead of per window.
//                       Level 2: the few dozen DISTINCT chunks are cut into their 16 k-mers
//                       (forward / reverse complement / canonical), each k-mer is looked up in
//                       a shared-memory open-addressing table and takes the chunk's whole
//                       W-word sample bitset.  The CTA ends by writing its distinct k-mers,
//                       popcounts and bitsets ("partial rows") to a slab in HBM: ~1/30 of the
//                       bytes the records would have taken, written once.  A row of one sample
//                       (most rows) is written as its key and a one-sample code, without the
//                       bitset (see slab_cnt).  Every run keeps its own slab, so the kernels
//                       after kA see per-run items.
//   kB1/kB3             a k-mer can start in two runs (indels, clamped flanks, paralogs,
//                       repeats), so the partial rows of one cluster are merged by FULL key in a
//                       per-cluster open-addressing table in global memory: the first row of a
//                       key owns it, later ones OR their bitset into the owner's; owners are
//                       filtered on their popcount with the integer MAF window and emitted.
//   kB4/kB5             with sample slices (S > 1024) kB1 merges per (cluster, slice); kB4
//                       links the slices of a k-mer and sums their popcounts, kB5 filters on the
//                       sum and assembles the full-width bitsets of the survivors.
//
// Exact for any input: nothing depends on the sequences being aligned — alignment only
// decides how few partial rows there are.  A run holding more distinct k-mers than the
// shared-memory tables take flags itself; the host reruns just those runs with larger tables
// and, past the largest, sends the batch through the record path (k2_extract_scatter +
// k3_local_direct / k3_local).
//
// Shared memory of kA: see ARunView.  The all-ones word marks an empty k-mer slot; it is a
// valid k-mer only for k = 32 in --non-canonical mode, which stays on the record path.
//
// Replaces the window loop and `cluster_dict[kmer][sortstrain[strain]] = 1` of
// /root/reference/panfeed/panfeed.py:54-88 and the filters of :190-204.
#pragma once
#include "pf_common.cuh"
#include "k1_extract.cuh"
#include "k3_local.cuh"

namespace pf {

struct SeqLite {           // 16 bytes: what kA needs of a sequence, one 128-bit load
  uint32_t word_off;       // first 64-bit word in the 2-bit plane
  uint32_t len;
  uint32_t sample_flags;   // sample rank | (ambiguous ? 1u << 31 : 0)
  uint32_t amb_word_off;   // first 32-bit word in the ambiguity bit plane
};
struct ClusterBlk {        // 16 bytes
  uint32_t seq_start, n_seqs, max_nwin, reserved;
};

#ifndef PF_KA_THREADS
#define PF_KA_THREADS 256
#endif
constexpr int kBlkThreads = PF_KA_THREADS;
constexpr int kBlkWarps = kBlkThreads / 32;
constexpr int kBlkRun = 16;                       // windows per task
constexpr uint32_t kBlkOverflow = 0xffffffffu;    // slab count of a block that did not fit
// slab_cnt[p], the state of partial row p:
//   popcount           (kA) two or more samples: the bitset is in slab_rows
//   kCntSingle | s     (kA) ONE sample, rank s < 1024 inside the slice: slab_rows holds nothing for p
//   kCntDead           (kB1) folded into an earlier row of the same k-mer
//   kCntDirty          (kB1) received another row's bits: recount from the row
//   kCntLocked         (kB1, transient) a one-sample owner whose bitset is being written out
constexpr uint32_t kCntSingle = 0x80000000u;
constexpr uint32_t kCntLocked = 0xfffffffdu, kCntDead = 0xfffffffeu, kCntDirty = 0xffffffffu;
__device__ __forceinline__ bool cnt_single(uint32_t code) { return (code & 0xfffffc00u) == kCntSingle; }
// the count of partial row p from its slab_cnt code; kCntDead for a row folded into another.
// Every reader of slab_cnt after kB1 goes through this.
__device__ __forceinline__ uint32_t partial_row_count(const uint32_t* __restrict__ slab_rows, uint32_t code,
                                                      size_t p, uint32_t WP) {
  if (cnt_single(code)) return 1u;
  if (code != kCntDirty) return code;          // popcount, or kCntDead
  const uint4* row = reinterpret_cast<const uint4*>(slab_rows + p * WP);
  uint32_t cnt = 0;
  for (uint32_t q = 0; q < WP / 4; ++q) {
    const uint4 x = row[q];
    cnt += __popc(x.x) + __popc(x.y) + __popc(x.z) + __popc(x.w);
  }
  return cnt;
}

__global__ void plan_seq_lite(const SeqDev* __restrict__ seqs, uint32_t n, SeqLite* __restrict__ out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const SeqDev d = seqs[i];
  SeqLite l;
  l.word_off = (uint32_t)(d.base_off >> 5);
  l.len = d.len;
  l.sample_flags = d.sample | ((d.flags & 2u) ? 0x80000000u : 0u);
  l.amb_word_off = (uint32_t)(d.amb_off >> 5);
  out[i] = l;
}

// ---------------------------------------------------------------------------
// Device-side planning of an upload ("lite" upload): the caller's pf_seq_desc array goes to the
// device as it is and ONE kernel does what the host planner does per sequence - validation
// (include/panfeed_b200.h: pf_seq_desc), rebasing to the sub-range, the 64-byte SeqDev and the
// 16-byte SeqLite - plus the batch totals.  The host then touches no descriptor at all: with
// several ranks sharing the host's cores the per-sequence planning (~15 ns per sequence and
// thread) was what bounded the end-to-end rate.  Only the block engine can run from it (no
// record offsets are computed); a batch that falls back to the record engine is re-planned on
// the host from the device copy of the descriptors.
// ---------------------------------------------------------------------------
struct LiteTotals {          // 64 bytes, zeroed (err = all ones) before the kernel
  unsigned long long bases, windows, pos_windows;
  unsigned long long err;    // min over bad sequences of (index << 32 | code); ~0 = none
  uint32_t pad[8];
};
enum : uint32_t { kLiteErrCluster = 1, kLiteErrClusterOrder, kLiteErrSample, kLiteErrSampleOrder, kLiteErrPresence,
                  kLiteErrAlign, kLiteErrPlane, kLiteErrStrand, kLiteErrAmbiguous, kLiteErrOrder };

__global__ void __launch_bounds__(256)
plan_from_raw(const pf_seq_desc* __restrict__ raw, uint32_t n, uint32_t cluster_base, uint64_t base_rebase,
              uint32_t n_clusters, uint32_t S, uint32_t W, const uint32_t* __restrict__ presence,
              uint64_t plane_bases, int k, uint32_t emit_positions, SeqDev* __restrict__ out,
              SeqLite* __restrict__ lite, LiteTotals* __restrict__ tot) {
  __shared__ unsigned long long s_sum[3][8];
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long bases = 0, windows = 0, posw = 0;
  if (i < n) {
    const pf_seq_desc q = raw[i];
    uint32_t err = 0;
    const uint32_t cluster = q.cluster - cluster_base;
    const uint64_t base_off = q.base_off - base_rebase;
    if (q.cluster < cluster_base || cluster >= n_clusters) err = kLiteErrCluster;
    else if (q.sample >= S) err = kLiteErrSample;
    else if (!((presence[(size_t)cluster * W + (q.sample >> 5)] >> (q.sample & 31u)) & 1u)) err = kLiteErrPresence;
    else if (q.base_off < base_rebase || (base_off & 63u)) err = kLiteErrAlign;
    else if (base_off + q.len > plane_bases) err = kLiteErrPlane;
    else if (q.strand != 1 && q.strand != -1) err = kLiteErrStrand;
    else if (q.flags & PF_SEQ_AMBIGUOUS) err = kLiteErrAmbiguous;
    else if (i) {
      const pf_seq_desc p = raw[i - 1];
      if (q.cluster < p.cluster) err = kLiteErrClusterOrder;
      else if (q.cluster == p.cluster && q.sample < p.sample) err = kLiteErrSampleOrder;
    }
    if (err) {
      atomicMin(&tot->err, ((unsigned long long)i << 32) | err);
    } else {
      const bool target = emit_positions && (q.flags & PF_SEQ_TARGET);
      SeqDev d;
      d.base_off = base_off; d.amb_off = 0; d.len = q.len; d.sample = q.sample; d.cluster = cluster;
      d.flags = target ? 1u : 0u;
      d.start = q.start; d.end = q.end; d.offset = q.offset; d.strand = q.strand;
      d.rec_off = 0; d.pos_off = 0; d.wrec_off = 0; d.pwide_off = 0;
      out[i] = d;
      SeqLite l;
      l.word_off = (uint32_t)(base_off >> 5); l.len = q.len; l.sample_flags = q.sample; l.amb_word_off = 0;
      lite[i] = l;
      const uint32_t nwin = q.len >= (uint32_t)k ? q.len - (uint32_t)k + 1u : 0u;
      bases = q.len; windows = nwin; posw = target ? nwin : 0u;
    }
  }
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) {
    bases += __shfl_xor_sync(kFull, bases, m);
    windows += __shfl_xor_sync(kFull, windows, m);
    posw += __shfl_xor_sync(kFull, posw, m);
  }
  if ((threadIdx.x & 31u) == 0) {
    s_sum[0][threadIdx.x >> 5] = bases; s_sum[1][threadIdx.x >> 5] = windows; s_sum[2][threadIdx.x >> 5] = posw;
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    unsigned long long t = 0;
    for (int w = 0; w < 8; ++w) t += s_sum[threadIdx.x][w];
    if (t) atomicAdd(threadIdx.x == 0 ? &tot->bases : threadIdx.x == 1 ? &tot->windows : &tot->pos_windows, t);
  }
}

// one warp per cluster: its sequence range (sequences are sorted by cluster), the
// longest window count and from it the number of position blocks
__global__ void plan_cluster_blocks(const SeqDev* __restrict__ seqs, uint32_t n_seqs, uint32_t n_clusters,
                                    int k, uint32_t block_windows, ClusterBlk* __restrict__ cb,
                                    uint32_t* __restrict__ n_items) {
  const uint32_t c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (c >= n_clusters) return;
  const uint32_t lane = lane_id();
  auto lower = [&](uint32_t v) {              // first sequence with cluster >= v
    uint32_t lo = 0, hi = n_seqs;
    while (lo < hi) {
      const uint32_t mid = (lo + hi) >> 1;
      if (seqs[mid].cluster < v) lo = mid + 1; else hi = mid;
    }
    return lo;
  };
  const uint32_t s0 = lower(c), s1 = lower(c + 1);
  uint32_t mx = 0;
  for (uint32_t s = s0 + lane; s < s1; s += 32) {
    const uint32_t len = seqs[s].len;
    if (len >= (uint32_t)k) mx = max(mx, len - (uint32_t)k + 1u);
  }
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) mx = max(mx, __shfl_xor_sync(kFull, mx, m));
  if (lane == 0) {
    ClusterBlk b;
    b.seq_start = s0; b.n_seqs = s1 - s0; b.max_nwin = mx; b.reserved = 0;
    cb[c] = b;
    n_items[c] = (mx + block_windows - 1) / block_windows;
  }
}

// one warp per cluster: first sequence of every sample slice (sequences are in sample order)
__global__ void plan_cluster_slices(const SeqDev* __restrict__ seqs, const ClusterBlk* __restrict__ cb,
                                    uint32_t n_clusters, uint32_t n_slices, uint32_t slice_samples,
                                    uint32_t* __restrict__ slice_seq) {
  const uint32_t c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (c >= n_clusters) return;
  const ClusterBlk b = cb[c];
  for (uint32_t s = lane_id(); s <= n_slices; s += 32) {
    const uint32_t first_sample = s * slice_samples;
    uint32_t lo = 0, hi = b.n_seqs;                 // first sequence with sample >= first_sample
    while (lo < hi) {
      const uint32_t mid = (lo + hi) >> 1;
      if (seqs[b.seq_start + mid].sample < first_sample) lo = mid + 1; else hi = mid;
    }
    slice_seq[(size_t)c * (n_slices + 1) + s] = s == n_slices ? b.n_seqs : lo;
  }
}

// one thread per kA work item (cluster, run, slice): everything the kernel needs to find its
// sequences, in one 16-byte load instead of a chain of three dependent ones
__global__ void plan_item_desc(const uint32_t* __restrict__ item_base, const uint32_t* __restrict__ item_cluster,
                               const ClusterBlk* __restrict__ cb, const uint32_t* __restrict__ slice_seq,
                               uint32_t n_run_items, uint32_t n_slices, uint32_t run_windows,
                               uint4* __restrict__ desc) {
  const uint32_t item = blockIdx.x * blockDim.x + threadIdx.x;
  if (item >= n_run_items * n_slices) return;
  const uint32_t run_item = item / n_slices, slice = item - run_item * n_slices;
  const uint32_t c = item_cluster[run_item];
  const ClusterBlk b = cb[c];
  uint32_t lo = 0, hi = b.n_seqs;
  if (n_slices > 1) {
    lo = slice_seq[(size_t)c * (n_slices + 1) + slice];
    hi = slice_seq[(size_t)c * (n_slices + 1) + slice + 1];
  }
  desc[item] = make_uint4(b.seq_start + lo, b.seq_start + hi, (run_item - item_base[c]) * run_windows, c);
}

// ---------------------------------------------------------------------------
// shared-memory table
// ---------------------------------------------------------------------------
struct BlkHead {           // 64 bytes at the start of kA's shared memory (see ARunView)
  uint32_t n_unique, overflow, n_pass, row_base, ok, work, seg[2], singles, pad[7];
};
__device__ __forceinline__ uint32_t ld_volatile_shared(const uint32_t* p) {
  return *reinterpret_cast<const volatile uint32_t*>(p);
}
__device__ __forceinline__ uint32_t blk_hash(uint32_t kh, uint32_t kl, uint32_t shift) {
  return ((kl ^ (kh * 0x85ebca6bu)) * 0x9e3779b1u) >> shift;
}

// ---------------------------------------------------------------------------
// kA
// ---------------------------------------------------------------------------
struct BlkPlan {
  const uint32_t* item_base;     // [n_clusters + 1] exclusive scan of blocks per cluster
  const uint32_t* item_cluster;  // [n_items] inverse of item_base
  const ClusterBlk* cblk;
  uint32_t n_clusters;
  uint32_t block_windows;        // B = kBlkRun
  uint32_t slots, cslots;        // k-mer table / chunk table sizes of kA (powers of two)
  uint32_t cap;                  // k-mer rows of kA (dense, handed out on insertion)
  uint32_t W, WP;                // bitset words of a partial row, slab row stride (W rounded up to 4)
  // sample slices (S > 1024): a work item is (cluster, run, slice); a partial row holds the
  // bits of `slice_samples` consecutive sample ranks only
  uint32_t n_slices;             // 1: no slicing
  uint32_t slice_samples;        // multiple of 32
  const uint32_t* slice_seq;     // [n_clusters][n_slices + 1] first sequence (cluster-relative) of every slice
  const uint4* item_desc;        // [n_items * n_slices] {first seq, end seq (absolute), first window, cluster}
  uint32_t n_run_items;          // (cluster, run) items of the batch
};

// Shared memory of kA.  Both tables hand out DENSE row ids on insertion, so the epilogue needs
// no compaction pass.  The tables are cleared once per CTA; after a run only what it touched is
// undone: the key slot of every k-mer row (rslot) and the state slot of every chunk id (cslot)
// are recorded on insertion, the pool rows are zeroed as they are copied out, and the chunk rows
// 0..n_chunks-1 are cleared.  An overflowing run may have claimed slots without a row; after it
// everything is cleared.
//
// chunk table: the R = k + 15 bases that the 16 windows of a run cover, as a 128-bit key
//   (top-aligned).  Sequences of a cluster are copies of a few haplotypes, so the ~500
//   sequences of a run collapse into a few dozen distinct chunks; only those are cut into
//   k-mers.  A slot's state word goes empty -> locked -> (full | chunk id).
// k-mer table: 64-bit keys claimed with one CAS; rowid[slot] is published afterwards
//   (0xffff = not yet), readers of a freshly claimed slot spin for those few cycles.
constexpr uint32_t kChunkEmpty = 0u, kChunkLocked = 1u, kChunkFull = 0x80000000u;
struct ARunView {
  BlkHead* h;              // n_unique = k-mer rows handed out, work = chunk ids handed out
  uint64_t* keys;          // [slots]
  uint64_t* rkey;          // [cap + 1]   key of row id
  uint64_t* ckhi;          // [ccap]
  uint64_t* cklo;          // [ccap]
  uint32_t* cstate;        // [cslots]
  uint32_t* pool;          // [(cap + 1) * WS]   row `cap` takes the ORs of an overflowing block
  uint32_t* crows;         // [ccap * WS]
  uint16_t* rowid;         // [slots]
  uint16_t* cmeta;         // [ccap]  low byte: bitset word of the chunk's first sample; bit 15: other words too
  uint16_t* rslot;         // [cap + 1]  key slot of row id
  uint16_t* cslot;         // [ccap]     state slot of chunk id
  uint32_t mask, shift, cmask, cshift, cap, ccap;
};
__host__ __device__ inline uint32_t blkA_ccap(uint32_t cslots) { return cslots * 3u / 4u; }
// slots: k-mer key slots (power of two); cap: k-mer rows (<= 13/16 slots); cslots: chunk slots
__host__ __device__ inline uint32_t blkA_smem_bytes(uint32_t slots, uint32_t cap, uint32_t cslots, uint32_t W) {
  const uint32_t ccap = blkA_ccap(cslots), WS = W | 1u;
  return (uint32_t)sizeof(BlkHead) + slots * 8u + (cap + 1u) * 8u + ccap * 16u + cslots * 4u +
         (cap + 1u) * WS * 4u + ccap * WS * 4u + slots * 2u + ccap * 2u + (cap + 1u) * 2u + ccap * 2u + 16u;
}
__device__ __forceinline__ ARunView arun_view(unsigned char* raw, uint32_t slots, uint32_t cap, uint32_t cslots, uint32_t W) {
  ARunView a;
  const uint32_t WS = W | 1u;
  a.cap = cap;
  a.ccap = blkA_ccap(cslots);
  a.h = reinterpret_cast<BlkHead*>(raw);
  a.keys = reinterpret_cast<uint64_t*>(raw + sizeof(BlkHead));
  a.rkey = a.keys + slots;
  a.ckhi = a.rkey + (a.cap + 1u);
  a.cklo = a.ckhi + a.ccap;
  a.cstate = reinterpret_cast<uint32_t*>(a.cklo + a.ccap);
  a.pool = a.cstate + cslots;
  a.crows = a.pool + (a.cap + 1u) * WS;
  a.rowid = reinterpret_cast<uint16_t*>(a.crows + a.ccap * WS);
  a.cmeta = a.rowid + slots;
  a.rslot = a.cmeta + a.ccap;
  a.cslot = a.rslot + (a.cap + 1u);
  a.mask = slots - 1u;
  a.shift = 32u - (uint32_t)__popc(a.mask);
  a.cmask = cslots - 1u;
  a.cshift = 32u - (uint32_t)__popc(a.cmask);
  return a;
}
// chunk id of (hi, lo); 0xffffffff if the chunk table is full (the caller then cuts the run
// into k-mers itself)
__device__ __noinline__ uint32_t chunk_find_or_insert(const ARunView a, uint64_t hi, uint64_t lo, uint32_t wofs) {
  const uint64_t m = (hi ^ (hi >> 29)) * 0x9e3779b97f4a7c15ULL + (lo ^ (lo >> 31)) * 0xc2b2ae3d27d4eb4fULL;
  uint32_t s = (uint32_t)(m >> 32) >> a.cshift;
  uint32_t spins = 0;
  for (uint32_t probes = 0; probes <= a.cmask;) {
    const uint32_t st = ld_volatile_shared(&a.cstate[s]);
    if (st & kChunkFull) {
      const uint32_t id = st & 0xffffu;
      if (*reinterpret_cast<const volatile uint64_t*>(&a.ckhi[id]) == hi &&
          *reinterpret_cast<const volatile uint64_t*>(&a.cklo[id]) == lo)
        return id;
      s = (s + 1u) & a.cmask;
      ++probes;
      continue;
    }
    if (st == kChunkEmpty) {
      if (atomicCAS(&a.cstate[s], kChunkEmpty, kChunkLocked) == kChunkEmpty) {
        const uint32_t id = atomicAdd(&a.h->work, 1u);
        if (id >= a.ccap) {                                   // no row left: give the slot back
          *reinterpret_cast<volatile uint32_t*>(&a.cstate[s]) = kChunkEmpty;
          return 0xffffffffu;
        }
        a.cmeta[id] = (uint16_t)wofs;
        a.cslot[id] = (uint16_t)s;
        *reinterpret_cast<volatile uint64_t*>(&a.ckhi[id]) = hi;
        *reinterpret_cast<volatile uint64_t*>(&a.cklo[id]) = lo;
        __threadfence_block();
        *reinterpret_cast<volatile uint32_t*>(&a.cstate[s]) = kChunkFull | id;
        return id;
      }
      continue;
    }
    if (++spins > (1u << 14)) break;          // locked: its owner publishes it in a few cycles
    __nanosleep(20);                          // (lets the owner run if it is a lane of this warp)
  }
  return 0xffffffffu;
}
// row id of a k-mer (insert if new); a.cap = the scratch row when the block overflows
__device__ __noinline__ uint32_t kmer_row_slow(const ARunView a, uint64_t key, uint32_t h, uint32_t WS) {
  const uint32_t limit = min(a.mask, 96u);
  bool found = false;
  for (uint32_t probes = 0; probes < limit; ++probes) {
    uint64_t cur = *reinterpret_cast<const volatile uint64_t*>(&a.keys[h]);
    if (cur == ~0ull) {
      cur = atomicCAS(reinterpret_cast<unsigned long long*>(&a.keys[h]), ~0ull, (unsigned long long)key);
      if (cur == ~0ull) {                                     // this thread owns the new slot
        uint32_t id = atomicAdd(&a.h->n_unique, 1u);
        if (id >= a.cap) { a.h->overflow = 1u; id = a.cap; }
        else a.rslot[id] = (uint16_t)h;
        a.rkey[id] = key;
        __threadfence_block();
        *reinterpret_cast<volatile uint16_t*>(&a.rowid[h]) = (uint16_t)id;
        return id;
      }
    }
    if (cur == key) { found = true; break; }
    h = (h + 1u) & a.mask;
  }
  if (!found) { a.h->overflow = 1u; return a.cap; }
  for (uint32_t spins = 0; spins < (1u << 14); ++spins) {
    const uint32_t id = *reinterpret_cast<const volatile uint16_t*>(&a.rowid[h]);
    if (id != 0xffffu) return id;
    __nanosleep(20);                          // (lets the owner run if it is a lane of this warp)
  }
  a.h->overflow = 1u;
  return a.cap;
}

#ifndef PF_KA_MIN_CTAS
#define PF_KA_MIN_CTAS 4
#endif
// A CTA walks SEGMENTS: `seg_runs` consecutive (cluster, run) items of one slice (item =
// run_item * n_slices + slice), taken from counters[LC_SEGMENT] after the first one; with an
// item list (a rescue launch) a segment is one listed item.  Every run still gets its own slab.
// Across the runs of a segment a thread keeps its first two sequences of the (cluster, slice) in
// registers: descriptor and the 64-bit words wi, wi + 1 of the run plus wi + 2, requested a run
// ahead of its use.  A run starts at a multiple of 16, so its R <= 47 bases lie in two words.
template <bool CANON>
__global__ void __launch_bounds__(kBlkThreads, PF_KA_MIN_CTAS)
kA_block_aggregate(const uint64_t* __restrict__ bases, const uint32_t* __restrict__ ambbits,
                   const SeqLite* __restrict__ seqs, BlkPlan plan, int k,
                   uint64_t* __restrict__ slab_keys, uint32_t* __restrict__ slab_rows,
                   uint32_t* __restrict__ slab_base, uint32_t* __restrict__ slab_count,
                   uint32_t* __restrict__ slab_cnt /* popcount or one-sample code of every partial row */,
                   uint32_t partial_capacity, uint32_t* __restrict__ counters,
                   const uint32_t* __restrict__ item_list /* null: segments of seg_runs runs */,
                   uint32_t n_segs, uint32_t seg_runs,
                   uint32_t* __restrict__ rescue_items /* out: items whose table overflowed */) {
  extern __shared__ __align__(16) unsigned char blk_raw[];
  const uint32_t W = plan.W, WS = W | 1u;
  const ARunView a = arun_view(blk_raw, plan.slots, plan.cap, plan.cslots, W);
  const uint32_t tid = threadIdx.x;

  auto clear_tables = [&]() {
    for (uint32_t i = tid; i < plan.slots; i += kBlkThreads) { a.keys[i] = ~0ull; a.rowid[i] = 0xffffu; }
    for (uint32_t i = tid; i < plan.cslots; i += kBlkThreads) a.cstate[i] = kChunkEmpty;
    for (uint32_t i = tid; i < (a.cap + 1u) * WS; i += kBlkThreads) a.pool[i] = 0u;
    for (uint32_t i = tid; i < a.ccap * WS; i += kBlkThreads) a.crows[i] = 0u;
  };
  clear_tables();
  if (tid == 0) { a.h->n_unique = 0; a.h->overflow = 0; a.h->work = 0; a.h->n_pass = 0; a.h->singles = 0; }
  __syncthreads();

  const uint32_t sh64 = 64u - 2u * (uint32_t)k;
  const uint32_t R = (uint32_t)k + (uint32_t)kBlkRun - 1u;      // bases a full run covers (<= 47)
  // top-aligned masks of the R bases
  const uint64_t cm_hi = R >= 32u ? ~0ull : (~0ull << (64u - 2u * R));
  const uint64_t cm_lo = R > 32u ? (~0ull << (64u - 2u * (R - 32u))) : 0ull;

  // one k-mer (in the low 2k bits) -> row, OR `nw` words starting at src into it
  auto put_bits = [&](uint64_t key, const uint32_t* src, uint32_t first_word, uint32_t nw) {
    const uint32_t h = blk_hash((uint32_t)(key >> 32), (uint32_t)key, a.shift);
    uint32_t id = 0xffffu;
    if (*reinterpret_cast<const volatile uint64_t*>(&a.keys[h]) == key)
      id = *reinterpret_cast<const volatile uint16_t*>(&a.rowid[h]);
    if (id == 0xffffu) id = kmer_row_slow(a, key, h, WS);
    uint32_t* dst = a.pool + id * WS + first_word;
    for (uint32_t w = 0; w < nw; ++w) {
      const uint32_t x = src[w];
      if (x) atomicOr(dst + w, x);
    }
  };
  auto put_kmer = [&](uint64_t fwd, const uint32_t* src, uint32_t first_word, uint32_t nw) {
    const uint64_t rc = revcomp2(fwd, k);
    if (CANON) put_bits(rc < fwd ? rc : fwd, src, first_word, nw);
    else { put_bits(fwd, src, first_word, nw); put_bits(rc, src, first_word, nw); }
  };

  // the thread's sequences j = 0, 1 of the (cluster, slice) whose first sequence is st_lo, at
  // word index st_wi: window count (0: none), sample | ambiguity flag, first word, words
  uint32_t st_lo = 0xffffffffu, st_wi = 0;
  uint32_t nw0 = 0, nw1 = 0, sf0 = 0, sf1 = 0, wo0 = 0, wo1 = 0;
  uint64_t c0 = 0, n0 = 0, p0 = 0, c1 = 0, n1 = 0, p1 = 0;

  uint32_t seg = blockIdx.x;
  for (uint32_t it = 0; seg < n_segs; ++it) {
    uint32_t r0 = 0, r1 = 1, slice = 0;
    if (!item_list) {
      slice = seg % plan.n_slices;
      r0 = seg / plan.n_slices * seg_runs;
      r1 = min(r0 + seg_runs, plan.n_run_items);
    }
    for (uint32_t r = r0; r < r1; ++r) {
      const uint32_t item = item_list ? item_list[seg] : r * plan.n_slices + slice;
      const uint4 desc = __ldg(plan.item_desc + item);
      const uint32_t seq_lo = desc.x, seq_hi = desc.y, s_rel = desc.z;   // sequences, first window of the run
      if (seq_lo == seq_hi) {                          // no sample of this slice carries the cluster
        if (tid == 0) { slab_count[item] = 0; slab_base[item] = 0; }
        continue;
      }
      const uint32_t sample0 = plan.n_slices > 1 ? (item % plan.n_slices) * plan.slice_samples : 0u;
      const uint32_t wi = s_rel >> 5;

      // ---- the register-held sequences at this run: new (cluster, slice) or position -> load,
      //      next word -> slide by one word and request the one after ---------------------------
      auto fetch = [&](uint32_t nw, uint32_t wo, uint64_t& c, uint64_t& n, uint64_t& p) {
        c = 0; n = 0; p = 0;
        if (s_rel < nw) {
          const uint64_t* w = bases + wo + wi;
          c = __ldg(w); n = __ldg(w + 1);
          if (32u * (wi + 1u) < nw) p = __ldg(w + 2);
        }
      };
      auto slide = [&](uint32_t nw, uint32_t wo, uint64_t& c, uint64_t& n, uint64_t& p) {
        c = n; n = p; p = 0;
        if (32u * (wi + 1u) < nw) p = __ldg(bases + wo + wi + 2u);
      };
      if (seq_lo != st_lo) {
        nw0 = 0; nw1 = 0;
        if (seq_lo + tid < seq_hi) {
          const uint4 raw = __ldg(reinterpret_cast<const uint4*>(seqs + seq_lo + tid));
          nw0 = raw.y >= (uint32_t)k ? raw.y - (uint32_t)k + 1u : 0u; sf0 = raw.z; wo0 = raw.x;
        }
        if (seq_lo + tid + kBlkThreads < seq_hi) {
          const uint4 raw = __ldg(reinterpret_cast<const uint4*>(seqs + seq_lo + tid + kBlkThreads));
          nw1 = raw.y >= (uint32_t)k ? raw.y - (uint32_t)k + 1u : 0u; sf1 = raw.z; wo1 = raw.x;
        }
      }
      if (seq_lo == st_lo && wi == st_wi + 1u) {
        slide(nw0, wo0, c0, n0, p0);
        slide(nw1, wo1, c1, n1, p1);
      } else if (seq_lo != st_lo || wi != st_wi) {
        fetch(nw0, wo0, c0, n0, p0);
        fetch(nw1, wo1, c1, n1, p1);
      }
      st_lo = seq_lo;
      st_wi = wi;

      // ---- phase 1: every sequence's run -> chunk table (or, for ragged / ambiguous runs and a
      //      full chunk table, straight into the k-mer table) ----------------------------------
      for (uint32_t j = 0, si = seq_lo + tid; si < seq_hi; ++j, si += kBlkThreads) {
        uint32_t nwin, sf;
        uint64_t w0, w1;
        if (j < 2u) {
          nwin = j ? nw1 : nw0; sf = j ? sf1 : sf0; w0 = j ? c1 : c0; w1 = j ? n1 : n0;
        } else {                                      // beyond 2 x threads: from global memory
          const uint4 raw = __ldg(reinterpret_cast<const uint4*>(seqs + si));
          nwin = raw.y >= (uint32_t)k ? raw.y - (uint32_t)k + 1u : 0u;
          sf = raw.z;
          w0 = 0; w1 = 0;
          if (s_rel < nwin) { const uint64_t* w = bases + raw.x + wi; w0 = __ldg(w); w1 = __ldg(w + 1); }
        }
        if (s_rel >= nwin) continue;
        const uint32_t nv = min((uint32_t)kBlkRun, nwin - s_rel);
        const uint32_t sample = (sf & 0x7fffffffu) - sample0;      // rank inside the slice
        const bool amb = (sf >> 31) != 0u;
        const uint32_t wofs = sample >> 5, bit = 1u << (sample & 31u);
        const uint32_t o0 = s_rel & 31u;
        uint64_t hi = w0, lo = w1;
        if (o0) {
          hi = (w0 << (2u * o0)) | (w1 >> (64u - 2u * o0));
          lo = w1 << (2u * o0);
        }
        uint32_t cs = 0xffffffffu;
        if (nv == (uint32_t)kBlkRun && !amb) cs = chunk_find_or_insert(a, hi & cm_hi, lo & cm_lo, wofs);
        if (cs != 0xffffffffu) {
          atomicOr(&a.crows[cs * WS + wofs], bit);
          const uint16_t meta = a.cmeta[cs];            // most chunks are one sample's: remember if not
          if ((meta & 0xffu) != wofs && !(meta & 0x8000u)) a.cmeta[cs] = meta | 0x8000u;
        } else {
          const uint32_t* ab = amb ? ambbits + seqs[si].amb_word_off : nullptr;
          for (uint32_t q = 0; q < nv; ++q) {
            bool dead = false;
            if (amb) {
              const uint32_t p = s_rel + q;
              const uint32_t wj = p >> 5, bs = p & 31u;
              const uint64_t two = ((uint64_t)ab[wj] << 32) | (uint64_t)ab[wj + 1];
              dead = ((two << bs) >> (64 - k)) != 0ull;
            }
            if (!dead) {
              const uint64_t x = q ? ((hi << (2u * q)) | (lo >> (64u - 2u * q))) : hi;
              put_kmer(x >> sh64, &bit, wofs, 1u);
            }
          }
        }
      }
      __syncthreads();

      // ---- phase 2: distinct chunks x 16 windows -> k-mer table, whole sample bitsets at a time ----
      const uint32_t n_chunks = min(a.h->work, a.ccap);
      const uint32_t n_pairs = n_chunks * (uint32_t)kBlkRun;
      // pairs cost very different amounts (a new k-mer is an insertion, a many-sample chunk ORs W
      // words): the first round is static, after it the warps take 32 pairs at a time from a counter
      for (uint32_t q0 = (tid & ~31u);;) {
        const uint32_t p = q0 + (tid & 31u);
        if (p < n_pairs) {
          const uint32_t cs = p >> 4, q = p & 15u;
          const uint64_t hi = a.ckhi[cs], lo = a.cklo[cs];
          const uint64_t x = q ? ((hi << (2u * q)) | (lo >> (64u - 2u * q))) : hi;
          const uint16_t meta = a.cmeta[cs];
          if (meta & 0x8000u) put_kmer(x >> sh64, a.crows + cs * WS, 0u, W);
          else put_kmer(x >> sh64, a.crows + cs * WS + (meta & 0xffu), meta & 0xffu, 1u);
        }
        __syncwarp();
        uint32_t nx = 0;
        if ((tid & 31u) == 0u) nx = atomicAdd(&a.h->n_pass, 32u);
        q0 = (uint32_t)kBlkThreads + __shfl_sync(kFull, nx, 0);
        if (q0 >= n_pairs) break;
      }
      __syncthreads();

      // ---- epilogue: the slab of this run (n partial rows from a bump allocator), then the
      //      tables are reset for the next run -----------------------------------------------
      const bool overflow = a.h->overflow != 0u;
      const uint32_t n = a.h->n_unique;
      if (tid == 0) {
        if (overflow) {
          slab_count[item] = kBlkOverflow;
          slab_base[item] = 0;
          atomicExch(&counters[LC_TABLE_OVERFLOW], 1u);
          rescue_items[atomicAdd(&counters[LC_RESCUE], 1u)] = item;
        } else {
          const uint32_t b = atomicAdd(&counters[LC_PARTIALS], n);
          a.h->row_base = b;
          a.h->ok = 1;
          slab_base[item] = b;
          slab_count[item] = n;
          if ((uint64_t)b + n > partial_capacity) {
            a.h->ok = 0;
            slab_count[item] = 0;
            atomicExch(&counters[LC_PARTIAL_OVERFLOW], 1u);
          }
        }
      }
      __syncthreads();
      if (tid == 0) { a.h->n_unique = 0; a.h->overflow = 0; a.h->work = 0; a.h->n_pass = 0; }
      if (!overflow && a.h->ok) {
        // a warp takes 32 rows: every lane writes its row's key and count code; a one-sample row
        // (most of them: the k-mers of a private SNP) is only that code, its bitset is never
        // written.  The other rows are listed (lane ids, in the chunk keys, which are dead until
        // the next run: ccap >= 16 gives 32 bytes per warp) and copied by L = WP / 4 lanes each,
        // one uint4 per lane, so a store instruction writes whole 16 * L-byte rows (W <= 32: L <= 8).
        const size_t base = a.h->row_base;
        const uint32_t WP = plan.WP, L = WP >> 2, lane = tid & 31u;
        const uint32_t lrow = lane / L, lq = 4u * (lane - lrow * L), per = 32u / L;
        uint8_t* list = reinterpret_cast<uint8_t*>(a.ckhi) + (tid & ~31u);
        for (uint32_t r0 = tid & ~31u; r0 < n; r0 += kBlkThreads) {
          const uint32_t r = r0 + lane;
          bool multi = false;
          if (r < n) {
            slab_keys[base + r] = a.rkey[r];
            uint32_t* src = a.pool + r * WS;
            uint32_t cnt = 0, wq = 0, orx = 0;         // one sample: it is bit ffs(orx) of word wq
            for (uint32_t q = 0; q < W; ++q) {
              const uint32_t x = src[q], c = __popc(x);
              cnt += c;
              wq += c * q;
              orx |= x;
            }
            multi = cnt != 1u;
            if (multi) {
              slab_cnt[base + r] = cnt;
            } else {
              slab_cnt[base + r] = kCntSingle | (wq << 5) | (uint32_t)(__ffs(orx) - 1);
              src[wq] = 0u;
            }
            const uint32_t h = a.rslot[r];
            a.keys[h] = ~0ull;
            a.rowid[h] = 0xffffu;
          }
          const uint32_t m = __ballot_sync(kFull, multi), nm = (uint32_t)__popc(m);
          if (multi) list[__popc(m & lanemask_lt())] = (uint8_t)lane;
          if (lane == 0 && nm < min(32u, n - r0)) atomicAdd(&a.h->singles, min(32u, n - r0) - nm);
          __syncwarp();
          for (uint32_t g = lrow; g < nm && lrow < per; g += per) {
            const uint32_t rr = r0 + list[g];
            uint32_t* src = a.pool + rr * WS + lq;
            uint4 x;
            x.x = src[0];                              // (lq < W: WP is W rounded up to 4)
            x.y = lq + 1 < W ? src[1] : 0u;
            x.z = lq + 2 < W ? src[2] : 0u;
            x.w = lq + 3 < W ? src[3] : 0u;
            reinterpret_cast<uint4*>(slab_rows + (base + rr) * WP + lq)[0] = x;
            src[0] = 0u;
            if (lq + 1 < W) src[1] = 0u;
            if (lq + 2 < W) src[2] = 0u;
            if (lq + 3 < W) src[3] = 0u;
          }
          __syncwarp();
        }
        for (uint32_t c = tid; c < n_chunks; c += kBlkThreads) a.cstate[a.cslot[c]] = kChunkEmpty;
        for (uint32_t i = tid; i < n_chunks * WS; i += kBlkThreads) a.crows[i] = 0u;
      } else {
        clear_tables();
      }
      __syncthreads();
    }
    if (item_list) {
      seg += gridDim.x;
    } else {
      if (tid == 0) a.h->seg[it & 1u] = gridDim.x + atomicAdd(&counters[LC_SEGMENT], 1u);
      __syncthreads();
      seg = a.h->seg[it & 1u];
    }
  }
  if (tid == 0 && a.h->singles) atomicAdd(&counters[LC_SINGLES], a.h->singles);
}

// ---------------------------------------------------------------------------
// kB: merge the partial rows of a cluster by k-mer, count, filter, emit rows
// ---------------------------------------------------------------------------
// A k-mer usually has ONE partial row (its windows start in one run of every sequence);
// indels, clamped flanks and paralogs give it a second one in a neighbouring run.  So the
// merge is a find-or-insert of every partial key into a per-cluster open-addressing table in
// global memory (L2-resident while the cluster's slabs are being inserted): the first row of
// a key becomes its owner, later rows OR their bitset into the owner's (rare), and the owners
// are counted, filtered with the cluster's integer MAF window and written out.
// Table entry: 64 bits = (32-bit fingerprint of the key) << 32 | index of the partial row that
// owns the slot; all ones = empty.  A fingerprint match is confirmed on the owner's full key
// (slab_keys), so nothing is ever merged on a hash.
typedef unsigned long long MergeEntry;

// one warp per (cluster, slice): partial rows -> table slots (eighths / 8 slots per row).  With
// slices, table2_ctas[c] additionally sizes the cluster's cross-slice table in units of 256
// slots (so that a CTA of kB5 belongs to one cluster).
__global__ void plan_merge_tables(const uint32_t* __restrict__ item_base, uint32_t n_clusters, uint32_t n_slices,
                                  const uint32_t* __restrict__ slab_count, uint32_t eighths /* slots per row x 8 */,
                                  uint32_t* __restrict__ n_slots, uint32_t* __restrict__ table2_ctas) {
  const uint32_t cs = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (cs >= n_clusters * n_slices) return;
  const uint32_t c = cs / n_slices, slice = cs - c * n_slices;
  const uint32_t lane = lane_id();
  uint32_t p = 0;
  for (uint32_t r = item_base[c] + lane; r < item_base[c + 1]; r += 32) {
    const uint32_t n = slab_count[(size_t)r * n_slices + slice];
    if (n != kBlkOverflow) p += n;
  }
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) p += __shfl_xor_sync(kFull, p, m);
  if (lane == 0) {
    n_slots[cs] = (uint32_t)(((uint64_t)p * eighths + 7u) >> 3) + 2u;
    if (table2_ctas) atomicAdd(&table2_ctas[c], p);       // partial rows of the cluster (all slices)
  }
}
// table2_ctas[c]: partial rows -> CTAs of 256 slots at load factor <= 2/3
__global__ void plan_table2_ctas(uint32_t* __restrict__ table2_ctas, uint32_t n_clusters) {
  const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_clusters) return;
  const uint32_t p = table2_ctas[c];
  table2_ctas[c] = (p + (p >> 1) + 2u + 255u) / 256u;
}

// expand an exclusive scan into its inverse map: out[base[c] + i] = c
__global__ void plan_expand_owner(const uint32_t* __restrict__ base, uint32_t n_clusters,
                                  uint32_t* __restrict__ out) {
  const uint32_t c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (c >= n_clusters) return;
  for (uint32_t i = base[c] + lane_id(); i < base[c + 1]; i += 32) out[i] = c;
}

// OR partial row p into row q (both WP words, WP a multiple of 4): the words are loaded four
// uint4 at a time before the first atomic goes out (one round trip, not one per word)
__device__ __forceinline__ void fold_partial_row(uint32_t* __restrict__ slab_rows, uint32_t p, uint32_t q, uint32_t WP) {
  const uint4* src = reinterpret_cast<const uint4*>(slab_rows + (size_t)p * WP);
  uint32_t* dst = slab_rows + (size_t)q * WP;
  const uint32_t n4 = WP >> 2;
  for (uint32_t w0 = 0; w0 < n4; w0 += 4) {
    uint4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = w0 + u < n4 ? src[w0 + u] : make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      uint32_t* d = dst + (size_t)(w0 + u) * 4;
      if (v[u].x) atomicOr(d + 0, v[u].x);
      if (v[u].y) atomicOr(d + 1, v[u].y);
      if (v[u].z) atomicOr(d + 2, v[u].z);
      if (v[u].w) atomicOr(d + 3, v[u].w);
    }
  }
}

// kB1: partial row p (a later row of the k-mer) goes into its owner q.  A one-sample row has no
// bitset in slab_rows: p's is one atomicOr; q's is written out first, by the first row that folds
// into it (single code -> kCntLocked by CAS, all WP words, kCntDirty), while other rows folding
// into q at the same time wait for kCntDirty.
__device__ __noinline__ void fold_into_owner(uint32_t* __restrict__ slab_rows, uint32_t* __restrict__ slab_cnt,
                                             uint32_t p, uint32_t q, uint32_t WP) {
  uint32_t* dst = slab_rows + (size_t)q * WP;
  for (;;) {
    const uint32_t code = *reinterpret_cast<volatile uint32_t*>(&slab_cnt[q]);
    if (cnt_single(code)) {
      if (atomicCAS(&slab_cnt[q], code, kCntLocked) != code) continue;
      for (uint32_t w = 0; w < WP; w += 4) *reinterpret_cast<uint4*>(dst + w) = make_uint4(0u, 0u, 0u, 0u);
      const uint32_t s = code & 0x3ffu;
      dst[s >> 5] = 1u << (s & 31u);
      __threadfence();
      *reinterpret_cast<volatile uint32_t*>(&slab_cnt[q]) = kCntDirty;
      break;
    }
    if (code != kCntLocked) { __threadfence(); break; }
    __nanosleep(32);                          // (lets the writer run if it is a lane of this warp)
  }
  const uint32_t pc = slab_cnt[p];
  if (cnt_single(pc)) atomicOr(dst + ((pc & 0x3ffu) >> 5), 1u << (pc & 31u));
  else fold_partial_row(slab_rows, p, q, WP);
  slab_cnt[p] = kCntDead;
  slab_cnt[q] = kCntDirty;
}

// kB1 in shared memory: one CTA per (cluster, slice).  The partial rows of a cluster number a few
// ten thousand, so the find-or-insert table of the merge fits shared memory when an entry is 32
// bits: a 15-bit fingerprint of the key and the 17-bit index of the owning row in the cluster's
// own numbering (prefix sums of its slabs' row counts, also in shared memory).  A fingerprint
// match is confirmed on the owner's full key.  Shared-memory CAS instead of one L2 atomic per
// row: 2.6 -> ~0.3 ms per step on BASELINE config #2.  A cluster with too many runs or rows for
// the table clears its region of the global table instead and sets spill[c]: kB1_insert, which
// runs next, takes exactly those.
constexpr uint32_t kMergeLocalThreads = 1024;
constexpr uint32_t kMergeLocalMaxItems = 2047;      // runs of one cluster (prefix array: 8 KB)
constexpr uint32_t kMergeLocalIdxBits = 17;
__host__ __device__ inline uint32_t merge_local_smem_bytes(uint32_t max_slots) {
  return (kMergeLocalMaxItems + 1u + max_slots) * 4u;
}

__global__ void __launch_bounds__(kMergeLocalThreads, 1)
kB1_local(const uint64_t* __restrict__ slab_keys, uint32_t* __restrict__ slab_rows,
          uint32_t* __restrict__ slab_cnt, const uint32_t* __restrict__ slab_base,
          const uint32_t* __restrict__ slab_count, const uint32_t* __restrict__ item_base /* [n_clusters + 1] */,
          uint32_t n_slices, const uint32_t* __restrict__ table_base /* [n_clusters * n_slices + 1] */,
          MergeEntry* __restrict__ table, uint16_t* __restrict__ pslice /* null without slices */,
          uint32_t WP, uint32_t* __restrict__ counters, uint32_t max_slots, uint8_t* __restrict__ spill,
          uint32_t fp_mask /* 0x7fff; fewer bits only to test the mismatch path */) {
  extern __shared__ uint32_t merge_sm[];
  uint32_t* prefix = merge_sm;                                  // [n_it + 1] rows before run i
  uint32_t* tab = merge_sm + kMergeLocalMaxItems + 1;           // [slots]
  __shared__ uint32_t s_wsum[32];
  __shared__ uint32_t s_dups, s_next;
  const uint32_t c = blockIdx.x;
  const uint32_t cluster = c / n_slices, slice = c - cluster * n_slices;
  const uint32_t it0 = item_base[cluster], n_it = item_base[cluster + 1] - it0;
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  bool spilled = n_it > kMergeLocalMaxItems;
  uint32_t total = 0;
  if (!spilled) {
    // prefix sums of the runs' row counts: 1024 runs per round, a warp per 32 of them
    for (uint32_t b0 = 0; b0 < n_it; b0 += kMergeLocalThreads) {
      const uint32_t i = b0 + tid;
      uint32_t v = 0;
      if (i < n_it) {
        v = slab_count[(size_t)(it0 + i) * n_slices + slice];
        if (v == kBlkOverflow) v = 0;
      }
      uint32_t x = v;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint32_t y = __shfl_up_sync(kFull, x, d);
        if ((int)lane >= d) x += y;
      }
      if (lane == 31) s_wsum[warp] = x;
      __syncthreads();
      uint32_t ws = s_wsum[lane], wx = ws;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint32_t y = __shfl_up_sync(kFull, wx, d);
        if ((int)lane >= d) wx += y;
      }
      const uint32_t before = __shfl_sync(kFull, wx - ws, warp);   // rows of the warps before this one
      if (i < n_it) prefix[i] = total + before + x - v;
      total += __shfl_sync(kFull, wx, 31);
      __syncthreads();
    }
    if (tid == 0) { prefix[n_it] = total; s_dups = 0; s_next = 0; }
    if (total == 0) { if (tid == 0) spill[c] = 0; return; }
    spilled = total >= (1u << kMergeLocalIdxBits) - 1u || total > max_slots / 16u * 13u;
  }
  if (spilled) {
    const uint32_t tb = table_base[c], te = table_base[c + 1];
    for (uint32_t i = tb + tid; i < te; i += kMergeLocalThreads) table[i] = ~0ull;
    if (tid == 0) spill[c] = 1;
    return;
  }
  if (tid == 0) spill[c] = 0;
  const uint32_t slots = min(max_slots, 2u * total + 2u);
  for (uint32_t i = tid; i < slots; i += kMergeLocalThreads) tab[i] = 0xffffffffu;
  __syncthreads();
  uint32_t dups = 0;
  // partial-row index of row `ql` of the cluster's numbering
  auto global_row = [&](uint32_t ql) -> uint32_t {
    uint32_t lo = 0, hi = n_it;                                 // last run with prefix <= ql
    while (hi - lo > 1) {
      const uint32_t mid = (lo + hi) >> 1;
      if (prefix[mid] <= ql) lo = mid; else hi = mid;
    }
    return slab_base[(size_t)(it0 + lo) * n_slices + slice] + (ql - prefix[lo]);
  };
  auto fold = [&](uint32_t p, uint32_t q) {
    fold_into_owner(slab_rows, slab_cnt, p, q, WP);
    ++dups;
  };
  // find-or-insert of one row: key, its index in the cluster's numbering, its partial-row index.
  // A fingerprint match is a row of the same k-mer but for one in 2^15; the full keys decide.
  // (Deferring the matches to a list that the whole CTA works off afterwards, so that their
  // global-memory round trips overlap, was measured and is slower: 84 vs 74 us per 200 clusters.)
  auto insert = [&](uint64_t key, uint32_t local, uint32_t p) {
    const uint64_t mixed = mix64(key);
    const uint32_t fp = (uint32_t)mixed & fp_mask;
    const uint32_t mine = (fp << kMergeLocalIdxBits) | local;
    uint32_t s = __umulhi((uint32_t)(mixed >> 32), slots);
    for (;;) {
      const uint32_t old = atomicCAS(&tab[s], 0xffffffffu, mine);
      if (old == 0xffffffffu) return;                           // this row owns the k-mer
      if ((old >> kMergeLocalIdxBits) == fp) {
        const uint32_t q = global_row(old & ((1u << kMergeLocalIdxBits) - 1u));
        if (slab_keys[q] == key) { fold(p, q); return; }        // an earlier row of the same k-mer
      }
      if (++s == slots) s = 0;
    }
  };
  // warps take half a run at a time (dynamic; ~128 rows: the tail of the CTA is short); the keys
  // of four rows per lane are loaded before the first of them is inserted
  for (;;) {
    uint32_t unit = 0;
    if (lane == 0) unit = atomicAdd(&s_next, 1u);
    unit = __shfl_sync(kFull, unit, 0);
    const uint32_t it = unit >> 1;
    if (it >= n_it) break;
    const size_t item = (size_t)(it0 + it) * n_slices + slice;
    const uint32_t n = slab_count[item];
    if (n == kBlkOverflow || n == 0) continue;
    const uint32_t half = (((n + 1u) >> 1) + 31u) & ~31u;
    const uint32_t r0 = (unit & 1u) * half, r1 = min(n, r0 + half);
    const uint32_t base = slab_base[item], lbase = prefix[it];
    for (uint32_t i0 = r0 + lane; i0 < r1; i0 += 128) {
      uint64_t key[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t i = i0 + 32u * u;
        key[u] = i < r1 ? slab_keys[base + i] : 0ull;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t i = i0 + 32u * u;
        if (i < r1) {
          if (pslice) pslice[base + i] = (uint16_t)slice;
          insert(key[u], lbase + i, base + i);
        }
      }
    }
  }
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) dups += __shfl_xor_sync(kFull, dups, m);
  if (lane == 0 && dups) atomicAdd(&s_dups, dups);
  __syncthreads();
  if (tid == 0 && s_dups) atomicAdd(&counters[LC_RESCUE], s_dups);   // (the rescue counter is free again after kA)
}

// kB1 in global memory, for the clusters kB1_local left (spill[c]; it has cleared their table
// regions): one warp per slab; every partial key finds or claims its slot.  A row that meets an
// earlier row of the same k-mer ORs its bitset into that one on the spot and is marked dead
// (counted: distinct k-mers = partial rows - dead rows); the owner's stored popcount is dirty.
__global__ void __launch_bounds__(256)
kB1_insert(const uint64_t* __restrict__ slab_keys, uint32_t* __restrict__ slab_rows,
           uint32_t* __restrict__ slab_cnt, const uint32_t* __restrict__ slab_base,
           const uint32_t* __restrict__ slab_count, const uint32_t* __restrict__ item_cluster,
           uint32_t n_items /* incl. slices */, uint32_t n_slices,
           const uint32_t* __restrict__ table_base /* [n_clusters * n_slices + 1] */,
           MergeEntry* __restrict__ table, uint16_t* __restrict__ pslice /* null without slices */,
           uint32_t WP, uint32_t* __restrict__ counters, const uint8_t* __restrict__ spill) {
  const uint32_t item = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (item >= n_items) return;
  const uint32_t run_item = n_slices > 1 ? item / n_slices : item;
  const uint32_t slice = item - run_item * n_slices;
  const uint32_t c = item_cluster[run_item] * n_slices + slice;
  if (!spill[c]) return;                     // merged in shared memory by kB1_local
  const uint32_t n = slab_count[item];
  if (n == kBlkOverflow || n == 0) return;
  const uint32_t tb = table_base[c], ts = table_base[c + 1] - tb;
  const uint32_t base = slab_base[item];
  if (pslice)
    for (uint32_t i = lane_id(); i < n; i += 32) pslice[base + i] = (uint16_t)slice;
  for (uint32_t i = lane_id(); i < n; i += 32) {
    const uint32_t p = base + i;
    const uint64_t key = slab_keys[p];
    const uint64_t mixed = mix64(key);
    const uint32_t fp = (uint32_t)mixed;
    const MergeEntry mine = ((MergeEntry)fp << 32) | p;
    uint32_t s = __umulhi((uint32_t)(mixed >> 32), ts);
    for (;;) {
      const MergeEntry old = atomicCAS(&table[tb + s], ~0ull, mine);
      if (old == ~0ull) break;                              // this row owns the k-mer
      if ((uint32_t)(old >> 32) == fp) {
        const uint32_t q = (uint32_t)old;
        if (slab_keys[q] == key) {                          // an earlier row of the same k-mer
          fold_into_owner(slab_rows, slab_cnt, p, q, WP);
          atomicAdd(&counters[LC_RESCUE], 1u);              // (the rescue counter is free again after kA)
          break;
        }
      }
      if (++s == ts) s = 0;
    }
  }
}

// kB3: one warp per slab; owners are counted, filtered and written out as rows.  Rows are
// handed out with ONE global atomic per CTA (a counter shared by 300,000 warps serialises).
__global__ void __launch_bounds__(256)
kB3_emit(const uint64_t* __restrict__ slab_keys, const uint32_t* __restrict__ slab_rows,
         const uint32_t* __restrict__ slab_base, const uint32_t* __restrict__ slab_count,
         const uint32_t* __restrict__ item_cluster, uint32_t n_items,
         const uint32_t* __restrict__ slab_cnt, const ClusterDev* __restrict__ clusters, RowOut out,
         uint32_t row_capacity, uint32_t* __restrict__ counters, uint32_t W, uint32_t WP) {
  __shared__ uint32_t w_pass[8];
  __shared__ uint32_t cta_base, cta_ok;
  const uint32_t item = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
  uint32_t n = 0, c = 0, base = 0;
  if (item < n_items) {
    n = slab_count[item];
    if (n == kBlkOverflow) n = 0;
    c = item_cluster[item];
    base = slab_base[item];
  }
  ClusterDev cl{};
  if (n) cl = clusters[c];
  auto row_of = [&](uint32_t i) { return reinterpret_cast<const uint4*>(slab_rows + (size_t)(base + i) * WP); };
  auto count_of = [&](uint32_t i, bool& owner) {
    const uint32_t cnt = i < n ? partial_row_count(slab_rows, slab_cnt[base + i], base + i, WP) : kCntDead;
    owner = cnt != kCntDead;
    return cnt;
  };
  // pass 1: rows this warp will write (verdicts of the first 256 partial rows stay in registers)
  uint32_t my = 0;
  uint32_t verdict[8];
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    verdict[it] = 0u;
    if ((uint32_t)it * 32u < n) {
      bool owner;
      const uint32_t cnt = count_of((uint32_t)it * 32u + lane, owner);
      const bool pass = owner && cnt >= cl.lo && cnt <= cl.hi;
      verdict[it] = pass ? (0x80000000u | cnt) : 0u;
      my += __popc(__ballot_sync(kFull, pass));
    }
  }
  for (uint32_t i0 = 256; i0 < n; i0 += 32) {
    bool owner;
    const uint32_t cnt = count_of(i0 + lane, owner);
    my += __popc(__ballot_sync(kFull, owner && cnt >= cl.lo && cnt <= cl.hi));
  }
  if (lane == 0) w_pass[warp] = my;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t total = 0;
    for (int w = 0; w < 8; ++w) { const uint32_t x = w_pass[w]; w_pass[w] = total; total += x; }
    uint32_t b = 0, ok = 1;
    if (total) {
      b = atomicAdd(&counters[LC_ROWS], total);
      if ((uint64_t)b + total > row_capacity) { ok = 0; atomicExch(&counters[LC_ROW_OVERFLOW], 1u); }
    }
    cta_base = b;
    cta_ok = ok;
  }
  __syncthreads();
  if (!cta_ok || my == 0) return;
  // pass 2: write them (the bitsets come back from L2)
  uint32_t g = cta_base + w_pass[warp];
  auto emit = [&](uint32_t i, bool pass, uint32_t cnt) {
    const uint32_t mp = __ballot_sync(kFull, pass);
    if (pass) {
      const size_t gi = (size_t)g + __popc(mp & lanemask_lt());
      out.cluster[gi] = cl.id;
      out.kmer[gi] = slab_keys[base + i];
      out.count[gi] = cnt;
      uint32_t* dst = out.cand + gi * out.key_words;
      const uint32_t code = cnt == 1u ? slab_cnt[base + i] : 0u;
      if (cnt_single(code)) {                  // one sample (a window with lo <= 1): no row to read
        const uint32_t s = code & 0x3ffu;
        for (uint32_t w = 0; w < W; ++w) dst[w] = w == (s >> 5) ? 1u << (s & 31u) : 0u;
      } else {
        // (one row per half-warp through shuffles, so that loads and stores are coalesced segments,
        //  was measured and is slower: kB 2.48 against 2.06 ms per config-2 step)
        const uint4* row = row_of(i);
        for (uint32_t q = 0; q < WP / 4; ++q) {
          const uint4 x = row[q];
          const uint32_t w = 4 * q;
          if (w < W) dst[w] = x.x;
          if (w + 1 < W) dst[w + 1] = x.y;
          if (w + 2 < W) dst[w + 2] = x.z;
          if (w + 3 < W) dst[w + 3] = x.w;
        }
      }
      if (out.key_words > W) dst[W] = out.cluster_pattern[c];
    }
    g += __popc(mp);
  };
#pragma unroll
  for (int it = 0; it < 8; ++it)
    if ((uint32_t)it * 32u < n) emit((uint32_t)it * 32u + lane, (verdict[it] >> 31) != 0u, verdict[it] & 0x7fffffffu);
  for (uint32_t i0 = 256; i0 < n; i0 += 32) {
    bool owner;
    const uint32_t cnt = count_of(i0 + lane, owner);
    emit(i0 + lane, owner && cnt >= cl.lo && cnt <= cl.hi, cnt);
  }
}


// ---------------------------------------------------------------------------
// sample slices: a k-mer's bitset is spread over up to n_slices partial rows (one per slice,
// after kB1 merged the rows of the same slice).  kB4 sums the popcounts per k-mer in a cross-slice
// table of the cluster; kB5 applies the MAF window to the sum, hands the survivors (~1 % of the
// k-mers at 10,000 samples) their output row and clears it; kB6 goes over the partial rows once
// more and copies those of a surviving k-mer to their place in its row.  (An earlier version
// chained the rows of a k-mer through a linked list and assembled the row by walking it: a
// dependent load per slice.  Now every step is parallel over rows or table slots.)
// ---------------------------------------------------------------------------
struct LinkEntry {         // 16 bytes, memset to 0xff: key empty, row nil, count = -1
  unsigned long long key;
  uint32_t row;            // kB5: output row of a surviving k-mer
  uint32_t count;          // (sum of popcounts) - 1
};

// one warp per kA work item, one row per lane and turn.  (Four rows per lane in flight measured
// slower, 0.49 against 0.39 ms on 48 clusters of 10,000 samples: the registers cost occupancy, and
// visiting the slices of a run far apart in time was slower still, 0.76 ms: the 20 slices of a
// k-mer hitting its entry together is what keeps the table in L2.)
__global__ void __launch_bounds__(256)
kB4_link(const uint64_t* __restrict__ slab_keys, const uint32_t* __restrict__ slab_rows,
         const uint32_t* __restrict__ slab_base, const uint32_t* __restrict__ slab_count,
         const uint32_t* __restrict__ item_cluster, uint32_t n_items, uint32_t n_slices,
         const uint32_t* __restrict__ slab_cnt, const uint32_t* __restrict__ table2_base /* CTAs of 256 slots */,
         LinkEntry* __restrict__ table2, uint32_t WP) {
  const uint32_t item = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (item >= n_items) return;
  const uint32_t n = slab_count[item];
  if (n == kBlkOverflow || n == 0) return;
  const uint32_t c = item_cluster[item / n_slices];
  const uint32_t tb = table2_base[c] * 256u, ts = (table2_base[c + 1] - table2_base[c]) * 256u;
  const uint32_t base = slab_base[item];
  for (uint32_t i = lane_id(); i < n; i += 32u) {
    const uint32_t cnt = partial_row_count(slab_rows, slab_cnt[base + i], base + i, WP);
    if (cnt == kCntDead) continue;              // folded into an earlier row of its slice
    const unsigned long long key = slab_keys[base + i];
    uint32_t s = __umulhi((uint32_t)(mix64(key) >> 32), ts);
    for (;;) {                                  // find or insert, linear probing
      const unsigned long long o = atomicCAS(&table2[tb + s].key, ~0ull, key);
      if (o == ~0ull || o == key) break;
      if (++s == ts) s = 0;
    }
    atomicAdd(&table2[tb + s].count, cnt);
  }
}

// one CTA per 256 slots of a cluster's cross-slice table
__global__ void __launch_bounds__(256)
kB5_emit(LinkEntry* __restrict__ table2, const uint32_t* __restrict__ cta_cluster,
         const uint32_t* __restrict__ table2_base, uint32_t* __restrict__ home_bits,
         const ClusterDev* __restrict__ clusters, RowOut out, uint32_t row_capacity,
         uint32_t* __restrict__ counters, uint32_t W) {
  __shared__ uint32_t w_pass[8], w_used[8];
  __shared__ uint32_t cta_base, cta_ok;
  const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
  const uint32_t c = cta_cluster[blockIdx.x];
  const ClusterDev cl = clusters[c];
  const size_t slot = (size_t)blockIdx.x * 256u + threadIdx.x;
  const LinkEntry e = table2[slot];
  const bool used = e.key != ~0ull;
  const uint32_t total = e.count + 1u;
  const bool pass = used && total >= cl.lo && total <= cl.hi;
  const uint32_t mp = __ballot_sync(kFull, pass), mu = __ballot_sync(kFull, used);
  if (lane == 0) { w_pass[warp] = (uint32_t)__popc(mp); w_used[warp] = (uint32_t)__popc(mu); }
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t tot = 0, tu = 0;
    for (int w = 0; w < 8; ++w) { const uint32_t x = w_pass[w]; w_pass[w] = tot; tot += x; tu += w_used[w]; }
    uint32_t b = 0, ok = 1;
    if (tu) atomicAdd(&counters[LC_UNIQUE], tu);
    if (tot) {
      b = atomicAdd(&counters[LC_ROWS], tot);
      if ((uint64_t)b + tot > row_capacity) { ok = 0; atomicExch(&counters[LC_ROW_OVERFLOW], 1u); }
    }
    cta_base = b;
    cta_ok = ok;
  }
  __syncthreads();
  if (!cta_ok || mp == 0u) return;
  const uint32_t g0 = cta_base + w_pass[warp];
  if (pass) {
    const size_t gi = (size_t)g0 + __popc(mp & lanemask_lt());
    out.cluster[gi] = cl.id;
    out.kmer[gi] = e.key;
    out.count[gi] = total;
    table2[slot].row = (uint32_t)gi;             // kB6 copies the k-mer's slices there
    // ... and finds the few survivors through one bit per table slot, set at the HOME slot of
    // the key (a few MB, resident in L2), instead of probing the table for every partial row
    const uint32_t tb = table2_base[c] * 256u, ts = (table2_base[c + 1] - table2_base[c]) * 256u;
    const uint32_t home = tb + __umulhi((uint32_t)(mix64(e.key) >> 32), ts);
    atomicOr(&home_bits[home >> 5], 1u << (home & 31));
  }
  // the warp clears its surviving rows one after the other, all lanes on one row
  for (uint32_t r = 0, n = (uint32_t)__popc(mp); r < n; ++r) {
    uint32_t* dst = out.cand + ((size_t)g0 + r) * out.key_words;
    for (uint32_t w = lane; w < W; w += 32) dst[w] = 0u;
    if (lane == 0 && out.key_words > W) dst[W] = out.cluster_pattern[c];
  }
}

// one warp per kA work item: the partial rows of surviving k-mers go to their slice of the row
__global__ void __launch_bounds__(256)
kB6_scatter(const uint64_t* __restrict__ slab_keys, const uint32_t* __restrict__ slab_rows,
            const uint32_t* __restrict__ slab_base, const uint32_t* __restrict__ slab_count,
            const uint32_t* __restrict__ item_cluster, uint32_t n_items, uint32_t n_slices,
            const uint32_t* __restrict__ slab_cnt, const uint32_t* __restrict__ table2_base,
            const LinkEntry* __restrict__ table2, const uint32_t* __restrict__ home_bits, RowOut out, uint32_t W,
            uint32_t Ws, uint32_t WP) {
  const uint32_t item = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (item >= n_items) return;
  const uint32_t n = slab_count[item];
  if (n == kBlkOverflow || n == 0) return;
  const uint32_t run_item = item / n_slices, slice = item - run_item * n_slices;
  const uint32_t c = item_cluster[run_item];
  const uint32_t tb = table2_base[c] * 256u, ts = (table2_base[c + 1] - table2_base[c]) * 256u;
  const uint32_t base = slab_base[item];
  const uint32_t w0 = slice * Ws;
  const uint32_t lane = lane_id();
  for (uint32_t i0 = 0; i0 < n; i0 += 32) {
    const uint32_t p = base + i0 + lane;
    uint32_t g = 0xffffffffu, code = 0;
    if (i0 + lane < n) code = slab_cnt[p];
    if (i0 + lane < n && partial_row_count(slab_rows, code, p, WP) != kCntDead) {   // (dead: folded into an earlier row of its slice)
      const unsigned long long key = slab_keys[p];
      uint32_t s = __umulhi((uint32_t)(mix64(key) >> 32), ts);
      if ((home_bits[(tb + s) >> 5] >> ((tb + s) & 31)) & 1u) {      // a survivor lives at this home slot
        uint32_t probes = 0;                             // (kB4 put the key there; bounded all the same)
        while (table2[tb + s].key != key && ++probes <= ts) { if (++s == ts) s = 0; }
        if (probes <= ts) g = table2[tb + s].row;        // nil: its k-mer did not pass the window
      }
    }
    // the rows of survivors (a fifth of the partial rows: surviving k-mers sit in most slices) are
    // copied by half-warps, two rows per instruction, 64 B coalesced: ms_count of config 4 129.0
    // against 135.7 ms with every lane copying its own row.  A one-sample row is one word: kB5
    // cleared the k-mer's row and its slice has no other live row
    const bool single = g != 0xffffffffu && cnt_single(code);
    if (single) {
      const uint32_t s = code & 0x3ffu;
      out.cand[(size_t)g * out.key_words + w0 + (s >> 5)] = 1u << (s & 31u);
    }
    uint32_t m = __ballot_sync(kFull, g != 0xffffffffu && !single);
    while (m) {
      const int l0 = __ffs(m) - 1;
      m &= m - 1;
      const int l1 = m ? __ffs(m) - 1 : -1;
      if (m) m &= m - 1;
      const int from = lane < 16 ? l0 : l1;
      const uint32_t gg = __shfl_sync(kFull, g, from < 0 ? 0 : from);
      const uint32_t pp = __shfl_sync(kFull, p, from < 0 ? 0 : from);
      if (from >= 0) {
        const uint32_t* src = slab_rows + (size_t)pp * WP;
        uint32_t* dst = out.cand + (size_t)gg * out.key_words + w0;
        for (uint32_t w = lane & 15u; w < Ws && w0 + w < W; w += 16u) dst[w] = src[w];
      }
    }
  }
}

}  // namespace pf
