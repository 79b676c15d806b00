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
//                       A chunk's key carries the run's live-window mask (ragged tails, N /
//                       IUPAC symbols), so every sequence takes this path.
//                       Level 2: the few dozen DISTINCT chunks are cut into their live k-mers
//                       (forward / reverse complement / canonical), each k-mer is looked up in
//                       a shared-memory open-addressing table and the (chunk, window) pair is
//                       pushed onto the k-mer row's list.  The CTA ends by writing its distinct
//                       k-mers, popcounts and bitsets ("partial rows", a bitset being the OR of
//                       the listed chunks' bitsets) to a slab in HBM: ~1/30 of the bytes the
//                       records would have taken, written once.  A row of one sample (most
//                       rows) is written as its key and a one-sample code, without the bitset
//                       (see slab_cnt).  Every run keeps its own slab, so the kernels after kA
//                       see per-run items.
//   kB1/kB3             a k-mer can start in two runs (indels, clamped flanks, paralogs,
//                       repeats), so the partial rows of one cluster are merged by FULL key in a
//                       per-cluster open-addressing table in global memory: the first row of a
//                       key owns it, later ones OR their bitset into the owner's; owners are
//                       filtered on their popcount with the integer MAF window and emitted,
//                       one CTA per cluster, with the cluster's distinct bitsets as K4's candidates.
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

// ---------------------------------------------------------------------------
// Device-side planning of an upload: the caller's pf_seq_desc array goes to the device as it is
// and ONE kernel validates every descriptor (include/panfeed_b200.h: pf_seq_desc), rebases it to
// the sub-range and writes the 64-byte SeqDev, the 16-byte SeqLite and the batch totals.  The host
// touches no descriptor: with several ranks sharing the host's cores, per-sequence host planning
// (~15 ns per sequence and thread) was what bounded the end-to-end rate.  The block engine runs
// from this alone; a batch that runs a record width also needs record offsets and tile lists,
// which plan_records (pf_upload.cuh) derives on the device from the SeqDev array.
// ---------------------------------------------------------------------------
struct PlanTotals {          // 128 bytes, zeroed (err = all ones) before plan_from_raw
  unsigned long long bases, windows, pos_windows;
  unsigned long long err;    // min over bad sequences of (index << 32 | code); ~0 = none
  // plan_records: totals of the per-sequence offsets (kOff* order), then per record width
  // (narrow, wide, 256-bit) the largest cluster and the sort tiles, and the local-reduce tiles
  uint32_t seq_tot[6], max_seg[3], n_tiles[3], n_ltiles;
  uint32_t pad[11];
};
static_assert(sizeof(PlanTotals) == 128, "PlanTotals");
enum : uint32_t { kPlanErrCluster = 1, kPlanErrClusterOrder, kPlanErrSample, kPlanErrSampleOrder, kPlanErrPresence,
                  kPlanErrAlign, kPlanErrPlane, kPlanErrStrand, kPlanErrNoAmbPlane, kPlanErrAmbAlign,
                  kPlanErrAmbPlane };

__global__ void __launch_bounds__(256)
plan_from_raw(const pf_seq_desc* __restrict__ raw, uint32_t n, uint32_t cluster_base, uint64_t base_rebase,
              uint64_t amb_rebase, uint32_t n_clusters, uint32_t S, uint32_t W, const uint32_t* __restrict__ presence,
              uint64_t plane_bases, bool has_amb_plane, uint64_t amb_plane_symbols, int k, uint32_t emit_positions,
              SeqDev* __restrict__ out, SeqLite* __restrict__ lite, PlanTotals* __restrict__ tot) {
  __shared__ unsigned long long s_sum[3][8];
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long bases = 0, windows = 0, posw = 0;
  if (i < n) {
    const pf_seq_desc q = raw[i];
    uint32_t err = 0;
    const uint32_t cluster = q.cluster - cluster_base;
    const uint64_t base_off = q.base_off - base_rebase;
    const bool amb = (q.flags & PF_SEQ_AMBIGUOUS) != 0;
    const uint64_t amb_off = amb ? q.amb_off - amb_rebase : 0;
    if (q.cluster < cluster_base || cluster >= n_clusters) err = kPlanErrCluster;
    else if (q.sample >= S) err = kPlanErrSample;
    else if (!((presence[(size_t)cluster * W + (q.sample >> 5)] >> (q.sample & 31u)) & 1u)) err = kPlanErrPresence;
    else if (q.base_off < base_rebase || (base_off & 63u)) err = kPlanErrAlign;
    else if (base_off + q.len > plane_bases) err = kPlanErrPlane;
    else if (q.strand != 1 && q.strand != -1) err = kPlanErrStrand;
    else if (amb && !has_amb_plane) err = kPlanErrNoAmbPlane;
    else if (amb && (amb_off & 31u)) err = kPlanErrAmbAlign;
    else if (amb && amb_off + q.len > amb_plane_symbols) err = kPlanErrAmbPlane;
    else if (i) {
      const pf_seq_desc p = raw[i - 1];
      if (q.cluster < p.cluster) err = kPlanErrClusterOrder;
      else if (q.cluster == p.cluster && q.sample < p.sample) err = kPlanErrSampleOrder;
    }
    if (err) {
      atomicMin(&tot->err, ((unsigned long long)i << 32) | err);
    } else {
      const bool target = emit_positions && (q.flags & PF_SEQ_TARGET);
      SeqDev d;
      d.base_off = base_off; d.amb_off = amb_off; d.len = q.len; d.sample = q.sample; d.cluster = cluster;
      d.flags = (target ? 1u : 0u) | (amb ? 2u : 0u);
      d.start = q.start; d.end = q.end; d.offset = q.offset; d.strand = q.strand;
      d.rec_off = 0; d.pos_off = 0; d.wrec_off = 0; d.pwide_off = 0;
      out[i] = d;
      SeqLite l;
      l.word_off = (uint32_t)(base_off >> 5); l.len = q.len;
      l.sample_flags = q.sample | (amb ? 0x80000000u : 0u);
      l.amb_word_off = (uint32_t)(amb_off >> 5);
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
// are recorded on insertion, row lists are emptied as the epilogue reads them, and the chunk
// rows 0..n_chunks-1 are cleared.  An overflowing run may have claimed slots without
// a row; after it everything is cleared.
//
// chunk table: the R = k + 15 bases that the 16 windows of a run cover, as a 128-bit key
//   (top-aligned, bases past the sequence's end zero) whose free low 16 bits hold the run's
//   live-window mask.  Sequences of a cluster are copies of a few haplotypes, so the ~500
//   sequences of a run collapse into a few dozen distinct chunks; only those are cut into
//   k-mers.  A chunk keeps the sample bitset of its sequences and its first sequence's sample,
//   or kChunkMixed once a sequence of another sample joins it.  A slot's state word goes
//   empty -> locked -> (full | chunk id).
// k-mer table: 64-bit keys claimed with one CAS; rowid[slot] is published afterwards
//   (0xffff = not yet), readers of a freshly claimed slot spin for those few cycles.  A row
//   holds no bitset, only a list of the (chunk, window[, strand]) nodes that carry its k-mer:
//   rhead[row] -> pnext[node] -> ... -> kNodeNil.  Node = chunk * 16 + window (canonical) or
//   2 * (chunk * 16 + window) + strand (--non-canonical).
constexpr uint32_t kChunkEmpty = 0u, kChunkLocked = 1u, kChunkFull = 0x80000000u;
constexpr uint32_t kNodeNil = 0xffffu, kChunkMixed = 0xffffu;
constexpr uint32_t kBlkRowBytes = 14u;   // shared memory of a k-mer row: rkey, rhead, rslot
struct ARunView {
  BlkHead* h;              // n_unique = k-mer rows handed out, work = chunk ids handed out
  uint32_t* crows;         // [ccap * WP]  sample bitset of chunk id (16-byte aligned rows)
  uint64_t* keys;          // [slots]
  uint64_t* rkey;          // [cap + 1]   key of row id (row `cap`: scratch of an overflowing run)
  uint64_t* ckhi;          // [ccap]
  uint64_t* cklo;          // [ccap]      low 16 bits: live-window mask
  uint32_t* cstate;        // [cslots]
  uint32_t* rhead;         // [cap]       first node of row id's list
  uint16_t* rowid;         // [slots]
  uint16_t* rslot;         // [cap + 1]   key slot of row id
  uint16_t* cslot;         // [ccap]      state slot of chunk id
  uint16_t* csample;       // [ccap]      sample rank of chunk id's sequences, or kChunkMixed
  uint16_t* pnext;         // [ccap * 16 * (CANON ? 1 : 2)]  next node of a row's list
  uint32_t mask, shift, cmask, cshift, cap, ccap;
};
__host__ __device__ inline uint32_t blkA_ccap(uint32_t cslots) { return cslots * 3u / 4u; }
// slots: k-mer key slots (power of two); cap: k-mer rows (<= 13/16 slots); cslots: chunk slots
// (power of two, <= 2048 so that node ids fit 16 bits); canon: one list node per (chunk, window)
__host__ __device__ inline uint32_t blkA_smem_bytes(uint32_t slots, uint32_t cap, uint32_t cslots, uint32_t W,
                                                   bool canon) {
  const uint32_t ccap = blkA_ccap(cslots), WP = (W + 3u) & ~3u;
  return (uint32_t)sizeof(BlkHead) + ccap * WP * 4u + slots * 8u + (cap + 1u) * 8u + ccap * 16u + cslots * 4u +
         cap * 4u + slots * 2u + (cap + 1u) * 2u + ccap * 4u +
         ccap * (uint32_t)kBlkRun * (canon ? 2u : 4u) + 16u;
}
__device__ __forceinline__ ARunView arun_view(unsigned char* raw, uint32_t slots, uint32_t cap, uint32_t cslots, uint32_t W) {
  ARunView a;
  const uint32_t WP = (W + 3u) & ~3u;
  a.cap = cap;
  a.ccap = blkA_ccap(cslots);
  a.h = reinterpret_cast<BlkHead*>(raw);
  a.crows = reinterpret_cast<uint32_t*>(raw + sizeof(BlkHead));
  a.keys = reinterpret_cast<uint64_t*>(a.crows + a.ccap * WP);
  a.rkey = a.keys + slots;
  a.ckhi = a.rkey + (a.cap + 1u);
  a.cklo = a.ckhi + a.ccap;
  a.cstate = reinterpret_cast<uint32_t*>(a.cklo + a.ccap);
  a.rhead = a.cstate + cslots;
  a.rowid = reinterpret_cast<uint16_t*>(a.rhead + a.cap);
  a.rslot = a.rowid + slots;
  a.cslot = a.rslot + (a.cap + 1u);
  a.csample = a.cslot + a.ccap;
  a.pnext = a.csample + a.ccap;
  a.mask = slots - 1u;
  a.shift = 32u - (uint32_t)__popc(a.mask);
  a.cmask = cslots - 1u;
  a.cshift = 32u - (uint32_t)__popc(a.cmask);
  return a;
}
// chunk id of (hi, lo), created with `sample` if new; 0xffffffff if the chunk table is full (the
// run then overflows)
__device__ __noinline__ uint32_t chunk_find_or_insert(const ARunView a, uint64_t hi, uint64_t lo, uint32_t sample) {
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
        a.cslot[id] = (uint16_t)s;
        a.csample[id] = (uint16_t)sample;
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
__device__ __noinline__ uint32_t kmer_row_slow(const ARunView a, uint64_t key, uint32_t h) {
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
#define PF_KA_MIN_CTAS 5      // 5 x 256 threads at 48 registers; ~30 KB of shared memory per CTA at S = 500
#endif
// A CTA walks SEGMENTS: `seg_runs` consecutive (cluster, run) items of one slice (item =
// run_item * n_slices + slice), taken from counters[LC_SEGMENT] after the first one; with an
// item list (a rescue launch) a segment is one listed item.  Every run still gets its own slab.
// Across the runs of a segment a thread keeps its first two sequences of the (cluster, slice) in
// registers: descriptor and the 64-bit words wi, wi + 1 of the run.  A run starts at a multiple
// of 16, so its R <= 47 bases lie in two words.
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
  const uint32_t W = plan.W, WP = plan.WP;
  const ARunView a = arun_view(blk_raw, plan.slots, plan.cap, plan.cslots, W);
  const uint32_t tid = threadIdx.x;

  auto clear_tables = [&]() {
    for (uint32_t i = tid; i < plan.slots; i += kBlkThreads) { a.keys[i] = ~0ull; a.rowid[i] = 0xffffu; }
    for (uint32_t i = tid; i < plan.cslots; i += kBlkThreads) a.cstate[i] = kChunkEmpty;
    for (uint32_t i = tid; i < a.cap; i += kBlkThreads) a.rhead[i] = kNodeNil;
    for (uint32_t i = tid; i < a.ccap * WP; i += kBlkThreads) a.crows[i] = 0u;
  };
  clear_tables();
  if (tid == 0) { a.h->n_unique = 0; a.h->overflow = 0; a.h->work = 0; a.h->n_pass = 0; a.h->singles = 0; }
  __syncthreads();

  const uint32_t sh64 = 64u - 2u * (uint32_t)k;
  const uint32_t R = (uint32_t)k + (uint32_t)kBlkRun - 1u;      // bases a full run covers (<= 47)
  // top-aligned masks of the R bases
  const uint64_t cm_hi = R >= 32u ? ~0ull : (~0ull << (64u - 2u * R));
  const uint64_t cm_lo = R > 32u ? (~0ull << (64u - 2u * (R - 32u))) : 0ull;

  // one k-mer (in the low 2k bits) -> row, `node` pushed onto the row's list
  auto put_node = [&](uint64_t key, uint32_t node) {
    const uint32_t h = blk_hash((uint32_t)(key >> 32), (uint32_t)key, a.shift);
    uint32_t id = 0xffffu;
    if (*reinterpret_cast<const volatile uint64_t*>(&a.keys[h]) == key)
      id = *reinterpret_cast<const volatile uint16_t*>(&a.rowid[h]);
    if (id == 0xffffu) id = kmer_row_slow(a, key, h);
    if (id < a.cap) a.pnext[node] = (uint16_t)atomicExch(&a.rhead[id], node);
  };

  // the thread's sequences j = 0, 1 of the (cluster, slice) whose first sequence is st_lo, at
  // word index st_wi: window count (0: none), sample | ambiguity flag, first word, words
  uint32_t st_lo = 0xffffffffu, st_wi = 0;
  uint32_t nw0 = 0, nw1 = 0, sf0 = 0, sf1 = 0, wo0 = 0, wo1 = 0;
  uint64_t c0 = 0, n0 = 0, c1 = 0, n1 = 0;

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
      auto fetch = [&](uint32_t nw, uint32_t wo, uint64_t& c, uint64_t& n) {
        c = 0; n = 0;
        if (s_rel < nw) {
          const uint64_t* w = bases + wo + wi;
          c = __ldg(w); n = __ldg(w + 1);
        }
      };
      auto slide = [&](uint32_t nw, uint32_t wo, uint64_t& c, uint64_t& n) {
        c = n; n = 0;
        if (s_rel < nw) n = __ldg(bases + wo + wi + 1u);
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
        slide(nw0, wo0, c0, n0);
        slide(nw1, wo1, c1, n1);
      } else if (seq_lo != st_lo || wi != st_wi) {
        fetch(nw0, wo0, c0, n0);
        fetch(nw1, wo1, c1, n1);
      }
      st_lo = seq_lo;
      st_wi = wi;

      // ---- phase 1: every sequence's run -> chunk table: the bases its live windows cover and
      //      the mask of those windows (a ragged tail, windows over N / IUPAC symbols) ---------
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
        const uint32_t o0 = s_rel & 31u;
        uint32_t live = (1u << nv) - 1u;                 // bit q: window s_rel + q exists, no N in it
        if (sf >> 31) {                                  // ambiguous: the N / IUPAC bit plane, MSB first
          const uint32_t* ab = ambbits + seqs[si].amb_word_off + wi;
          const uint64_t t = (((uint64_t)ab[0] << 32) | (uint64_t)ab[1]) << o0;
          for (uint32_t q = 0; q < nv; ++q)
            if ((t << q) >> (64 - k)) live &= ~(1u << q);
          if (!live) continue;
        }
        uint64_t hi = w0, lo = w1;
        if (o0) {
          hi = (w0 << (2u * o0)) | (w1 >> (64u - 2u * o0));
          lo = w1 << (2u * o0);
        }
        // the bases the run covers (top-aligned; those past the sequence's end cleared, so
        // equal ragged tails meet) and the live-window mask in the free low bits of lo
        if (nv == (uint32_t)kBlkRun) {
          hi &= cm_hi; lo &= cm_lo;
        } else {
          const uint32_t nb = nv + (uint32_t)k - 1u;
          hi &= nb >= 32u ? ~0ull : ~0ull << (64u - 2u * nb);
          lo &= nb > 32u ? ~0ull << (64u - 2u * (nb - 32u)) : 0ull;
        }
        const uint32_t cs = chunk_find_or_insert(a, hi, lo | live, sample);
        if (cs == 0xffffffffu) { a.h->overflow = 1u; continue; }
        atomicOr(&a.crows[cs * WP + (sample >> 5)], 1u << (sample & 31u));
        if (a.csample[cs] != sample) a.csample[cs] = (uint16_t)kChunkMixed;   // (a paralog of the same sample is not)
      }
      __syncthreads();

      // ---- phase 2: distinct chunks x live windows -> k-mer table; a (chunk, window) pair only
      //      adds itself to its k-mer row's list -------------------------------------------------
      const uint32_t n_chunks = min(a.h->work, a.ccap);
      const uint32_t n_pairs = a.h->overflow ? 0u : n_chunks * (uint32_t)kBlkRun;
      // pairs cost very different amounts (a new k-mer is an insertion): the first round is
      // static, after it the warps take 32 pairs at a time from a counter
      for (uint32_t q0 = (tid & ~31u);;) {
        const uint32_t p = q0 + (tid & 31u);
        if (p < n_pairs) {
          const uint32_t cs = p >> 4, q = p & 15u;
          const uint64_t lo = a.cklo[cs];
          if ((lo >> q) & 1u) {
            const uint64_t hi = a.ckhi[cs];
            const uint64_t x = q ? ((hi << (2u * q)) | (lo >> (64u - 2u * q))) : hi;
            const uint64_t fwd = x >> sh64, rc = revcomp2(fwd, k);
            if (CANON) put_node(rc < fwd ? rc : fwd, p);
            else { put_node(fwd, 2u * p); put_node(rc, 2u * p + 1u); }
          }
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
        // a warp takes 32 rows: every lane writes its row's key, takes its list and empties it.
        // A list of ONE node whose chunk has one sample (most rows: the k-mers of a private SNP)
        // is a one-sample row: its code comes from the chunk, no bitset is read or written.  The
        // other rows are listed (lane ids, in the chunk keys, which are dead until the next run:
        // ccap >= 16 gives 32 bytes per warp) and built by L lanes each, L = WP / 4 rounded up to
        // a power of two: they walk the row's list together, OR one uint4 slice of every listed
        // chunk's row, and sum the popcount by shuffles.  A row whose OR has one bit (two chunks
        // of one sample's paralogs) is still written as a one-sample code.
        const size_t base = a.h->row_base;
        const uint32_t L = WP > 16u ? 8u : WP > 8u ? 4u : WP > 4u ? 2u : 1u, lane = tid & 31u;
        const uint32_t lrow = lane / L, lq = 4u * (lane & (L - 1u)), per = 32u / L;
        const uint32_t nsh = CANON ? 4u : 5u;            // node -> chunk id
        uint8_t* list = reinterpret_cast<uint8_t*>(a.ckhi) + (tid & ~31u);
        uint32_t singles = 0;
        for (uint32_t r0 = tid & ~31u; r0 < n; r0 += kBlkThreads) {
          const uint32_t r = r0 + lane;
          bool multi = false;
          uint32_t head = kNodeNil;
          if (r < n) {
            slab_keys[base + r] = a.rkey[r];
            head = a.rhead[r];
            a.rhead[r] = kNodeNil;
            const uint32_t c = head >> nsh;
            const uint32_t s1 = a.csample[c];
            multi = a.pnext[head] != kNodeNil || s1 == kChunkMixed;
            if (!multi) slab_cnt[base + r] = kCntSingle | s1;
            const uint32_t h = a.rslot[r];
            a.keys[h] = ~0ull;
            a.rowid[h] = 0xffffu;
          }
          const uint32_t m = __ballot_sync(kFull, multi), nm = (uint32_t)__popc(m);
          if (multi) list[__popc(m & lanemask_lt())] = (uint8_t)lane;
          singles += min(32u, n - r0) - nm;
          __syncwarp();
          for (uint32_t g0 = 0; g0 < nm; g0 += per) {
            const uint32_t g = g0 + lrow;
            const uint32_t src = g < nm ? list[g] : 0u;
            uint32_t node = __shfl_sync(kFull, head, src);
            uint4 x = make_uint4(0u, 0u, 0u, 0u);
            if (g < nm && lq < WP) {
              for (; node != kNodeNil; node = a.pnext[node]) {
                const uint4 y = *reinterpret_cast<const uint4*>(a.crows + (node >> nsh) * WP + lq);
                x.x |= y.x; x.y |= y.y; x.z |= y.z; x.w |= y.w;
              }
            }
            uint32_t cnt = __popc(x.x) + __popc(x.y) + __popc(x.z) + __popc(x.w);
            uint32_t one = x.x ? 32u * lq + __ffs(x.x) - 1u : x.y ? 32u * (lq + 1u) + __ffs(x.y) - 1u
                         : x.z ? 32u * (lq + 2u) + __ffs(x.z) - 1u : x.w ? 32u * (lq + 3u) + __ffs(x.w) - 1u : 0u;
            for (uint32_t o = 1; o < L; o <<= 1) {
              cnt += __shfl_xor_sync(kFull, cnt, o);
              one |= __shfl_xor_sync(kFull, one, o);
            }
            singles += __popc(__ballot_sync(kFull, g < nm && lq == 0u && cnt == 1u));
            if (g < nm) {
              const size_t p = base + r0 + src;
              if (lq == 0u) slab_cnt[p] = cnt == 1u ? kCntSingle | one : cnt;
              if (cnt != 1u && lq < WP) reinterpret_cast<uint4*>(slab_rows + p * WP + lq)[0] = x;
            }
          }
          __syncwarp();
        }
        if (lane == 0 && singles) atomicAdd(&a.h->singles, singles);
        __syncthreads();                                 // chunk rows are read until here
        for (uint32_t c = tid; c < n_chunks; c += kBlkThreads) a.cstate[a.cslot[c]] = kChunkEmpty;
        for (uint32_t i = tid; i < n_chunks * WP; i += kBlkThreads) a.crows[i] = 0u;
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

// kB3: one CTA per cluster; owners are counted, filtered and written out as rows, and the rows'
// bitsets are deduplicated inside the cluster before K4 sees them.  All k-mers of a stretch of a
// cluster carry the same sample set until a SNP enters or leaves the window, so ~4 surviving rows
// share each pattern; patterns of different clusters rarely coincide.  K4 gets one candidate per
// pattern of a cluster instead of one per row (row_cand maps a row to its candidate) and still
// deduplicates the candidates globally on the full key, so the result does not depend on how
// many rows share a candidate.
//   pass 1  verdict of every partial row (owner, count in [lo, hi]); the survivors are listed in
//           shared memory; ONE atomic takes the cluster's rows
//   pass 2  the rows, one survivor per thread; each bitset is found or inserted in a
//           shared-memory table of the cluster's patterns (entry: 16-bit hash fingerprint |
//           candidate id; a candidate remembers the survivor that created it, and a match is
//           confirmed on all words: nothing is merged on a hash).  Lanes of a warp with equal
//           hashes (neighbouring k-mers of one stretch) compare with their leader instead.
//   pass 3  ONE atomic takes the candidates; their bitsets and row_cand are written
// A cluster with more survivors than the list takes (PF_PATTERN_SMEM_KB) makes every row its own
// candidate, written on a second walk over its partial rows.
constexpr uint32_t kEmitThreads = 512;
constexpr uint32_t kEmitWarps = kEmitThreads / 32;
constexpr uint32_t kPatEmpty = 0xffffffffu, kPatLocked = 0xfffffffeu;
constexpr uint32_t kPatMaxCand = 0xfff0u;          // candidate ids stay below the two marks' low halves
constexpr uint32_t kNoOne = 0xffffu;               // a survivor whose bitset is a row of slab_rows
// survivors of a cluster that `smem` bytes take: per survivor its partial row (4 bytes), count and
// one-sample code (4), 1.5 table slots (6) and, as a candidate, the survivor that created it (2)
__host__ __device__ inline uint32_t pattern_table_rows(uint32_t smem) {
  const uint32_t n = smem >= 16u ? (smem - 16u) / 16u : 0u;
  return n < kPatMaxCand ? n : kPatMaxCand;
}

// words 4q .. 4q + 3 of a pattern: partial row p of slab_rows (W rounded up to WP with zeros),
// or the one-hot bitset of sample `one` (a one-sample row has no bitset in slab_rows)
__device__ __forceinline__ uint4 pattern_quad(const uint32_t* __restrict__ slab_rows, uint32_t p, uint32_t one,
                                              uint32_t q, uint32_t WP) {
  if (one == kNoOne) return __ldg(reinterpret_cast<const uint4*>(slab_rows + (size_t)p * WP) + q);
  uint4 x = make_uint4(0u, 0u, 0u, 0u);
  if ((one >> 7) == q) {
    const uint32_t b = 1u << (one & 31u);
    switch ((one >> 5) & 3u) {
      case 0: x.x = b; break;
      case 1: x.y = b; break;
      case 2: x.z = b; break;
      default: x.w = b; break;
    }
  }
  return x;
}

__global__ void __launch_bounds__(kEmitThreads)
kB3_cluster_emit(const uint64_t* __restrict__ slab_keys, const uint32_t* __restrict__ slab_rows,
                 const uint32_t* __restrict__ slab_base, const uint32_t* __restrict__ slab_count,
                 const uint32_t* __restrict__ item_base /* [n_clusters + 1] */,
                 const uint32_t* __restrict__ slab_cnt, const ClusterDev* __restrict__ clusters, RowOut out,
                 uint32_t row_capacity, uint32_t* __restrict__ counters, uint32_t W, uint32_t WP,
                 uint32_t cap /* pattern_table_rows(dynamic shared memory) */) {
  extern __shared__ uint32_t pat_sm[];
  __shared__ uint32_t s_total, s_emit, s_row_base, s_mode, s_cand_base, s_n_cand;
  const uint32_t c = blockIdx.x, tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  const uint32_t it0 = item_base[c], it1 = item_base[c + 1];
  const ClusterDev cl = clusters[c];
  const uint32_t NQ = WP >> 2;
  uint32_t* list_p = pat_sm;                  // [cap] partial row of survivor j
  uint32_t* list_c = list_p + cap;            // [cap] one-sample code << 16 | count (pass 2: | candidate)
  if (tid == 0) { s_total = 0; s_emit = 0; s_n_cand = 0; }
  __syncthreads();

  // every survivor of the cluster: visit(partial row, count, one-sample code, index j from *next).
  // A warp takes every kEmitWarps-th slab, 128 rows per turn (four loads in flight per lane).
  auto walk = [&](uint32_t* next, auto&& visit) {
    for (uint32_t it = it0 + warp; it < it1; it += kEmitWarps) {
      uint32_t n = slab_count[it];
      if (n == kBlkOverflow) n = 0;
      const uint32_t base = slab_base[it];
      for (uint32_t i0 = 0; i0 < n; i0 += 128) {
        uint32_t code[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const uint32_t i = i0 + 32u * u + lane;
          code[u] = i < n ? slab_cnt[base + i] : kCntDead;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const uint32_t p = base + i0 + 32u * u + lane;
          const uint32_t cnt = partial_row_count(slab_rows, code[u], p, WP);     // kCntDead past n
          const bool pass = cnt != kCntDead && cnt >= cl.lo && cnt <= cl.hi;
          const uint32_t mp = __ballot_sync(kFull, pass);
          if (!mp) continue;
          uint32_t b = 0;
          if (lane == 0) b = atomicAdd(next, (uint32_t)__popc(mp));
          b = __shfl_sync(kFull, b, 0);
          if (pass) visit(p, cnt, cnt_single(code[u]) ? (code[u] & 0x3ffu) : kNoOne, b + __popc(mp & lanemask_lt()));
        }
      }
    }
  };
  auto write_row = [&](uint32_t gi, uint32_t p, uint32_t cnt) {
    out.cluster[gi] = cl.id;
    out.kmer[gi] = slab_keys[p];
    out.count[gi] = cnt;
  };
  auto write_cand = [&](uint32_t id, uint32_t p, uint32_t one) {
    uint32_t* dst = out.cand + (size_t)id * out.key_words;
    for (uint32_t q = 0; q < NQ; ++q) {
      const uint4 x = pattern_quad(slab_rows, p, one, q, WP);
      const uint32_t w = 4 * q;
      if (w < W) dst[w] = x.x;
      if (w + 1 < W) dst[w + 1] = x.y;
      if (w + 2 < W) dst[w + 2] = x.z;
      if (w + 3 < W) dst[w + 3] = x.w;
    }
    if (out.key_words > W) dst[W] = out.cluster_pattern[c];       // the same word for every row of c
  };

  // ---- pass 1: list the survivors ----------------------------------------------------------------
  walk(&s_total, [&](uint32_t p, uint32_t cnt, uint32_t one, uint32_t j) {
    if (j < cap) { list_p[j] = p; list_c[j] = (one << 16) | cnt; }
  });
  __syncthreads();
  if (tid == 0) {
    const uint32_t total = s_total;
    uint32_t b = 0, mode = 0;                       // 0: nothing to write, 1: table, 2: a candidate per row
    if (total) {
      b = atomicAdd(&counters[LC_ROWS], total);
      if ((uint64_t)b + total > row_capacity) atomicExch(&counters[LC_ROW_OVERFLOW], 1u);
      else if (total <= cap) mode = 1;
      else { mode = 2; s_cand_base = atomicAdd(&counters[LC_CAND], total); }
    }
    s_row_base = b;
    s_mode = mode;
  }
  __syncthreads();
  const uint32_t mode = s_mode, total = s_total, row_base = s_row_base;
  if (mode == 0) return;
  if (mode == 2) {                                  // too many survivors: walk again, rows are candidates
    const uint32_t cand_base = s_cand_base;
    walk(&s_emit, [&](uint32_t p, uint32_t cnt, uint32_t one, uint32_t j) {
      write_row(row_base + j, p, cnt);
      write_cand(cand_base + j, p, one);
      out.row_cand[row_base + j] = cand_base + j;
    });
    return;
  }

  // ---- pass 2: rows, and the candidate of each ------------------------------------------------
  const uint32_t slots = total + (total >> 1) + 1u;
  uint32_t* tab = list_c + cap;                                     // [slots]
  uint16_t* cand = reinterpret_cast<uint16_t*>(tab + slots);        // [<= total] survivor that created it
  for (uint32_t i = tid; i < slots; i += kEmitThreads) tab[i] = kPatEmpty;
  __syncthreads();
  auto same = [&](uint32_t p, uint32_t one, uint32_t p2, uint32_t one2) {
    if (one != kNoOne && one2 != kNoOne) return one == one2;
    for (uint32_t q = 0; q < NQ; ++q) {
      const uint4 a = pattern_quad(slab_rows, p, one, q, WP), b = pattern_quad(slab_rows, p2, one2, q, WP);
      if (a.x != b.x || a.y != b.y || a.z != b.z || a.w != b.w) return false;
    }
    return true;
  };
  auto new_cand = [&](uint32_t j) {
    const uint32_t id = atomicAdd(&s_n_cand, 1u);   // each survivor takes at most one: ids < total
    cand[id] = (uint16_t)j;
    return id;
  };
  // local candidate id of survivor j's pattern (inserted if new)
  auto find_or_insert = [&](uint32_t j, uint32_t p, uint32_t one, uint64_t h) -> uint32_t {
    const uint32_t fp = (uint32_t)h & 0xffffu;
    uint32_t s = __umulhi((uint32_t)(h >> 32), slots);
    for (uint32_t probes = 0, spins = 0; probes < slots;) {
      const uint32_t e = ld_volatile_shared(&tab[s]);
      if (e == kPatEmpty) {
        if (atomicCAS(&tab[s], kPatEmpty, kPatLocked) == kPatEmpty) {
          const uint32_t id = new_cand(j);
          __threadfence_block();
          *reinterpret_cast<volatile uint32_t*>(&tab[s]) = (fp << 16) | id;
          return id;
        }
        continue;
      }
      if (e == kPatLocked) {                    // its owner publishes it in a few cycles
        if (++spins > (1u << 14)) break;
        __nanosleep(20);
        continue;
      }
      if ((e >> 16) == fp) {
        const uint32_t id = e & 0xffffu;
        const uint32_t j2 = *reinterpret_cast<volatile uint16_t*>(&cand[id]);
        if (same(p, one, list_p[j2], list_c[j2] >> 16)) return id;
      }
      if (++s == slots) s = 0;
      ++probes;
    }
    return new_cand(j);                         // no slot: a candidate of its own (K4 merges it)
  };
  for (uint32_t j0 = warp * 32u; j0 < total; j0 += kEmitThreads) {
    const uint32_t j = j0 + lane;
    const bool live = j < total;
    uint32_t p = 0, one = kNoOne;
    uint64_t h = ~0ull;
    if (live) {
      p = list_p[j];
      const uint32_t lc = list_c[j];
      one = lc >> 16;
      write_row(row_base + j, p, lc & 0xffffu);
      h = 0;
      for (uint32_t q = 0; q < NQ; ++q) {
        const uint4 x = pattern_quad(slab_rows, p, one, q, WP);
        h += word_hash(x.x, 4 * q) + word_hash(x.y, 4 * q + 1) + word_hash(x.z, 4 * q + 2) + word_hash(x.w, 4 * q + 3);
      }
      h = fmix64(h);
    }
    const uint32_t lm = __ballot_sync(kFull, live);
    uint32_t leader = lane;
    if (live) leader = __ffs(__match_any_sync(lm, h)) - 1;
    uint32_t id = 0;
    if (live && lane == leader) id = find_or_insert(j, p, one, h);
    const uint32_t lid = __shfl_sync(kFull, id, leader);
    const uint32_t lp = __shfl_sync(kFull, p, leader), lone = __shfl_sync(kFull, one, leader);
    if (live && lane != leader) id = same(p, one, lp, lone) ? lid : find_or_insert(j, p, one, h);
    if (live) list_c[j] = (one << 16) | id;     // (the count is written; readers use the high half)
  }
  __syncthreads();

  // ---- pass 3: the candidates ---------------------------------------------------------------------
  if (tid == 0) s_cand_base = atomicAdd(&counters[LC_CAND], s_n_cand);
  __syncthreads();
  const uint32_t cand_base = s_cand_base, n_cand = s_n_cand;
  for (uint32_t id = tid; id < n_cand; id += kEmitThreads) {
    const uint32_t j = cand[id];
    write_cand(cand_base + id, list_p[j], list_c[j] >> 16);
  }
  for (uint32_t j = tid; j < total; j += kEmitThreads) out.row_cand[row_base + j] = cand_base + (list_c[j] & 0xffffu);
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
