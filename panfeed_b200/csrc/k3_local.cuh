// K3 (partition mode) — per-k-mer sample presence from PARTIALLY sorted records.
//
// After `p` radix passes the records of a cluster are ordered by the leading
// 8p bits of the mixed key only.  Instead of spending more global passes, one
// CTA takes all prefix-runs that START inside its 2048-record tile (a handful
// of buckets, typically a few thousand records and ~100 distinct k-mers),
// streams their records through a shared-memory open-addressing table keyed on
// the FULL 64-bit key, and does the whole reduction on chip.  Two variants:
//
// k3_local_direct (S <= 1024): every distinct key gets a dense id and a W-word
//   bitset in shared memory; each record is one table probe + one atomicOr.  The
//   sample count is the popcount, so record order is irrelevant.  One pass over
//   the records.
//
// k3_local (any S): bitsets for every key would not fit, so
//   phase 1  find-or-insert the key, count its distinct samples.  Records of one
//            key arrive in ascending sample order (stable passes, sample-ordered
//            packing): across 2048-record chunks only "equal to the last sample
//            seen" can repeat; inside a chunk a (slot, sample) pair set removes
//            duplicates exactly.
//   phase 2  keys whose count lies in the cluster's integer MAF window get a row.
//   phase 3  the records are streamed again (L2-resident) and the surviving keys'
//            sample bits are OR-ed into shared-memory bitsets, as many rows per
//            round as fit, then written out coalesced.
//
// Replaces `cluster_dict[kmer][sortstrain[strain]] = 1` and the filters of
// /root/reference/panfeed/panfeed.py:77-88,190-204.  Exact for any input: a CTA
// that meets more distinct keys than it can hold raises a flag; the host falls
// back from the direct to the general variant, and from there re-runs the batch
// with 8 more sorted bits (at 64 bits a tile holds at most 2048 + 1 distinct
// keys, which always fits the general table).
#pragma once
#include "pf_common.cuh"
#include "k3_reduce.cuh"

namespace pf {

constexpr int kLocalThreads = 256;
constexpr int kLocalItems = 8;
constexpr int kLocalTile = kLocalThreads * kLocalItems;   // 2048 records
constexpr uint64_t kEmptyKey = ~0ull;
constexpr uint32_t kNoRow = 0xffffffffu;
enum { LC_ROWS = 0, LC_UNIQUE = 1, LC_TABLE_OVERFLOW = 2, LC_ROW_OVERFLOW = 3, LC_RESCUE = 4,
       LC_PARTIALS = 5, LC_PARTIAL_OVERFLOW = 6, LC_SEGMENT = 7 /* kA's segment counter */,
       LC_SINGLES = 8 /* one-sample partial rows kA wrote */,
       LC_CAND = 9 /* K4 candidates of kB3_cluster_emit: patterns distinct within a cluster */, LC_COUNT = 10 };

// prefix-runs of one radix pass are the digit buckets: their starts are the
// scanned histogram itself.  first_run[t] = first bucket starting at or after tile t.
__global__ void k3_tiles_from_hist(const TileDev* __restrict__ ltiles, uint32_t n_ltiles,
                                   const uint32_t* __restrict__ digit_start /* [seg][256] */,
                                   uint32_t n_seg, uint32_t* __restrict__ tile_first_run) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t > n_ltiles) return;
  if (t == n_ltiles) { tile_first_run[t] = n_seg * kRadix; return; }
  const TileDev td = ltiles[t];
  const uint32_t* s = digit_start + (size_t)td.seg * kRadix;
  uint32_t lo = 0, hi = kRadix;                 // first d with s[d] >= td.start
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (s[mid] < td.start) lo = mid + 1; else hi = mid;
  }
  tile_first_run[t] = td.seg * kRadix + lo;
}

// ---------------------------------------------------------------------------
// direct variant
// ---------------------------------------------------------------------------
constexpr int kDirectTile = 4096;                // records per CTA tile (2 chunks of 2048)
constexpr int kDirectSlots = 2048;
constexpr int kDirectPoolWords = 12288;          // 48 KB of bitsets
constexpr uint32_t kDirectMaxUnique = 768;
constexpr uint32_t kDirectMaxWords = 32;         // S <= 1024

struct DirectSmem {
  uint64_t keys[kDirectSlots + 1];     // slot kDirectSlots: home of the key equal to kEmptyKey
  alignas(16) uint32_t pool[kDirectPoolWords];   // dense id x W words
  uint16_t id[kDirectSlots + 2];       // slot -> dense id
  uint16_t slot_of[kDirectMaxUnique];  // dense id -> slot
  uint16_t row_id[kDirectMaxUnique];   // surviving row -> dense id
  uint32_t n_unique, n_pass, row_base, special_used, overflow, ok;
};

__global__ void __launch_bounds__(kLocalThreads, 3)
k3_local_direct(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ vals,
                const TileDev* __restrict__ ltiles, uint32_t n_ltiles,
                const uint32_t* __restrict__ tile_first_run /* [n_ltiles + 1] */,
                const uint32_t* __restrict__ run_start, uint32_t n_records,
                const ClusterDev* __restrict__ clusters, RowOut out, uint32_t row_capacity,
                uint32_t* __restrict__ counters,
                uint32_t* __restrict__ rescue_runs /* out: runs of tiles that did not fit */,
                const uint32_t* __restrict__ run_list /* null, or: one run per CTA (rescue launch) */,
                const uint32_t* __restrict__ run_seg /* null: seg = run / 256 (runs from the histogram) */) {
  extern __shared__ __align__(16) unsigned char local_raw[];
  DirectSmem& sm = *reinterpret_cast<DirectSmem*>(local_raw);
  const uint32_t tid = threadIdx.x;
  const uint32_t n_runs = tile_first_run[n_ltiles];
  uint32_t r0, r1, seg;
  if (run_list) {
    r0 = run_list[blockIdx.x];
    r1 = r0 + 1;
    seg = run_seg ? run_seg[r0] : r0 / kRadix;
  } else {
    r0 = tile_first_run[blockIdx.x];
    r1 = tile_first_run[blockIdx.x + 1];
    if (r0 == r1) return;
    seg = ltiles[blockIdx.x].seg;
  }
  const uint32_t a = run_start[r0];
  const uint32_t b = (r1 < n_runs) ? run_start[r1] : n_records;
  if (a >= b) return;
  const ClusterDev cl = clusters[seg];
  const uint32_t W = out.pattern_words;
  // bitset rows are W words at an ODD stride: the records a warp handles together mostly
  // carry the same sample (same word index), so distinct rows must fall in distinct banks
  const uint32_t WS = W | 1u;
  const uint32_t max_unique = min(kDirectMaxUnique, (uint32_t)kDirectPoolWords / WS);

  for (uint32_t i = tid; i <= kDirectSlots; i += kLocalThreads) sm.keys[i] = kEmptyKey;
  if (tid == 0) { sm.n_unique = 0; sm.n_pass = 0; sm.special_used = 0; sm.overflow = 0; sm.ok = 1; }
  __syncthreads();

  for (uint32_t c0 = a; c0 < b; c0 += kLocalTile) {
    uint64_t key[kLocalItems];
    uint32_t val[kLocalItems];
    uint16_t slot[kLocalItems];
    uint32_t inserted = 0;
#pragma unroll
    for (int j = 0; j < kLocalItems; ++j) {
      const uint32_t i = c0 + j * kLocalThreads + tid;
      val[j] = kInvalidSample;
      key[j] = 0;
      if (i < b) { key[j] = keys[i]; val[j] = vals[i]; }
    }
    const int n_items = (int)min((uint32_t)kLocalItems, (b - c0 + kLocalThreads - 1) / kLocalThreads);   // CTA-uniform
    // (i) find or insert
#pragma unroll
    for (int j = 0; j < kLocalItems; ++j) {
      slot[j] = 0xffff;
      if (j >= n_items) break;
      if (val[j] == kInvalidSample) continue;
      const uint64_t k = key[j];
      if (k == kEmptyKey) {
        if (atomicExch(&sm.special_used, 1u) == 0u) inserted |= 1u << j;
        slot[j] = kDirectSlots;
        continue;
      }
      uint32_t h = (uint32_t)k & (kDirectSlots - 1);
      for (int probes = 0; probes < kDirectSlots; ++probes) {
        const uint64_t cur = sm.keys[h];
        if (cur == k) { slot[j] = (uint16_t)h; break; }
        if (cur == kEmptyKey) {
          const uint64_t old = atomicCAS(reinterpret_cast<unsigned long long*>(&sm.keys[h]),
                                         (unsigned long long)kEmptyKey, (unsigned long long)k);
          if (old == kEmptyKey) { slot[j] = (uint16_t)h; inserted |= 1u << j; break; }
          if (old == k) { slot[j] = (uint16_t)h; break; }
        }
        h = (h + 1) & (kDirectSlots - 1);
      }
      if (slot[j] == 0xffff) sm.overflow = 1;
    }
    __syncthreads();
    // (ii) dense ids for the keys this thread inserted
    const uint32_t id_first = sm.n_unique;          // read by everyone before anyone adds
    __syncthreads();
    if (inserted) {
#pragma unroll
      for (int j = 0; j < kLocalItems; ++j) {
        if (inserted >> j & 1u) {
          const uint32_t id = atomicAdd(&sm.n_unique, 1u);
          if (id < max_unique) {
            sm.id[slot[j]] = (uint16_t)id;
            sm.slot_of[id] = slot[j];
          } else {
            sm.overflow = 1;
          }
        }
      }
    }
    __syncthreads();
    // bitsets of the new ids are zeroed on demand, by the whole CTA
    {
      const uint32_t id_last = min(sm.n_unique, max_unique);
      for (uint32_t i = id_first * WS + tid; i < id_last * WS; i += kLocalThreads) sm.pool[i] = 0;
    }
    __syncthreads();
    if (sm.overflow) {
      // too many distinct keys for one CTA: hand the tile's runs to the rescue launch
      // (one CTA per run); a single run that does not fit needs more sorted bits
      if (run_list || r1 - r0 == 1) {
        if (tid == 0) atomicExch(&counters[LC_TABLE_OVERFLOW], 1u);
      } else {
        if (tid == 0) sm.row_base = atomicAdd(&counters[LC_RESCUE], r1 - r0);
        __syncthreads();
        for (uint32_t r = r0 + tid; r < r1; r += kLocalThreads) rescue_runs[sm.row_base + (r - r0)] = r;
      }
      return;
    }
    // (iii) one OR per record
#pragma unroll
    for (int j = 0; j < kLocalItems; ++j) {
      if (j >= n_items) break;
      if (slot[j] == 0xffff) continue;
      const uint32_t v = val[j];
      atomicOr(&sm.pool[(uint32_t)sm.id[slot[j]] * WS + (v >> 5)], 1u << (v & 31u));
    }
  }
  __syncthreads();

  // ---- counts, filter, rows ---------------------------------------------------------
  const uint32_t n_unique = sm.n_unique;
  for (uint32_t id = tid; id < n_unique; id += kLocalThreads) {
    const uint32_t* bits = sm.pool + id * WS;
    uint32_t c = 0;
    for (uint32_t w = 0; w < W; ++w) c += __popc(bits[w]);
    if (c >= cl.lo && c <= cl.hi) sm.row_id[atomicAdd(&sm.n_pass, 1u)] = (uint16_t)id;
  }
  __syncthreads();
  if (tid == 0) {
    atomicAdd(&counters[LC_UNIQUE], n_unique);
    if (sm.n_pass) {
      const uint32_t base = atomicAdd(&counters[LC_ROWS], sm.n_pass);
      sm.row_base = base;
      if ((uint64_t)base + sm.n_pass > row_capacity) {
        sm.ok = 0;
        atomicExch(&counters[LC_ROW_OVERFLOW], 1u);
      }
    }
  }
  __syncthreads();
  const uint32_t n_pass = sm.n_pass;
  if (n_pass == 0 || !sm.ok) return;
  const uint32_t base = sm.row_base;
  for (uint32_t r = tid; r < n_pass; r += kLocalThreads) {
    const uint32_t id = sm.row_id[r];
    const uint32_t s = sm.slot_of[id];
    const uint32_t* bits = sm.pool + id * WS;
    uint32_t c = 0;
    for (uint32_t w = 0; w < W; ++w) c += __popc(bits[w]);
    const size_t g = (size_t)base + r;
    out.cluster[g] = cl.id;
    out.kmer[g] = unmix64(s < kDirectSlots ? sm.keys[s] : kEmptyKey);
    out.count[g] = c;
    if (out.key_words > W) out.cand[g * out.key_words + W] = out.cluster_pattern[seg];
  }
  for (uint32_t i = tid; i < n_pass * W; i += kLocalThreads) {
    const uint32_t r = i / W, w = i - r * W;
    out.cand[((size_t)base + r) * out.key_words + w] = sm.pool[(uint32_t)sm.row_id[r] * WS + w];
  }
}

// ---------------------------------------------------------------------------
// general variant
// ---------------------------------------------------------------------------
constexpr int kLocalSlots = 4096;                         // >= 2 * kLocalTile
constexpr uint32_t kLocalMaxUnique = 3072;
constexpr uint32_t kEmptyPair = 0xffffffffu;
constexpr uint32_t kLocalMaxSamples = 1u << 19;           // (slot:13 | sample:19) pair word
constexpr int kLocalPoolWords = 2 * kLocalSlots;          // 32 KB of bitsets per round

struct LocalSmem {
  uint64_t keys[kLocalSlots + 1];      // slot kLocalSlots: home of the key equal to kEmptyKey
  uint32_t cnt[kLocalSlots + 1];       // distinct samples
  uint32_t last[kLocalSlots + 1];      // 1 + largest sample of earlier chunks; phase 2+: row index
  uint32_t pairs[kLocalSlots];         // chunk-local (slot, sample) set   } phase 3: bitset pool
  uint32_t pool_tail[kLocalSlots];     //                                  }
  uint32_t n_unique, n_pass, row_base, special_used, overflow, ok;
};

__device__ __forceinline__ uint32_t local_find_or_insert(LocalSmem& sm, uint64_t key) {
  if (key == kEmptyKey) {
    if (atomicExch(&sm.special_used, 1u) == 0u) atomicAdd(&sm.n_unique, 1u);
    return kLocalSlots;
  }
  uint32_t h = (uint32_t)key & (kLocalSlots - 1);
  for (int probes = 0; probes < kLocalSlots; ++probes) {
    const uint64_t cur = sm.keys[h];
    if (cur == key) return h;
    if (cur == kEmptyKey) {
      const uint64_t old = atomicCAS(reinterpret_cast<unsigned long long*>(&sm.keys[h]),
                                     (unsigned long long)kEmptyKey, (unsigned long long)key);
      if (old == kEmptyKey) { atomicAdd(&sm.n_unique, 1u); return h; }
      if (old == key) return h;
    }
    h = (h + 1) & (kLocalSlots - 1);
  }
  sm.overflow = 1;
  return kNoRow;
}

__device__ __forceinline__ uint32_t local_find(const LocalSmem& sm, uint64_t key) {
  if (key == kEmptyKey) return kLocalSlots;
  uint32_t h = (uint32_t)key & (kLocalSlots - 1);
  while (sm.keys[h] != key) h = (h + 1) & (kLocalSlots - 1);
  return h;
}

__global__ void __launch_bounds__(kLocalThreads, 2)
k3_local(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ vals,
         const TileDev* __restrict__ ltiles, uint32_t n_ltiles,
         const uint32_t* __restrict__ tile_first_run /* [n_ltiles + 1] */,
         const uint32_t* __restrict__ run_start, uint32_t n_records,
         const ClusterDev* __restrict__ clusters, RowOut out, uint32_t row_capacity,
         uint32_t* __restrict__ counters) {
  extern __shared__ __align__(16) unsigned char local_raw[];
  LocalSmem& sm = *reinterpret_cast<LocalSmem*>(local_raw);
  const uint32_t tid = threadIdx.x;
  const uint32_t t = blockIdx.x;
  const uint32_t r0 = tile_first_run[t], r1 = tile_first_run[t + 1];
  if (r0 == r1) return;                       // no prefix-run starts in this tile
  const uint32_t n_runs = tile_first_run[n_ltiles];
  const uint32_t a = run_start[r0];
  const uint32_t b = (r1 < n_runs) ? run_start[r1] : n_records;
  if (a >= b) return;
  const uint32_t seg = ltiles[t].seg;
  const ClusterDev cl = clusters[seg];
  const uint32_t W = out.pattern_words;

  for (uint32_t i = tid; i <= kLocalSlots; i += kLocalThreads) {
    sm.keys[i] = kEmptyKey;
    sm.cnt[i] = 0;
    sm.last[i] = 0;
  }
  for (uint32_t i = tid; i < kLocalSlots; i += kLocalThreads) sm.pairs[i] = kEmptyPair;
  if (tid == 0) { sm.n_unique = 0; sm.n_pass = 0; sm.special_used = 0; sm.overflow = 0; sm.ok = 1; }
  __syncthreads();

  // ---- phase 1: group by full key, count distinct samples ---------------------
  for (uint32_t c0 = a; c0 < b; c0 += kLocalTile) {
    uint64_t key[kLocalItems];
    uint32_t val[kLocalItems];
    uint16_t slot[kLocalItems], pair_at[kLocalItems];
#pragma unroll
    for (int j = 0; j < kLocalItems; ++j) {
      const uint32_t i = c0 + j * kLocalThreads + tid;
      val[j] = kInvalidSample;
      key[j] = 0;
      if (i < b) { key[j] = keys[i]; val[j] = vals[i]; }
    }
#pragma unroll
    for (int j = 0; j < kLocalItems; ++j) {
      pair_at[j] = 0xffff;
      const uint32_t v = val[j];
      if (v == kInvalidSample) continue;
      const uint32_t s = local_find_or_insert(sm, key[j]);
      if (s == kNoRow) continue;
      slot[j] = (uint16_t)s;
      const uint32_t e = (s << 19) | v;
      uint32_t h = (e * 0x9e3779b1u) >> 20;              // 12 bits
      for (;;) {
        const uint32_t old = atomicCAS(&sm.pairs[h], kEmptyPair, e);
        if (old == kEmptyPair) { pair_at[j] = (uint16_t)h; break; }
        if (old == e) break;
        h = (h + 1) & (kLocalSlots - 1);
      }
      if (pair_at[j] != 0xffff && sm.last[s] != v + 1u) atomicAdd(&sm.cnt[s], 1u);
    }
    __syncthreads();
    if (sm.overflow || sm.n_unique > kLocalMaxUnique) {
      if (tid == 0) atomicExch(&counters[LC_TABLE_OVERFLOW], 1u);
      return;
    }
    // fold this chunk's samples into `last`, release the pair entries this thread set
#pragma unroll
    for (int j = 0; j < kLocalItems; ++j) {
      if (pair_at[j] != 0xffff) {
        atomicMax(&sm.last[slot[j]], val[j] + 1u);
        sm.pairs[pair_at[j]] = kEmptyPair;
      }
    }
    __syncthreads();
  }

  // ---- phase 2: which keys survive, row allocation -----------------------------
  for (uint32_t i = tid; i <= kLocalSlots; i += kLocalThreads) {
    const bool used = (i < kLocalSlots) ? (sm.keys[i] != kEmptyKey) : (sm.special_used != 0u);
    uint32_t row = kNoRow;
    if (used) {
      const uint32_t c = sm.cnt[i];
      if (c >= cl.lo && c <= cl.hi) row = atomicAdd(&sm.n_pass, 1u);
    }
    sm.last[i] = row;
  }
  __syncthreads();
  if (tid == 0) {
    atomicAdd(&counters[LC_UNIQUE], sm.n_unique);
    if (sm.n_pass) {
      const uint32_t base = atomicAdd(&counters[LC_ROWS], sm.n_pass);
      sm.row_base = base;
      if ((uint64_t)base + sm.n_pass > row_capacity) {
        sm.ok = 0;
        atomicExch(&counters[LC_ROW_OVERFLOW], 1u);
      }
    }
  }
  __syncthreads();
  const uint32_t n_pass = sm.n_pass;
  if (n_pass == 0 || !sm.ok) return;
  const uint32_t base = sm.row_base;
  for (uint32_t i = tid; i <= kLocalSlots; i += kLocalThreads) {
    const uint32_t row = sm.last[i];
    if (row != kNoRow) {
      const size_t g = (size_t)base + row;
      out.cluster[g] = cl.id;
      out.kmer[g] = unmix64(i < kLocalSlots ? sm.keys[i] : kEmptyKey);
      out.count[g] = sm.cnt[i];
      if (out.key_words > W) out.cand[g * out.key_words + W] = out.cluster_pattern[seg];
    }
  }

  // ---- phase 3: bitsets of the surviving keys, `per_round` rows at a time ----------
  uint32_t* pool = sm.pairs;                     // pairs + pool_tail are contiguous
  const uint32_t WS = (W | 1u) <= (uint32_t)kLocalPoolWords ? (W | 1u) : W;   // odd stride: no bank aliasing between rows
  const uint32_t per_round = max(1u, (uint32_t)kLocalPoolWords / WS);
  for (uint32_t lo = 0; lo < n_pass; lo += per_round) {
    const uint32_t rows = min(per_round, n_pass - lo);
    __syncthreads();
    for (uint32_t i = tid; i < rows * WS; i += kLocalThreads) pool[i] = 0;
    __syncthreads();
    for (uint32_t c0 = a; c0 < b; c0 += kLocalTile) {
      uint64_t key[kLocalItems];
      uint32_t val[kLocalItems];
#pragma unroll
      for (int j = 0; j < kLocalItems; ++j) {
        const uint32_t i = c0 + j * kLocalThreads + tid;
        val[j] = kInvalidSample;
        key[j] = 0;
        if (i < b) { key[j] = keys[i]; val[j] = vals[i]; }
      }
#pragma unroll
      for (int j = 0; j < kLocalItems; ++j) {
        const uint32_t v = val[j];
        if (v == kInvalidSample) continue;
        const uint32_t row = sm.last[local_find(sm, key[j])];
        if (row - lo < rows)                      // also false for kNoRow
          atomicOr(&pool[(row - lo) * WS + (v >> 5)], 1u << (v & 31u));
      }
    }
    __syncthreads();
    for (uint32_t i = tid; i < rows * W; i += kLocalThreads) {
      const uint32_t r = i / W, w = i - r * W;
      out.cand[((size_t)base + lo + r) * out.key_words + w] = pool[r * WS + w];
    }
  }
}

}  // namespace pf
