// K3 — segmented reduction of the sorted records into per-k-mer sample
// presence bitsets.  Replaces `cluster_dict[kmer][sortstrain[strain]] = 1`
// (/root/reference/panfeed/panfeed.py:77-88), the MAF test (:190-200) and the
// same-as-cluster test (:202-204).
//
//   k3_mark_runs   one streaming pass: a record starts a run if it is the first
//                  of its segment or its sorted prefix differs from its left
//                  neighbour's; run starts are compacted with warp ballots and a
//                  decoupled look-back across tiles.
//   k3_runs<COUNT> one warp per run: distinct-sample count (records of one key
//                  arrive in ascending sample order because the sort is stable),
//                  compared with the cluster's integer window [lo, hi] that the
//                  host derived from the reference's float64 expression.
//   k3_runs<EMIT>  only for surviving runs: the warp ORs sample bits into a
//                  shared-memory bitset (lanes that hit the same word are merged
//                  with match/reduce_or before one lane touches the word), then
//                  streams the W words out next to (cluster, un-mixed k-mer, count).
//
// A run is defined by the sorted PREFIX only.  If a run holds more than one
// distinct full key (probability ~2^-sort_bits per pair) or records that belong
// to the other key width, the warp walks its distinct keys in ascending order
// and treats each exactly; nothing is ever merged on a hash alone.
#pragma once
#include "pf_common.cuh"
#include "k2_onesweep.cuh"

namespace pf {

constexpr uint64_t kFlag64Agg = 1ull << 62;
constexpr uint64_t kFlag64Incl = 2ull << 62;
constexpr uint64_t kFlag64Mask = 3ull << 62;

template <typename KeyT, int ITEMS>
__global__ void __launch_bounds__(kSortThreads)
k3_mark_runs(const KeyT* __restrict__ keys, const TileDev* __restrict__ tiles, uint32_t n_tiles,
             int sort_bits, uint32_t* __restrict__ run_start, uint32_t* __restrict__ run_seg,
             uint32_t* __restrict__ tile_first_run /* [n_tiles + 1] or null */,
             uint64_t* __restrict__ lookback /* [n_tiles], zeroed */,
             uint32_t* __restrict__ ticket, uint32_t* __restrict__ n_runs_out,
             uint32_t* __restrict__ err) {
  constexpr int kWarps = kSortThreads / 32;
  constexpr int kGroups = ITEMS * kWarps;              // 32-record groups per tile
  __shared__ uint32_t group_count[kGroups];
  __shared__ uint32_t group_off[kGroups];
  __shared__ uint32_t s_tile;
  __shared__ uint64_t s_base;
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  if (tid == 0) s_tile = atomicAdd(ticket, 1u);
  __syncthreads();
  const uint32_t tile = s_tile;
  if (tile >= n_tiles) return;
  const TileDev td = tiles[tile];

  uint32_t heads[ITEMS];
#pragma unroll
  for (int j = 0; j < ITEMS; ++j) {
    const uint32_t idx = j * kSortThreads + tid;       // group g = j*kWarps + warp, tile order
    bool head = false;
    if (idx < td.count) {
      const size_t g = (size_t)td.start + idx;
      if (idx == 0 && tile == td.first_tile) head = true;
      else head = key_prefix(keys[g], sort_bits) != key_prefix(keys[g - 1], sort_bits);
    }
    heads[j] = __ballot_sync(kFull, head);
    if (lane == 0) group_count[j * kWarps + warp] = __popc(heads[j]);
  }
  __syncthreads();
  if (warp == 0) {                                      // scan 128 group counts
    uint32_t v[kGroups / 32], sum = 0;
#pragma unroll
    for (int i = 0; i < kGroups / 32; ++i) { v[i] = group_count[lane * (kGroups / 32) + i]; sum += v[i]; }
    uint32_t incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t n = __shfl_up_sync(kFull, incl, o);
      if (lane >= (uint32_t)o) incl += n;
    }
    uint32_t run = incl - sum;
#pragma unroll
    for (int i = 0; i < kGroups / 32; ++i) { group_off[lane * (kGroups / 32) + i] = run; run += v[i]; }
    const uint32_t total = __shfl_sync(kFull, incl, 31);
    if (lane == 0) {
      uint64_t prev = 0;
      if (tile != 0) {
        st_relaxed(&lookback[tile], kFlag64Agg | (uint64_t)total);
        uint32_t j = tile, spins = 0;
        for (;;) {
          --j;
          uint64_t x = ld_relaxed(&lookback[j]);
          bool failed = false;
          while ((x & kFlag64Mask) == 0ull) {
            if (++spins > kSpinLimit) { failed = true; break; }
            __nanosleep(40);
            x = ld_relaxed(&lookback[j]);
          }
          if (failed) { atomicExch(err, 2u); break; }
          prev += x & ~kFlag64Mask;
          if ((x & kFlag64Mask) == kFlag64Incl || j == 0) break;
        }
      }
      st_relaxed(&lookback[tile], kFlag64Incl | (prev + total));
      s_base = prev;
      if (tile_first_run) tile_first_run[tile] = (uint32_t)prev;
      if (tile == n_tiles - 1) {
        *n_runs_out = (uint32_t)(prev + total);
        if (tile_first_run) tile_first_run[n_tiles] = (uint32_t)(prev + total);
      }
    }
  }
  __syncthreads();
  const uint32_t base = (uint32_t)s_base;
#pragma unroll
  for (int j = 0; j < ITEMS; ++j) {
    if (heads[j] >> lane & 1u) {
      const uint32_t slot = base + group_off[j * kWarps + warp] + __popc(heads[j] & lanemask_lt());
      run_start[slot] = td.start + j * kSortThreads + tid;
      run_seg[slot] = td.seg;
    }
  }
}

// ---- warp helpers ----------------------------------------------------------
__device__ __forceinline__ uint64_t shfl_key(uint64_t k, int src) { return __shfl_sync(kFull, k, src); }
__device__ __forceinline__ Key128 shfl_key(const Key128& k, int src) {
  return Key128{__shfl_sync(kFull, k.hi, src), __shfl_sync(kFull, k.lo, src)};
}
__device__ __forceinline__ Key256 shfl_key(const Key256& k, int src) {
  return Key256{{__shfl_sync(kFull, k.w[0], src), __shfl_sync(kFull, k.w[1], src),
                 __shfl_sync(kFull, k.w[2], src), __shfl_sync(kFull, k.w[3], src)}};
}
__device__ __forceinline__ uint64_t shfl_xor_key(uint64_t k, int m) { return __shfl_xor_sync(kFull, k, m); }
__device__ __forceinline__ Key128 shfl_xor_key(const Key128& k, int m) {
  return Key128{__shfl_xor_sync(kFull, k.hi, m), __shfl_xor_sync(kFull, k.lo, m)};
}
__device__ __forceinline__ Key256 shfl_xor_key(const Key256& k, int m) {
  return Key256{{__shfl_xor_sync(kFull, k.w[0], m), __shfl_xor_sync(kFull, k.w[1], m),
                 __shfl_xor_sync(kFull, k.w[2], m), __shfl_xor_sync(kFull, k.w[3], m)}};
}
// minimum over lanes whose `has` is set; returns whether any lane had one
template <typename KeyT>
__device__ __forceinline__ bool warp_min_key(KeyT& key, bool has) {
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) {
    const KeyT ok = shfl_xor_key(key, m);
    const bool oh = __shfl_xor_sync(kFull, (int)has, m) != 0;
    if (oh && (!has || ok < key)) { key = ok; has = true; }
  }
  return has;
}
__device__ __forceinline__ uint64_t unmix_key(uint64_t k) { return unmix64(k); }
__device__ __forceinline__ Key128 unmix_key(const Key128& k) { return unmix128(k); }
__device__ __forceinline__ Key256 unmix_key(const Key256& k) { return unmix256(k); }

struct RowOut {
  uint32_t* cluster;
  uint64_t* kmer;          // 1 word per row (narrow), 2 (wide) or 4 (256-bit keys)
  uint32_t* count;
  uint32_t* cand;          // rows x key_words
  uint32_t key_words;      // W (+1 with consider_missing)
  uint32_t pattern_words;  // W
  const uint32_t* cluster_pattern;   // batch-local cluster -> cluster-pattern id (or null)
  uint32_t row_base;       // first row of this key width in the shared row arrays
  uint32_t cand_base;      // first candidate of this key width: row_base, or less after a per-cluster emit
  uint32_t* row_cand;      // kB3_cluster_emit: candidate of every row (rows share candidates); else null
};

// OR the sample bits of every live record of [a,b) whose key equals `cur` into
// `bits` (W words of this warp's shared memory); returns the popcount.
template <typename KeyT>
__device__ __forceinline__ uint32_t build_bitset(const KeyT* __restrict__ keys,
                                                 const uint32_t* __restrict__ vals, uint32_t a,
                                                 uint32_t b, const KeyT& cur, uint32_t* bits,
                                                 uint32_t W) {
  const uint32_t lane = lane_id();
  for (uint32_t w = lane; w < W; w += 32) bits[w] = 0;
  __syncwarp();
  for (uint32_t i0 = a; i0 < b; i0 += 32) {
    const uint32_t i = i0 + lane;
    bool live = false;
    uint32_t v = 0;
    if (i < b) {
      v = vals[i];
      live = (v != kInvalidSample) && (keys[i] == cur);
    }
    const uint32_t word = live ? (v >> 5) : (0xffff0000u + lane);
    const uint32_t peers = __match_any_sync(kFull, word);
    const uint32_t ored = __reduce_or_sync(peers, live ? (1u << (v & 31u)) : 0u);
    if (live && (int)lane == __ffs(peers) - 1) bits[word] |= ored;
    __syncwarp();
  }
  uint32_t c = 0;
  for (uint32_t w = lane; w < W; w += 32) c += __popc(bits[w]);
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) c += __shfl_xor_sync(kFull, c, m);
  return c;
}

template <typename KeyT, bool EMIT>
__global__ void __launch_bounds__(256)
k3_runs(const KeyT* __restrict__ keys, const uint32_t* __restrict__ vals,
        const uint32_t* __restrict__ run_start, const uint32_t* __restrict__ run_seg,
        uint32_t n_runs, uint32_t n_records, const ClusterDev* __restrict__ clusters,
        uint32_t* __restrict__ nrows /* COUNT: out counts; EMIT: exclusive offsets (n_runs+1) */,
        RowOut out,
        uint32_t* __restrict__ n_unique = nullptr /* COUNT: += distinct live keys (may be null) */) {
  extern __shared__ uint32_t k3_smem[];
  const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
  const uint32_t W = out.pattern_words;
  uint32_t* bits = k3_smem + (size_t)warp * W;
  const uint32_t total_warps = gridDim.x * (blockDim.x >> 5);
  uint32_t distinct = 0;                 // live keys of this warp's runs (n_unique only)
  for (uint32_t r = blockIdx.x * (blockDim.x >> 5) + warp; r < n_runs; r += total_warps) {
    uint32_t row0 = 0;
    if (EMIT) {
      row0 = nrows[r];
      if (nrows[r + 1] == row0) continue;
    }
    const uint32_t a = run_start[r];
    const uint32_t b = (r + 1 < n_runs) ? run_start[r + 1] : n_records;
    const uint32_t seg = run_seg[r];
    const ClusterDev cl = clusters[seg];

    if (!EMIT) {
      // fast path: one key, no foreign records -> count sample changes
      const KeyT k0 = keys[a];
      bool same = true, clean = true;
      uint32_t cnt = 0, prev_last = kInvalidSample;
      for (uint32_t i0 = a; i0 < b; i0 += 32) {
        const uint32_t i = i0 + lane;
        const bool in = i < b;
        uint32_t v = kInvalidSample - 1u;
        if (in) {
          v = vals[i];
          same &= (keys[i] == k0);
          clean &= (v != kInvalidSample);
        }
        uint32_t up = __shfl_up_sync(kFull, v, 1);
        if (lane == 0) up = prev_last;
        cnt += __popc(__ballot_sync(kFull, in && (i == a || v != up)));
        prev_last = __shfl_sync(kFull, v, 31);
      }
      same = __all_sync(kFull, same);
      clean = __all_sync(kFull, clean);
      if (same && clean) {
        if (lane == 0) nrows[r] = (cnt >= cl.lo && cnt <= cl.hi) ? 1u : 0u;
        ++distinct;
        continue;
      }
    }
    // general path: distinct live keys in ascending order
    uint32_t n_out = 0;
    KeyT cur = KeyTraits<KeyT>::zero();
    bool have_cur = false;
    for (;;) {
      KeyT best = KeyTraits<KeyT>::zero();
      bool has = false;
      for (uint32_t i0 = a; i0 < b; i0 += 32) {
        const uint32_t i = i0 + lane;
        if (i < b && vals[i] != kInvalidSample) {
          const KeyT kk = keys[i];
          if ((!have_cur || cur < kk) && (!has || kk < best)) { best = kk; has = true; }
        }
      }
      if (!warp_min_key(best, has)) break;
      cur = best;
      have_cur = true;
      ++distinct;
      const uint32_t c = build_bitset(keys, vals, a, b, cur, bits, W);
      if (c >= cl.lo && c <= cl.hi && c > 0u) {
        if (EMIT) {
          const size_t row = (size_t)row0 + n_out;
          if (lane == 0) {
            out.cluster[out.row_base + row] = cl.id;
            store_kmer(out.kmer, row, unmix_key(cur));
            out.count[out.row_base + row] = c;
          }
          uint32_t* dst = out.cand + (out.cand_base + row) * out.key_words;
          for (uint32_t w = lane; w < W; w += 32) dst[w] = bits[w];
          if (out.key_words > W && lane == 0) dst[W] = out.cluster_pattern[seg];
        }
        ++n_out;
      }
      __syncwarp();
    }
    if (!EMIT && lane == 0) nrows[r] = n_out;
  }
  if (!EMIT && n_unique && lane == 0 && distinct) atomicAdd(n_unique, distinct);
}

// ---- in-place exclusive scan of a u32 array (three small kernels) ----------
constexpr int kScanBlock = 2048;   // elements per CTA (256 threads x 8)

__global__ void __launch_bounds__(256)
scan_block_sums(const uint32_t* __restrict__ data, uint32_t n, uint32_t* __restrict__ bsum) {
  __shared__ uint32_t ws[8];
  const uint32_t base = blockIdx.x * kScanBlock;
  uint32_t s = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const uint32_t i = base + j * 256 + threadIdx.x;
    if (i < n) s += data[i];
  }
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) s += __shfl_xor_sync(kFull, s, m);
  if (lane_id() == 0) ws[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t t = 0;
    for (int i = 0; i < 8; ++i) t += ws[i];
    bsum[blockIdx.x] = t;
  }
}

// single CTA: exclusive scan of bsum[0..nb) in place, total to bsum[nb] and *total_out
__global__ void __launch_bounds__(1024)
scan_of_sums(uint32_t* __restrict__ bsum, uint32_t nb, uint32_t* __restrict__ total_out) {
  __shared__ uint32_t ws[32];
  __shared__ uint32_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (uint32_t base = 0; base < nb; base += 1024) {
    const uint32_t i = base + threadIdx.x;
    const uint32_t v = i < nb ? bsum[i] : 0u;
    uint32_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t n = __shfl_up_sync(kFull, incl, o);
      if (lane_id() >= (uint32_t)o) incl += n;
    }
    if (lane_id() == 31) ws[threadIdx.x >> 5] = incl;
    __syncthreads();
    if (threadIdx.x < 32) {
      uint32_t x = ws[threadIdx.x], xi = x;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t n = __shfl_up_sync(kFull, xi, o);
        if (threadIdx.x >= (uint32_t)o) xi += n;
      }
      ws[threadIdx.x] = xi - x;
    }
    __syncthreads();
    const uint32_t excl = carry + ws[threadIdx.x >> 5] + incl - v;
    if (i < nb) bsum[i] = excl;
    __syncthreads();
    if (threadIdx.x == 1023) carry = excl + v;
    __syncthreads();
  }
  if (threadIdx.x == 0) { bsum[nb] = carry; *total_out = carry; }
}

// exclusive scan inside each CTA's 2048 elements + the CTA offset; also writes
// data[n] = grand total so callers can take differences.
__global__ void __launch_bounds__(256)
scan_apply(uint32_t* __restrict__ data, uint32_t n, const uint32_t* __restrict__ bsum, uint32_t nb) {
  __shared__ uint32_t ws[8];
  const uint32_t base = blockIdx.x * kScanBlock + threadIdx.x * 8;   // blocked: 8 consecutive per thread
  uint32_t v[8], s = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) { v[j] = (base + j < n) ? data[base + j] : 0u; s += v[j]; }
  uint32_t incl = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t x = __shfl_up_sync(kFull, incl, o);
    if (lane_id() >= (uint32_t)o) incl += x;
  }
  if (lane_id() == 31) ws[threadIdx.x >> 5] = incl;
  __syncthreads();
  uint32_t woff = 0;
  for (uint32_t w = 0; w < (threadIdx.x >> 5); ++w) woff += ws[w];
  uint32_t run = bsum[blockIdx.x] + woff + incl - s;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    if (base + j < n) data[base + j] = run;
    run += v[j];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) data[n] = bsum[nb];
}

}  // namespace pf
