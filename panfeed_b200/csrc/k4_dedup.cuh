// K4 — global pattern deduplication in a GPU open-addressing table keyed on
// the FULL bitset.  Replaces `if khash in patterns: continue; patterns.add()`
// (/root/reference/panfeed/panfeed.py:179-180,210-212) where the reference keys
// a Python set on base64(md5(vector bytes)): here two different patterns can
// never be merged, whatever their hashes.
//
// The table holds 32-bit entries: an index into the persistent pattern pool,
// or (top bit set) the index of a candidate row of the current batch.  One warp
// per candidate: hash W words cooperatively, linear-probe, claim an empty slot
// with one atomicCAS, and on an occupied slot compare all W words against the
// occupant (pool entry or another candidate of this batch).  After the kernel
// the winners are numbered by a scan and copied to the pool in that order.
#pragma once
#include "pf_common.cuh"

namespace pf {

constexpr uint32_t kEmptySlot = 0xffffffffu;
constexpr uint32_t kTentative = 0x80000000u;

// A row is handled by a group of L lanes (L = 4, 8, 16 or 32, chosen so that a lane
// holds at most a few words): short keys (S = 500 -> 16 words) would leave most of a
// full warp idle and, worse, give the memory system one row per warp to chew on.
template <int L>
__device__ __forceinline__ uint32_t group_mask() {
  return L == 32 ? kFull : (((1u << L) - 1u) << (lane_id() & ~(uint32_t)(L - 1)));
}

template <int L>
__device__ __forceinline__ uint64_t group_hash_words(const uint32_t* __restrict__ key, uint32_t n) {
  const uint32_t gl = lane_id() & (L - 1);
  uint64_t h = 0;
  for (uint32_t w = gl; w < n; w += L) h += word_hash(key[w], w);
#pragma unroll
  for (int m = L / 2; m >= 1; m >>= 1) h += __shfl_xor_sync(group_mask<L>(), h, m, L);
  return fmix64(h);
}
__device__ __forceinline__ uint64_t warp_hash_words(const uint32_t* __restrict__ key, uint32_t n) {
  return group_hash_words<32>(key, n);
}

template <int L>
__device__ __forceinline__ bool group_equal_words(const uint32_t* __restrict__ a,
                                                  const uint32_t* __restrict__ b, uint32_t n) {
  const uint32_t gl = lane_id() & (L - 1);
  for (uint32_t w0 = 0; w0 < n; w0 += L) {
    const uint32_t w = w0 + gl;
    const bool ok = (w >= n) || (a[w] == b[w]);
    if (!__all_sync(group_mask<L>(), ok)) return false;
  }
  return true;
}

// rep[row]  : pool index of an existing equal pattern, or kTentative|q where q
//             is the candidate row that claimed the slot (q == row: this row won)
// slot_of[row] (winners only): the table slot it claimed
template <int L>
__global__ void __launch_bounds__(256)
k4_probe(const uint32_t* __restrict__ cand, uint32_t n_rows, uint32_t key_words,
         const uint32_t* __restrict__ pool, uint32_t* __restrict__ table, uint32_t table_mask,
         uint32_t* __restrict__ rep, uint32_t* __restrict__ slot_of,
         uint32_t* __restrict__ winner_flag) {
  const uint32_t gl = lane_id() & (L - 1);
  const uint32_t groups_per_block = 256 / L;
  const uint32_t total_groups = gridDim.x * groups_per_block;
  const uint32_t gmask = group_mask<L>();
  // every group of a warp runs the same number of iterations (the *_sync calls need all
  // their lanes), so rows past the end are clamped and their results dropped
  const uint32_t n_iter = (n_rows + total_groups - 1) / total_groups;
  uint32_t row = blockIdx.x * groups_per_block + threadIdx.x / L;
  for (uint32_t it = 0; it < n_iter; ++it, row += total_groups) {
    const bool live = row < n_rows;
    const uint32_t r = live ? row : 0u;
    const uint32_t* key = cand + (size_t)r * key_words;
    uint32_t slot = (uint32_t)group_hash_words<L>(key, key_words) & table_mask;
    uint32_t result = kEmptySlot;
    bool won = false;
    for (;;) {
      uint32_t e = 0;
      if (gl == 0) {
        e = *reinterpret_cast<volatile uint32_t*>(table + slot);
        if (e == kEmptySlot && live) {
          const uint32_t old = atomicCAS(table + slot, kEmptySlot, kTentative | row);
          if (old == kEmptySlot) { won = true; e = kTentative | row; }
          else e = old;
        }
      }
      e = __shfl_sync(gmask, e, 0, L);
      won = __shfl_sync(gmask, (int)won, 0, L) != 0;
      if (won || e == kEmptySlot) { result = e; break; }      // (e == empty only for clamped rows)
      const uint32_t* other = (e & kTentative)
                                  ? cand + (size_t)(e & ~kTentative) * key_words
                                  : pool + (size_t)e * key_words;
      if (group_equal_words<L>(key, other, key_words)) { result = e; break; }
      slot = (slot + 1u) & table_mask;
    }
    if (gl == 0 && live) {
      rep[row] = result;
      winner_flag[row] = won ? 1u : 0u;
      if (won) slot_of[row] = slot;
    }
  }
}

// winners: copy the candidate into the pool at pool_base + rank, fix the slot.
// everyone: translate rep into a final pool index.
template <int L>
__global__ void __launch_bounds__(256)
k4_commit(const uint32_t* __restrict__ cand, uint32_t n_rows, uint32_t key_words,
          uint32_t* __restrict__ pool, uint32_t pool_base, uint32_t* __restrict__ table,
          const uint32_t* __restrict__ rep, const uint32_t* __restrict__ slot_of,
          const uint32_t* __restrict__ winner_rank /* exclusive scan of winner_flag, n_rows+1 */,
          uint32_t* __restrict__ row_pattern) {
  const uint32_t gl = lane_id() & (L - 1);
  const uint32_t groups_per_block = 256 / L;
  const uint32_t total_groups = gridDim.x * groups_per_block;
  for (uint32_t row = blockIdx.x * groups_per_block + threadIdx.x / L; row < n_rows; row += total_groups) {
    const uint32_t r = rep[row];
    uint32_t id;
    if (r & kTentative) {
      const uint32_t q = r & ~kTentative;
      id = pool_base + winner_rank[q];
      if (q == row) {
        const uint32_t* src = cand + (size_t)row * key_words;
        uint32_t* dst = pool + (size_t)id * key_words;
        for (uint32_t w = gl; w < key_words; w += L) dst[w] = src[w];
        if (gl == 0) table[slot_of[row]] = id;
      }
    } else {
      id = r;
    }
    if (gl == 0) row_pattern[row] = id;
  }
}

// pattern id of every row from its candidate's: the first n_mapped rows (kB3_cluster_emit) name
// their candidate in row_cand, row r after them owns candidate r - shift
__global__ void __launch_bounds__(256)
k4_gather(const uint32_t* __restrict__ row_cand, uint32_t n_mapped, uint32_t shift,
          const uint32_t* __restrict__ cand_pattern, uint32_t n_rows, uint32_t* __restrict__ row_pattern) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_rows) return;
  row_pattern[r] = cand_pattern[r < n_mapped ? row_cand[r] : r - shift];
}

// re-insert pool entries [0, n) into a fresh (larger) table; entries are distinct
__global__ void __launch_bounds__(256)
k4_rehash(const uint32_t* __restrict__ pool, uint32_t n, uint32_t key_words,
          uint32_t* __restrict__ table, uint32_t table_mask) {
  const uint32_t lane = lane_id();
  const uint32_t total_warps = gridDim.x * (blockDim.x >> 5);
  for (uint32_t e = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); e < n; e += total_warps) {
    uint32_t slot = (uint32_t)warp_hash_words(pool + (size_t)e * key_words, key_words) & table_mask;
    if (lane == 0) {
      while (atomicCAS(table + slot, kEmptySlot, e) != kEmptySlot) slot = (slot + 1u) & table_mask;
    }
  }
}

}  // namespace pf
