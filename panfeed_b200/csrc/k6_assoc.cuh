// K6 — the post-GWAS join of a second pass run with --associations: which k-mer instances of the
// target strains carry a pattern that passed the association threshold.  This is what the
// reference's panfeed-get-kmers does with kmers.tsv and kmers_to_hashes.tsv in pandas
// (/root/reference/panfeed/get_kmers.py:108-145), done while the batch is still on the device:
//
//   K6a  pattern -> association row: the MD5 id of every new pattern (K5's loop), looked up in an
//        open-addressing table of the passing digests (full 128 bits compared);
//   K6b  an open-addressing table over the batch's surviving rows, keyed on (cluster, k-mer);
//   K6c  every window of a target sequence: its k-mer (the strand K1 chose in canonical mode, both
//        strands otherwise), its row in the table above, that row's association row.
//
// A k-mer is looked up in the width its row was written in: one word (k <= 32, ACGT only), two
// words (k <= 32 with N/IUPAC symbols: 4 bits per symbol; k = 33..64 ACGT: 2 bits per base), four
// words (k = 33..64 with N/IUPAC symbols); most significant word first, first symbol on top.
#pragma once
#include "pf_common.cuh"
#include "k1_extract.cuh"
#include "k5_md5.cuh"

namespace pf {

constexpr uint32_t kAssocNone = 0xffffffffu;

struct AssocTable {          // passing digests: capacity mask + 1 >= 2 n, a free slot always remains
  const uint4* key;
  const uint32_t* val;       // association row, kAssocNone = free slot
  uint32_t mask;
};

__device__ __forceinline__ uint32_t assoc_find(const AssocTable& t, const uint32_t (&d)[4]) {
  for (uint32_t s = d[0] & t.mask;; s = (s + 1u) & t.mask) {      // (MD5 words are uniform)
    const uint32_t v = t.val[s];
    if (v == kAssocNone) return kAssocNone;
    const uint4 k = t.key[s];
    if (k.x == d[0] && k.y == d[1] && k.z == d[2] && k.w == d[3]) return v;
  }
}

// K6a: pattern_assoc[first + i] for the patterns [first, first + count) of a pool (same arguments as
// k5_md5_ids: the digest is computed the same way, then looked up instead of copied out)
__global__ void __launch_bounds__(128)
k6_pattern_assoc(const uint32_t* __restrict__ pool, uint32_t first, uint32_t count, uint32_t key_words,
                 uint32_t W, uint32_t S, int as_int64, const uint32_t* __restrict__ nan_pool, AssocTable t,
                 uint32_t* __restrict__ pattern_assoc) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const uint32_t* bits = pool + (size_t)(first + i) * key_words;
  const uint32_t* present = (key_words > W && nan_pool) ? nan_pool + (size_t)bits[W] * W : nullptr;
  uint32_t st[4];
  md5_pattern(bits, present, S, as_int64, st);
  pattern_assoc[first + i] = assoc_find(t, st);
}

// The rows of a batch as pf_collect returns them: narrow, then wide, then 256-bit
struct AssocRows {
  const uint32_t* cluster;   // [n_nar + n_wid + n_xwd]
  const uint32_t* pattern;   // k-mer pattern of every row
  const uint64_t* nar;       // 1 word per row
  const uint64_t* wid;       // 2 words
  const uint64_t* xwd;       // 4 words
  uint32_t n_nar, n_wid, n_xwd;
};

template <int NW>
__device__ __forceinline__ uint64_t row_hash(uint32_t cluster, const uint64_t (&w)[4]) {
  uint64_t h = fmix64(((uint64_t)cluster << 3 | (uint64_t)NW) + 0x9e3779b97f4a7c15ULL);
#pragma unroll
  for (int i = 0; i < NW; ++i) h = fmix64(h ^ (w[i] + 0xd1b54a32d192ed03ULL * (uint64_t)(i + 1)));
  return h;
}

// K6b: row r at the first free slot from its hash.  Rows are unique per (cluster, k-mer).
__global__ void __launch_bounds__(256)
k6_row_index(AssocRows rows, uint32_t* __restrict__ table, uint32_t mask, const uint32_t* __restrict__ kp_assoc,
             uint8_t* __restrict__ cluster_pass) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t n = rows.n_nar + rows.n_wid + rows.n_xwd;
  if (r >= n) return;
  const uint32_t c = rows.cluster[r];
  uint64_t w[4] = {0, 0, 0, 0};
  uint64_t h;
  if (r < rows.n_nar) {
    w[0] = rows.nar[r];
    h = row_hash<1>(c, w);
  } else if (r < rows.n_nar + rows.n_wid) {
    const uint64_t* p = rows.wid + 2 * (size_t)(r - rows.n_nar);
    w[0] = p[0]; w[1] = p[1];
    h = row_hash<2>(c, w);
  } else {
    const uint64_t* p = rows.xwd + 4 * (size_t)(r - rows.n_nar - rows.n_wid);
    w[0] = p[0]; w[1] = p[1]; w[2] = p[2]; w[3] = p[3];
    h = row_hash<4>(c, w);
  }
  for (uint32_t s = (uint32_t)h & mask;; s = (s + 1u) & mask)
    if (atomicCAS(table + s, kAssocNone, r) == kAssocNone) break;
  if (kp_assoc[rows.pattern[r]] != kAssocNone) cluster_pass[c] = 1;       // (benign: every writer stores 1)
}

// the row of (cluster, k-mer w) of width NW words, or kAssocNone
template <int NW>
__device__ __forceinline__ uint32_t row_find(const AssocRows& rows, const uint32_t* __restrict__ table, uint32_t mask,
                                             uint32_t cluster, const uint64_t (&w)[4]) {
  const uint32_t lo = NW == 1 ? 0u : NW == 2 ? rows.n_nar : rows.n_nar + rows.n_wid;
  const uint32_t hi = NW == 1 ? rows.n_nar : NW == 2 ? rows.n_nar + rows.n_wid : rows.n_nar + rows.n_wid + rows.n_xwd;
  const uint64_t* keys = NW == 1 ? rows.nar : NW == 2 ? rows.wid : rows.xwd;
  for (uint32_t s = (uint32_t)row_hash<NW>(cluster, w) & mask;; s = (s + 1u) & mask) {
    const uint32_t r = table[s];
    if (r == kAssocNone) return kAssocNone;
    if (r < lo || r >= hi || rows.cluster[r] != cluster) continue;
    const uint64_t* p = keys + (size_t)NW * (r - lo);
    bool eq = true;
#pragma unroll
    for (int i = 0; i < NW; ++i) eq &= p[i] == w[i];
    if (eq) return r;
  }
}

// 4-bit codes of PF_AMB_ALPHABET ("ABCDGHKMNRSTVWXY") -> code of the complement symbol, a nibble each
constexpr uint64_t kAmbComplement = 0x9ed10af8673254cbULL;

// window p of sequence d in the 4-bit plane, NW words, the strand `rc` (reverse complement)
template <int NW>
__device__ __forceinline__ void amb_window_key(const uint64_t* __restrict__ amb, const SeqDev& d, uint32_t p, int k,
                                               bool rc, uint64_t (&w)[4]) {
#pragma unroll
  for (int i = 0; i < 4; ++i) w[i] = 0;
  for (int s = 0; s < k; ++s) {
    const uint64_t i = d.amb_off + p + (uint64_t)(rc ? k - 1 - s : s);
    uint32_t code = (uint32_t)(amb[i >> 4] >> (60 - 4 * (i & 15u))) & 15u;
    if (rc) code = (uint32_t)(kAmbComplement >> (4 * code)) & 15u;
#pragma unroll
    for (int j = 0; j < NW - 1; ++j) w[j] = (w[j] << 4) | (w[j + 1] >> 60);
    w[NW - 1] = (w[NW - 1] << 4) | code;
  }
}

// K6c: one warp per target sequence of a cluster that has a passing hash; lane l owns window
// 32 * it + l.  A window whose row passes is listed as ((base_off + p) << 1 | rc, association row)
// - rc only in --non-canonical mode, where both strands are rows of kmers.tsv - and marks its row.
template <bool CANON>
__global__ void __launch_bounds__(kK1Warps * 32)
k6_window_join(const uint64_t* __restrict__ bases, const uint64_t* __restrict__ amb,
               const uint32_t* __restrict__ ambbits, const SeqDev* __restrict__ seqs, uint32_t n_seqs, int k,
               const uint32_t* __restrict__ strand_bits, AssocRows rows, const uint32_t* __restrict__ table,
               uint32_t mask, const uint32_t* __restrict__ kp_assoc, const uint8_t* __restrict__ cluster_pass,
               uint8_t* __restrict__ row_seen, uint64_t* __restrict__ out_win, uint32_t* __restrict__ out_assoc,
               uint32_t* __restrict__ out_count) {
  const uint32_t lane = lane_id();
  const uint32_t stride = gridDim.x * kK1Warps;
  for (uint32_t s = blockIdx.x * kK1Warps + (threadIdx.x >> 5); s < n_seqs; s += stride) {
    const SeqDev d = seqs[s];
    if (!(d.flags & 1u) || d.len < (uint32_t)k || !cluster_pass[d.cluster]) continue;
    const uint32_t nwin = d.len - (uint32_t)k + 1u;
    const uint32_t* ab = (d.flags & 2u) ? ambbits + (d.amb_off >> 5) : nullptr;
    for (uint32_t it = 0; it * 32u < nwin; ++it) {
      const uint32_t p = it * 32u + lane;
      const bool valid = p < nwin;
      const uint64_t i = d.base_off + p;
      bool is_amb = false;
      if (ab && valid) {                       // any non-ACGT symbol in [p, p + k)?
        const uint32_t wi = p >> 5, bs = p & 31u;
        const uint64_t two = ((uint64_t)ab[wi] << 32) | (uint64_t)ab[wi + 1];
        if (k <= 32) {
          is_amb = ((two << bs) >> (64 - k)) != 0ull;
        } else {
          const uint64_t x = (two << bs) | (((uint64_t)ab[wi + 2] << bs) >> 32);
          is_amb = (k >= 64 ? x : x >> (64 - k)) != 0ull;
        }
      }
      // the 64 bases from base p, first base on top (x0) and the 64 after them (x1)
      const uint64_t* wp = bases + (i >> 5);
      const uint32_t sh = 2u * (uint32_t)(i & 31u);
      const uint64_t x0 = valid ? (wp[0] << sh) | ((wp[1] >> 1) >> (63u - sh)) : 0ull;
      const uint64_t x1 = valid && k > 32 ? (wp[1] << sh) | ((wp[2] >> 1) >> (63u - sh)) : 0ull;
      const bool use_rc = CANON && valid && ((strand_bits[i >> 5] >> (i & 31u)) & 1u);
#pragma unroll
      for (int o = 0; o < (CANON ? 1 : 2); ++o) {
        const bool rc = CANON ? use_rc : o == 1;
        uint32_t row = kAssocNone;
        if (valid) {
          uint64_t w[4] = {0, 0, 0, 0};
          if (is_amb) {
            if (k <= 32) { amb_window_key<2>(amb, d, p, k, rc, w); row = row_find<2>(rows, table, mask, d.cluster, w); }
            else { amb_window_key<4>(amb, d, p, k, rc, w); row = row_find<4>(rows, table, mask, d.cluster, w); }
          } else if (k <= 32) {
            const uint64_t fwd = x0 >> (64 - 2 * k);
            w[0] = rc ? revcomp2(fwd, k) : fwd;
            row = row_find<1>(rows, table, mask, d.cluster, w);
          } else {
            const uint32_t drop = 128u - 2u * (uint32_t)k;                   // 0..62
            const uint64_t lo = x1 & (drop ? ~0ull << drop : ~0ull);          // the window, left-aligned
            if (!rc) {
              w[0] = drop ? x0 >> drop : x0;
              w[1] = drop ? (lo >> drop) | (x0 << (64u - drop)) : lo;
            } else {                                                          // padding becomes leading T's
              w[0] = revcomp2(lo, 32);
              w[1] = revcomp2(x0, 32);
              if (2u * (uint32_t)k - 64u < 64u) w[0] &= (1ull << (2u * (uint32_t)k - 64u)) - 1ull;
            }
            row = row_find<2>(rows, table, mask, d.cluster, w);
          }
        }
        const uint32_t a = row != kAssocNone ? kp_assoc[rows.pattern[row]] : kAssocNone;
        const bool hit = a != kAssocNone;
        if (hit) row_seen[row] = 1;
        const uint32_t ballot = __ballot_sync(kFull, hit);
        if (!ballot) continue;
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(out_count, (uint32_t)__popc(ballot));
        base = __shfl_sync(kFull, base, 0);
        if (hit) {
          const uint32_t at = base + (uint32_t)__popc(ballot & lanemask_lt());
          out_win[at] = (i << 1) | (CANON ? 0ull : (uint64_t)o);
          out_assoc[at] = a;
        }
      }
    }
  }
}

// K6d: the passing rows of the batch, (row, association row, seen in a target window)
__global__ void __launch_bounds__(256)
k6_passing_rows(const uint32_t* __restrict__ row_pattern, uint32_t n_rows, const uint32_t* __restrict__ kp_assoc,
                const uint8_t* __restrict__ row_seen, uint32_t* __restrict__ out_row, uint32_t* __restrict__ out_assoc,
                uint8_t* __restrict__ out_seen, uint32_t* __restrict__ out_count) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t a = r < n_rows ? kp_assoc[row_pattern[r]] : kAssocNone;
  const bool hit = a != kAssocNone;
  const uint32_t ballot = __ballot_sync(kFull, hit);
  if (!ballot) return;
  uint32_t base = 0;
  if (lane_id() == 0) base = atomicAdd(out_count, (uint32_t)__popc(ballot));
  base = __shfl_sync(kFull, base, 0);
  if (hit) {
    const uint32_t at = base + (uint32_t)__popc(ballot & lanemask_lt());
    out_row[at] = r;
    out_assoc[at] = a;
    out_seen[at] = row_seen[r];
  }
}

// K6e: per cluster of the batch, the association row of its own (cluster-row) pattern and whether
// any of its hashes passes (initialises cluster_pass before K6b adds the rows)
__global__ void __launch_bounds__(256)
k6_cluster_assoc(const uint32_t* __restrict__ cl_pattern, uint32_t n_clusters, const uint32_t* __restrict__ cp_assoc,
                 uint32_t* __restrict__ cluster_assoc, uint8_t* __restrict__ cluster_pass) {
  const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_clusters) return;
  const uint32_t a = cp_assoc[cl_pattern[c]];
  cluster_assoc[c] = a;
  cluster_pass[c] = a != kAssocNone ? 1 : 0;
}

}  // namespace pf
