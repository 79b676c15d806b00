// Shared device helpers and internal device-side descriptors.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace pf {

constexpr uint32_t kInvalidSample = 0xffffffffu;  // record of a window that belongs to the other key width
constexpr int kWarp = 32;
constexpr uint32_t kFull = 0xffffffffu;

// ---- bijective 64-bit mixers and their inverses -----------------------------
// The radix sort orders only the leading `sort_bits` of mix(kmer); mixing makes
// those bits a uniform hash of the whole k-mer, so near-identical k-mers (SNP
// neighbours) do not share a prefix.  K3 resolves the rare shared prefix
// exactly and un-mixes the key when it emits a row.
constexpr uint64_t kMulA = 0xff51afd7ed558ccdULL;
constexpr uint64_t kMulB = 0xc4ceb9fe1a85ec53ULL;
constexpr uint64_t inv_odd(uint64_t a) {
  uint64_t x = a;                       // Newton iteration mod 2^64
  for (int i = 0; i < 6; ++i) x *= 2 - a * x;
  return x;
}
constexpr uint64_t kInvA = inv_odd(kMulA);
constexpr uint64_t kInvB = inv_odd(kMulB);
static_assert(kMulA * kInvA == 1ULL && kMulB * kInvB == 1ULL, "inverse");

// full-strength mixer (murmur3 finaliser): pattern hashing, synthetic data, wide keys
__host__ __device__ __forceinline__ uint64_t fmix64(uint64_t x) {
  x ^= x >> 33; x *= kMulA; x ^= x >> 33; x *= kMulB; x ^= x >> 33;
  return x;
}
// k-mer key mixer on the hot path: one odd multiply (every bit of the k-mer reaches
// the leading digits) and one xor-shift (the leading half reaches the low bits the
// shared-memory tables index with).  Bijective; exactness never depends on its quality.
constexpr uint64_t kMulK = 0x9e3779b97f4a7c15ULL;
constexpr uint64_t kInvK = inv_odd(kMulK);
static_assert(kMulK * kInvK == 1ULL, "inverse");
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t x) {
  x *= kMulK;
  return x ^ (x >> 32);
}
__host__ __device__ __forceinline__ uint64_t unmix64(uint64_t x) {
  x ^= x >> 32;
  return x * kInvK;
}

// 128-bit key for windows holding N/IUPAC symbols (4 bits per symbol, k <= 32).
struct Key128 {
  uint64_t hi, lo;
};
__host__ __device__ __forceinline__ bool operator==(const Key128& a, const Key128& b) {
  return a.hi == b.hi && a.lo == b.lo;
}
__host__ __device__ __forceinline__ bool operator!=(const Key128& a, const Key128& b) {
  return !(a == b);
}
__host__ __device__ __forceinline__ bool operator<(const Key128& a, const Key128& b) {
  return a.hi < b.hi || (a.hi == b.hi && a.lo < b.lo);
}
// Feistel-free bijection on 128 bits: mix each half with the other (invertible
// step by step), enough to make the leading bits a hash of all 128.
__host__ __device__ __forceinline__ Key128 mix128(Key128 k) {
  k.hi ^= fmix64(k.lo + 0x9e3779b97f4a7c15ULL);
  k.lo ^= fmix64(k.hi + 0xd1b54a32d192ed03ULL);
  k.hi ^= fmix64(k.lo + 0x8cb92ba72f3d8dd7ULL);
  return k;
}
__host__ __device__ __forceinline__ Key128 unmix128(Key128 k) {
  k.hi ^= fmix64(k.lo + 0x8cb92ba72f3d8dd7ULL);
  k.lo ^= fmix64(k.hi + 0xd1b54a32d192ed03ULL);
  k.hi ^= fmix64(k.lo + 0x9e3779b97f4a7c15ULL);
  return k;
}

// 256-bit key for windows of 33..64 symbols holding N/IUPAC symbols: 4 bits per symbol (codes of
// PF_AMB_ALPHABET), first symbol in the top used bits, w[0] the most significant word.  Unsigned
// comparison over the words is the reference's string order, as for Key128.
struct Key256 {
  uint64_t w[4];
};
__host__ __device__ __forceinline__ bool operator==(const Key256& a, const Key256& b) {
  return a.w[0] == b.w[0] && a.w[1] == b.w[1] && a.w[2] == b.w[2] && a.w[3] == b.w[3];
}
__host__ __device__ __forceinline__ bool operator!=(const Key256& a, const Key256& b) {
  return !(a == b);
}
__host__ __device__ __forceinline__ bool operator<(const Key256& a, const Key256& b) {
  if (a.w[0] != b.w[0]) return a.w[0] < b.w[0];
  if (a.w[1] != b.w[1]) return a.w[1] < b.w[1];
  if (a.w[2] != b.w[2]) return a.w[2] < b.w[2];
  return a.w[3] < b.w[3];
}
// Bijection on 256 bits: the last word takes a hash of the first three, then the leading word a
// hash of the (new) last one, which by then depends on all 256 bits.
__host__ __device__ __forceinline__ Key256 mix256(Key256 k) {
  k.w[3] ^= fmix64(k.w[0] + 0x9e3779b97f4a7c15ULL) ^ fmix64(k.w[1] + 0xd1b54a32d192ed03ULL) ^
            fmix64(k.w[2] + 0x8cb92ba72f3d8dd7ULL);
  k.w[0] ^= fmix64(k.w[3] + 0xa0761d6478bd642fULL);
  return k;
}
__host__ __device__ __forceinline__ Key256 unmix256(Key256 k) {
  k.w[0] ^= fmix64(k.w[3] + 0xa0761d6478bd642fULL);
  k.w[3] ^= fmix64(k.w[0] + 0x9e3779b97f4a7c15ULL) ^ fmix64(k.w[1] + 0xd1b54a32d192ed03ULL) ^
            fmix64(k.w[2] + 0x8cb92ba72f3d8dd7ULL);
  return k;
}

// Leading `bits` of a key, right-aligned digit extraction for the radix passes.
__device__ __forceinline__ uint32_t key_digit(uint64_t k, int shift) {
  return (uint32_t)(k >> shift) & 255u;
}
__device__ __forceinline__ uint32_t key_digit(const Key128& k, int shift) {
  // shift counts from bit 0 of the 128-bit value; sorted bits are the leading
  // ones, so shift >= 64 whenever sort_bits <= 64 (always).
  return (uint32_t)(k.hi >> (shift - 64)) & 255u;
}
__device__ __forceinline__ uint32_t key_digit(const Key256& k, int shift) {
  return (uint32_t)(k.w[0] >> (shift - 192)) & 255u;      // (the same on the leading word)
}
__device__ __forceinline__ uint64_t key_prefix(uint64_t k, int sort_bits) {
  return sort_bits >= 64 ? k : (k >> (64 - sort_bits));
}
__device__ __forceinline__ uint64_t key_prefix(const Key128& k, int sort_bits) {
  return sort_bits >= 64 ? k.hi : (k.hi >> (64 - sort_bits));
}
__device__ __forceinline__ uint64_t key_prefix(const Key256& k, int sort_bits) {
  return sort_bits >= 64 ? k.w[0] : (k.w[0] >> (64 - sort_bits));
}
// k-mer `row` of an output array of 1, 2 or 4 words per k-mer, most significant word first
__device__ __forceinline__ void store_kmer(uint64_t* out, size_t row, uint64_t k) { out[row] = k; }
__device__ __forceinline__ void store_kmer(uint64_t* out, size_t row, const Key128& k) {
  out[2 * row] = k.hi; out[2 * row + 1] = k.lo;
}
__device__ __forceinline__ void store_kmer(uint64_t* out, size_t row, const Key256& k) {
#pragma unroll
  for (int i = 0; i < 4; ++i) out[4 * row + i] = k.w[i];
}
template <typename K> struct KeyTraits;
template <> struct KeyTraits<uint64_t> {
  static constexpr int kBits = 64;
  __device__ static __forceinline__ uint64_t zero() { return 0; }
};
template <> struct KeyTraits<Key128> {
  static constexpr int kBits = 128;
  __device__ static __forceinline__ Key128 zero() { return Key128{0, 0}; }
};
template <> struct KeyTraits<Key256> {
  static constexpr int kBits = 256;
  __device__ static __forceinline__ Key256 zero() { return Key256{{0, 0, 0, 0}}; }
};

// ---- relaxed gpu-scope accesses for the decoupled look-back chains --------
__device__ __forceinline__ uint32_t ld_relaxed(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed(uint32_t* p, uint32_t v) {
  asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint64_t ld_relaxed(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed(uint64_t* p, uint64_t v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// Streaming 128-bit load of read-once data (packed bases).
__device__ __forceinline__ uint4 ld_stream128(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }
__device__ __forceinline__ uint32_t lanemask_lt() { return (1u << lane_id()) - 1u; }

// ---- hash of a pattern key (W words); commutative over words so a warp can
// reduce it in any order.  Same function picks the owner rank in the exchange.
__host__ __device__ __forceinline__ uint64_t word_hash(uint32_t w, uint32_t i) {
  // one odd multiply of (position, word) + one xor-shift: the sum over the words is
  // finalised with fmix64 by the caller, and table / owner decisions never rest on the hash
  const uint64_t x = (((uint64_t)(i + 1u) << 32) | (uint64_t)w) * 0x9e3779b97f4a7c15ULL;
  return x ^ (x >> 29);
}

// ---- device-side descriptors (built on the host in pf_upload) -------------
struct SeqDev {          // 64 bytes
  uint64_t base_off;     // bases
  uint64_t amb_off;      // symbols in the 4-bit plane
  uint32_t len;
  uint32_t sample;
  uint32_t cluster;      // batch-local
  uint32_t flags;
  int32_t start, end, offset, strand;
  uint32_t rec_off;      // first record in the narrow record arrays; k > 32 (no narrow records):
                         // first record in the 256-bit record arrays (sequences with N/IUPAC)
  uint32_t pos_off;      // first positional record
  uint32_t wrec_off;     // first record in the wide record arrays
  uint32_t pwide_off;    // first slot in the wide positional k-mer array (targets with N/IUPAC)
};
static_assert(sizeof(SeqDev) == 64, "SeqDev");

struct ClusterDev {      // 40 bytes
  uint32_t rec_start, rec_end;   // narrow record range (a segment of the sort)
  uint32_t id;
  uint32_t lo, hi;               // surviving sample counts, filters folded in
  uint32_t n_present;
  uint32_t wrec_start, wrec_end; // wide record range
  uint32_t xrec_start, xrec_end; // 256-bit record range (k > 32, windows with N/IUPAC symbols)
};

struct TileDev {         // 16 bytes: one sort tile, never crossing a segment
  uint32_t start;        // first record
  uint32_t count;
  uint32_t seg;          // batch-local cluster
  uint32_t first_tile;   // first tile of the segment
};

constexpr int kSortThreads = 256;
constexpr int kSortItems = 16;
constexpr int kSortTile = kSortThreads * kSortItems;   // 4096 records
constexpr int kRadix = 256;

}  // namespace pf
