// K5 — reference-identical pattern ids.  The reference names a pattern
// base64(md5(raw bytes of its vector))[:24]: int64 bytes for a cluster's own row
// (/root/reference/panfeed/panfeed.py:175-176), float64 bytes for k-mer rows
// (:206-207), NaN where the cluster is absent under --consider-missing (:16-20).
// One thread per pattern expands its bits on the fly into those 8-byte little-endian
// images (0.0 = 00..00, 1.0 = ..F0 3F, NaN = ..F8 7F, int 1 = 01 00..) and runs MD5
// over the 8*S bytes; the 16-byte digest goes back to the host, which only base64s it.
#pragma once
#include "pf_common.cuh"

namespace pf {

__constant__ uint32_t kMd5K[64] = {
    0xd76aa478, 0xe8c7b756, 0x242070db, 0xc1bdceee, 0xf57c0faf, 0x4787c62a, 0xa8304613, 0xfd469501,
    0x698098d8, 0x8b44f7af, 0xffff5bb1, 0x895cd7be, 0x6b901122, 0xfd987193, 0xa679438e, 0x49b40821,
    0xf61e2562, 0xc040b340, 0x265e5a51, 0xe9b6c7aa, 0xd62f105d, 0x02441453, 0xd8a1e681, 0xe7d3fbc8,
    0x21e1cde6, 0xc33707d6, 0xf4d50d87, 0x455a14ed, 0xa9e3e905, 0xfcefa3f8, 0x676f02d9, 0x8d2a4c8a,
    0xfffa3942, 0x8771f681, 0x6d9d6122, 0xfde5380c, 0xa4beea44, 0x4bdecfa9, 0xf6bb4b60, 0xbebfbc70,
    0x289b7ec6, 0xeaa127fa, 0xd4ef3085, 0x04881d05, 0xd9d4d039, 0xe6db99e5, 0x1fa27cf8, 0xc4ac5665,
    0xf4292244, 0x432aff97, 0xab9423a7, 0xfc93a039, 0x655b59c3, 0x8f0ccc92, 0xffeff47d, 0x85845dd1,
    0x6fa87e4f, 0xfe2ce6e0, 0xa3014314, 0x4e0811a1, 0xf7537e82, 0xbd3af235, 0x2ad7d2bb, 0xeb86d391};

__device__ __forceinline__ void md5_block(uint32_t (&s)[4], const uint32_t (&m)[16]) {
  constexpr int R[64] = {7, 12, 17, 22, 7, 12, 17, 22, 7, 12, 17, 22, 7, 12, 17, 22,
                         5, 9,  14, 20, 5, 9,  14, 20, 5, 9,  14, 20, 5, 9,  14, 20,
                         4, 11, 16, 23, 4, 11, 16, 23, 4, 11, 16, 23, 4, 11, 16, 23,
                         6, 10, 15, 21, 6, 10, 15, 21, 6, 10, 15, 21, 6, 10, 15, 21};
  uint32_t a = s[0], b = s[1], c = s[2], d = s[3];
#pragma unroll
  for (int i = 0; i < 64; ++i) {
    uint32_t f;
    int g;
    if (i < 16) { f = (b & c) | (~b & d); g = i; }
    else if (i < 32) { f = (d & b) | (~d & c); g = (5 * i + 1) & 15; }
    else if (i < 48) { f = b ^ c ^ d; g = (3 * i + 5) & 15; }
    else { f = c ^ (b | ~d); g = (7 * i) & 15; }
    f = f + a + kMd5K[i] + m[g];
    a = d; d = c; c = b;
    b = b + __funnelshift_l(f, f, R[i]);
  }
  s[0] += a; s[1] += b; s[2] += c; s[3] += d;
}

// MD5 state of one pattern: its bits expanded on the fly into the 8-byte little-endian images the
// reference hashes.  present (may be null): the NaN plane of a k-mer pattern under --consider-missing.
__device__ __forceinline__ void md5_pattern(const uint32_t* __restrict__ bits, const uint32_t* __restrict__ present,
                                            uint32_t S, int as_int64, uint32_t (&st)[4]) {
  st[0] = 0x67452301u; st[1] = 0xefcdab89u; st[2] = 0x98badcfeu; st[3] = 0x10325476u;
  uint32_t m[16];
  const uint64_t total_bytes = (uint64_t)S * 8;
  const uint32_t n_blocks = (uint32_t)((total_bytes + 9 + 63) / 64);     // message + 0x80 + 64-bit length
  for (uint32_t blk = 0; blk < n_blocks; ++blk) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint32_t smp = blk * 8 + j;
      uint32_t lo = 0, hi = 0;
      if (smp < S) {
        const uint32_t bit = (bits[smp >> 5] >> (smp & 31)) & 1u;
        if (as_int64) lo = bit;
        else {
          hi = bit ? 0x3ff00000u : 0u;
          if (present && !((present[smp >> 5] >> (smp & 31)) & 1u)) hi = 0x7ff80000u;
        }
      } else if (smp == S) {
        lo = 0x80u;                                    // padding starts right after the message
      }
      m[2 * j] = lo;
      m[2 * j + 1] = hi;
    }
    if (blk == n_blocks - 1) {                          // length in bits, little-endian
      const uint64_t nbits = total_bytes * 8;
      m[14] = (uint32_t)nbits;
      m[15] = (uint32_t)(nbits >> 32);
    }
    md5_block(st, m);
  }
}

// pool: n x key_words.  as_int64: cluster namespace.  nan_pool / nan_words: cluster pattern
// pool used for the NaN plane when key_words == W + 1 (consider_missing).
__global__ void __launch_bounds__(128)
k5_md5_ids(const uint32_t* __restrict__ pool, uint32_t first, uint32_t count, uint32_t key_words,
           uint32_t W, uint32_t S, int as_int64, const uint32_t* __restrict__ nan_pool,
           uint8_t* __restrict__ digests) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const uint32_t* bits = pool + (size_t)(first + i) * key_words;
  const uint32_t* present = (key_words > W && nan_pool) ? nan_pool + (size_t)bits[W] * W : nullptr;
  uint32_t st[4];
  md5_pattern(bits, present, S, as_int64, st);
  uint32_t* out = reinterpret_cast<uint32_t*>(digests + (size_t)i * 16);
  out[0] = st[0]; out[1] = st[1]; out[2] = st[2]; out[3] = st[3];
}

}  // namespace pf
