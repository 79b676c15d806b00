// K1 — k-mer extraction.  Replaces the window loop of the reference's
// cluster_cutter (/root/reference/panfeed/panfeed.py:54-88) and its positional
// branch (:90-107).
//
// One warp walks one cut sequence.  The packed 2-bit plane is read with
// coalesced 128-bit loads (32 lanes x 16 B = 2048 bases per step) into a
// per-warp shared-memory stage together with a 2-word halo (the k-1 bases the
// last windows of the step reach into); the next step's loads are issued
// before the current step is consumed.  Lane l of iteration `it` owns the
// window starting at base 32*it + l of the stage, so all lanes read the same
// two staged words (a broadcast) and differ only in the funnel-shift amount.
// Stores are fully coalesced: 32 consecutive 8-byte keys / 4-byte sample ranks.
#pragma once
#include "pf_common.cuh"

namespace pf {

constexpr int kK1Warps = 8;
constexpr int kK1StageWords = 64 + 2;      // 2048 bases + halo

struct PosOut {
  uint64_t* kmer;
  uint32_t* seq;
  int32_t* contig_start;
  int32_t* gene_start;
  uint8_t* flags;
};

// reverse complement of a k-mer held in the low 2k bits (first base on top)
__device__ __forceinline__ uint64_t revcomp2(uint64_t fwd, int k) {
  uint64_t v = __brevll(~fwd);                       // reverses bases AND the 2 bits inside each
  v = ((v & 0xaaaaaaaaaaaaaaaaULL) >> 1) | ((v & 0x5555555555555555ULL) << 1);
  return v >> (64 - 2 * k);
}

// RECORDS = false: positional records only (target sequences); the k-mer records are
// produced by the fused first pass (k1_fused.cuh) instead.
template <bool CANON, bool RECORDS>
__global__ void __launch_bounds__(kK1Warps * 32)
k1_extract(const uint64_t* __restrict__ bases, const uint32_t* __restrict__ ambbits,
           const SeqDev* __restrict__ seqs, uint32_t n_seqs, int k,
           uint64_t* __restrict__ keys, uint32_t* __restrict__ vals, PosOut pos) {
  __shared__ __align__(16) uint64_t stage_all[kK1Warps][kK1StageWords];
  const uint32_t lane = lane_id();
  const uint32_t warp = threadIdx.x >> 5;
  uint64_t* stage = stage_all[warp];
  const uint32_t stride = gridDim.x * kK1Warps;
  const int kshift = 64 - 2 * k;

  for (uint32_t s = blockIdx.x * kK1Warps + warp; s < n_seqs; s += stride) {
    const SeqDev d = seqs[s];
    if (d.len < (uint32_t)k) continue;
    const uint32_t nwin = d.len - (uint32_t)k + 1u;
    const uint64_t* w = bases + (d.base_off >> 5);
    const bool target = (d.flags & 1u) != 0u && pos.kmer != nullptr;
    if (!RECORDS && !target) continue;
    const bool amb = (d.flags & 2u) != 0u;
    const uint32_t* ab = amb ? (ambbits + (d.amb_off >> 5)) : nullptr;

    // prefetch step 0
    uint4 cur = ld_stream128(w + 2 * lane);
    uint4 halo = make_uint4(0, 0, 0, 0);
    if (lane == 0) halo = ld_stream128(w + 64);
    for (uint32_t c0 = 0; c0 < nwin; c0 += 2048u) {
      __syncwarp();
      reinterpret_cast<uint4*>(stage)[lane] = cur;
      if (lane == 0) reinterpret_cast<uint4*>(stage)[32] = halo;
      __syncwarp();
      const uint32_t next = c0 + 2048u;
      if (next < nwin) {                       // overlap the next step's loads
        const uint64_t* wn = w + (next >> 5);
        cur = ld_stream128(wn + 2 * lane);
        if (lane == 0) halo = ld_stream128(wn + 64);
      }
      const uint32_t iters = min(64u, (nwin - c0 + 31u) >> 5);
      for (uint32_t it = 0; it < iters; ++it) {
        const uint32_t p = c0 + it * 32u + lane;
        const bool valid = p < nwin;
        const uint64_t w0 = stage[it], w1 = stage[it + 1];
        const uint32_t sh = 2u * lane;
        const uint64_t x = (w0 << sh) | ((w1 >> 1) >> (63u - sh));
        const uint64_t fwd = x >> kshift;
        const uint64_t rc = revcomp2(fwd, k);
        if (!valid) continue;
        bool is_amb = false;
        if (amb) {                              // any non-ACGT symbol in [p, p+k)?
          const uint32_t wi = p >> 5, bs = p & 31u;
          const uint64_t two = ((uint64_t)ab[wi] << 32) | (uint64_t)ab[wi + 1];
          is_amb = ((two << bs) >> (64 - k)) != 0ull;
        }
        if (CANON) {
          const bool use_rc = rc < fwd;          // reference: fwd <= rc keeps fwd (+1)
          const uint64_t canon = use_rc ? rc : fwd;
          if (RECORDS) {
            const size_t r = (size_t)d.rec_off + p;
            keys[r] = is_amb ? 0ull : mix64(canon);
            vals[r] = is_amb ? kInvalidSample : d.sample;
          }
          if (target) {
            const size_t q = (size_t)d.pos_off + p;
            pos.kmer[q] = is_amb ? (uint64_t)(d.pwide_off + p) : canon;
            pos.seq[q] = s;
            pos.contig_start[q] = d.strand > 0 ? d.start + (int32_t)p : d.end - (int32_t)p - k;
            pos.gene_start[q] = (int32_t)p - d.offset;
            pos.flags[q] = (uint8_t)((use_rc ? 1u : 0u) | (is_amb ? 2u : 0u));
          }
        } else {
          if (RECORDS) {
            const size_t r = (size_t)d.rec_off + 2 * (size_t)p;
            ulonglong2 kk;
            kk.x = is_amb ? 0ull : mix64(fwd);
            kk.y = is_amb ? 0ull : mix64(rc);
            *reinterpret_cast<ulonglong2*>(keys + r) = kk;
            const uint32_t sv = is_amb ? kInvalidSample : d.sample;
            *reinterpret_cast<uint2*>(vals + r) = make_uint2(sv, sv);
          }
          if (target) {
            const size_t q = (size_t)d.pos_off + p;
            pos.kmer[q] = is_amb ? (uint64_t)(d.pwide_off + p) : fwd;
            pos.seq[q] = s;
            pos.contig_start[q] = d.strand > 0 ? d.start + (int32_t)p : d.end - (int32_t)p - k;
            pos.gene_start[q] = (int32_t)p - d.offset;
            pos.flags[q] = (uint8_t)(is_amb ? 2u : 0u);
          }
        }
      }
    }
  }
}

// Compact positional form (pf_params.emit_positions == 2, canonical mode): the only fact about a
// window of a --targets sequence that its descriptor and position do not already give is which
// strand was the canonical one (used_strand, panfeed.py:69-75).  One warp per target sequence,
// lane l owns window 32 * it + l: the 32 verdicts of an iteration are one ballot = one word of
// the bit plane, which is indexed like the packed plane (bit (i & 31) of word (i >> 5),
// i = base_off + pos; sequences start on 64-base boundaries, so words are never shared).
__global__ void __launch_bounds__(kK1Warps * 32)
k1_strand_bits(const uint64_t* __restrict__ bases, const SeqDev* __restrict__ seqs, uint32_t n_seqs, int k,
               uint32_t* __restrict__ strand_bits) {
  const uint32_t lane = lane_id();
  const uint32_t stride = gridDim.x * kK1Warps;
  const int kshift = 64 - 2 * k;
  for (uint32_t s = blockIdx.x * kK1Warps + (threadIdx.x >> 5); s < n_seqs; s += stride) {
    const SeqDev d = seqs[s];
    if (!(d.flags & 1u) || d.len < (uint32_t)k) continue;
    const uint32_t nwin = d.len - (uint32_t)k + 1u;
    const uint64_t* w = bases + (d.base_off >> 5);
    uint32_t* out = strand_bits + (d.base_off >> 5);
    for (uint32_t it = 0; it * 32u < nwin; ++it) {
      const uint64_t w0 = __ldg(w + it), w1 = __ldg(w + it + 1);       // the same two words for the whole warp
      const uint32_t sh = 2u * lane;
      const uint64_t x = (w0 << sh) | ((w1 >> 1) >> (63u - sh));
      const uint64_t fwd = x >> kshift;
      const bool use_rc = (it * 32u + lane < nwin) && revcomp2(fwd, k) < fwd;
      const uint32_t word = __ballot_sync(kFull, use_rc);
      if (lane == 0) out[it] = word;
    }
  }
}

// ---- k = 33..64: a k-mer is 2k <= 128 bits ------------------------------------------------
// The reference takes any -k (its k-mers are Python strings, panfeed.py:59-88).  Up to 32 bases a
// k-mer is one 64-bit word and goes through the engines above; from 33 to 64 it is a Key128 (2 bits
// per base, first base in the top USED bits) and every window goes through the 128-bit record
// pipeline that the N/IUPAC windows use (radix sort of mixed keys + run reduction).  One warp
// walks one sequence; lane l of iteration `it` owns the window starting at base 32 * it + l: the
// three words it needs are the same for the whole warp.
// A window of a sequence flagged ambiguous that touches a non-ACGT symbol (whose 2-bit code is
// that of A) is written as a dead record here: k1_extract_wide<Key256> owns it, and runs after
// this kernel on the same stream to correct its positional record / strand bit.
template <bool CANON>
__global__ void __launch_bounds__(kK1Warps * 32)
k1_extract_long(const uint64_t* __restrict__ bases, const uint32_t* __restrict__ ambbits,
                const SeqDev* __restrict__ seqs, uint32_t n_seqs, int k,
                Key128* __restrict__ keys, uint32_t* __restrict__ vals, PosOut pos,
                uint64_t* __restrict__ pos_wide, uint32_t* __restrict__ strand_bits) {
  const uint32_t lane = lane_id();
  const uint32_t stride = gridDim.x * kK1Warps;
  const uint32_t drop = 128u - 2u * (uint32_t)k;                  // unused low bits of the 64-base string (0..62)
  const uint64_t top_mask = (2u * (uint32_t)k - 64u) >= 64u ? ~0ull : ((1ull << (2u * (uint32_t)k - 64u)) - 1ull);
  for (uint32_t s = blockIdx.x * kK1Warps + (threadIdx.x >> 5); s < n_seqs; s += stride) {
    const SeqDev d = seqs[s];
    if (d.len < (uint32_t)k) continue;
    const uint32_t nwin = d.len - (uint32_t)k + 1u;
    const uint64_t* w = bases + (d.base_off >> 5);
    const bool target = (d.flags & 1u) != 0u;
    const uint32_t* ab = (d.flags & 2u) ? ambbits + (d.amb_off >> 5) : nullptr;
    for (uint32_t it = 0; it * 32u < nwin; ++it) {
      const uint32_t p = it * 32u + lane;
      const bool valid = p < nwin;
      const uint64_t w0 = __ldg(w + it), w1 = __ldg(w + it + 1), w2 = __ldg(w + it + 2);
      bool is_amb = false;
      if (ab && valid) {                   // any non-ACGT symbol in [p, p + k)?  (k <= 64: 3 bit words)
        const uint32_t wi = p >> 5, bs = p & 31u;
        const uint64_t two = ((uint64_t)ab[wi] << 32) | (uint64_t)ab[wi + 1];
        const uint64_t x = (two << bs) | (((uint64_t)ab[wi + 2] << bs) >> 32);    // bits [p, p + 64)
        is_amb = (k >= 64 ? x : x >> (64 - k)) != 0ull;
      }
      const uint32_t sh = 2u * lane;
      // the 64 bases from base p, first base on top
      uint64_t hi = w0, lo = w1;
      if (sh) { hi = (w0 << sh) | (w1 >> (64u - sh)); lo = (w1 << sh) | (w2 >> (64u - sh)); }
      if (drop) lo &= ~0ull << drop;                               // the k-mer's own bases only
      Key128 f, r;
      f.hi = drop ? hi >> drop : hi;
      f.lo = drop ? (lo >> drop) | (hi << (64u - drop)) : lo;
      // reverse complement of the 64-base string: the k-mer's is its last k bases
      r.hi = revcomp2(lo, 32) & top_mask;
      r.lo = revcomp2(hi, 32);
      const bool use_rc = r < f;                                   // reference: fwd <= rc keeps fwd (+1)
      if (CANON && strand_bits && target) {
        const uint32_t word = __ballot_sync(kFull, valid && use_rc);
        if (lane == 0) strand_bits[(d.base_off >> 5) + it] = word;
      }
      if (!valid) continue;
      if (CANON) {
        const Key128 canon = use_rc ? r : f;
        const size_t rec = (size_t)d.wrec_off + p;
        keys[rec] = is_amb ? Key128{0, 0} : mix128(canon);
        vals[rec] = is_amb ? kInvalidSample : d.sample;
        if (target && pos.kmer) {
          const size_t q = (size_t)d.pos_off + p, wq = (size_t)d.pwide_off + p;
          pos.kmer[q] = (uint64_t)wq;
          pos.seq[q] = s;
          pos.contig_start[q] = d.strand > 0 ? d.start + (int32_t)p : d.end - (int32_t)p - k;
          pos.gene_start[q] = (int32_t)p - d.offset;
          pos.flags[q] = (uint8_t)((use_rc ? 1u : 0u) | 2u);
          pos_wide[2 * wq] = canon.hi;
          pos_wide[2 * wq + 1] = canon.lo;
        }
      } else {
        const size_t rec = (size_t)d.wrec_off + 2 * (size_t)p;
        keys[rec] = is_amb ? Key128{0, 0} : mix128(f);
        keys[rec + 1] = is_amb ? Key128{0, 0} : mix128(r);
        vals[rec] = vals[rec + 1] = is_amb ? kInvalidSample : d.sample;
        if (target && pos.kmer) {
          const size_t q = (size_t)d.pos_off + p, wq = (size_t)d.pwide_off + p;
          pos.kmer[q] = (uint64_t)wq;
          pos.seq[q] = s;
          pos.contig_start[q] = d.strand > 0 ? d.start + (int32_t)p : d.end - (int32_t)p - k;
          pos.gene_start[q] = (int32_t)p - d.offset;
          pos.flags[q] = 2u;
          pos_wide[2 * wq] = f.hi;
          pos_wide[2 * wq + 1] = f.lo;
        }
      }
    }
  }
}

// ---- 4-bit plane: ambiguity bits and the wide (128-bit) extraction --------
// One ambiguity bit per symbol, 32 per word, first symbol in the top bit.
__global__ void k1_amb_bits(const uint64_t* __restrict__ amb_codes, uint64_t n_amb_words,
                            uint32_t* __restrict__ ambbits, uint64_t n_bit_words) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_bit_words) return;
  uint32_t out = 0;
  for (int h = 0; h < 2; ++h) {
    const uint64_t wi = 2 * i + h;
    const uint64_t w = wi < n_amb_words ? amb_codes[wi] : 0ull;
    for (int j = 0; j < 16; ++j) {
      const uint32_t c = (uint32_t)(w >> (60 - 4 * j)) & 15u;
      const bool acgt = (c == 0u) | (c == 2u) | (c == 4u) | (c == 11u);
      out |= (acgt ? 0u : 1u) << (31 - (16 * h + j));
    }
  }
  ambbits[i] = out;
}

// complement of the 16 symbols "ABCDGHKMNRSTVWXY" (pyfaidx table), nibble i = comp(i)
__device__ __forceinline__ uint32_t comp4(uint32_t c) {
  // A->T(11) B->V(12) C->G(4) D->H(5) G->C(2) H->D(3) K->M(7) M->K(6) N->N(8)
  // R->Y(15) S->S(10) T->A(0) V->B(1) W->W(13) X->X(14) Y->R(9)
  constexpr uint64_t kTable = 0x9ED10AF86732'54CBULL;
  return (uint32_t)(kTable >> (4 * c)) & 15u;
}

// 4-bit keys, built one symbol at a time: push4 appends a symbol at the bottom (the forward
// k-mer), set4 ORs a symbol into nibble i from the bottom (the reverse complement)
__device__ __forceinline__ void push4(Key128& key, uint32_t c) {
  key.hi = (key.hi << 4) | (key.lo >> 60);
  key.lo = (key.lo << 4) | c;
}
__device__ __forceinline__ void push4(Key256& key, uint32_t c) {
  key.w[0] = (key.w[0] << 4) | (key.w[1] >> 60);
  key.w[1] = (key.w[1] << 4) | (key.w[2] >> 60);
  key.w[2] = (key.w[2] << 4) | (key.w[3] >> 60);
  key.w[3] = (key.w[3] << 4) | c;
}
__device__ __forceinline__ void set4(Key128& key, int i, uint64_t c) {
  if (i < 16) key.lo |= c << (4 * i); else key.hi |= c << (4 * (i - 16));
}
__device__ __forceinline__ void set4(Key256& key, int i, uint64_t c) {
  const uint64_t v = c << (4 * (i & 15));
  const int j = i >> 4;                    // (a branch per word keeps the key in registers)
  if (j == 0) key.w[3] |= v; else if (j == 1) key.w[2] |= v; else if (j == 2) key.w[1] |= v; else key.w[0] |= v;
}
__device__ __forceinline__ Key128 mix_key(const Key128& key) { return mix128(key); }
__device__ __forceinline__ Key256 mix_key(const Key256& key) { return mix256(key); }

// One thread per window of a flagged sequence; only windows that touch a non-ACGT symbol produce
// a live record (the narrow kernel owns the others).  KeyT = Key128: k <= 32, records at wrec_off,
// positional k-mers at pwide_off (pos_flags bit 1).  KeyT = Key256: k = 33..64, records at rec_off,
// positional k-mers at pos_slot[list entry] (pos_flags bit 2; the positional record's k-mer index
// is rewritten too) - after k1_extract_long, which wrote the windows' 2-bit records as dead ones.
template <bool CANON, typename KeyT>
__global__ void k1_extract_wide(const uint64_t* __restrict__ amb_codes,
                                const SeqDev* __restrict__ seqs,
                                const uint32_t* __restrict__ wide_seqs, uint32_t n_wide_seqs,
                                int k, KeyT* __restrict__ keys, uint32_t* __restrict__ vals,
                                uint64_t* __restrict__ pos_wide, uint8_t* __restrict__ pos_flags,
                                uint32_t* __restrict__ strand_bits /* compact positional form, else null */,
                                uint64_t* __restrict__ pos_kmer = nullptr, const uint32_t* __restrict__ pos_slot = nullptr) {
  constexpr bool kX = sizeof(KeyT) == sizeof(Key256);
  constexpr uint8_t kFlag = kX ? 4u : 2u;
  const uint32_t lane = lane_id();
  const uint32_t warp = threadIdx.x >> 5;
  const uint32_t stride = gridDim.x * (blockDim.x >> 5);
  for (uint32_t wsi = blockIdx.x * (blockDim.x >> 5) + warp; wsi < n_wide_seqs; wsi += stride) {
    const uint32_t s = wide_seqs[wsi];
    const SeqDev d = seqs[s];
    if (d.len < (uint32_t)k) continue;
    const uint32_t nwin = d.len - (uint32_t)k + 1u;
    const bool target = (d.flags & 1u) != 0u;
    const uint32_t rec0 = kX ? d.rec_off : d.wrec_off;
    const uint32_t slot0 = kX ? (pos_slot ? pos_slot[wsi] : 0u) : d.pwide_off;
    for (uint32_t p = lane; p < nwin; p += 32u) {
      KeyT f = KeyTraits<KeyT>::zero(), r = KeyTraits<KeyT>::zero();
      bool is_amb = false;
      for (int i = 0; i < k; ++i) {
        const uint64_t sym = d.amb_off + p + (uint32_t)i;
        const uint32_t c = (uint32_t)(amb_codes[sym >> 4] >> (60 - 4 * (sym & 15u))) & 15u;
        is_amb |= !((c == 0u) | (c == 2u) | (c == 4u) | (c == 11u));
        push4(f, c);                 // forward: first symbol ends up in the top used nibble
        set4(r, i, comp4(c));        // reverse complement: symbol i becomes nibble i from the bottom
      }
      // r has comp(sym_i) at nibble i (LSB side) = reversed order: top nibble (k-1) holds
      // comp(sym_{k-1}) which is the first symbol of the reverse complement.
      const size_t slot = (size_t)slot0 + p;
      if (CANON) {
        const bool use_rc = r < f;
        const KeyT canon = use_rc ? r : f;
        const size_t rec = (size_t)rec0 + p;
        keys[rec] = is_amb ? mix_key(canon) : KeyTraits<KeyT>::zero();
        vals[rec] = is_amb ? d.sample : kInvalidSample;
        if (target && is_amb && strand_bits) {
          // runs after k1_strand_bits / k1_extract_long on the same stream: the strand choice of
          // an ambiguous window must come from the 4-bit comparison
          const uint64_t i = d.base_off + p;
          if (use_rc) atomicOr(&strand_bits[i >> 5], 1u << (i & 31u));
          else atomicAnd(&strand_bits[i >> 5], ~(1u << (i & 31u)));
        } else if (target && is_amb) {
          store_kmer(pos_wide, slot, canon);
          // runs after the narrow / long kernel on the same stream: the strand choice of an
          // ambiguous window must come from the 4-bit comparison
          pos_flags[(size_t)d.pos_off + p] = (uint8_t)((use_rc ? 1u : 0u) | kFlag);
          if (kX) pos_kmer[(size_t)d.pos_off + p] = slot;
        }
      } else {
        const size_t rec = (size_t)rec0 + 2 * (size_t)p;
        keys[rec] = is_amb ? mix_key(f) : KeyTraits<KeyT>::zero();
        keys[rec + 1] = is_amb ? mix_key(r) : KeyTraits<KeyT>::zero();
        vals[rec] = vals[rec + 1] = is_amb ? d.sample : kInvalidSample;
        if (target && is_amb && pos_wide) {
          store_kmer(pos_wide, slot, f);
          if (kX) {
            pos_flags[(size_t)d.pos_off + p] = kFlag;
            pos_kmer[(size_t)d.pos_off + p] = slot;
          }
        }
      }
    }
  }
}

}  // namespace pf
