// Native (multi-threaded, host) text formatting of the positional records: the kmers.tsv rows
// the reference's cluster_cutter writes at /root/reference/panfeed/panfeed.py:90-107,
//
//   {idx}\t{strain}\t{gene_id}\t{contig}\t{strand}\t{truestart}\t{trueend}\t{genestart}\t{geneend}\t{used_strand}\t{kmer}\n
//
// from the binary records pf_collect returns (21 bytes per k-mer instance).  A second pass
// over a few hundred clusters yields 1e8 rows; formatting them in the Python host costs minutes,
// here it is a memory-bound loop over host threads.  No device code in this file.
#include <algorithm>
#include <atomic>
#include <cstdint>
#include <cstring>
#include <thread>
#include <vector>

#include <zlib.h>

#include "../../include/panfeed_b200.h"
#include "pf_host.h"

namespace {

const char kAcgt[5] = "ACGT";
const char kAmb[17] = PF_AMB_ALPHABET;
// complement of the 16 symbols (pyfaidx table restricted to upper case, as input.py:448-452 uses it)
inline char comp_symbol(char c) {
  switch (c) {
    case 'A': return 'T'; case 'C': return 'G'; case 'T': return 'A'; case 'G': return 'C';
    case 'N': return 'N'; case 'Y': return 'R'; case 'R': return 'Y'; case 'W': return 'W';
    case 'S': return 'S'; case 'K': return 'M'; case 'M': return 'K'; case 'D': return 'H';
    case 'V': return 'B'; case 'H': return 'D'; case 'B': return 'V'; case 'X': return 'X';
    default: return c;
  }
}

inline int put_int(char* p, int64_t v) {          // decimal, like Python's str(int); returns the length
  char tmp[24];
  int n = 0;
  uint64_t u = v < 0 ? (uint64_t)(-v) : (uint64_t)v;
  do { tmp[n++] = (char)('0' + u % 10); u /= 10; } while (u);
  int len = 0;
  if (v < 0) p[len++] = '-';
  while (n) p[len++] = tmp[--n];
  return len;
}
inline int len_int(int64_t v) {
  int len = v < 0 ? 1 : 0;
  uint64_t u = v < 0 ? (uint64_t)(-v) : (uint64_t)v;
  do { ++len; u /= 10; } while (u);
  return len;
}

// text of a k-mer of n_words words (most significant first), first symbol in the top used bits:
// 4 bits per symbol (codes of PF_AMB_ALPHABET) when k symbols fit that way (two words: N/IUPAC
// k-mers of k <= 32; four words: k <= 64), else 2 bits per base (two words, k > 32)
inline void wide_kmer_text(const uint64_t* w, uint32_t n_words, uint32_t k, char* out) {
  const uint32_t bits = k <= 16 * n_words ? 4u : 2u;
  const char* alphabet = bits == 4u ? kAmb : kAcgt;
  const uint64_t mask = (1ull << bits) - 1ull;
  for (uint32_t s = 0; s < k; ++s) {
    const uint32_t pos = bits * (k - 1 - s);              // from bit 0 of the last word
    out[s] = alphabet[(w[n_words - 1 - pos / 64] >> (pos % 64)) & mask];
  }
}

struct Job {
  const pf_batch_result* r;
  uint32_t k;
  int canonical;
  const char* lead_blob;
  const uint64_t* lead_off;
  const int32_t* seq_strand;
};

// k-mer text of record i into `out` (k bytes)
inline void kmer_text(const Job& j, uint64_t i, char* out) {
  const uint32_t k = j.k;
  if (j.r->pos_flags[i] & 4u) {
    wide_kmer_text(j.r->pos_xwide_kmer + 4 * j.r->pos_kmer[i], 4, k, out);
  } else if (j.r->pos_flags[i] & 2u) {
    wide_kmer_text(j.r->pos_wide_kmer + 2 * j.r->pos_kmer[i], 2, k, out);
  } else {
    const uint64_t v = j.r->pos_kmer[i];
    for (uint32_t s = 0; s < k; ++s) out[s] = kAcgt[(v >> (2 * (k - 1 - s))) & 3u];
  }
}

inline uint64_t row_len(const Job& j, uint64_t i) {
  const uint32_t seq = j.r->pos_seq[i];
  const uint64_t lead = j.lead_off[seq + 1] - j.lead_off[seq];
  const int64_t c0 = j.r->pos_contig_start[i], g0 = j.r->pos_gene_start[i];
  const uint64_t coords = (uint64_t)len_int(c0) + len_int(c0 + j.k) + len_int(g0) + len_int(g0 + j.k) + 4;
  if (j.canonical) {
    const int used = (j.r->pos_flags[i] & 1u) ? 2 : 1;                  // "-1" / "1"
    return lead + coords + used + 1 + j.k + 1;
  }
  const int32_t st = j.seq_strand[seq];                                  // rows for st and -st
  return 2 * (lead + coords + 1 + j.k + 1) + len_int(st) + len_int(-(int64_t)st);
}

inline char* write_row(const Job& j, uint64_t i, char* p) {
  const uint32_t seq = j.r->pos_seq[i];
  const uint64_t lead = j.lead_off[seq + 1] - j.lead_off[seq];
  const int64_t c0 = j.r->pos_contig_start[i], g0 = j.r->pos_gene_start[i];
  char km[72];
  kmer_text(j, i, km);
  auto head = [&](char* q) {
    memcpy(q, j.lead_blob + j.lead_off[seq], lead);
    q += lead;
    q += put_int(q, c0); *q++ = '\t';
    q += put_int(q, c0 + j.k); *q++ = '\t';
    q += put_int(q, g0); *q++ = '\t';
    q += put_int(q, g0 + j.k); *q++ = '\t';
    return q;
  };
  if (j.canonical) {
    p = head(p);
    if (j.r->pos_flags[i] & 1u) { *p++ = '-'; *p++ = '1'; } else { *p++ = '1'; }
    *p++ = '\t';
    memcpy(p, km, j.k); p += j.k;
    *p++ = '\n';
    return p;
  }
  const int32_t st = j.seq_strand[seq];
  p = head(p);
  p += put_int(p, st); *p++ = '\t';
  memcpy(p, km, j.k); p += j.k;
  *p++ = '\n';
  p = head(p);
  p += put_int(p, -(int64_t)st); *p++ = '\t';
  for (uint32_t s = 0; s < j.k; ++s) p[s] = comp_symbol(km[j.k - 1 - s]);   // reverse complement
  p += j.k;
  *p++ = '\n';
  return p;
}

}  // namespace

extern "C" int pf_format_positions(const pf_batch_result* r, uint32_t k, int canonical, uint64_t first,
                                   uint64_t count, const char* lead_blob, const uint64_t* lead_off,
                                   const int32_t* seq_strand, char* out, uint64_t out_cap, uint64_t* out_len,
                                   uint32_t n_threads) {
  if (!r || !out_len || k < 1 || k > 64) return PF_ERR_INVALID;
  if (first + count > r->n_pos) return PF_ERR_INVALID;
  *out_len = 0;
  if (count == 0) return PF_OK;
  if (!lead_blob || !lead_off || (!canonical && !seq_strand)) return PF_ERR_INVALID;
  Job j{r, k, canonical, lead_blob, lead_off, seq_strand};
  const uint32_t hw = pf_host_threads();
  uint32_t nt = n_threads ? n_threads : hw;
  nt = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(nt, (count + 65535) / 65536));
  const uint64_t per = (count + nt - 1) / nt;
  std::vector<uint64_t> bytes(nt, 0);
  auto run = [&](auto&& fn) {
    if (nt == 1) { fn(0u); return; }
    std::vector<std::thread> th;
    for (uint32_t t = 0; t < nt; ++t) th.emplace_back(fn, t);
    for (auto& x : th) x.join();
  };
  run([&](uint32_t t) {
    const uint64_t a = first + std::min<uint64_t>(count, t * per), b = first + std::min<uint64_t>(count, (t + 1) * per);
    uint64_t s = 0;
    for (uint64_t i = a; i < b; ++i) s += row_len(j, i);
    bytes[t] = s;
  });
  uint64_t total = 0;
  std::vector<uint64_t> start(nt, 0);
  for (uint32_t t = 0; t < nt; ++t) { start[t] = total; total += bytes[t]; }
  *out_len = total;
  if (!out) return PF_OK;                       // sizing call
  if (out_cap < total) return PF_ERR_NOMEM;
  run([&](uint32_t t) {
    const uint64_t a = first + std::min<uint64_t>(count, t * per), b = first + std::min<uint64_t>(count, (t + 1) * per);
    char* p = out + start[t];
    for (uint64_t i = a; i < b; ++i) p = write_row(j, i, p);
  });
  return PF_OK;
}

// ---------------------------------------------------------------------------
// Compact positional form (pf_params.emit_positions == 2): the device returns one bit per
// window (was the reverse complement the canonical k-mer?); everything else of a kmers.tsv
// row is a function of the caller's own batch.
// ---------------------------------------------------------------------------
namespace {
struct CJob {
  const pf_batch* b;
  const uint32_t* bits;
  uint32_t k;
  int canonical;
  const char* lead_blob;
  const uint64_t* lead_off;
};
// A coordinate that moves by one from row to row, kept as its decimal text: a step touches the
// last digit (and the carry's) instead of dividing the number down again.  Anything unusual - a
// negative value, a change of the number of digits - goes through put_int.
struct DecCounter {
  char text[24];
  int len = 0;
  int64_t v = 0;
  void set(int64_t x) { v = x; len = put_int(text, x); }
  void step(int d) {                                 // d = +1 or -1
    const int64_t nv = v + d;
    if (v > 0 && nv > 0) {
      int i = len - 1;
      if (d > 0) {
        while (i >= 0 && text[i] == '9') text[i--] = '0';
        if (i >= 0) { ++text[i]; v = nv; return; }
      } else {
        while (i >= 0 && text[i] == '0') text[i--] = '9';
        if (i > 0 || (i == 0 && text[0] > '1') || len == 1) { --text[i]; v = nv; return; }
      }
    }
    set(nv);                                         // (the digits touched above are rewritten in full)
  }
  char* put(char* o) const { for (int i = 0; i < len; ++i) o[i] = text[i]; return o + len; }
};
inline bool strand_bit(const CJob& j, const pf_seq_desc& q, uint32_t p) {
  const uint64_t i = q.base_off + p;
  return (j.bits[i >> 5] >> (i & 31u)) & 1u;
}
inline uint64_t seq_rows_len(const CJob& j, uint32_t si) {
  const pf_seq_desc& q = j.b->seqs[si];
  if (!(q.flags & PF_SEQ_TARGET) || q.len < j.k) return 0;
  const uint32_t nwin = q.len - j.k + 1;
  const uint64_t lead = j.lead_off[si + 1] - j.lead_off[si];
  uint64_t total = 0;
  for (uint32_t p = 0; p < nwin; ++p) {
    const int64_t c0 = q.strand > 0 ? (int64_t)q.start + p : (int64_t)q.end - p - j.k, g0 = (int64_t)p - q.offset;
    const uint64_t coords = (uint64_t)len_int(c0) + len_int(c0 + j.k) + len_int(g0) + len_int(g0 + j.k) + 4;
    if (j.canonical) total += lead + coords + (strand_bit(j, q, p) ? 2 : 1) + 1 + j.k + 1;
    else total += 2 * (lead + coords + 1 + j.k + 1) + len_int(q.strand) + len_int(-(int64_t)q.strand);
  }
  return total;
}
inline char* write_seq_rows(const CJob& j, uint32_t si, char* p) {
  const pf_seq_desc& q = j.b->seqs[si];
  if (!(q.flags & PF_SEQ_TARGET) || q.len < j.k) return p;
  const uint32_t nwin = q.len - j.k + 1, k = j.k;
  const uint64_t lead = j.lead_off[si + 1] - j.lead_off[si];
  const char* lead_p = j.lead_blob + j.lead_off[si];
  // the sequence's symbols once, and their reverse complement once: windows are slices of both
  std::vector<char> text((size_t)q.len), rc_text((size_t)q.len);
  if (q.flags & PF_SEQ_AMBIGUOUS) {
    for (uint32_t s = 0; s < q.len; ++s) {
      const uint64_t i = q.amb_off + s;
      text[s] = kAmb[(j.b->amb_codes[i >> 4] >> (60 - 4 * (i & 15u))) & 15u];
    }
  } else {
    for (uint32_t s = 0; s < q.len; ++s) {
      const uint64_t i = q.base_off + s;
      text[s] = kAcgt[(j.b->packed_bases[i >> 5] >> (62 - 2 * (i & 31u))) & 3u];
    }
  }
  for (uint32_t s = 0; s < q.len; ++s) rc_text[s] = comp_symbol(text[q.len - 1 - s]);
  // the four coordinates of a row move by one from window to window
  const int dir = q.strand > 0 ? 1 : -1;
  DecCounter c_lo, c_hi, g_lo, g_hi;
  {
    const int64_t c0 = q.strand > 0 ? (int64_t)q.start : (int64_t)q.end - k, g0 = -(int64_t)q.offset;
    c_lo.set(c0); c_hi.set(c0 + k); g_lo.set(g0); g_hi.set(g0 + k);
  }
  char strand_fwd[24], strand_rev[24];
  const int sf = put_int(strand_fwd, q.strand), sr = put_int(strand_rev, -(int64_t)q.strand);
  for (uint32_t w = 0; w < nwin; ++w) {
    auto head = [&](char* o) {
      memcpy(o, lead_p, lead);
      o += lead;
      o = c_lo.put(o); *o++ = '\t';
      o = c_hi.put(o); *o++ = '\t';
      o = g_lo.put(o); *o++ = '\t';
      o = g_hi.put(o); *o++ = '\t';
      return o;
    };
    const char* fwd = text.data() + w;
    const char* rev = rc_text.data() + (q.len - w - k);        // reverse complement of window w
    if (j.canonical) {
      const bool rc = strand_bit(j, q, w);
      p = head(p);
      if (rc) { *p++ = '-'; *p++ = '1'; } else { *p++ = '1'; }
      *p++ = '\t';
      memcpy(p, rc ? rev : fwd, k);
      p += k;
      *p++ = '\n';
    } else {
      p = head(p);
      memcpy(p, strand_fwd, sf); p += sf; *p++ = '\t';
      memcpy(p, fwd, k); p += k;
      *p++ = '\n';
      p = head(p);
      memcpy(p, strand_rev, sr); p += sr; *p++ = '\t';
      memcpy(p, rev, k); p += k;
      *p++ = '\n';
    }
    c_lo.step(dir); c_hi.step(dir); g_lo.step(1); g_hi.step(1);
  }
  return p;
}
}  // namespace

extern "C" int pf_format_positions_compact(const pf_batch* b, const uint32_t* strand_bits, uint32_t k, int canonical,
                                           uint32_t seq_first, uint32_t seq_count, const char* lead_blob,
                                           const uint64_t* lead_off, char* out, uint64_t out_cap, uint64_t* out_len,
                                           uint32_t n_threads) {
  if (!b || !out_len || k < 1 || k > 64) return PF_ERR_INVALID;
  if ((uint64_t)seq_first + seq_count > b->n_seqs) return PF_ERR_INVALID;
  *out_len = 0;
  if (seq_count == 0) return PF_OK;
  if (!b->seqs || !b->packed_bases || !lead_blob || !lead_off || (canonical && !strand_bits)) return PF_ERR_INVALID;
  for (uint32_t i = seq_first; i < seq_first + seq_count; ++i)
    if ((b->seqs[i].flags & PF_SEQ_TARGET) && (b->seqs[i].flags & PF_SEQ_AMBIGUOUS) && !b->amb_codes) return PF_ERR_INVALID;
  CJob j{b, strand_bits, k, canonical, lead_blob, lead_off};
  const uint32_t hw = pf_host_threads();
  uint32_t nt = n_threads ? n_threads : hw;
  nt = std::max(1u, std::min<uint32_t>(nt, (seq_count + 63u) / 64u));
  const uint32_t per = (seq_count + nt - 1) / nt;
  std::vector<uint64_t> bytes(nt, 0);
  auto run = [&](auto&& fn) {
    if (nt == 1) { fn(0u); return; }
    std::vector<std::thread> th;
    for (uint32_t t = 0; t < nt; ++t) th.emplace_back(fn, t);
    for (auto& x : th) x.join();
  };
  run([&](uint32_t t) {
    const uint32_t a = seq_first + std::min(seq_count, t * per), e = seq_first + std::min(seq_count, (t + 1) * per);
    uint64_t s = 0;
    for (uint32_t i = a; i < e; ++i) s += seq_rows_len(j, i);
    bytes[t] = s;
  });
  uint64_t total = 0;
  std::vector<uint64_t> start(nt, 0);
  for (uint32_t t = 0; t < nt; ++t) { start[t] = total; total += bytes[t]; }
  *out_len = total;
  if (!out) return PF_OK;                       // sizing call
  if (out_cap < total) return PF_ERR_NOMEM;
  run([&](uint32_t t) {
    const uint32_t a = seq_first + std::min(seq_count, t * per), e = seq_first + std::min(seq_count, (t + 1) * per);
    char* p = out + start[t];
    for (uint32_t i = a; i < e; ++i) p = write_seq_rows(j, i, p);
  });
  return PF_OK;
}

// ---------------------------------------------------------------------------
// --associations: the lines of panfeed-get-kmers (get_kmers.py:108-145) from the compact positional
// form and the device join (pf_assoc_collect).  The association columns arrive as one text snippet
// per passing association, formatted by the caller (pandas prints them, so pandas formats them);
// a line is a concatenation of the cluster tag, the k-mer, a snippet and the positional fields.
// ---------------------------------------------------------------------------
namespace {
struct AJob {
  const pf_batch* b;
  const uint32_t* bits;
  uint32_t k;
  int canonical;
  const pf_batch_result* rows;
  const pf_assoc_result* a;
  const char* tag_blob;
  const uint64_t* tag_off;
  const char* lead_blob;
  const uint64_t* lead_off;
  const char* snip_blob;
  const uint64_t* snip_off;
  uint32_t empty_snip;          // tabs of a snippet where nothing passes
  bool only_passing, floats;
  std::vector<std::pair<uint64_t, uint32_t>> win;     // (window, association row), sorted
};

inline uint64_t snip_len(const AJob& j, uint32_t a) {
  return a == PF_ASSOC_NONE ? j.empty_snip : j.snip_off[a + 1] - j.snip_off[a];
}
inline char* put_snip(const AJob& j, uint32_t a, char* p) {
  if (a == PF_ASSOC_NONE) { memset(p, '\t', j.empty_snip); return p + j.empty_snip; }
  const uint64_t n = j.snip_off[a + 1] - j.snip_off[a];
  memcpy(p, j.snip_blob + j.snip_off[a], n);
  return p + n;
}
inline char* put_num(const AJob& j, char* p, int64_t v) {
  p += put_int(p, v);
  if (j.floats) { *p++ = '.'; *p++ = '0'; }
  return p;
}
// the window entries of sequence q: [lo, hi) of j.win
inline std::pair<size_t, size_t> seq_windows(const AJob& j, const pf_seq_desc& q) {
  auto lo = std::lower_bound(j.win.begin(), j.win.end(), std::make_pair(q.base_off << 1, 0u));
  auto hi = std::lower_bound(lo, j.win.end(), std::make_pair((q.base_off + q.len) << 1, 0u));
  return {(size_t)(lo - j.win.begin()), (size_t)(hi - j.win.begin())};
}
// Bytes (out == NULL) or the lines of target sequence si.  Right join: every window row of a
// passing cluster; left join: the passing ones.
inline uint64_t annot_seq(const AJob& j, uint32_t si, char* out) {
  const pf_seq_desc& q = j.b->seqs[si];
  if (!(q.flags & PF_SEQ_TARGET) || q.len < j.k || !j.a->cluster_pass[q.cluster]) return 0;
  const uint32_t k = j.k, nwin = q.len - k + 1;
  auto range = seq_windows(j, q);
  if (j.only_passing && range.first == range.second) return 0;
  const uint64_t tl = j.tag_off[q.cluster + 1] - j.tag_off[q.cluster];
  const char* tag = j.tag_blob + j.tag_off[q.cluster];
  const uint64_t ll = j.lead_off[si + 1] - j.lead_off[si];
  const char* lead = j.lead_blob + j.lead_off[si];
  const uint32_t fl = j.floats ? 2 : 0;
  std::vector<char> text, rc_text;
  if (out) {
    text.resize(q.len);
    rc_text.resize(q.len);
    if (q.flags & PF_SEQ_AMBIGUOUS) {
      for (uint32_t s = 0; s < q.len; ++s) {
        const uint64_t i = q.amb_off + s;
        text[s] = kAmb[(j.b->amb_codes[i >> 4] >> (60 - 4 * (i & 15u))) & 15u];
      }
    } else {
      for (uint32_t s = 0; s < q.len; ++s) {
        const uint64_t i = q.base_off + s;
        text[s] = kAcgt[(j.b->packed_bases[i >> 5] >> (62 - 2 * (i & 31u))) & 3u];
      }
    }
    for (uint32_t s = 0; s < q.len; ++s) rc_text[s] = comp_symbol(text[q.len - 1 - s]);
  }
  uint64_t total = 0;
  char* p = out;
  size_t at = range.first;
  auto line = [&](uint32_t w, bool rc, int64_t used, uint32_t a) {
    const int64_t c0 = q.strand > 0 ? (int64_t)q.start + w : (int64_t)q.end - w - k, g0 = (int64_t)w - q.offset;
    if (!out) {
      total += tl + 1 + k + 1 + snip_len(j, a) + 1 + ll + len_int(q.strand) + len_int(c0) + len_int(c0 + k) +
               len_int(g0) + len_int(g0 + k) + len_int(used) + 6 * fl + 6;
      return;
    }
    memcpy(p, tag, tl); p += tl; *p++ = '\t';
    memcpy(p, rc ? rc_text.data() + (q.len - w - k) : text.data() + w, k); p += k; *p++ = '\t';
    p = put_snip(j, a, p); *p++ = '\t';
    memcpy(p, lead, ll); p += ll;
    p = put_num(j, p, q.strand); *p++ = '\t';
    p = put_num(j, p, c0); *p++ = '\t';
    p = put_num(j, p, c0 + k); *p++ = '\t';
    p = put_num(j, p, g0); *p++ = '\t';
    p = put_num(j, p, g0 + k); *p++ = '\t';
    p = put_num(j, p, used); *p++ = '\n';
  };
  auto emit = [&](uint32_t w, uint32_t o) {          // window w, row o (canonical: the one row)
    const uint64_t id = ((q.base_off + w) << 1) | o;
    while (at < range.second && j.win[at].first < id) ++at;
    const uint32_t a = at < range.second && j.win[at].first == id ? j.win[at].second : PF_ASSOC_NONE;
    if (j.only_passing && a == PF_ASSOC_NONE) return;
    if (j.canonical) {
      const uint64_t i = q.base_off + w;
      const bool rc = (j.bits[i >> 5] >> (i & 31u)) & 1u;
      line(w, rc, rc ? -1 : 1, a);
    } else {
      line(w, o == 1, o == 1 ? -(int64_t)q.strand : (int64_t)q.strand, a);
    }
  };
  if (j.only_passing) {                               // only the listed windows
    for (size_t e = range.first; e < range.second; ++e) {
      if (e > range.first && j.win[e].first == j.win[e - 1].first) continue;
      const uint64_t id = j.win[e].first;
      emit((uint32_t)((id >> 1) - q.base_off), (uint32_t)(id & 1u));
    }
  } else {
    for (uint32_t w = 0; w < nwin; ++w)
      for (uint32_t o = 0; o < (j.canonical ? 1u : 2u); ++o) emit(w, o);
  }
  return out ? (uint64_t)(p - out) : total;
}
// --only-passing: the passing rows no window carries and the passing cluster-row hashes
inline uint64_t annot_unseen(const AJob& j, char* out) {
  const pf_batch_result* r = j.rows;
  const uint64_t nn = r->n_rows, nw = r->n_wide_rows;
  uint64_t total = 0;
  char* p = out;
  auto line = [&](uint32_t c, const char* kmer, uint32_t a) {
    const uint64_t tl = j.tag_off[c + 1] - j.tag_off[c];
    const uint64_t kl = kmer ? j.k : 0;
    if (!out) { total += tl + 1 + kl + 1 + snip_len(j, a) + 9 + 1; return; }
    memcpy(p, j.tag_blob + j.tag_off[c], tl); p += tl; *p++ = '\t';
    if (kmer) { memcpy(p, kmer, kl); p += kl; }
    *p++ = '\t';
    p = put_snip(j, a, p);
    memset(p, '\t', 9); p += 9;
    *p++ = '\n';
  };
  char km[72];
  for (uint64_t e = 0; e < j.a->n_rows; ++e) {
    if (j.a->row_seen[e]) continue;
    const uint64_t i = j.a->row[e];
    uint32_t c;
    if (i < nn) {
      c = r->row_cluster[i];
      for (uint32_t s = 0; s < j.k; ++s) km[s] = kAcgt[(r->row_kmer[i] >> (2 * (j.k - 1 - s))) & 3u];
    } else if (i < nn + nw) {
      c = r->wide_row_cluster[i - nn];
      wide_kmer_text(r->wide_row_kmer + 2 * (i - nn), 2, j.k, km);
    } else {
      c = r->xwide_row_cluster[i - nn - nw];
      wide_kmer_text(r->xwide_row_kmer + 4 * (i - nn - nw), 4, j.k, km);
    }
    line(c, km, j.a->row_assoc[e]);
  }
  for (uint32_t c = 0; c < j.a->n_clusters; ++c)
    if (j.a->cluster_assoc[c] != PF_ASSOC_NONE) line(c, nullptr, j.a->cluster_assoc[c]);
  return out ? (uint64_t)(p - out) : total;
}
}  // namespace

extern "C" int pf_format_annotated(const pf_batch* b, const uint32_t* strand_bits, uint32_t k, int canonical,
                                   const pf_batch_result* rows, const pf_assoc_result* assoc, const char* tag_blob,
                                   const uint64_t* tag_off, const char* lead_blob, const uint64_t* lead_off,
                                   const char* snip_blob, const uint64_t* snip_off, uint64_t n_snips,
                                   uint32_t snip_fields, uint32_t flags, char* out, uint64_t out_cap,
                                   uint64_t* out_len, uint32_t n_threads) {
  if (!b || !rows || !assoc || !out_len || k < 1 || k > 64 || snip_fields < 1) return PF_ERR_INVALID;
  *out_len = 0;
  if (assoc->n_clusters != b->n_clusters || rows->n_clusters != b->n_clusters) return PF_ERR_INVALID;
  if (b->n_clusters && (!tag_blob || !tag_off || !assoc->cluster_pass || !assoc->cluster_assoc)) return PF_ERR_INVALID;
  if (b->n_seqs && (!b->seqs || !b->packed_bases || !lead_blob || !lead_off || (canonical && !strand_bits)))
    return PF_ERR_INVALID;
  if (n_snips && (!snip_blob || !snip_off)) return PF_ERR_INVALID;
  if (assoc->n_windows && (!assoc->window || !assoc->window_assoc)) return PF_ERR_INVALID;
  if (assoc->n_rows && (!assoc->row || !assoc->row_assoc || !assoc->row_seen)) return PF_ERR_INVALID;
  const uint64_t n_all_rows = rows->n_rows + rows->n_wide_rows + rows->n_xwide_rows;
  for (uint64_t e = 0; e < assoc->n_windows; ++e) if (assoc->window_assoc[e] >= n_snips) return PF_ERR_INVALID;
  for (uint64_t e = 0; e < assoc->n_rows; ++e)
    if (assoc->row_assoc[e] >= n_snips || assoc->row[e] >= n_all_rows) return PF_ERR_INVALID;
  for (uint32_t c = 0; c < b->n_clusters; ++c) {
    const uint32_t a = assoc->cluster_assoc[c];
    if ((a != PF_ASSOC_NONE && a >= n_snips) || tag_off[c + 1] < tag_off[c]) return PF_ERR_INVALID;
  }
  for (uint32_t i = 0; i < b->n_seqs; ++i) {
    const pf_seq_desc& q = b->seqs[i];
    if (q.cluster >= b->n_clusters) return PF_ERR_INVALID;
    if ((q.flags & PF_SEQ_TARGET) && (q.flags & PF_SEQ_AMBIGUOUS) && !b->amb_codes) return PF_ERR_INVALID;
  }
  AJob j{b, strand_bits, k, canonical, rows, assoc, tag_blob, tag_off, lead_blob, lead_off, snip_blob, snip_off,
         snip_fields - 1, (flags & PF_ANNOT_ONLY_PASSING) != 0, (flags & PF_ANNOT_FLOAT_POSITIONS) != 0, {}};
  j.win.resize(assoc->n_windows);
  for (uint64_t e = 0; e < assoc->n_windows; ++e) j.win[e] = {assoc->window[e], assoc->window_assoc[e]};
  std::sort(j.win.begin(), j.win.end());
  const uint32_t n = b->n_seqs;
  const uint32_t hw = pf_host_threads();
  uint32_t nt = n_threads ? n_threads : hw;
  nt = std::max(1u, std::min<uint32_t>(nt, (n + 63u) / 64u));
  const uint32_t per = (n + nt - 1) / nt;
  auto run = [&](auto&& fn) {
    if (nt == 1) { fn(0u); return; }
    std::vector<std::thread> th;
    for (uint32_t t = 0; t < nt; ++t) th.emplace_back(fn, t);
    for (auto& x : th) x.join();
  };
  std::vector<uint64_t> bytes(nt + 1, 0);
  run([&](uint32_t t) {
    const uint32_t a = std::min(n, t * per), e = std::min(n, (t + 1) * per);
    uint64_t s = 0;
    for (uint32_t i = a; i < e; ++i) s += annot_seq(j, i, nullptr);
    bytes[t] = s;
  });
  if (j.only_passing) bytes[nt] = annot_unseen(j, nullptr);
  std::vector<uint64_t> start(nt + 1, 0);
  uint64_t total = 0;
  for (uint32_t t = 0; t <= nt; ++t) { start[t] = total; total += bytes[t]; }
  *out_len = total;
  if (!out) return PF_OK;
  if (out_cap < total) return PF_ERR_NOMEM;
  run([&](uint32_t t) {
    const uint32_t a = std::min(n, t * per), e = std::min(n, (t + 1) * per);
    char* p = out + start[t];
    for (uint32_t i = a; i < e; ++i) p += annot_seq(j, i, p);
  });
  if (j.only_passing) annot_unseen(j, out + start[nt]);
  return PF_OK;
}

// ---------------------------------------------------------------------------
// Native packer: ASCII sequences -> the 2-bit / 4-bit planes of a pf_batch (what
// panfeed_b200/packer.py:pack_batch does with numpy look-up tables), host threads.
// ---------------------------------------------------------------------------
namespace {
struct Lut {
  uint8_t two[256], four[256];
  Lut() {
    memset(two, 255, sizeof two);
    memset(four, 255, sizeof four);
    two[(unsigned char)'A'] = 0; two[(unsigned char)'C'] = 1; two[(unsigned char)'G'] = 2; two[(unsigned char)'T'] = 3;
    for (int i = 0; i < 16; ++i) four[(unsigned char)kAmb[i]] = (uint8_t)i;
  }
};
const Lut kLut;

template <typename F>
void parallel_for(uint32_t n, uint32_t n_threads, F&& fn) {
  const uint32_t hw = pf_host_threads();
  uint32_t nt = n_threads ? n_threads : hw;
  nt = std::max(1u, std::min<uint32_t>(nt, (n + 4095u) / 4096u));
  if (nt == 1) { fn(0u, n); return; }
  const uint32_t per = (n + nt - 1) / nt;
  std::vector<std::thread> th;
  for (uint32_t t = 0; t < nt; ++t) th.emplace_back(fn, std::min(n, t * per), std::min(n, (t + 1) * per));
  for (auto& x : th) x.join();
}
}  // namespace

extern "C" int pf_pack_plan(const uint64_t* seq_off, uint32_t n_seqs, uint64_t* base_off, uint64_t* n_words) {
  if (!seq_off || !base_off || !n_words) return PF_ERR_INVALID;
  uint64_t pos = 0;
  for (uint32_t i = 0; i < n_seqs; ++i) {
    if (seq_off[i + 1] < seq_off[i]) return PF_ERR_INVALID;
    base_off[i] = pos;
    pos += (seq_off[i + 1] - seq_off[i] + 63) / 64 * 64;     // every sequence starts on a 64-base boundary
  }
  *n_words = pos / 32;
  return PF_OK;
}

extern "C" int pf_pack_2bit(const char* ascii, const uint64_t* seq_off, uint32_t n_seqs, const uint64_t* base_off,
                            uint64_t* packed, uint8_t* is_amb, uint32_t n_threads) {
  if (!seq_off || !base_off || !packed || !is_amb || (n_seqs && !ascii)) return PF_ERR_INVALID;
  parallel_for(n_seqs, n_threads, [&](uint32_t a, uint32_t b) {
    for (uint32_t i = a; i < b; ++i) {
      const unsigned char* s = reinterpret_cast<const unsigned char*>(ascii) + seq_off[i];
      const uint64_t len = seq_off[i + 1] - seq_off[i];
      uint64_t* out = packed + base_off[i] / 32;
      const uint64_t words = (len + 63) / 64 * 2;
      bool amb = false;
      for (uint64_t w = 0; w < words; ++w) {
        uint64_t v = 0;
        const uint64_t p0 = w * 32;
        for (uint32_t j = 0; j < 32; ++j) {
          const uint64_t p = p0 + j;
          uint32_t c = 0;                                   // padding and non-ACGT symbols pack as A
          if (p < len) {
            c = kLut.two[s[p]];
            if (c == 255u) { amb = true; c = 0; }
          }
          v = (v << 2) | c;
        }
        out[w] = v;
      }
      is_amb[i] = amb ? 1 : 0;
    }
  });
  return PF_OK;
}

extern "C" int pf_pack_4bit(const char* ascii, const uint64_t* seq_off, uint32_t n_seqs, const uint8_t* is_amb,
                            uint64_t* amb_off, uint64_t* amb_plane, uint64_t* n_amb_words, int* bad_symbol) {
  if (!seq_off || !is_amb || !amb_off || !n_amb_words) return PF_ERR_INVALID;
  if (bad_symbol) *bad_symbol = 0;
  uint64_t pos = 0;                                         // in symbols; 64-symbol blocks like the 2-bit plane
  for (uint32_t i = 0; i < n_seqs; ++i) {
    amb_off[i] = 0;
    if (!is_amb[i]) continue;
    const unsigned char* s = reinterpret_cast<const unsigned char*>(ascii) + seq_off[i];
    const uint64_t len = seq_off[i + 1] - seq_off[i];
    const uint64_t padded = (len + 63) / 64 * 64;
    amb_off[i] = pos;
    if (amb_plane) {
      uint64_t* out = amb_plane + pos / 16;
      for (uint64_t w = 0; w < padded / 16; ++w) {
        uint64_t v = 0;
        for (uint32_t j = 0; j < 16; ++j) {
          const uint64_t p = w * 16 + j;
          uint32_t c = kLut.four[(unsigned char)'A'];       // padding packs as A
          if (p < len) {
            c = kLut.four[s[p]];
            if (c == 255u) { if (bad_symbol) *bad_symbol = s[p]; return PF_ERR_UNSUPPORTED; }
          }
          v = (v << 4) | c;
        }
        out[w] = v;
      }
    }
    pos += padded;
  }
  *n_amb_words = pos / 16;
  return PF_OK;
}

// ---------------------------------------------------------------------------
// hashes_to_patterns rows (panfeed.py:183-187,217-223): id, then one field per sample:
// '0' / '1', or empty where the vector holds NaN (cluster absent, --consider-missing).
// ---------------------------------------------------------------------------
namespace {
struct OctetLut {                                  // the fields of eight samples: tab + '0' / '1', bit 0 first
  char t[256][16];
  OctetLut() {
    for (int b = 0; b < 256; ++b)
      for (int j = 0; j < 8; ++j) { t[b][2 * j] = '\t'; t[b][2 * j + 1] = (char)('0' + ((b >> j) & 1)); }
  }
};
const OctetLut kOctet;
struct NibbleLut {                                 // four samples with NaN cells: index = bits | present << 4
  char t[256][8];
  uint8_t len[256];
  NibbleLut() {
    for (int k = 0; k < 256; ++k) {
      int n = 0;
      for (int j = 0; j < 4; ++j) {
        t[k][n++] = '\t';
        if ((k >> (4 + j)) & 1) t[k][n++] = (char)('0' + ((k >> j) & 1));
      }
      len[k] = (uint8_t)n;
      for (; n < 8; ++n) t[k][n] = '\t';
    }
  }
};
const NibbleLut kNibble;
}  // namespace

extern "C" int pf_format_patterns(const uint32_t* pattern_words, uint64_t n, uint32_t stride_words,
                                  uint32_t n_samples, const char* ids, const uint32_t* present_words,
                                  uint32_t present_stride, char* out, uint64_t out_cap, uint64_t* out_len,
                                  uint32_t n_threads) {
  if (!out_len || (n && (!pattern_words || !ids)) || n_samples == 0) return PF_ERR_INVALID;
  const uint32_t W = (n_samples + 31u) / 32u;
  if (stride_words < W || (present_words && present_stride < W)) return PF_ERR_INVALID;
  *out_len = 0;
  if (n == 0) return PF_OK;
  if (n >= (1ull << 32)) return PF_ERR_INVALID;
  std::vector<uint64_t> len(n + 1, 0);
  parallel_for((uint32_t)n, n_threads, [&](uint32_t a, uint32_t b) {
    for (uint32_t i = a; i < b; ++i) {
      uint64_t cells = n_samples;
      if (present_words) {
        cells = 0;
        const uint32_t* pw = present_words + (size_t)i * present_stride;
        for (uint32_t w = 0; w < W; ++w) {
          uint32_t x = pw[w];
          if (w == W - 1 && (n_samples & 31u)) x &= (1u << (n_samples & 31u)) - 1u;
          cells += (uint64_t)__builtin_popcount(x);
        }
      }
      len[i + 1] = 24 + (uint64_t)n_samples + cells + 1;
    }
  });
  for (uint64_t i = 0; i < n; ++i) len[i + 1] += len[i];
  *out_len = len[n];
  if (!out) return PF_OK;
  if (out_cap < len[n]) return PF_ERR_NOMEM;
  parallel_for((uint32_t)n, n_threads, [&](uint32_t a, uint32_t b) {
    for (uint32_t i = a; i < b; ++i) {
      char* p = out + len[i];
      memcpy(p, ids + (size_t)i * 24, 24);
      p += 24;
      const uint32_t* bits = pattern_words + (size_t)i * stride_words;
      const uint32_t* pw = present_words ? present_words + (size_t)i * present_stride : nullptr;
      if (pw) {
        // NaN (cluster absent): an empty field.  Branch-free: the digit is always written and
        // only kept (p moves past it) where the sample is present; the byte after a dropped
        // digit is rewritten by the next tab or the closing newline of this same row
        // four samples per look-up while at least eight fields (>= 8 bytes of this row) remain:
        // the 8-byte copy never leaves the row
        uint32_t s = 0;
        for (; s + 8 <= n_samples; s += 4) {
          const uint32_t key = ((bits[s >> 5] >> (s & 31u)) & 15u) | (((pw[s >> 5] >> (s & 31u)) & 15u) << 4);
          memcpy(p, kNibble.t[key], 8);
          p += kNibble.len[key];
        }
        for (; s < n_samples; ++s) {
          const uint32_t present = (pw[s >> 5] >> (s & 31u)) & 1u;
          p[0] = '\t';
          p[1] = (char)('0' + ((bits[s >> 5] >> (s & 31u)) & 1u));
          p += 1 + present;
        }
      } else {
        // eight samples per table look-up: "\t0\t1..." of a byte of presence bits (bit 0 first)
        uint32_t s = 0;
        for (; s + 8 <= n_samples; s += 8, p += 16)
          memcpy(p, kOctet.t[(bits[s >> 5] >> (s & 31u)) & 255u], 16);
        for (; s < n_samples; ++s) {
          *p++ = '\t';
          *p++ = (char)('0' + ((bits[s >> 5] >> (s & 31u)) & 1u));
        }
      }
      *p++ = '\n';
    }
  });
  return PF_OK;
}

// ---------------------------------------------------------------------------
// kmers_to_hashes rows (panfeed.py:177 "<idx>\t\t<cluster hash>", :208 "<idx>\t<kmer>\t<hash>"):
// per cluster of the batch, in order, the header row and then its k-mer rows — the plain ones in
// alphabetical (= numeric) k-mer order, then those holding N/IUPAC symbols in the numeric order of
// their 4-bit codes.  (The reference's order inside a cluster is that of a Python dict of
// k-mers filled in window order; consumers key on the k-mer, not on the row order.)
// ---------------------------------------------------------------------------
namespace {
struct KeyedRow { uint64_t kmer; uint32_t row; };
struct QuadLut {                                   // the four bases of a byte of 2-bit codes, first base in the top bits
  char t[256][4];
  QuadLut() {
    for (int b = 0; b < 256; ++b)
      for (int j = 0; j < 4; ++j) t[b][j] = "ACGT"[(b >> (6 - 2 * j)) & 3];
  }
};
const QuadLut kQuad;

// (k-mer, row) pairs in k-mer order, ties by row.  Rows enter in ascending row order, so a STABLE
// sort on the k-mer alone keeps the ties right: least-significant-digit radix passes of 11 bits
// over the `bits` the k-mers use (6 passes for k = 31; a comparison sort of a few thousand random
// keys mispredicts every other branch).  Small inputs go to std::sort.
inline void sort_keyed(std::vector<KeyedRow>& v, std::vector<KeyedRow>& tmp, uint32_t bits) {
  const size_t n = v.size();
  if (n < 256) {
    std::sort(v.begin(), v.end(), [](const KeyedRow& a, const KeyedRow& b) {
      return a.kmer != b.kmer ? a.kmer < b.kmer : a.row < b.row;
    });
    return;
  }
  tmp.resize(n);
  KeyedRow* src = v.data();
  KeyedRow* dst = tmp.data();
  uint32_t count[2048];
  for (uint32_t shift = 0; shift < bits; shift += 11) {
    memset(count, 0, sizeof count);
    for (size_t i = 0; i < n; ++i) ++count[(src[i].kmer >> shift) & 2047u];
    uint32_t at = 0;
    for (uint32_t d = 0; d < 2048; ++d) { const uint32_t c = count[d]; count[d] = at; at += c; }
    for (size_t i = 0; i < n; ++i) dst[count[(src[i].kmer >> shift) & 2047u]++] = src[i];
    std::swap(src, dst);
  }
  if (src != v.data()) memcpy(v.data(), src, n * sizeof(KeyedRow));
}
}  // namespace

extern "C" int pf_format_kmer_rows(const pf_batch_result* r, uint32_t k, const char* tag_blob,
                                   const uint64_t* tag_off, const char* kmer_ids, uint64_t n_kmer_ids,
                                   const char* cluster_ids, uint64_t n_cluster_ids, char* out, uint64_t out_cap,
                                   uint64_t* out_len, uint64_t* cluster_off, uint32_t n_threads) {
  if (!r || !out_len || !tag_off || k == 0 || k > 64) return PF_ERR_INVALID;
  const uint64_t nc = r->n_clusters, nn = r->n_rows, nw = r->n_wide_rows, nx = r->n_xwide_rows;
  *out_len = 0;
  if (nc >= (1ull << 32) || nn >= (1ull << 32) || nw >= (1ull << 32) || nx >= (1ull << 32)) return PF_ERR_INVALID;
  if (nc && (!tag_blob || !cluster_ids || !r->cluster_pattern)) return PF_ERR_INVALID;
  if (nn && (!r->row_cluster || !r->row_kmer || !r->row_pattern || !kmer_ids)) return PF_ERR_INVALID;
  if (nw && (!r->wide_row_cluster || !r->wide_row_kmer || !r->wide_row_pattern || !kmer_ids)) return PF_ERR_INVALID;
  if (nx && (!r->xwide_row_cluster || !r->xwide_row_kmer || !r->xwide_row_pattern || !kmer_ids)) return PF_ERR_INVALID;
  if (nc == 0) return (nn || nw || nx) ? PF_ERR_INVALID : PF_OK;
  if (nn && k > 32) return PF_ERR_INVALID;             // one-word k-mers hold at most 32 bases
  // rows of every cluster (narrow rows; the wide ones, few, below).  The block engine writes the
  // rows of a cluster as ONE run (a CTA per cluster reserves them with one atomic), clusters in any
  // order: then a scan for the run boundaries is all it takes - no counting pass, no scatter of
  // row indices, which were the serial part of this function.  Anything else (a cluster in
  // several runs: the record engines, sample slices) goes through a counting sort.
  std::vector<uint32_t> first(nc + 1, 0), first_w(nc + 1, 0);
  std::vector<uint32_t> run_at(nc, 0);                  // direct: first row of cluster c's run
  std::vector<uint32_t> order;
  bool direct = true;
  {
    std::vector<uint8_t> seen(nc, 0);
    uint64_t i = 0;
    while (i < nn) {
      const uint32_t c = r->row_cluster[i];
      if (c >= nc) return PF_ERR_INVALID;
      uint64_t j = i + 1;
      while (j < nn && r->row_cluster[j] == c) ++j;
      if (seen[c]) { direct = false; break; }
      seen[c] = 1;
      run_at[c] = (uint32_t)i;
      first[c + 1] = (uint32_t)(j - i);
      i = j;
    }
  }
  if (!direct) {
    std::fill(first.begin(), first.end(), 0u);
    for (uint64_t i = 0; i < nn; ++i) {
      if (r->row_cluster[i] >= nc) return PF_ERR_INVALID;
      ++first[r->row_cluster[i] + 1];
    }
  }
  // the wide and xwide rows (few) of every cluster: a counting sort
  std::vector<uint32_t> first_x(nx ? nc + 1 : 0, 0);
  for (uint64_t i = 0; i < nw; ++i) {
    if (r->wide_row_cluster[i] >= nc || r->wide_row_pattern[i] >= n_kmer_ids) return PF_ERR_INVALID;
    ++first_w[r->wide_row_cluster[i] + 1];
  }
  for (uint64_t i = 0; i < nx; ++i) {
    if (r->xwide_row_cluster[i] >= nc || r->xwide_row_pattern[i] >= n_kmer_ids) return PF_ERR_INVALID;
    ++first_x[r->xwide_row_cluster[i] + 1];
  }
  for (uint64_t c = 0; c < nc; ++c) {
    if (r->cluster_pattern[c] >= n_cluster_ids || tag_off[c + 1] < tag_off[c]) return PF_ERR_INVALID;
    first[c + 1] += first[c];
    first_w[c + 1] += first_w[c];
    if (nx) first_x[c + 1] += first_x[c];
  }
  auto n_xrows = [&](uint64_t c) -> uint32_t { return nx ? first_x[c + 1] - first_x[c] : 0u; };
  std::vector<uint32_t> order_w(nw), order_x(nx);
  {
    std::vector<uint32_t> at_w(first_w.begin(), first_w.end() - 1);
    for (uint64_t i = 0; i < nw; ++i) order_w[at_w[r->wide_row_cluster[i]]++] = (uint32_t)i;
    if (nx) {
      std::vector<uint32_t> at_x(first_x.begin(), first_x.end() - 1);
      for (uint64_t i = 0; i < nx; ++i) order_x[at_x[r->xwide_row_cluster[i]]++] = (uint32_t)i;
    }
    if (!direct) {
      order.resize(nn);
      std::vector<uint32_t> at(first.begin(), first.end() - 1);
      for (uint64_t i = 0; i < nn; ++i) order[at[r->row_cluster[i]]++] = (uint32_t)i;
    }
  }
  // byte offsets of the clusters' texts
  std::vector<uint64_t> off(nc + 1, 0);
  for (uint64_t c = 0; c < nc; ++c) {
    const uint64_t tag = tag_off[c + 1] - tag_off[c];
    const uint64_t rows = (uint64_t)(first[c + 1] - first[c]) + (first_w[c + 1] - first_w[c]) + n_xrows(c);
    off[c + 1] = off[c] + (tag + 2 + 24 + 1) + rows * (tag + 1 + k + 1 + 24 + 1);
  }
  *out_len = off[nc];
  if (cluster_off) memcpy(cluster_off, off.data(), (nc + 1) * sizeof(uint64_t));
  if (!out) return PF_OK;
  if (out_cap < off[nc]) return PF_ERR_NOMEM;
  // clusters are taken one at a time by the threads (they differ in rows): sort, then write
  const uint32_t hw = pf_host_threads();
  uint32_t nt = n_threads ? n_threads : hw;
  nt = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(nt, (nn + nw + nx + nc + 16383) / 16384));
  std::atomic<uint32_t> next{0};
  std::atomic<uint32_t> bad_pattern{0};
  auto work = [&]() {
    std::vector<KeyedRow> keyed, scratch;
    for (;;) {
      const uint32_t c = next.fetch_add(1);
      if (c >= nc) return;
      // (k-mer, row) pairs side by side: the sort compares values it already holds instead of
      // chasing row indices into the result arrays
      const uint32_t n = first[c + 1] - first[c];
      keyed.resize(n);
      if (direct) {
        const uint32_t a = run_at[c];
        for (uint32_t j = 0; j < n; ++j) keyed[j] = KeyedRow{r->row_kmer[a + j], a + j};
      } else {
        const uint32_t* o = order.data() + first[c];
        for (uint32_t j = 0; j < n; ++j) keyed[j] = KeyedRow{r->row_kmer[o[j]], o[j]};
      }
      bool ok = true;
      for (uint32_t j = 0; j < n; ++j) ok &= r->row_pattern[keyed[j].row] < n_kmer_ids;
      if (!ok) { bad_pattern.store(1); continue; }
      sort_keyed(keyed, scratch, 2 * k);
      // the k-mers of n_words words (most significant first) of rows `o`, sorted
      auto sort_rows = [](uint32_t* o, uint32_t n_o, const uint64_t* kmers, uint32_t n_words) {
        std::sort(o, o + n_o, [&](uint32_t a, uint32_t b) {
          const uint64_t* x = kmers + (uint64_t)n_words * a;
          const uint64_t* y = kmers + (uint64_t)n_words * b;
          for (uint32_t i = 0; i < n_words; ++i)
            if (x[i] != y[i]) return x[i] < y[i];
          return a < b;
        });
      };
      uint32_t* ow = order_w.data() + first_w[c];
      const uint32_t n_w = first_w[c + 1] - first_w[c];
      sort_rows(ow, n_w, r->wide_row_kmer, 2);
      uint32_t* ox = nx ? order_x.data() + first_x[c] : nullptr;
      const uint32_t n_x = n_xrows(c);
      if (n_x) sort_rows(ox, n_x, r->xwide_row_kmer, 4);
      const char* tag = tag_blob + tag_off[c];
      const uint64_t tl = tag_off[c + 1] - tag_off[c];
      char* p = out + off[c];
      memcpy(p, tag, tl); p += tl;
      *p++ = '\t'; *p++ = '\t';
      memcpy(p, cluster_ids + (size_t)r->cluster_pattern[c] * 24, 24); p += 24;
      *p++ = '\n';
      for (uint32_t j = 0; j < n; ++j) {
        const uint32_t i = keyed[j].row;
        memcpy(p, tag, tl); p += tl;
        *p++ = '\t';
        // four bases per table look-up, first base in the top bits; the up to three letters written
        // past the k-th are overwritten by the rest of the row (a tab and a 24-character id follow)
        uint64_t u = keyed[j].kmer << (64 - 2 * k);
        for (uint32_t s4 = 0; s4 < k; s4 += 4, u <<= 8) memcpy(p + s4, kQuad.t[u >> 56], 4);
        p += k;
        *p++ = '\t';
        memcpy(p, kmer_ids + (size_t)r->row_pattern[i] * 24, 24); p += 24;
        *p++ = '\n';
      }
      auto write_rows = [&](const uint32_t* o, uint32_t n_o, const uint64_t* kmers, const uint32_t* pattern,
                            uint32_t n_words) {
        for (uint32_t j = 0; j < n_o; ++j) {
          const uint32_t i = o[j];
          memcpy(p, tag, tl); p += tl;
          *p++ = '\t';
          wide_kmer_text(kmers + (uint64_t)n_words * i, n_words, k, p);
          p += k;
          *p++ = '\t';
          memcpy(p, kmer_ids + (size_t)pattern[i] * 24, 24); p += 24;
          *p++ = '\n';
        }
      };
      write_rows(ow, n_w, r->wide_row_kmer, r->wide_row_pattern, 2);
      if (n_x) write_rows(ox, n_x, r->xwide_row_kmer, r->xwide_row_pattern, 4);
    }
  };
  if (nt == 1) work();
  else {
    std::vector<std::thread> th;
    for (uint32_t t = 0; t < nt; ++t) th.emplace_back(work);
    for (auto& x : th) x.join();
  }
  return bad_pattern.load() ? PF_ERR_INVALID : PF_OK;          // a row_pattern past the id table
}

// ---------------------------------------------------------------------------
// Pattern ids: base64 of the 16-byte MD5 digests K5 computed (panfeed.py:175-176, 206-207:
// binascii.b2a_base64(md5(vector bytes).digest())[:24]) - 24 characters, the last two '='.
// ---------------------------------------------------------------------------
extern "C" int pf_base64_ids(const uint8_t* digests, uint64_t n, char* out, uint32_t n_threads) {
  if (n && (!digests || !out)) return PF_ERR_INVALID;
  if (n >= (1ull << 32)) return PF_ERR_INVALID;
  static const char* kB64 = "ABCDEFGHIJKLMNOPQRSTUVWXYZabcdefghijklmnopqrstuvwxyz0123456789+/";
  parallel_for((uint32_t)n, n_threads, [&](uint32_t a, uint32_t b) {
    for (uint32_t i = a; i < b; ++i) {
      const uint8_t* d = digests + (size_t)i * 16;
      char* o = out + (size_t)i * 24;
      for (int g = 0; g < 5; ++g) {
        const uint32_t t = ((uint32_t)d[3 * g] << 16) | ((uint32_t)d[3 * g + 1] << 8) | d[3 * g + 2];
        o[4 * g] = kB64[t >> 18]; o[4 * g + 1] = kB64[(t >> 12) & 63]; o[4 * g + 2] = kB64[(t >> 6) & 63];
        o[4 * g + 3] = kB64[t & 63];
      }
      const uint32_t t = (uint32_t)d[15] << 16;               // the 16th byte and two bytes of padding
      o[20] = kB64[t >> 18]; o[21] = kB64[(t >> 12) & 63]; o[22] = '='; o[23] = '=';
    }
  });
  return PF_OK;
}

// ---------------------------------------------------------------------------
// --compress: the reference opens its three outputs with gzip.open(..., "wt", compresslevel=9)
// (input.py:235-259) and deflates every row on the one writer process; with --cores > 2 its
// writers interleave and the file is corrupt (SURVEY App. A).  Here a text buffer is cut into
// members of `member_bytes`, every member is deflated by a host thread into a complete gzip member
// (RFC 1952 allows any number of members per file: zcat, Python's gzip and pandas read them as one
// stream), and the members are concatenated in order.
// ---------------------------------------------------------------------------
extern "C" int pf_gzip_members(const char* text, uint64_t len, int level, uint64_t member_bytes, char* out,
                               uint64_t out_cap, uint64_t* out_len, uint32_t n_threads) {
  if (!out_len || (len && !text) || level < 0 || level > 9) return PF_ERR_INVALID;
  if (member_bytes == 0) member_bytes = 4ull << 20;
  if (member_bytes > (1ull << 30)) member_bytes = 1ull << 30;          // zlib counts in 32 bits
  const uint64_t n_members = std::max<uint64_t>(1, (len + member_bytes - 1) / member_bytes);
  if (n_members >= (1ull << 31)) return PF_ERR_INVALID;
  // worst-case size of every member (deflateBound + gzip header / trailer)
  z_stream probe;
  memset(&probe, 0, sizeof probe);
  if (deflateInit2(&probe, level, Z_DEFLATED, 15 + 16, 8, Z_DEFAULT_STRATEGY) != Z_OK) return PF_ERR_INTERNAL;
  const uint64_t bound_full = deflateBound(&probe, (uLong)std::min<uint64_t>(member_bytes, len)) + 32;
  deflateEnd(&probe);
  *out_len = n_members * bound_full;                                    // an upper bound when out == NULL
  if (!out) return PF_OK;
  std::vector<std::vector<unsigned char>> parts(n_members);
  std::vector<int> rc(n_members, Z_OK);
  const uint32_t hw = pf_host_threads();
  uint32_t nt = n_threads ? n_threads : hw;
  nt = (uint32_t)std::min<uint64_t>(nt, n_members);
  std::atomic<uint32_t> next{0};
  auto work = [&]() {
    for (;;) {
      const uint32_t m = next.fetch_add(1);
      if (m >= n_members) return;
      const uint64_t a = (uint64_t)m * member_bytes, b = std::min(len, a + member_bytes);
      z_stream z;
      memset(&z, 0, sizeof z);
      if (deflateInit2(&z, level, Z_DEFLATED, 15 + 16, 8, Z_DEFAULT_STRATEGY) != Z_OK) { rc[m] = Z_MEM_ERROR; continue; }
      parts[m].resize(deflateBound(&z, (uLong)(b - a)) + 32);
      z.next_in = reinterpret_cast<Bytef*>(const_cast<char*>(text ? text + a : ""));
      z.avail_in = (uInt)(b - a);
      z.next_out = parts[m].data();
      z.avail_out = (uInt)parts[m].size();
      const int r = deflate(&z, Z_FINISH);
      rc[m] = r == Z_STREAM_END ? Z_OK : (r == Z_OK ? Z_BUF_ERROR : r);
      parts[m].resize(z.total_out);
      deflateEnd(&z);
    }
  };
  if (nt <= 1) work();
  else {
    std::vector<std::thread> th;
    for (uint32_t t = 0; t < nt; ++t) th.emplace_back(work);
    for (auto& x : th) x.join();
  }
  uint64_t total = 0;
  for (uint64_t m = 0; m < n_members; ++m) {
    if (rc[m] != Z_OK) return PF_ERR_INTERNAL;
    total += parts[m].size();
  }
  *out_len = total;
  if (out_cap < total) return PF_ERR_NOMEM;
  uint64_t at = 0;
  for (uint64_t m = 0; m < n_members; ++m) {
    memcpy(out + at, parts[m].data(), parts[m].size());
    at += parts[m].size();
  }
  return PF_OK;
}
