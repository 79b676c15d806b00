/*
 * panfeed_b200.h — C-ABI of the B200-native k-mer streaming hot path.
 *
 * This is the drop-in boundary for the path BASELINE.json's north_star names:
 * the two Python callables of the reference that are bound with
 * functools.partial in /root/reference/panfeed/__main__.py:277-297 and invoked
 * per cluster at __main__.py:351-356 (single process) or inside worker()/
 * writer() at __main__.py:39-81:
 *
 *     cluster_cutter   /root/reference/panfeed/panfeed.py:23-113
 *     pattern_hasher   /root/reference/panfeed/panfeed.py:132-235
 *     init_presabs_vector              panfeed.py:16-20
 *
 * The reference has no FFI; every entry point below states which reference
 * lines it replaces.  Plain pointers and sizes only: no torch, no CUDA types.
 * One pf_ctx per GPU, driven by one host thread.  Every call returns PF_OK (0)
 * or a negative pf_status; pf_last_error() gives the message.  The library
 * never frees caller memory; result pointers are owned by the context and stay
 * valid until the next pf_collect()/pf_destroy() on it.
 *
 * There is no CPU fallback: without a CUDA device pf_create() fails.
 */
#ifndef PANFEED_B200_H
#define PANFEED_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* 2: pf_batch_result gained the xwide_row_* and pos_xwide_kmer fields (k = 33..64 with N/IUPAC) */
#define PF_ABI_VERSION 2

typedef enum pf_status {
  PF_OK = 0,
  PF_ERR_INVALID = -1,      /* bad argument / malformed batch              */
  PF_ERR_CUDA = -2,         /* CUDA runtime error (no device, launch, ...) */
  PF_ERR_NOMEM = -3,        /* host or device allocation failed            */
  PF_ERR_UNSUPPORTED = -4,  /* k outside 1..64; a symbol outside PF_AMB_ALPHABET (packer) */
  PF_ERR_STATE = -5,        /* call order violated                         */
  PF_ERR_INTERNAL = -6      /* device-side watchdog / invariant violated   */
} pf_status;

typedef struct pf_ctx pf_ctx;

/* Options bound into the two reference callables at __main__.py:277-297. */
typedef struct pf_params {
  uint32_t abi_version;          /* PF_ABI_VERSION                                  */
  uint32_t k;                    /* -k/--kmer-length, 1..64: up to 32 a k-mer is one 64-bit word
                                    (all engines); 33..64 two words, through the 128-bit record
                                    engine, rows come back as wide rows (2 bits per base); there
                                    a k-mer holding N/IUPAC symbols takes four words (4 bits per
                                    symbol, 256-bit records) and comes back as an xwide row     */
  uint32_t n_samples;            /* S = number of strain columns of the panaroo CSV */
  uint32_t canonical;            /* 1 unless --non-canonical (panfeed.py:69-88)     */
  uint32_t consider_missing;     /* --consider-missing (panfeed.py:16-20,192-196)   */
  uint32_t cluster_equal_filter; /* 1 iff --no-filter GIVEN: the reference runs the
                                    "same as cluster" filter only when patfilt is
                                    False (panfeed.py:202-204, __main__.py:292)     */
  uint32_t emit_positions;       /* 0: none.  Non-zero if any --targets strain exists (panfeed.py:90):
                                    1 = one 21-byte record per k-mer instance of a target sequence
                                        (pos_* arrays of the result);
                                    2 = compact: only what the input does not already determine
                                        leaves the device - the used_strand bit of every window
                                        (pos_strand_bits); pf_format_positions_compact derives the
                                        k-mer text and the coordinates from the caller's own packed
                                        plane and descriptors (panfeed.py:91-102 are affine in pos) */
  uint32_t sort_bits;            /* 0 = auto; else number of leading bits of the
                                    mixed key the radix sort orders (multiple of 8,
                                    8..64); the rest is resolved exactly in K3     */
  uint32_t mode;                 /* 0 = partition: few radix passes, then per-tile grouping
                                    in a shared-memory hash table (default);
                                    1 = full sort: LSD passes over sort_bits, then a
                                    segmented run reduction                          */
  uint32_t debug_flags;          /* bit 0: do not fuse K1 into the histogram / first pass;
                                    bit 1: no block aggregation (always go through records)  */
  double   maf;                  /* --maf, compared in float64 exactly as
                                    panfeed.py:190-200 (see pf_maf_window)          */
} pf_params;

/* One cut, gene-oriented sequence = one reference Seqinfo (classes.py:11-18,
 * built at input.py:455-459).  Bases live in the packed plane. */
typedef struct pf_seq_desc {
  uint64_t base_off;  /* index of the first base in the packed plane; multiple of 64 */
  uint32_t len;       /* number of bases                                              */
  uint32_t cluster;   /* batch-local cluster index; non-decreasing over the array     */
  uint32_t sample;    /* rank of the strain in sorted(strains) (panfeed.py:47-48);
                         non-decreasing inside a cluster                              */
  uint32_t flags;     /* PF_SEQ_* */
  int32_t  start;     /* Seqinfo.start (1-based contig coordinate of the cut window)  */
  int32_t  end;       /* Seqinfo.end                                                  */
  int32_t  offset;    /* Seqinfo.offset (upstream bases actually included)            */
  int32_t  strand;    /* +1 / -1                                                      */
  uint64_t amb_off;   /* if PF_SEQ_AMBIGUOUS: index of this sequence's first base in
                         the 4-bit plane (multiple of 32)                              */
} pf_seq_desc;        /* 48 bytes */

#define PF_SEQ_TARGET    1u  /* strain in --targets: emit positional records (panfeed.py:90-107) */
#define PF_SEQ_AMBIGUOUS 2u  /* sequence holds non-ACGT symbols (N / IUPAC)                       */

/* 4-bit symbol codes of the ambiguous plane: rank in ASCII order, so that the
 * unsigned comparison of packed k-mers equals the reference's string "<=". */
#define PF_AMB_ALPHABET "ABCDGHKMNRSTVWXY"

typedef struct pf_cluster_desc {
  uint32_t id;        /* caller's cluster number, echoed in result rows */
  uint32_t reserved;
} pf_cluster_desc;

/* One batch of whole gene clusters = the items iter_gene_clusters yields
 * (input.py:468) for those clusters. */
typedef struct pf_batch {
  const uint64_t*        packed_bases;   /* 2-bit plane: base i in word i>>5 at bits
                                            [63-2*(i&31)-1, 63-2*(i&31)], A=0 C=1 G=2 T=3 */
  uint64_t               n_words;        /* length of packed_bases                         */
  const pf_seq_desc*     seqs;
  uint32_t               n_seqs;
  const pf_cluster_desc* clusters;
  uint32_t               n_clusters;
  const uint32_t*        cluster_presence; /* n_clusters x pf_pattern_words(S) words: bit
                                              (s&31) of word (s>>5) = clusterpresab[s]
                                              (input.py:371-377)                          */
  const uint64_t*        amb_codes;      /* 4-bit plane (16 symbols per word, first symbol
                                            in the top nibble) for PF_SEQ_AMBIGUOUS
                                            sequences; NULL if none                        */
  uint64_t               n_amb_words;
} pf_batch;

/* Result of one batch.  Rows are the lines pattern_hasher writes to
 * kmers_to_hashes (panfeed.py:177,208); patterns the lines it writes to
 * hashes_to_patterns (panfeed.py:187,223); positional records the lines
 * cluster_cutter formats for kmers.tsv (panfeed.py:104-107). */
typedef struct pf_batch_result {
  /* k-mer rows that survived the MAF / same-as-cluster filters (U') */
  uint64_t        n_rows;
  const uint32_t* row_cluster;     /* pf_cluster_desc.id                                   */
  const uint64_t* row_kmer;        /* 2-bit k-mer, first base in the top used bits          */
  const uint32_t* row_count;       /* number of samples carrying it                         */
  const uint32_t* row_pattern;     /* index into the context's k-mer pattern pool           */
  /* rows whose k-mer takes two words: N/IUPAC symbols (k <= 32, 4 bits per symbol, codes of
     PF_AMB_ALPHABET) or any k-mer of 33..64 bases (2 bits per base); first symbol in the top
     used bits of [hi, lo] */
  uint64_t        n_wide_rows;
  const uint32_t* wide_row_cluster;
  const uint64_t* wide_row_kmer;   /* 2 words per row: [hi, lo]                             */
  const uint32_t* wide_row_count;
  const uint32_t* wide_row_pattern;
  /* the cluster's own row ("idx\t\tid", panfeed.py:175-187) */
  uint32_t        n_clusters;
  const uint32_t* cluster_pattern; /* index into the cluster pattern pool (int64 namespace) */
  /* patterns first seen in this batch, appended to the pools in this order */
  uint64_t        kmer_pattern_base;    /* pool index of the first new k-mer pattern        */
  uint64_t        n_new_kmer_patterns;
  const uint32_t* new_kmer_patterns;    /* n x pf_kmer_pattern_words(): presence words,
                                           then (consider_missing only) one word = index of
                                           the cluster pattern giving the NaN plane          */
  uint64_t        cluster_pattern_base;
  uint64_t        n_new_cluster_patterns;
  const uint32_t* new_cluster_patterns; /* n x pf_pattern_words(S)                           */
  /* positional records, one per k-mer instance of PF_SEQ_TARGET sequences */
  uint64_t        n_pos;
  const uint64_t* pos_kmer;        /* canonical mode: the canonical k-mer; else the forward one */
  const uint32_t* pos_seq;         /* index into pf_batch.seqs                                   */
  const int32_t*  pos_contig_start;/* contig_end  = contig_start + k (panfeed.py:91-99)          */
  const int32_t*  pos_gene_start;  /* gene_end    = gene_start + k   (panfeed.py:101-102)        */
  const uint8_t*  pos_flags;       /* bit0: reverse complement was the canonical one
                                      (used_strand = -1); bit1: two-word k-mer (N/IUPAC at
                                      k <= 32, any k-mer at k > 32), pos_kmer holds an index
                                      into pos_wide_kmer; bit2 (k > 32, k-mer holds N/IUPAC
                                      symbols; bit1 is then clear): pos_kmer holds an index
                                      into pos_xwide_kmer                                      */
  const uint64_t* pos_wide_kmer;   /* 2 words per two-word positional k-mer                   */
  uint64_t        n_pos_wide;
  /* emit_positions == 2: n_pos still counts the instances, the pos_* arrays above are NULL and
   * bit (i & 31) of pos_strand_bits[i >> 5], i = pf_seq_desc.base_off + pos, is 1 iff the reverse
   * complement was the canonical k-mer of the window starting at `pos` of that sequence
   * (used_strand = -1, panfeed.py:69-75).  Words of sequences without PF_SEQ_TARGET are
   * undefined; with canonical == 0 nothing is needed and the plane is empty. */
  const uint32_t* pos_strand_bits;
  uint64_t        n_pos_bit_words; /* pf_batch.n_words (one bit per base position), or 0      */
  /* k = 33..64: rows whose k-mer holds N/IUPAC symbols, 4 bits per symbol (codes of
     PF_AMB_ALPHABET), first symbol in the top used bits of [w0, w1, w2, w3].  Their patterns are
     numbered with those of the other rows (one pattern, one id).  Empty (0 / NULL) otherwise. */
  uint64_t        n_xwide_rows;
  const uint32_t* xwide_row_cluster;
  const uint64_t* xwide_row_kmer;  /* 4 words per row, most significant first                */
  const uint32_t* xwide_row_count;
  const uint32_t* xwide_row_pattern;
  const uint64_t* pos_xwide_kmer;  /* 4 words per positional k-mer with pos_flags bit 2       */
  uint64_t        n_pos_xwide;
} pf_batch_result;

typedef struct pf_stats {
  uint64_t batches;
  uint64_t bases;            /* N: sum of pf_seq_desc.len                           */
  uint64_t instances;        /* M: k-mer records extracted                          */
  uint64_t unique_kmers;     /* U: distinct (cluster, k-mer)                        */
  uint64_t rows;             /* U'                                                  */
  uint64_t kmer_patterns;    /* P (k-mer namespace)                                 */
  uint64_t cluster_patterns; /* P (cluster namespace)                               */
  uint32_t sort_passes;      /* radix passes used by the last batch                  */
  uint32_t launches;         /* kernels launched by the last batch                   */
  /* device time of the last batch, CUDA events on the context stream:
     h2d | K1 extract | K2 histogram | K2 onesweep passes | K3 mark runs |
     K3 count (incl. the host sync for the run count) | K3 emit + cluster-row
     dedup (incl. the host sync for the row count) | K4 dedup | d2h | K1..K4.
     Engine 2: ms_sort = kA_block_aggregate, ms_count = kB_merge (incl. the host sync). */
  float ms_h2d, ms_extract, ms_hist, ms_sort, ms_mark, ms_count, ms_reduce, ms_dedup, ms_d2h, ms_total;
  uint64_t total_launches;   /* kernels launched since pf_create                     */
  /* engine the last batch went through: 0 = records, partition mode (K1 fused into one radix
     pass + shared-memory grouping); 1 = records, full sort; 2 = block aggregation (per run of
     16 window positions the sequences of a cluster are grouped as 128-bit chunks, the distinct
     chunks are cut into k-mers and per-k-mer sample bitsets are built in shared memory: no
     records; above 1024 samples in slices of 512 samples) */
  uint32_t engine;
  uint32_t block_windows;    /* engine 2: windows per position block                  */
  uint32_t block_slots;      /* engine 2: shared-memory table slots per block         */
  uint32_t sub_batches;      /* sub-batches the last pf_submit was pipelined through (1 = not split) */
  uint64_t partial_rows;     /* engine 2: (k-mer, bitset) partial rows of the last batch */
} pf_stats;

/* ---- lifetime ---- */
int  pf_create(pf_ctx** out, int device, const pf_params* params);
void pf_destroy(pf_ctx* ctx);
const char* pf_last_error(const pf_ctx* ctx);   /* ctx may be NULL: create errors */
int  pf_abi_version(void);

/* ---- the hot path ---- */
/* pf_submit = pf_upload + pf_execute.  Host buffers of the batch must stay
 * valid until pf_upload / pf_submit returns.  A batch of >= ~400,000 sequences without
 * N/IUPAC symbols is cut by pf_submit into sub-batches of whole clusters that flow through
 * two device slots: the H2D of sub-batch j+1 and the D2H of sub-batch j-1 run under the
 * kernels of sub-batch j (results are those of the one big batch; PF_PIPELINE_SEQS sets the
 * sub-batch size, 0 disables).  For that, sequences must lie in the packed plane in array
 * order (base_off non-decreasing), as panfeed_b200/packer.py and pf_synth_fill produce. */
int pf_upload(pf_ctx* ctx, const pf_batch* batch);   /* validate, H2D, plan tiles   */
int pf_execute(pf_ctx* ctx);                         /* K1..K4 on the resident batch */
int pf_submit(pf_ctx* ctx, const pf_batch* batch);
int pf_collect(pf_ctx* ctx, pf_batch_result* out);   /* sync + D2H                  */

/* Forget all patterns (the `patterns = set()` reset of --multiple-files,
 * panfeed.py:165; also used between benchmark repetitions). */
int pf_reset_patterns(pf_ctx* ctx);

/* ---- helpers that are part of the contract ---- */
uint32_t pf_pattern_words(uint32_t n_samples);            /* ceil(S/32)               */
uint32_t pf_kmer_pattern_words(const pf_ctx* ctx);        /* + 1 if consider_missing   */
/* Integer window [lo, hi] of sample counts c that survive
 *   af = c / n; if af >= 0.5: af = 1 - af; drop if af < maf
 * evaluated in IEEE double exactly as panfeed.py:190-200.  Returns 0 and
 * lo > hi if nothing survives. */
int pf_maf_window(double maf, uint32_t n, uint32_t* lo, uint32_t* hi);
/* Device-side pool access (full bitsets of every pattern seen so far). */
int pf_patterns_export(pf_ctx* ctx, int cluster_namespace, uint64_t first,
                       uint64_t count, uint32_t* host_out);
/* K5: the reference's pattern ids.  16-byte MD5 digests of the int64 (cluster namespace,
 * panfeed.py:175) or float64 (k-mer namespace, panfeed.py:206, NaN where the cluster is
 * absent) expansion of patterns [first, first+count); id = base64(digest)[:24]. */
int pf_pattern_ids(pf_ctx* ctx, int cluster_namespace, uint64_t first, uint64_t count,
                   uint8_t* host_digests);
int pf_stats_get(pf_ctx* ctx, pf_stats* out);
/* sizeof of the ABI structs as the library was built: 0 pf_params, 1 pf_seq_desc,
 * 2 pf_cluster_desc, 3 pf_batch, 4 pf_batch_result, 5 pf_stats, 6 pf_synth_params,
 * 7 pf_cut_result; 0 for an unknown id.  Lets a binding check its own struct mirrors. */
uint32_t pf_struct_size(int which);
/* CUDA stream the context launches on, as an opaque handle (cudaStream_t). */
void* pf_stream(pf_ctx* ctx);

/* ---- native text formatting of the positional records (host threads, no device work) ----
 * The kmers.tsv rows cluster_cutter writes at panfeed.py:90-107,
 *   {idx}\t{strain}\t{gene_id}\t{contig}\t{strand}\t{truestart}\t{trueend}\t{genestart}\t{geneend}\t{used_strand}\t{kmer}\n
 * for records [first, first + count) of a result.  lead_blob / lead_off give, per sequence of the
 * batch, the first five fields with their tabs ("idx\tstrain\tgene_id\tcontig\tstrand\t");
 * seq_strand the Seqinfo.strand of every sequence (only read when canonical == 0, where every
 * record yields two rows: the forward k-mer on `strand`, its reverse complement on `-strand`).
 * out == NULL: only *out_len (bytes needed) is computed.  n_threads == 0: all host cores. */
int pf_format_positions(const pf_batch_result* result, uint32_t k, int canonical, uint64_t first,
                        uint64_t count, const char* lead_blob, const uint64_t* lead_off,
                        const int32_t* seq_strand, char* out, uint64_t out_cap, uint64_t* out_len,
                        uint32_t n_threads);

/* The same rows from the compact form (emit_positions == 2): for sequences [seq_first, seq_first +
 * seq_count) of `batch` that carry PF_SEQ_TARGET, in array order, every window in ascending
 * position.  The k-mer text comes from the batch's own planes (the 4-bit plane for sequences
 * flagged PF_SEQ_AMBIGUOUS), the coordinates from the descriptors:
 *   contig_start = strand > 0 ? start + pos : end - pos - k,  gene_start = pos - offset,
 * used_strand from strand_bits (canonical) or +-pf_seq_desc.strand (two rows, canonical == 0;
 * strand_bits may then be NULL).  lead_blob / lead_off index the sequences of the batch. */
int pf_format_positions_compact(const pf_batch* batch, const uint32_t* strand_bits, uint32_t k,
                                int canonical, uint32_t seq_first, uint32_t seq_count,
                                const char* lead_blob, const uint64_t* lead_off, char* out,
                                uint64_t out_cap, uint64_t* out_len, uint32_t n_threads);

/* The hashes_to_patterns rows of n patterns (panfeed.py:183-187,217-223): ids (n x 24 chars,
 * e.g. from pf_pattern_ids + base64), then per sample a tab and '0' / '1' — or nothing where
 * present_words (n x present_stride words, bit s = sample s's cluster is present; NULL = all
 * present) has a 0: the reference writes NaN cells as empty fields with --consider-missing. */
int pf_format_patterns(const uint32_t* pattern_words, uint64_t n, uint32_t stride_words,
                       uint32_t n_samples, const char* ids, const uint32_t* present_words,
                       uint32_t present_stride, char* out, uint64_t out_cap, uint64_t* out_len,
                       uint32_t n_threads);

/* The kmers_to_hashes rows of a batch (panfeed.py:177 "<idx>\t\t<cluster hash>", :208
 * "<idx>\t<kmer>\t<hash>"): for every cluster of `result`, in order, the header row and then its
 * k-mer rows — the plain ones in alphabetical k-mer order, then the wide ones, then the xwide ones
 * (k > 32 with N/IUPAC symbols), each group sorted (the reference's order inside a cluster is the
 * insertion order of a Python dict; consumers key on the k-mer).  tag_blob + tag_off[c .. c+1]:
 * the text of the first column for cluster c.
 * kmer_ids / cluster_ids: 24 characters per pattern, indexed by row_pattern / cluster_pattern
 * (all patterns numbered so far, e.g. from pf_pattern_ids + base64).  cluster_off (may be NULL):
 * [n_clusters + 1] byte offsets of every cluster's text.  out == NULL: only *out_len (and
 * cluster_off).  Uses row_*, wide_row_*, xwide_row_*, cluster_pattern and n_clusters of the result. */
int pf_format_kmer_rows(const pf_batch_result* result, uint32_t k, const char* tag_blob,
                        const uint64_t* tag_off, const char* kmer_ids, uint64_t n_kmer_ids,
                        const char* cluster_ids, uint64_t n_cluster_ids, char* out,
                        uint64_t out_cap, uint64_t* out_len, uint64_t* cluster_off,
                        uint32_t n_threads);

/* --compress (input.py:235-259: gzip.open(..., "wt", compresslevel=9) on the three outputs):
 * `text` is cut into members of member_bytes (0 = 4 MiB), every member becomes a complete gzip
 * member deflated at `level` by a host thread, the members are concatenated in order — a valid
 * gzip file or a piece of one (RFC 1952: any number of members; zcat / Python gzip / pandas read
 * them as one stream).  len == 0 yields one empty member.  out == NULL: *out_len = an upper bound
 * of the size; otherwise *out_len = the bytes written (PF_ERR_NOMEM if out_cap is too small). */
int pf_gzip_members(const char* text, uint64_t len, int level, uint64_t member_bytes, char* out,
                    uint64_t out_cap, uint64_t* out_len, uint32_t n_threads);

/* ---- native packer (host threads): ASCII sequences -> the planes of a pf_batch ----
 * What the feeder has after cutting (input.py:455-459: Seqinfo.sequence, upper case) goes into
 * the 2-bit plane; sequences holding N/IUPAC symbols are flagged and additionally packed into
 * the 4-bit plane.  ascii / seq_off: the sequences of the batch back to back, sequence i =
 * [seq_off[i], seq_off[i+1]).  pf_pack_plan lays the sequences out (base_off[i], multiples of 64;
 * n_words of the 2-bit plane); pf_pack_2bit fills the plane and is_amb[i]; pf_pack_4bit lays out
 * and fills the 4-bit plane (amb_plane == NULL: only amb_off / n_amb_words), returning
 * PF_ERR_UNSUPPORTED and the offending byte in *bad_symbol for symbols outside PF_AMB_ALPHABET. */
int pf_pack_plan(const uint64_t* seq_off, uint32_t n_seqs, uint64_t* base_off, uint64_t* n_words);
int pf_pack_2bit(const char* ascii, const uint64_t* seq_off, uint32_t n_seqs, const uint64_t* base_off,
                 uint64_t* packed, uint8_t* is_amb, uint32_t n_threads);
int pf_pack_4bit(const char* ascii, const uint64_t* seq_off, uint32_t n_seqs, const uint8_t* is_amb,
                 uint64_t* amb_off, uint64_t* amb_plane, uint64_t* n_amb_words, int* bad_symbol);

/* ---- synthetic pangenome (SURVEY.md §8(d)), generated on the device ---- */
typedef struct pf_synth_params {
  uint64_t seed;
  uint32_t n_samples;
  uint32_t n_clusters;       /* clusters in this batch                              */
  uint32_t first_cluster;    /* global index of the first (for the RNG stream)      */
  uint32_t gene_len;         /* ancestral length incl. flanks (e.g. 1200)           */
  uint32_t n_founders;       /* 8                                                   */
  float    founder_div;      /* 0.01                                                */
  float    private_div;      /* 0.001                                               */
  float    core_fraction;    /* 0.6: probability that a cluster is core (present w.p. 0.99) */
  float    paralog_rate;     /* 0.01                                                */
  uint32_t total_clusters;   /* C of the whole pangenome (core/accessory split)     */
  uint32_t all_targets;      /* 1: flag every sequence PF_SEQ_TARGET                */
} pf_synth_params;
/* Sizes of the batch pf_synth_fill will write. */
int pf_synth_plan(const pf_synth_params* p, uint32_t* n_seqs, uint64_t* n_words);
/* Fill caller-provided HOST buffers (seqs, clusters, presence, packed bases)
 * with a deterministic synthetic batch; bases are generated on `device`. */
int pf_synth_fill(int device, const pf_synth_params* p, pf_seq_desc* seqs,
                  pf_cluster_desc* clusters, uint32_t* presence,
                  uint64_t* packed_bases);

/* ---- multi-GPU global pattern dedup (SURVEY.md §8(e)) ----
 * Clusters are sharded over ranks; the only global state is the reference's
 * `patterns` set (__main__.py:70).  Owner of a pattern = hash(bitset) % world.
 * The caller moves the buffers between ranks (NCCL all-to-all on the context's
 * stream, see pf_stream); all pointers in this group are DEVICE pointers owned
 * by the caller unless named *_host.  Order of one namespace:
 *   pf_exchange_pack      local patterns bucketed by owner -> send buffer; bucket sizes on the host
 *                         (the one host sync: they are the split sizes of the all-to-all)
 *   [all-to-all of the keys]
 *   pf_exchange_dedup     owner side: unique index of every received key (bit 31 set on the first
 *                         copy of a pattern: its sender is the one that writes the pattern row),
 *                         the number of unique keys to a device word (asynchronous) and/or the host
 *   [all-gather of the unique counts -> exclusive scan = owner_base; reverse all-to-all of the indices]
 *   pf_exchange_unpack    local_to_global[i] = owner_base[owner(i)] + unique index; writer[i] = bit 31
 *                         (asynchronous on the context's stream) */
int pf_exchange_pack(pf_ctx* ctx, int cluster_namespace, uint32_t world,
                     const uint32_t* mask_remap_dev, /* local->global cluster-pattern ids, or NULL */
                     uint32_t* send_words_dev, uint64_t capacity_patterns,
                     uint64_t* counts_host /* [world] */);
int pf_exchange_dedup(pf_ctx* ctx, int cluster_namespace,
                      const uint32_t* recv_words_dev, uint64_t n_recv,
                      uint32_t* recv_unique_index_dev,
                      uint32_t* n_unique_dev /* one word, may be NULL */,
                      uint64_t* n_unique_host /* may be NULL: then the call does not synchronise */,
                      uint32_t keep_unique_keys /* 1: keep the owner-side unique keys (n_unique x words
                                                   of device memory) for pf_exchange_unique_export */);
int pf_exchange_unique_count(pf_ctx* ctx, int cluster_namespace, uint64_t* n_unique_host);
int pf_exchange_unique_export(pf_ctx* ctx, int cluster_namespace,
                              uint32_t* host_out /* n_unique x words */);
int pf_exchange_unpack(pf_ctx* ctx, int cluster_namespace,
                       const uint32_t* returned_ids_dev, /* in send order */
                       const uint32_t* owner_base_dev /* [world] or NULL (ids already global) */,
                       uint32_t* local_to_global_dev /* [n local patterns] */,
                       uint8_t* writer_dev /* [n local patterns] or NULL */);

/* The same exchange over peer memory (ranks of one box): the keys go straight from the local
 * pattern pool into the OWNER's receive buffer with NVLink peer stores - no send buffer, no
 * all-to-all of the keys.  Order of one namespace:
 *   pf_exchange_classify     owners and bucket positions of the local patterns; bucket sizes on
 *                            the host (one sync)
 *   [all-gather of every rank's bucket sizes: rank r's bucket for owner o starts at row
 *    sum of counts[r' -> o] over r' < r of o's receive buffer, which holds sum over all r']
 *   pf_exchange_recv_buffer  this rank's receive buffer (library-owned, grows; a growth
 *                            invalidates earlier handles: peers close their mappings first) and
 *                            its CUDA IPC handle, which the caller passes to the peers
 *   pf_exchange_open_peer    map a peer's receive buffer (cudaIpcOpenMemHandle); cache the result
 *   pf_exchange_scatter      every local key to owner_buffer[owner] + (row0[owner] + position);
 *                            asynchronous on the context's stream
 *   [a barrier of all ranks on that stream: every scatter has completed]
 *   pf_exchange_dedup on the receive buffer, then as above */
int pf_exchange_classify(pf_ctx* ctx, int cluster_namespace, uint32_t world,
                         const uint32_t* mask_remap_dev, uint64_t* counts_host /* [world] */);
int pf_exchange_recv_buffer(pf_ctx* ctx, int cluster_namespace, uint64_t min_rows, void** dev_ptr,
                            uint64_t* capacity_rows, unsigned char* ipc_handle_out /* 64 bytes */);
int pf_exchange_open_peer(pf_ctx* ctx, const unsigned char* ipc_handle /* 64 bytes */, void** mapped);
int pf_exchange_close_peer(pf_ctx* ctx, void* mapped);
int pf_exchange_scatter(pf_ctx* ctx, int cluster_namespace, uint32_t world,
                        const uint32_t* mask_remap_dev, void* const* dest_ptrs /* [world]: device
                        pointers, the own buffer or pf_exchange_open_peer mappings */,
                        const uint64_t* dest_row0 /* [world] */);

/* Pattern ids as text (host threads): out[24 * i ..] = base64 of the 16-byte digest i, as
 * binascii.b2a_base64(md5(...).digest())[:24] gives them (panfeed.py:175-176, 206-207). */
int pf_base64_ids(const uint8_t* digests /* [n][16], pf_pattern_ids */, uint64_t n, char* out /* [n][24] */,
                  uint32_t n_threads);

/* ---- native feeder (host threads of the caller): GFF3 + FASTA -> cut sequences of a cluster ----
 * Replaces, for the feeding side of the path, the reference's parse_gff (input.py:274-332), its
 * pyfaidx contigs (input.py:262-266) and the per-strain loop of iter_gene_clusters
 * (input.py:335-468, window arithmetic :413-446).  Genomes are parsed once; a cluster is cut by one
 * call into ASCII sequences + descriptors that pf_pack_plan / pf_pack_2bit / pf_pack_4bit read as
 * they are.  Semantics are those of the reference line by line (malformed GFF lines are skipped
 * and counted, a repeated feature id / contig name replaces the earlier one, slices clamp like
 * Python's, the minus strand is reverse-complemented with pyfaidx's table). */
typedef struct pf_feeder pf_feeder;

typedef struct pf_cut_result {
  uint32_t n_seqs;
  const char*     ascii;      /* the sequences, back to back (upper case as read)                    */
  const uint64_t* seq_off;    /* [n_seqs + 1] offsets into ascii                                     */
  const uint32_t* cell;       /* [n_seqs] index of the panaroo cell (= strain) the sequence is from  */
  const uint32_t* feature;    /* [n_seqs] feature index inside that strain's genome (pf_feeder_feature) */
  const int32_t*  start;      /* Seqinfo.start / end / offset / strand (classes.py:11-18)            */
  const int32_t*  end;
  const int32_t*  offset;
  const int32_t*  strand;
  uint32_t n_missing;         /* feature ids (kind 0) / contigs (kind 1) that were not found:        */
  const uint32_t* missing_cell;   /* the reference logs a warning and skips the gene (input.py:396-411) */
  const uint8_t*  missing_kind;
  const char*     missing_text;   /* names, back to back                                             */
  const uint64_t* missing_off;    /* [n_missing + 1]                                                 */
} pf_cut_result;

int  pf_feeder_create(pf_feeder** out);
void pf_feeder_destroy(pf_feeder* f);
const char* pf_feeder_last_error(const pf_feeder* f);
/* One genome: CDS features with an ID= attribute from the GFF3 (up to "##FASTA"), contigs from
 * fasta_path or, if NULL, from the GFF's ##FASTA section.  Returns the genome's index (>= 0, in
 * order of the calls) or a negative PF_ERR_*.  skipped_lines (may be NULL): malformed GFF lines. */
int  pf_feeder_add_genome(pf_feeder* f, const char* name, const char* gff_path, const char* fasta_path,
                          uint32_t* skipped_lines);
int  pf_feeder_add_genome_text(pf_feeder* f, const char* name, const char* gff, uint64_t gff_len,
                               const char* fasta /* NULL: ##FASTA section of gff */, uint64_t fasta_len,
                               uint32_t* skipped_lines);
/* n genomes, read and parsed on host threads, appended in the order given; returns the index of
 * the first (the others follow).  fasta_paths NULL, or NULL entries: the GFF's ##FASTA section. */
int  pf_feeder_add_genomes(pf_feeder* f, uint32_t n, const char* const* names, const char* const* gff_paths,
                           const char* const* fasta_paths, uint32_t* skipped_lines, uint32_t n_threads);
int  pf_feeder_genome_info(const pf_feeder* f, uint32_t genome, uint32_t* n_features, uint32_t* n_contigs,
                           uint64_t* n_bases);
int  pf_feeder_feature(const pf_feeder* f, uint32_t genome, uint32_t feature, const char** id,
                       const char** contig, int64_t* start, int64_t* end, int32_t* strand);
/* Contig `contig` of a genome (in order of first appearance): its name, its length and whether it
 * is used IN PLACE - a FASTA record whose lines all have one width (a shorter last one allowed)
 * stays where it lies in the mapped file text, case folded when a window is cut; any other record
 * is copied line by line, stripped and upper-cased as the reference's pyfaidx contigs are. */
int  pf_feeder_contig(const pf_feeder* f, uint32_t genome, uint32_t contig, const char** name,
                      uint64_t* n_bases, uint32_t* in_place);
/* One cluster: cells_blob = the n_cells panaroo cells (';'-separated feature ids) of the strains
 * that have the cluster, joined with '\n'; genome[i] = genome index of cell i.  The result (valid
 * until the next call on this feeder) lists the sequences cell by cell, genes in cell order. */
int  pf_feeder_cut(pf_feeder* f, uint32_t n_cells, const uint32_t* genome, const char* cells_blob,
                   uint64_t cells_len, int32_t up, int32_t down, int32_t down_start_codon,
                   pf_cut_result* out);

/* The same cut with the sequences packed on the spot (host threads; n_threads 0 = all cores):
 * the windows go from the contigs straight into the planes of a pf_batch - the layout of
 * pf_pack_plan (every sequence on a 64-base boundary), the codes of pf_pack_2bit and, for
 * sequences holding N / IUPAC symbols, pf_pack_4bit - without the ASCII copy in between.
 * out->ascii is NULL; out->seq_off still gives the lengths.  A symbol outside the 16 IUPAC codes:
 * PF_ERR_UNSUPPORTED, planes->bad_symbol names it.  Valid until the next call on this feeder. */
typedef struct pf_cut_planes {
  const uint64_t* packed;     /* 2-bit plane, n_words words of 32 bases                              */
  uint64_t n_words;
  const uint64_t* base_off;   /* [n_seqs] first base of a sequence in the plane                      */
  const uint8_t*  is_amb;     /* [n_seqs] 1: the sequence holds a symbol outside ACGT                 */
  const uint64_t* amb_plane;  /* 4-bit plane of the flagged sequences, or NULL                       */
  uint64_t n_amb_words;
  const uint64_t* amb_off;    /* [n_seqs] first symbol in the 4-bit plane (0 when not flagged)       */
  int32_t bad_symbol;
} pf_cut_planes;
int  pf_feeder_cut_packed(pf_feeder* f, uint32_t n_cells, const uint32_t* genome, const char* cells_blob,
                          uint64_t cells_len, int32_t up, int32_t down, int32_t down_start_codon,
                          uint32_t n_threads, pf_cut_result* out, pf_cut_planes* planes);

/* ---- the pangenome table (host threads): panaroo's gene_presence_absence.csv ----
 * What the reference reads with pd.read_csv(path, sep=",", index_col=0, low_memory=False)
 * .drop(columns=["Non-unique Gene name", "Annotation"]) (input.py:198-201) and walks with
 * iterrows() (input.py:352).  The file is mapped, a cell is an (offset, length) into it; RFC-4180
 * quoting, blank lines skipped, short rows padded with missing cells; a cell that is empty or
 * one of na_values (the caller passes pandas' STR_NA_VALUES) is absent.  Escaped quotes inside a
 * row label or a kept cell are refused (PF_ERR_INVALID + pf_table_last_error). */
typedef struct pf_table pf_table;
int  pf_table_create(pf_table** out);
void pf_table_destroy(pf_table* t);
const char* pf_table_last_error(const pf_table* t);
int  pf_table_load(pf_table* t, const char* path, const char* const* drop_columns, uint32_t n_drop,
                   const char* const* na_values, uint32_t n_na, uint32_t n_threads);
int  pf_table_shape(const pf_table* t, uint64_t* n_rows, uint32_t* n_cols);
/* names back to back with their offsets [n + 1]: the kept columns (row_labels 0) or the row labels */
int  pf_table_names(const pf_table* t, int row_labels, const char** blob, const uint64_t** off);
int  pf_table_row_counts(const pf_table* t, uint32_t* n_present /* [n_rows] */);
/* The cells of rows[0 .. n_sel) with the columns in the order col_order (col_order[j] = table
 * column at position j, NULL = table order): present[i * n_cols + j] (may be NULL) and the
 * present cells row by row joined with '\n' - the cells_blob of pf_feeder_cut.  blob and present
 * NULL: sizing only (blob_len, n_cells). */
int  pf_table_cells(const pf_table* t, const uint64_t* rows, uint64_t n_sel, const uint32_t* col_order,
                    uint8_t* present, char* blob, uint64_t blob_cap, uint64_t* blob_len, uint64_t* n_cells);

/* ---- row filter over the TSV outputs (host threads): the scans of the post-GWAS joins ----
 * panfeed-get-clusters / panfeed-get-kmers (get_clusters.py:90-101, get_kmers.py:108-145) keep the
 * rows of kmers_to_hashes.tsv whose hashed_pattern, and of kmers.tsv whose cluster, is in a set
 * (pandas, 100,000 rows at a time).  pf_tsv_filter maps the file, scans pieces of it on host
 * threads and returns the matching lines in file order ('\n'-terminated, header excluded when
 * skip_header) in a buffer the caller releases with pf_free.  column: 0-based, tab-separated,
 * no quoting.  keys: n_keys strings back to back (keys_blob, key_off[n_keys + 1]). */
int  pf_tsv_filter(const char* path, uint32_t column, const char* keys_blob, const uint64_t* key_off,
                   uint64_t n_keys, int skip_header, char** out, uint64_t* out_len, uint64_t* n_rows,
                   uint32_t n_threads);
void pf_free(void* p);

#ifdef __cplusplus
}
#endif
#endif /* PANFEED_B200_H */
