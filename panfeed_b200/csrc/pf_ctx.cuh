// pf_ctx.cuh — context and batch state, device-side planning kernels, error / buffer helpers.
// Part of libpanfeed_b200.so's single translation unit: included once, in order, by pf_api.cu.

namespace pf {
// ---- planning helpers that run on the device (tile lists are pure functions of the
//      per-cluster record ranges; generating them there saves host loops and H2D) -------
__global__ void plan_expand_tiles(const ClusterDev* __restrict__ clusters, uint32_t n_clusters,
                                  const uint32_t* __restrict__ tile_base, uint32_t tile_size,
                                  int width /* record range: 0 narrow, 1 wide, 2 256-bit */,
                                  TileDev* __restrict__ tiles) {
  const uint32_t c = blockIdx.x;
  if (c >= n_clusters) return;
  const ClusterDev& cd = clusters[c];
  const uint32_t lo = width == 2 ? cd.xrec_start : width ? cd.wrec_start : cd.rec_start;
  const uint32_t hi = width == 2 ? cd.xrec_end : width ? cd.wrec_end : cd.rec_end;
  const uint32_t first = tile_base[c];
  const uint32_t n = (hi - lo + tile_size - 1) / tile_size;
  for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
    TileDev t;
    t.start = lo + i * tile_size;
    t.count = min(tile_size, hi - t.start);
    t.seg = c;
    t.first_tile = first;
    tiles[first + i] = t;
  }
}
__global__ void plan_seq_rec_off(const SeqDev* __restrict__ seqs, uint32_t n_seqs, uint32_t total,
                                 uint32_t* __restrict__ out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_seqs) out[i] = seqs[i].rec_off;
  else if (i == n_seqs) out[i] = total;
}
// Counter read-back without a copy engine: the D2H engine may be busy with the previous
// batch's rows, and a 64-byte memcpy queued behind them would stall the pipeline's host side.
// `dst` is pinned host memory (device-accessible under UVA).
__global__ void mirror_counters(uint32_t* __restrict__ dst, const uint32_t* __restrict__ src, uint32_t n) {
  if (threadIdx.x < n) dst[threadIdx.x] = src[threadIdx.x];
  __threadfence_system();
}
// pipelined submit: positional records of a sub-batch index its own sequences / wide k-mers
__global__ void pos_rebase(uint32_t* __restrict__ pos_seq, uint64_t* __restrict__ pos_kmer,
                           const uint8_t* __restrict__ pos_flags, uint32_t n, uint32_t seq_base,
                           uint64_t wide_base) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  pos_seq[i] += seq_base;
  if (wide_base && (pos_flags[i] & 2u)) pos_kmer[i] += wide_base;
}
// sequence holding the first record of every tile (last s with rec_off[s] <= start, non-empty)
__global__ void plan_tile_first_seq(const TileDev* __restrict__ tiles, uint32_t n_tiles,
                                    const uint32_t* __restrict__ seq_rec_off, uint32_t n_seqs,
                                    uint32_t* __restrict__ out) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t > n_tiles) return;
  if (t == n_tiles) { out[t] = n_seqs ? n_seqs - 1 : 0; return; }
  const uint32_t r = tiles[t].start;
  uint32_t lo = 0, hi = n_seqs;                   // first index in [0, n_seqs] with rec_off > r
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (seq_rec_off[mid] <= r) lo = mid + 1; else hi = mid;
  }
  out[t] = lo ? lo - 1 : 0;
}
}  // namespace pf

namespace {

thread_local std::string g_create_error;

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};
struct PinBuf {
  void* p = nullptr;
  size_t cap = 0;
  template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

// The pattern pools only ever grow, up to tens of GB (50,000 samples: 6 kB per pattern).  Growing a
// cudaMalloc'ed array means allocate + copy + free of everything numbered so far, and cudaFree
// stalls the whole device; instead the pool reserves a range of virtual addresses once and maps
// more physical memory behind what is already there (CUDA virtual memory management, driver entry
// points fetched through the runtime: no link-time dependency on libcuda).  Pointers into the pool
// stay valid, nothing is copied.  Falls back to the copying DevBuf if the driver refuses.
struct PoolBuf : DevBuf {
  bool vmm = false;
  CUdeviceptr base = 0;
  size_t reserved = 0;
  std::vector<std::pair<CUmemGenericAllocationHandle, size_t>> chunks;
  // growth ahead of need on the context's grower thread (mapping memory costs 10-30 ms in a process
  // with NCCL peers): `cap` is what the calling thread may use, `growing` marks a mapping in flight
  // that raises it when joined
  bool growing = false;
  size_t grown_cap = 0;
  bool big_step_done = false;
};

struct PatternSpace {
  uint32_t key_words = 0;
  PoolBuf pool;           // n x key_words
  uint64_t n = 0;         // committed patterns
  DevBuf table;           // table_size x u32
  uint32_t table_size = 0;
  // exchange state
  DevBuf x_owner, x_pos, x_perm, x_counts, x_unique, x_table, x_rep, x_slot, x_winner, x_recv;
  uint64_t x_n_unique = 0;
  bool x_have_unique = false;           // x_unique holds the owner-side unique keys of the last exchange
  bool x_unique_pending = false;        // x_n_unique still sits in the pinned mirror below
  const uint32_t* x_unique_mirror = nullptr;
};

struct WidthState {       // per key width (narrow u64 / wide Key128 / Key256)
  DevBuf keys[2], vals[2];
  DevBuf tiles, seg_start, seg_hist, lookback, cursors;
  DevBuf ltiles, tile_first_run;     // partition mode: 2048-record tiles of the local reduce
  PinBuf h_tiles, h_seg_start, h_ltiles;       // h_tiles / h_ltiles now hold per-cluster tile bases
  DevBuf d_tile_base, d_ltile_base;
  uint32_t n_tiles = 0, n_ltiles = 0, max_seg = 0;
  uint32_t n_records = 0;
  uint32_t n_runs = 0;
  uint32_t n_rows = 0;
  int sort_bits = 0, passes = 0;
  int final_buf = 0;      // which of keys[]/vals[] holds the sorted records
};

enum Ev { EV_START, EV_EXTRACT, EV_HIST, EV_SORT, EV_MARK, EV_COUNTED, EV_REDUCE, EV_DEDUP, EV_END, EV_COUNT };

}  // namespace

// Everything that belongs to ONE batch of whole clusters: what pf_upload builds, the record /
// row buffers of that batch and its result arrays on the device.  A context holds three of these
// so that the uploads of sub-batches j+1 and j+2 and the D2H of sub-batch j-1 can overlap the
// kernels of sub-batch j (pf_submit on a large batch; see submit_pipelined).
struct BatchState {
  bool have_batch = false, executed = false;
  uint32_t n_seqs = 0, n_clusters = 0, n_wide_seqs = 0;
  uint64_t n_words = 0, n_amb_words = 0, n_bases = 0;
  uint32_t n_pos = 0, n_pos_wide = 0, n_pos_xwide = 0;
  PinBuf h_seqs, h_clusters, h_wide_seqs;
  PinBuf h_xpos_slot;            // k > 32: first positional 256-bit slot of every listed ambiguous sequence
  DevBuf d_bases, d_amb, d_ambbits, d_seqs, d_clusters, d_wide_seqs, d_presence, d_xpos_slot;
  WidthState nar, wid;
  WidthState xwd;                // k > 32: the windows holding N/IUPAC symbols, Key256 records
  // rows (narrow first, then wide, then 256-bit)
  DevBuf d_row_cluster, d_row_kmer, d_wrow_kmer, d_xrow_kmer, d_row_count, d_row_pattern;
  DevBuf d_cl_pattern;
  DevBuf d_pos_kmer, d_pos_seq, d_pos_cstart, d_pos_gstart, d_pos_flags, d_pos_wide, d_pos_xwide;
  DevBuf d_pos_bits;             // compact positional form: used_strand bit plane, indexed like d_bases
  DevBuf d_seq_rec_off, d_tile_first_seq;
  PinBuf h_seq_rec_off, h_tile_first_seq;
  std::vector<std::pair<uint32_t, uint32_t>> nar_ranges;   // narrow record range of every cluster
  uint32_t n_items = 0;          // (cluster, block) work items of the batch (block aggregation)
  DevBuf d_seq_lite, d_cblk, d_item_base, d_item_cluster, d_plan_total, d_bsum_slot, d_slice_seq, d_item_desc;
  PinBuf h_plan;
  uint64_t kp_base = 0, cp_base = 0;   // pool sizes before the batch
  bool rows_prefetched = false;
  uint64_t row_cap = 0;          // capacity of the row arrays above
  cudaEvent_t ev[EV_COUNT]{};    // stage timestamps of the batch's pf_execute
  cudaEvent_t ev_h2d[2]{};       // around the batch's H2D
  // pipelined submit: the upload has been enqueued / the kernels are done with the slot's inputs /
  // the slot's result arrays have left the device
  cudaEvent_t ev_up_done = nullptr, ev_exec_end = nullptr, ev_out_done = nullptr;
  PinBuf h_done;                 // pinned mirror of the batch's new k-mer pattern count (K4)
  // device-side planning ("lite" upload, plan_from_raw): the caller's descriptors as uploaded, the
  // totals the kernel computed, and what a later fall-back to the record engine needs to re-plan
  // the batch on the host
  bool lite = false;
  DevBuf d_raw, d_lite_tot;
  PinBuf h_raw, h_lite_tot;
  std::vector<pf_cluster_desc> lite_clusters;
  std::vector<uint32_t> lite_presence;
  const pf_seq_desc* lite_src = nullptr;     // caller's descriptors of the sub-range (valid during the call)
  uint32_t lite_c0 = 0;                      // rebasing of the sub-range (cluster index, first base)
  uint64_t lite_b0 = 0;
};


// Host worker threads that stay alive with the context: the per-sequence planning of an upload
// runs on them (a std::thread per chunk and phase cost more than the planning of a sub-batch),
// and one of them enqueues the uploads of the pipelined submit.
class WorkerPool {
 public:
  ~WorkerPool() {
    { std::lock_guard<std::mutex> lk(mu_); stop_ = true; }
    cv_go_.notify_all();
    for (auto& t : th_) t.join();
  }
  // fn(t) for t in [0, n), on up to n - 1 workers and the calling thread; returns when all ran
  void parallel(unsigned n, const std::function<void(unsigned)>& fn) {
    if (n <= 1) { if (n) fn(0); return; }
    std::lock_guard<std::mutex> one(call_mu_);
    {
      std::lock_guard<std::mutex> lk(mu_);
      while (th_.size() + 1 < n) th_.emplace_back([this]() { worker(); });
      fn_ = &fn; n_tasks_ = n; next_ = 0; done_ = 0; ++gen_;
    }
    cv_go_.notify_all();
    run_tasks();
    std::unique_lock<std::mutex> lk(mu_);
    cv_done_.wait(lk, [&]() { return done_ == n_tasks_; });
    fn_ = nullptr;
  }

 private:
  void run_tasks() {
    std::unique_lock<std::mutex> lk(mu_);
    while (fn_ && next_ < n_tasks_) {
      const unsigned t = next_++;
      const std::function<void(unsigned)>* f = fn_;
      lk.unlock();
      (*f)(t);
      lk.lock();
      if (++done_ == n_tasks_) cv_done_.notify_all();
    }
  }
  void worker() {
    uint64_t seen = 0;
    for (;;) {
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_go_.wait(lk, [&]() { return stop_ || gen_ != seen; });
        if (stop_) return;
        seen = gen_;
      }
      run_tasks();
    }
  }
  std::vector<std::thread> th_;
  std::mutex mu_, call_mu_;
  std::condition_variable cv_go_, cv_done_;
  const std::function<void(unsigned)>* fn_ = nullptr;
  unsigned n_tasks_ = 0, next_ = 0, done_ = 0;
  uint64_t gen_ = 0;
  bool stop_ = false;
};

// One thread that runs one job at a time, started and joined by its owner.
class AsyncWorker {
 public:
  ~AsyncWorker() {
    { std::lock_guard<std::mutex> lk(mu_); stop_ = true; }
    cv_.notify_all();
    if (th_.joinable()) th_.join();
  }
  void start(std::function<void()> job) {
    std::unique_lock<std::mutex> lk(mu_);
    cv_.wait(lk, [&]() { return !busy_; });
    if (!th_.joinable()) th_ = std::thread([this]() { loop(); });
    job_ = std::move(job);
    busy_ = true;
    cv_.notify_all();
  }
  void join() {
    std::unique_lock<std::mutex> lk(mu_);
    cv_.wait(lk, [&]() { return !busy_; });
  }

 private:
  void loop() {
    std::unique_lock<std::mutex> lk(mu_);
    for (;;) {
      cv_.wait(lk, [&]() { return stop_ || busy_; });
      if (stop_) return;
      std::function<void()> job = std::move(job_);
      lk.unlock();
      job();
      lk.lock();
      busy_ = false;
      cv_.notify_all();
    }
  }
  std::thread th_;
  std::mutex mu_;
  std::condition_variable cv_;
  std::function<void()> job_;
  bool busy_ = false, stop_ = false;
};

struct pf_ctx : BatchState {
  pf_params prm{};
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;   // D2H of finished row arrays while K4 still runs
  cudaStream_t up_stream = nullptr;     // H2D of the next sub-batch while the current one computes
  cudaEvent_t ev_rows = nullptr;
  std::string err;
  uint32_t W = 0, Wk = 0;
  std::unordered_map<uint32_t, std::pair<uint32_t, uint32_t>> maf_cache;
  std::mutex maf_mu;       // the upload helper thread of the pipelined submit shares the cache
  WorkerPool pool;         // planning threads
  AsyncWorker uploader;    // enqueues the uploads of the pipelined submit
  AsyncWorker grower;      // maps more memory behind a pattern pool before it is needed

  BatchState alt, alt2;    // the other batch slots (pipelined submit)
  DevBuf d_counters;       // u32[C_COUNT]: tickets, n_runs, errors, totals
  PinBuf h_counters;
  DevBuf d_bsum;
  DevBuf d_cand;
  DevBuf d_rep, d_slot_of, d_winner;
  DevBuf d_cl_rep, d_cl_slot, d_cl_winner;
  bool partition = true;   // mode 0: few radix passes + shared-memory hash grouping (k3_local)
  bool use_direct = true;  // S <= 1024: bitsets for every distinct key in shared memory
  bool runs_from_hist = false;   // one pass: prefix-runs are the digit buckets of the histogram
  uint32_t local_tile = 0;       // records per tile of the local reduce (4096 direct / 2048 general)
  bool fused = false;            // K1 fused into the histogram and the first pass (no record write in K1)
  DevBuf d_digests;
  int extra_bits = 0;      // sort bits added after a table overflow (sticky)
  double row_ratio = 1.0 / 48;   // surviving rows per record, learned from earlier batches (pf_create scales
                                 // the first guess with 1 / n_samples: rows per cluster do not grow with S, records do)
  bool row_ratio_learned = false;
  uint64_t unique_last = 0;
  uint32_t rescued_last = 0;
  // block aggregation (k3_block.cuh): no records, partial (k-mer, bitset) rows per position block
  bool block_mode = false;       // S <= 1024 and not disabled: kA_block_aggregate + kB1..kB3
  uint32_t block_windows = 16;   // windows per position block (= kBlkRun)
  uint32_t blk_slots = 1024, blk_cap = 448, blk_cslots = 128;   // shared memory of kA: k-mer key slots / rows, chunk slots
  uint32_t ka_seg_runs = 0;      // runs per kA segment (PF_KA_SEG_RUNS); 0: chosen from the batch
  uint32_t n_slices = 1, slice_samples = 0, Ws = 0;   // sample slices of the block engine (S > 1024): slices,
                                                       // samples per slice, bitset words of a partial row
  uint32_t block_fallbacks = 0;
  double partial_ratio = 1.0 / 16;   // partial rows per window, learned from earlier batches
  uint64_t partial_cap = 0;
  uint64_t partials_last = 0;
  bool used_block = false;       // the last batch went through kA/kB
  DevBuf d_slab_base, d_slab_count, d_slab_keys, d_slab_rows,
      d_group_base /* merge-table offsets per (cluster, slice) */, d_mtable,
      d_table2_base, d_table2, d_home_bits, d_cta_cluster, d_slab_cnt, d_rescue[2],
      d_spill /* (cluster, slice) merged in the global table */;
  uint32_t merge_fp_mask = 0x7fffu;   // PF_MERGE_FP_BITS (tests: a 1-bit fingerprint exercises the mismatch path)
  uint32_t merge_slots = 49152;  // shared-memory merge table of kB1_local (PF_MERGE_SMEM_KB)
  PatternSpace kp, cp;     // k-mer patterns, cluster patterns
  // pinned results
  PinBuf r_row_cluster, r_row_kmer, r_wrow_kmer, r_xrow_kmer, r_row_count, r_row_pattern, r_cl_pattern;
  PinBuf r_new_kp, r_new_cp, r_pos_kmer, r_pos_seq, r_pos_cstart, r_pos_gstart, r_pos_flags,
      r_pos_wide, r_pos_xwide, r_pos_bits;
  PinBuf r_wrow_cluster, r_wrow_count, r_wrow_pattern;   // pipelined submit: wide rows apart
  cudaEvent_t ev_d2h[2]{};
  pf_stats stats{};
  // the k-mer pattern count of the last pf_execute is folded into kp.n lazily (its K4 may still run)
  bool kp_pending = false;
  uint64_t kp_pending_base = 0;
  const uint32_t* kp_pending_count = nullptr;
  std::atomic<uint32_t> launches{0};
  // pipelined submit (submit_pipelined / collect_pipelined)
  bool prefetch_rows = false;    // start the D2H of the row arrays under K4 (PF_PREFETCH_ROWS=1): off by
                                 // default, the copy engine it occupies delays every small read-back that
                                 // follows (multi-GPU exchange), and large submits are pipelined anyway
  bool pipe_pending = false;     // results of a pipelined submit wait for pf_collect
  uint32_t pipe_subs = 1;        // sub-batches of the last submit
  bool pipe_mode = false;        // inside submit_pipelined: pf_execute leaves the D2H to it
  double pipe_ms[10] = {0};      // stage times summed over the sub-batches
  uint64_t pipe_rows = 0, pipe_wide_rows = 0, pipe_pos = 0, pipe_pos_wide = 0, pipe_bit_words = 0;
  uint32_t pipe_clusters = 0;
  uint64_t pipe_kp_base = 0, pipe_cp_base = 0, pipe_kp_copied = 0;
  uint64_t pipe_row_cap = 0, pipe_wide_cap = 0;
  cudaEvent_t ev_pipe[2]{};
  std::vector<std::array<cudaEvent_t, 5>> dbg_ev;   // PF_DEBUG_PIPE: per sub-batch {upload start, upload end, kernels start, kernels end, D2H end}
  uint32_t pipe_min_seqs = 200000;   // batches with fewer sequences are not split
  uint32_t pipe_target_seqs = 262144;   // sequences per sub-batch
  uint32_t pipe_first_seqs = 98304;     // ... of the first one (its upload is not hidden)
  bool lite_ok = true;           // device-side planning of uploads (PF_LITE=0 disables; off after a record fall-back)
};

namespace {

int fail(pf_ctx* c, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (c) c->err = buf; else g_create_error = buf;
  return code;
}

#define CU(call)                                                                       \
  do {                                                                                 \
    cudaError_t e_ = (call);                                                           \
    if (e_ != cudaSuccess)                                                             \
      return fail(ctx, PF_ERR_CUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_),   \
                  __FILE__, __LINE__);                                                 \
  } while (0)

// PF_DEBUG_ALLOC=1: report every (re)allocation - in the steady state there must be none
inline bool debug_alloc() { static const bool v = getenv("PF_DEBUG_ALLOC") != nullptr; return v; }

int dev_ensure(pf_ctx* ctx, DevBuf& b, size_t bytes, bool keep = false) {
  if (bytes <= b.cap) return PF_OK;
  if (debug_alloc()) fprintf(stderr, "[pf] alloc: device buffer %zu -> %zu bytes%s\n", b.cap, bytes, keep ? " (copy)" : "");
  size_t want = std::max(bytes, b.cap + b.cap / 2);
  want = (want + 255) & ~size_t(255);
  void* np = nullptr;
  CU(cudaMalloc(&np, want));
  if (keep && b.p && b.cap) {
    CU(cudaMemcpyAsync(np, b.p, b.cap, cudaMemcpyDeviceToDevice, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
  }
  if (b.p) CU(cudaFree(b.p));
  b.p = np;
  b.cap = want;
  return PF_OK;
}
int pin_ensure(pf_ctx* ctx, PinBuf& b, size_t bytes) {
  if (bytes <= b.cap) return PF_OK;
  if (debug_alloc()) fprintf(stderr, "[pf] alloc: pinned buffer %zu -> %zu bytes\n", b.cap, bytes);
  size_t want = std::max(bytes, b.cap + b.cap / 2);
  want = (want + 4095) & ~size_t(4095);
  if (b.p) CU(cudaFreeHost(b.p));
  b.p = nullptr; b.cap = 0;
  CU(cudaMallocHost(&b.p, want));
  b.cap = want;
  return PF_OK;
}
#define TRY(x) do { int r_ = (x); if (r_ != PF_OK) return r_; } while (0)

struct VmmApi {
  CUresult (*reserve)(CUdeviceptr*, size_t, size_t, CUdeviceptr, unsigned long long) = nullptr;
  CUresult (*addr_free)(CUdeviceptr, size_t) = nullptr;
  CUresult (*create)(CUmemGenericAllocationHandle*, size_t, const CUmemAllocationProp*, unsigned long long) = nullptr;
  CUresult (*release)(CUmemGenericAllocationHandle) = nullptr;
  CUresult (*map)(CUdeviceptr, size_t, size_t, CUmemGenericAllocationHandle, unsigned long long) = nullptr;
  CUresult (*unmap)(CUdeviceptr, size_t) = nullptr;
  CUresult (*set_access)(CUdeviceptr, size_t, const CUmemAccessDesc*, size_t) = nullptr;
  CUresult (*granularity)(size_t*, const CUmemAllocationProp*, CUmemAllocationGranularity_flags) = nullptr;
  bool ok = false;
};
const VmmApi& vmm_api() {
  static const VmmApi api = []() {
    VmmApi a;
    if (getenv("PF_NO_VMM")) return a;
    auto get = [](const char* name, void** fn) {
      cudaDriverEntryPointQueryResult st;
      return cudaGetDriverEntryPoint(name, fn, cudaEnableDefault, &st) == cudaSuccess &&
             st == cudaDriverEntryPointSuccess && *fn != nullptr;
    };
    a.ok = get("cuMemAddressReserve", (void**)&a.reserve) && get("cuMemAddressFree", (void**)&a.addr_free) &&
           get("cuMemCreate", (void**)&a.create) && get("cuMemRelease", (void**)&a.release) &&
           get("cuMemMap", (void**)&a.map) && get("cuMemUnmap", (void**)&a.unmap) &&
           get("cuMemSetAccess", (void**)&a.set_access) &&
           get("cuMemGetAllocationGranularity", (void**)&a.granularity);
    if (!a.ok) cudaGetLastError();
    return a;
  }();
  return api;
}

void pool_free(PoolBuf& b) {          // (the context's grower thread has been joined)
  if (b.vmm) {
    const VmmApi& api = vmm_api();
    size_t off = 0;
    for (auto& c : b.chunks) { api.unmap(b.base + off, c.second); api.release(c.first); off += c.second; }
    if (b.base) api.addr_free(b.base, b.reserved);
    b.chunks.clear();
    b.base = 0; b.reserved = 0; b.vmm = false;
  } else if (b.p) {
    cudaFree(b.p);
  }
  b.p = nullptr; b.cap = 0;
}

// map physical memory behind a VMM pool up to `want` bytes (rounded up); *cap_out = the new size.
// Touches nothing below the current end, so it may run while kernels use the pool.
int pool_map_to(pf_ctx* ctx, PoolBuf& b, size_t cur_cap, size_t want, size_t floor_bytes, size_t* cap_out) {
  const VmmApi& api = vmm_api();
  CUmemAllocationProp prop{};
  prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
  prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
  prop.location.id = ctx->device;
  size_t gran = 0;
  if (api.granularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED) != CUDA_SUCCESS || gran == 0) return PF_ERR_CUDA;
  want = std::min((want + gran - 1) / gran * gran, b.reserved);
  floor_bytes = (floor_bytes + gran - 1) / gran * gran;
  if (floor_bytes > b.reserved) return PF_ERR_NOMEM;
  CUmemGenericAllocationHandle h = 0;
  const auto t0 = std::chrono::steady_clock::now();
  CUresult r = want > cur_cap ? api.create(&h, want - cur_cap, &prop, 0) : CUDA_ERROR_INVALID_VALUE;
  if (r != CUDA_SUCCESS && floor_bytes > cur_cap && floor_bytes < want) {     // no room for the generous step: the exact one
    want = floor_bytes;
    r = api.create(&h, want - cur_cap, &prop, 0);
  }
  if (r != CUDA_SUCCESS) return PF_ERR_NOMEM;
  const size_t got = want - cur_cap;
  CUmemAccessDesc acc{};
  acc.location = prop.location;
  acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
  if (api.map(b.base + cur_cap, got, 0, h, 0) != CUDA_SUCCESS || api.set_access(b.base + cur_cap, got, &acc, 1) != CUDA_SUCCESS) {
    api.release(h);
    return PF_ERR_CUDA;
  }
  b.chunks.emplace_back(h, got);
  *cap_out = want;
  if (debug_alloc())
    fprintf(stderr, "[pf] alloc: mapped %zu MB behind a pool (now %zu MB) in %.1f ms\n", got >> 20, want >> 20,
            std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
  return PF_OK;
}

// a growth started ahead of need has to be over before the pool's size is looked at again
void pool_join(pf_ctx* ctx, PoolBuf& b) {
  if (!b.growing) return;
  ctx->grower.join();
  b.growing = false;
  if (b.grown_cap > b.cap) b.cap = b.grown_cap;
}

// grow a pattern pool to at least `bytes`, keeping its contents (and, with VMM, its address).
// Small pools double; a pool that outgrows 256 MB takes one big step, and once 7/8 of that is in
// use the next quarter is mapped on the grower thread while the kernels run.
int pool_ensure(pf_ctx* ctx, PoolBuf& b, size_t bytes) {
  constexpr size_t kMinStep = (size_t)256 << 20;
  // doubling up to 4 GB, then a quarter at a time: the exchange of a sharded run needs room for
  // two more copies of every pattern next to the pool
  // (mapping costs 10-40 ms per call in a process with NCCL peers, whatever the size, and stalls
  //  the device: a pool that outgrows 256 MB takes a quarter of the free memory, up to 48 GB, in
  //  ONE call; after that a quarter of its size at a time)
  auto grow_step = [&](size_t cap) -> size_t {
    if (!b.big_step_done) {
      size_t free_b = 0, total_b = 0;
      if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); free_b = (size_t)8 << 30; }
      b.big_step_done = true;
      return std::max<size_t>(cap, std::min<size_t>(free_b / 4, (size_t)48 << 30));
    }
    return std::max<size_t>((size_t)2 << 30, cap / 4);
  };
  auto prefetch = [&]() {
    if (!b.vmm || b.growing || b.cap < kMinStep || bytes <= b.cap / 8 * 7 || b.cap >= b.reserved) return;
    const size_t cur = b.cap, want = cur + grow_step(cur);
    b.growing = true;
    b.grown_cap = cur;
    ctx->grower.start([ctx, &b, cur, want]() {
      cudaSetDevice(ctx->device);
      size_t got = cur;
      if (pool_map_to(ctx, b, cur, want, cur, &got) == PF_OK) b.grown_cap = got;
    });
  };
  if (bytes <= b.cap) { prefetch(); return PF_OK; }
  pool_join(ctx, b);
  if (bytes <= b.cap) { prefetch(); return PF_OK; }
  const VmmApi& api = vmm_api();
  if (debug_alloc()) fprintf(stderr, "[pf] alloc: pattern pool %zu -> %zu bytes\n", b.cap, bytes);
  if (api.ok && (b.vmm || !b.p)) {
    if (!b.p) {
      CUmemAllocationProp prop{};
      prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
      prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
      prop.location.id = ctx->device;
      size_t gran = 0, free_b = 0, total_b = 0;
      if (api.granularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED) == CUDA_SUCCESS && gran > 0 &&
          cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) {
        const size_t want_va = (total_b + gran - 1) / gran * gran;      // a pool cannot outgrow the device
        CUdeviceptr base = 0;
        if (api.reserve(&base, want_va, gran, 0, 0) == CUDA_SUCCESS) {
          b.base = base; b.reserved = want_va; b.p = reinterpret_cast<void*>(base); b.cap = 0; b.vmm = true;
        }
      }
    }
    if (b.vmm) {
      // small pools (cluster patterns, tests) take what they need; big ones double
      const size_t step = std::max(bytes, b.cap) < kMinStep ? std::max<size_t>(b.cap, (size_t)8 << 20) : grow_step(b.cap);
      size_t got = b.cap;
      const int rc = pool_map_to(ctx, b, b.cap, std::max(bytes, b.cap + step), bytes, &got);
      if (rc == PF_ERR_NOMEM) return fail(ctx, PF_ERR_NOMEM, "no device memory left for %zu bytes of patterns", bytes);
      if (rc != PF_OK) return fail(ctx, PF_ERR_CUDA, "mapping more memory behind the pattern pool failed");
      b.cap = got;
      return PF_OK;
    }
  }
  return dev_ensure(ctx, b, bytes, true);       // copying fallback
}

// PF_DEBUG_SYNC=1: synchronise after every stage so a device fault names its kernel.
bool debug_sync(const char* name) {
  static const char* v = getenv("PF_DEBUG_SYNC");
  return v && (v[0] == '1' || strstr(name, v) != nullptr);
}
// PF_DEBUG_TIME=1: synchronise after every stage and print the wall-clock time since the previous
// stage boundary (host work + device work of the stage).
inline double pf_now_ms() {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}
inline bool debug_time() { static const bool v = getenv("PF_DEBUG_TIME") != nullptr; return v; }
static thread_local double g_stage_tick = 0;
#define STAGE(name)                                                                      \
  do {                                                                                   \
    if (debug_sync(name) || debug_time()) {                                              \
      cudaError_t e_ = cudaStreamSynchronize(ctx->stream);                               \
      if (e_ != cudaSuccess)                                                             \
        return fail(ctx, PF_ERR_CUDA, "stage %s: %s", name, cudaGetErrorString(e_));     \
      if (debug_time()) {                                                                \
        const double t_ = pf_now_ms();                                                   \
        fprintf(stderr, "[pf] stage %-28s %8.3f ms\n", name, t_ - g_stage_tick);         \
        g_stage_tick = t_;                                                               \
      }                                                                                  \
    }                                                                                    \
  } while (0)

inline uint32_t cdiv(uint64_t a, uint64_t b) { return (uint32_t)((a + b - 1) / b); }
constexpr int kGridPersist = 148 * 4;
constexpr uint32_t kBlkMaxSmem = 220u * 1024u;   // largest kA table we ask for

// counters layout in d_counters
enum { C_TICKET_N = 0, C_TICKET_W = 1, C_RUNS_N = 2, C_RUNS_W = 3, C_ERR = 4, C_ROWS_N = 5,
       C_ROWS_W = 6, C_NEW_KP = 7, C_NEW_CP = 8, C_TICKET_MARK_N = 9, C_TICKET_MARK_W = 10,
       C_LOCAL = 11 /* LC_COUNT words: rows, unique, table overflow, row overflow, rescue runs,
                        partial rows, partial overflow, kA segments, one-sample partial rows */,
       C_X_UNIQUE_KP = 20, C_X_UNIQUE_CP = 21 /* owner-side unique counts of the exchange */,
       C_TICKET_X = 22, C_RUNS_X = 23, C_ROWS_X = 24, C_TICKET_MARK_X = 25 /* 256-bit keys (k > 32) */,
       C_UNIQUE_WX = 26 /* distinct live keys of the wide and 256-bit records (k > 32 with N/IUPAC) */,
       C_COUNT = 28 };
static_assert(C_COUNT <= 32, "mirror_counters copies one warp's worth");
static_assert(C_LOCAL + LC_COUNT <= C_X_UNIQUE_KP, "counter layout");

bool keep_count(double maf, uint32_t c, uint32_t n) {
  double af = (double)c / (double)n;      // numpy: vec.sum() / vec.shape[0]
  if (af >= 0.5) af = 1 - af;
  return !(af < maf);
}

}  // namespace
