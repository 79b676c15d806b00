// pf_upload.cuh — host-side planning of a batch (tiles, offsets, MAF windows), H2D, pf_upload.
// Part of libpanfeed_b200.so's single translation unit: included once, in order, by pf_api.cu.

namespace {

int auto_sort_bits(const pf_ctx* ctx, uint32_t max_seg_records, bool narrow) {
  if (ctx->prm.sort_bits) return std::min(64, (int)ctx->prm.sort_bits + (narrow ? ctx->extra_bits : 0));
  if (narrow && ctx->partition) {
    // enough 8-bit passes that a prefix bucket of the largest cluster averages <= 4096 records
    int passes = 1;
    uint64_t buckets = 256;
    while ((uint64_t)max_seg_records / buckets > 4096 && passes < 8) { ++passes; buckets <<= 8; }
    return std::min(64, 8 * passes + ctx->extra_bits);
  }
  int lg = 0;
  while ((1ull << lg) < (uint64_t)std::max<uint32_t>(max_seg_records, 1)) ++lg;
  int bits = ((lg + 12 + 7) / 8) * 8;      // expected shared prefixes per segment <= n / 8192
  return std::min(64, std::max(16, bits));
}

// Build the tile list of one key width from the per-cluster record ranges.
// Tile list of the local reduce (partition mode): 8192-record tiles for the direct
// variant, 2048 for the general one (its exactness guarantee needs <= 2048).
int plan_local_tiles(pf_ctx* ctx, BatchState& B, cudaStream_t st) {
  WidthState& w = B.nar;
  if (!ctx->partition) { w.n_ltiles = 0; return PF_OK; }
  const uint32_t tile = ctx->use_direct ? (uint32_t)kDirectTile : (uint32_t)kLocalTile;
  ctx->local_tile = tile;
  const uint32_t nc = (uint32_t)B.nar_ranges.size();
  TRY(pin_ensure(ctx, w.h_ltiles, std::max<size_t>(1, nc) * 4));
  uint32_t* base = w.h_ltiles.as<uint32_t>();
  uint64_t nl = 0;
  for (uint32_t c = 0; c < nc; ++c) {
    base[c] = (uint32_t)nl;
    nl += cdiv(B.nar_ranges[c].second - B.nar_ranges[c].first, tile);
  }
  w.n_ltiles = (uint32_t)nl;
  if (w.n_ltiles) {
    TRY(dev_ensure(ctx, w.ltiles, (size_t)w.n_ltiles * sizeof(TileDev)));
    TRY(dev_ensure(ctx, w.tile_first_run, ((size_t)w.n_ltiles + 1) * 4));
    TRY(dev_ensure(ctx, w.lookback, std::max<size_t>((size_t)w.n_tiles * kRadix * 4, (size_t)w.n_ltiles * 8)));
    TRY(dev_ensure(ctx, w.d_ltile_base, (size_t)nc * 4));
    CU(cudaMemcpyAsync(w.d_ltile_base.p, base, (size_t)nc * 4, cudaMemcpyHostToDevice, st));
    // needs d_clusters: the caller uploads it first
    plan_expand_tiles<<<nc, 128, 0, st>>>(B.d_clusters.as<ClusterDev>(), nc, w.d_ltile_base.as<uint32_t>(),
                                                   tile, 0, w.ltiles.as<TileDev>());
    ctx->launches++;     // (the pinned `base` array must not be rewritten before this copy ran:
                         //  pf_upload ends with a sync, the re-plan in pf_execute syncs itself)
  }
  return PF_OK;
}

int plan_tiles(pf_ctx* ctx, WidthState& w, const std::vector<std::pair<uint32_t, uint32_t>>& ranges, bool narrow) {
  uint64_t n_tiles = 0;
  uint32_t max_seg = 0;
  for (auto& r : ranges) {
    n_tiles += cdiv(r.second - r.first, kSortTile);
    max_seg = std::max(max_seg, r.second - r.first);
  }
  if (max_seg >= (1u << 30))
    return fail(ctx, PF_ERR_INVALID, "a cluster has %u k-mer records; the limit per cluster is 2^30", max_seg);
  w.n_tiles = (uint32_t)n_tiles;
  w.max_seg = max_seg;
  w.sort_bits = auto_sort_bits(ctx, max_seg, narrow);
  w.passes = w.sort_bits / 8;
  TRY(pin_ensure(ctx, w.h_tiles, std::max<size_t>(1, ranges.size()) * 4));
  TRY(pin_ensure(ctx, w.h_seg_start, std::max<size_t>(1, ranges.size()) * sizeof(uint32_t)));
  uint32_t* tb = w.h_tiles.as<uint32_t>();
  uint32_t* ss = w.h_seg_start.as<uint32_t>();
  uint32_t ti = 0;
  for (uint32_t c = 0; c < ranges.size(); ++c) {
    ss[c] = ranges[c].first;
    tb[c] = ti;
    ti += cdiv(ranges[c].second - ranges[c].first, kSortTile);
  }
  return PF_OK;
}

}  // namespace

namespace {
int plan_blocks(pf_ctx* ctx, BatchState& B, cudaStream_t st, bool sync);
int plan_blocks_finish(pf_ctx* ctx, BatchState& B, cudaStream_t st, bool sync = true);
int scan_inplace(pf_ctx* ctx, uint32_t* data, uint32_t n, uint32_t* total_dev, cudaStream_t st = nullptr, DevBuf* scratch = nullptr);
}

namespace {
// A sub-range of a caller batch: sequences [s0,s1) of clusters [c0,c1), whose bases are words
// [w0,w1) of the 2-bit plane and [a0,a1) of the 4-bit plane.
struct SubRange { uint32_t s0, s1, c0, c1; uint64_t w0, w1, a0, a1; };

// The per-sequence checks of an upload for ONE sequence of the (sub-)batch: the message the host
// planner would give.  The lite upload validates on the device and calls this for the first bad index.
std::string describe_bad_seq(const pf_ctx* ctx, const pf_batch* b, uint32_t i, uint32_t rc, uint64_t rb, uint64_t ra) {
  const uint32_t S = ctx->prm.n_samples, W = ctx->W;
  char buf[256];
  pf_seq_desc q = b->seqs[i];
  q.cluster -= rc; q.base_off -= rb; q.amb_off -= (q.flags & PF_SEQ_AMBIGUOUS) ? ra : 0;
  auto f = [&](const char* fmt, uint32_t a1, uint32_t a2 = 0, uint32_t a3 = 0) { snprintf(buf, sizeof buf, fmt, a1, a2, a3); return std::string(buf); };
  if (q.cluster >= b->n_clusters) return f("seq %u: cluster %u out of range", i, q.cluster);
  if (i && q.cluster + rc < b->seqs[i - 1].cluster) return f("seq %u: clusters must be non-decreasing", i);
  if (q.sample >= S) return f("seq %u: sample rank %u >= n_samples %u", i, q.sample, S);
  if (i && q.cluster + rc == b->seqs[i - 1].cluster && q.sample < b->seqs[i - 1].sample)
    return f("seq %u: sample ranks must be non-decreasing inside a cluster", i);
  if (!((b->cluster_presence[(size_t)q.cluster * W + (q.sample >> 5)] >> (q.sample & 31)) & 1u))
    return f("seq %u: sample %u is not marked present in cluster %u", i, q.sample, q.cluster);
  if (q.base_off & 63u) return f("seq %u: base_off must be a multiple of 64", i);
  if (q.base_off + q.len > b->n_words * 32ull) return f("seq %u: bases run past the packed plane", i);
  if (q.strand != 1 && q.strand != -1) return f("seq %u: strand must be +1/-1", i);
  if (q.flags & PF_SEQ_AMBIGUOUS) return f("seq %u is flagged ambiguous but the batch has no 4-bit plane", i);
  return f("seq %u: malformed descriptor", i);
}

// ClusterDev of every cluster of the (sub-)batch: presence popcount, MAF window, filters folded in.
// rec ranges stay zero unless `nr` / `wr` / `xr` give them (record engines).
int build_clusters(pf_ctx* ctx, const pf_batch* b, ClusterDev* hc, const std::pair<uint32_t, uint32_t>* nr,
                   const std::pair<uint32_t, uint32_t>* wr, const std::pair<uint32_t, uint32_t>* xr = nullptr) {
  const pf_params& P = ctx->prm;
  const uint32_t S = P.n_samples, W = ctx->W;
  for (uint32_t c = 0; c < b->n_clusters; ++c) {
    uint32_t np = 0;
    for (uint32_t w = 0; w < W; ++w) {
      uint32_t word = b->cluster_presence[(size_t)c * W + w];
      if (w == W - 1 && (S & 31u)) {
        if (word >> (S & 31u)) return fail(ctx, PF_ERR_INVALID, "cluster %u: presence bits beyond n_samples", c);
      }
      np += (uint32_t)__builtin_popcount(word);
    }
    ClusterDev& d = hc[c];
    d.rec_start = nr ? nr[c].first : 0; d.rec_end = nr ? nr[c].second : 0;
    d.wrec_start = wr ? wr[c].first : 0; d.wrec_end = wr ? wr[c].second : 0;
    d.xrec_start = xr ? xr[c].first : 0; d.xrec_end = xr ? xr[c].second : 0;
    d.id = b->clusters[c].id; d.n_present = np;
    const uint32_t n = P.consider_missing ? np : S;
    uint32_t lo, hi;
    {
      std::lock_guard<std::mutex> lk(ctx->maf_mu);
      auto it = ctx->maf_cache.find(n);
      if (it == ctx->maf_cache.end()) {
        uint32_t wl, wh;
        pf_maf_window(P.maf, n, &wl, &wh);
        it = ctx->maf_cache.emplace(n, std::make_pair(wl, wh)).first;
      }
      lo = it->second.first; hi = it->second.second;
    }
    // "same as cluster" (panfeed.py:202-204): k-mer bits are a subset of the
    // cluster's, so equality <=> count == n_present; NaN entries never compare equal.
    if (P.cluster_equal_filter && (!P.consider_missing || np == S)) {
      if (np == 0) { lo = 1; hi = 0; }
      else hi = std::min(hi, np - 1);
    }
    if (lo == 0) lo = 1;                    // a k-mer row always has >= 1 sample
    d.lo = lo; d.hi = hi;
  }
  return PF_OK;
}

// Lite upload: no per-sequence host work.  H2D of the packed plane and of the caller's descriptors
// as they are, one device kernel validates and builds SeqDev / SeqLite and the totals
// (plan_from_raw), then the block planning kernels.  upload_finish* reads the totals.
int upload_async_lite(pf_ctx* ctx, BatchState& B, const pf_batch* b, uint32_t rc, uint64_t rb, cudaStream_t st) {
  const pf_params& P = ctx->prm;
  const uint32_t W = ctx->W, n = b->n_seqs, nc = b->n_clusters;
  B.lite = true;
  B.lite_src = b->seqs; B.lite_c0 = rc; B.lite_b0 = rb;
  B.lite_clusters.assign(b->clusters, b->clusters + nc);
  B.lite_presence.assign(b->cluster_presence, b->cluster_presence + (size_t)nc * W);
  const size_t slack_words = 80;
  TRY(dev_ensure(ctx, B.d_bases, (b->n_words + slack_words) * 8));
  CU(cudaEventRecord(B.ev_h2d[0], st));
  if (b->n_words) CU(cudaMemcpyAsync(B.d_bases.p, b->packed_bases, b->n_words * 8, cudaMemcpyHostToDevice, st));
  CU(cudaMemsetAsync((char*)B.d_bases.p + b->n_words * 8, 0, slack_words * 8, st));
  // descriptors: straight from the caller's array if it is pinned, else through the slot's pinned
  // staging buffer (a plain copy on the planning threads; a pageable cudaMemcpyAsync would block)
  TRY(dev_ensure(ctx, B.d_raw, (size_t)n * sizeof(pf_seq_desc)));
  const void* src = b->seqs;
  cudaPointerAttributes attr{};
  const bool pinned = cudaPointerGetAttributes(&attr, b->seqs) == cudaSuccess && attr.type == cudaMemoryTypeHost;
  if (!pinned) {
    cudaGetLastError();
    TRY(pin_ensure(ctx, B.h_raw, (size_t)n * sizeof(pf_seq_desc)));
    static const uint32_t host_thr = []() { const char* e = getenv("PF_HOST_THREADS"); const int v = e ? atoi(e) : 0;
                                            return v > 0 ? (uint32_t)v : 8u; }();
    const uint32_t n_thr = std::max(1u, std::min<uint32_t>(std::min(host_thr, std::thread::hardware_concurrency()),
                                                           (n + 65535u) / 65536u));
    const uint32_t per = (n + n_thr - 1) / n_thr;
    char* dst = B.h_raw.as<char>();
    const char* from = reinterpret_cast<const char*>(b->seqs);
    ctx->pool.parallel(n_thr, [&](uint32_t t) {
      const size_t i0 = std::min<size_t>(n, (size_t)t * per), i1 = std::min<size_t>(n, i0 + per);
      memcpy(dst + i0 * sizeof(pf_seq_desc), from + i0 * sizeof(pf_seq_desc), (i1 - i0) * sizeof(pf_seq_desc));
    });
    src = dst;
  }
  CU(cudaMemcpyAsync(B.d_raw.p, src, (size_t)n * sizeof(pf_seq_desc), cudaMemcpyHostToDevice, st));
  // clusters
  TRY(pin_ensure(ctx, B.h_clusters, std::max<size_t>(1, nc) * sizeof(ClusterDev)));
  TRY(build_clusters(ctx, b, B.h_clusters.as<ClusterDev>(), nullptr, nullptr));
  TRY(dev_ensure(ctx, B.d_seqs, std::max<size_t>(1, n) * sizeof(SeqDev)));
  TRY(dev_ensure(ctx, B.d_seq_lite, std::max<size_t>(1, n) * sizeof(SeqLite)));
  TRY(dev_ensure(ctx, B.d_clusters, std::max<size_t>(1, nc) * sizeof(ClusterDev)));
  TRY(dev_ensure(ctx, B.d_presence, std::max<size_t>(1, (size_t)nc * W) * 4));
  TRY(dev_ensure(ctx, ctx->d_counters, C_COUNT * 4));
  TRY(pin_ensure(ctx, ctx->h_counters, C_COUNT * 4 + 64 * 4));
  TRY(dev_ensure(ctx, B.d_lite_tot, sizeof(LiteTotals)));
  TRY(pin_ensure(ctx, B.h_lite_tot, sizeof(LiteTotals)));
  CU(cudaMemcpyAsync(B.d_clusters.p, B.h_clusters.p, (size_t)nc * sizeof(ClusterDev), cudaMemcpyHostToDevice, st));
  // (the presence words come from the slot's own copy: the caller's array may be pageable)
  CU(cudaMemcpyAsync(B.d_presence.p, B.lite_presence.data(), (size_t)nc * W * 4, cudaMemcpyHostToDevice, st));
  CU(cudaMemsetAsync(B.d_lite_tot.p, 0, 24, st));
  CU(cudaMemsetAsync((char*)B.d_lite_tot.p + 24, 0xff, 8, st));
  plan_from_raw<<<cdiv(n, 256), 256, 0, st>>>(B.d_raw.as<pf_seq_desc>(), n, rc, rb, nc, P.n_samples, W,
                                               B.d_presence.as<uint32_t>(), b->n_words * 32ull, (int)P.k,
                                               P.emit_positions, B.d_seqs.as<SeqDev>(), B.d_seq_lite.as<SeqLite>(),
                                               B.d_lite_tot.as<LiteTotals>());
  ctx->launches++;
  mirror_counters<<<1, 32, 0, st>>>(B.h_lite_tot.as<uint32_t>(), B.d_lite_tot.as<uint32_t>(), 16);
  B.n_seqs = n; B.n_clusters = nc; B.n_wide_seqs = 0;
  B.n_words = b->n_words; B.n_amb_words = 0;
  B.n_bases = 0; B.n_pos = 0; B.n_pos_wide = 0; B.n_pos_xwide = 0;   // totals: upload_finish*
  B.nar.n_records = 0; B.wid.n_records = 0; B.xwd.n_records = 0; B.xwd.n_tiles = 0;
  B.nar.n_tiles = B.wid.n_tiles = 0; B.nar.n_ltiles = 0; B.nar.max_seg = B.wid.max_seg = 0;
  B.nar.passes = B.wid.passes = 1; B.nar.sort_bits = B.wid.sort_bits = 8;
  B.nar_ranges.clear();
  CU(cudaEventRecord(B.ev_h2d[1], st));
  TRY(plan_blocks(ctx, B, st, false));
  CU(cudaEventRecord(B.ev_up_done, st));
  CU(cudaGetLastError());
  return PF_OK;
}

// After the stream has passed a lite upload: errors and totals of plan_from_raw
int lite_finish(pf_ctx* ctx, BatchState& B) {
  if (!B.lite) return PF_OK;
  const LiteTotals& t = *B.h_lite_tot.as<LiteTotals>();
  if (t.err != ~0ull) {
    const uint32_t i = (uint32_t)(t.err >> 32);
    if (B.lite_src && i < B.n_seqs) {        // the host planner's message for that sequence
      pf_batch v{};
      v.seqs = B.lite_src; v.n_seqs = B.n_seqs; v.n_clusters = B.n_clusters; v.n_words = B.n_words;
      v.cluster_presence = B.lite_presence.data();
      return fail(ctx, PF_ERR_INVALID, "%s", describe_bad_seq(ctx, &v, i, B.lite_c0, B.lite_b0, 0).c_str());
    }
    return fail(ctx, PF_ERR_INVALID, "seq %u: malformed descriptor (check %u)", i, (uint32_t)t.err);
  }
  const uint64_t mult = ctx->prm.canonical ? 1u : 2u;
  if (t.windows * mult >= (1ull << 32) - kSortTile) return fail(ctx, PF_ERR_INVALID, "batch holds more than 2^32 k-mer records; split it");
  if (t.pos_windows >= (1ull << 32)) return fail(ctx, PF_ERR_INVALID, "more than 2^32 positional records; split the batch");
  B.n_bases = t.bases;
  B.nar.n_records = (uint32_t)(t.windows * mult);
  B.n_pos = (uint32_t)t.pos_windows;
  return PF_OK;
}

// Validate + plan + H2D of the sub-range into the CURRENT batch slot, all asynchronous on `st`
// (the caller's buffers must stay valid until `st` has passed).  upload_finish completes it.
int upload_async(pf_ctx* ctx, BatchState& B, const pf_batch* full, const SubRange& r, cudaStream_t st,
                 bool force_full = false, bool have_bases = false) {
  const double t_dbg_in = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
  pf_batch view = *full;
  view.seqs = full->seqs ? full->seqs + r.s0 : nullptr;
  view.n_seqs = r.s1 - r.s0;
  view.clusters = full->clusters ? full->clusters + r.c0 : nullptr;
  view.n_clusters = r.c1 - r.c0;
  view.cluster_presence = full->cluster_presence ? full->cluster_presence + (size_t)r.c0 * ctx->W : nullptr;
  view.packed_bases = full->packed_bases ? full->packed_bases + r.w0 : nullptr;
  view.n_words = r.w1 - r.w0;
  view.amb_codes = full->amb_codes ? full->amb_codes + r.a0 : nullptr;
  view.n_amb_words = r.a1 - r.a0;
  const pf_batch* b = &view;
  const uint32_t rc = r.c0;                       // rebase of cluster indices
  const uint64_t rb = r.w0 * 32ull, ra = r.a0 * 16ull;   // ... of base / symbol offsets
  B.have_batch = false;
  B.executed = false;
  const pf_params& P = ctx->prm;
  const uint32_t k = P.k, S = P.n_samples, W = ctx->W;
  if (b->n_seqs && (!b->seqs || (!b->packed_bases && !have_bases))) return fail(ctx, PF_ERR_INVALID, "null seqs/packed_bases");
  if (b->n_clusters && (!b->clusters || !b->cluster_presence))
    return fail(ctx, PF_ERR_INVALID, "null clusters/cluster_presence");
  if (b->n_clusters == 0 && b->n_seqs) return fail(ctx, PF_ERR_INVALID, "sequences without clusters");
  B.lite = false;
  if (!force_full && ctx->lite_ok && ctx->block_mode && P.emit_positions != 1u && b->n_amb_words == 0 && b->n_seqs &&
      b->n_words < (1ull << 32))
    return upload_async_lite(ctx, B, b, rc, rb, st);

  TRY(pin_ensure(ctx, B.h_seqs, std::max<size_t>(1, b->n_seqs) * sizeof(SeqDev)));
  TRY(pin_ensure(ctx, B.h_clusters, std::max<size_t>(1, b->n_clusters) * sizeof(ClusterDev)));
  TRY(pin_ensure(ctx, B.h_wide_seqs, std::max<size_t>(1, b->n_seqs) * sizeof(uint32_t)));
  SeqDev* hs = B.h_seqs.as<SeqDev>();
  ClusterDev* hc = B.h_clusters.as<ClusterDev>();
  uint32_t* hw = B.h_wide_seqs.as<uint32_t>();

  const uint32_t mult = P.canonical ? 1u : 2u;
  // two-word k-mers: every window is a record of the 128-bit pipeline; the windows of a sequence
  // with N/IUPAC symbols are ALSO records of the 256-bit pipeline (4 bits per symbol), and each
  // pipeline kills the records of the windows the other one owns
  const bool long_k = k > 32;
  // the packed plane is the bulk of the transfer: start it before the host-side planning
  const size_t slack_words = 80;
  TRY(dev_ensure(ctx, B.d_bases, (b->n_words + slack_words) * 8));
  CU(cudaEventRecord(B.ev_h2d[0], st));
  if (b->n_words && !have_bases) CU(cudaMemcpyAsync(B.d_bases.p, b->packed_bases, b->n_words * 8, cudaMemcpyHostToDevice, st));
  if (!have_bases) CU(cudaMemsetAsync((char*)B.d_bases.p + b->n_words * 8, 0, slack_words * 8, st));

  static const bool dbg_up = getenv("PF_DEBUG_PIPE") != nullptr;
  auto now_ms = []() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t_dbg0 = now_ms();
  // ---- planning, in parallel over chunks of sequences --------------------------------
  // phase A: validate + per-sequence sizes, per-chunk sums; phase B: prefix over chunks;
  // phase C: offsets.  Cluster ranges come from the first sequence of every cluster.
  uint64_t rec = 0, wrec = 0, xrec = 0, pos = 0, pwide = 0, pxwide = 0, bases = 0;
  uint32_t n_wide = 0;                 // sequences with N/IUPAC symbols (listed in h_wide_seqs)
  std::vector<std::pair<uint32_t, uint32_t>> nr(b->n_clusters), wr(b->n_clusters), xr(b->n_clusters);
  {
    const uint32_t n = b->n_seqs;
    // PF_HOST_THREADS caps the planning threads (several contexts / ranks share the host's cores)
    static const uint32_t host_thr = []() { const char* e = getenv("PF_HOST_THREADS"); const int v = e ? atoi(e) : 0;
                                            return v > 0 ? (uint32_t)v : 16u; }();
    const uint32_t n_thr = std::max(1u, std::min<uint32_t>(std::min(host_thr, std::thread::hardware_concurrency()),
                                                           (n + 16383u) / 16384u));
    struct Part { uint64_t rec = 0, wrec = 0, xrec = 0, pos = 0, pwide = 0, pxwide = 0, bases = 0; uint32_t wide = 0; std::string err; };
    std::vector<Part> parts(n_thr);
    const uint32_t per = (n + n_thr - 1) / std::max(1u, n_thr);
    auto run = [&](const std::function<void(uint32_t)>& fn) { ctx->pool.parallel(n_thr, fn); };
    auto errf = [](Part& p, const char* fmt, uint32_t i, uint32_t a2 = 0, uint32_t a3 = 0) {
      char buf[256];
      snprintf(buf, sizeof buf, fmt, i, a2, a3);
      p.err = buf;
    };
    run([&](uint32_t t) {
      Part& p = parts[t];
      const uint32_t i0 = std::min(n, t * per), i1 = std::min(n, i0 + per);
      for (uint32_t i = i0; i < i1; ++i) {
        pf_seq_desc q = b->seqs[i];
        q.cluster -= rc; q.base_off -= rb; q.amb_off -= (q.flags & PF_SEQ_AMBIGUOUS) ? ra : 0;
        if (q.cluster >= b->n_clusters) return errf(p, "seq %u: cluster %u out of range", i, q.cluster);
        if (i && q.cluster + rc < b->seqs[i - 1].cluster) return errf(p, "seq %u: clusters must be non-decreasing", i);
        if (q.sample >= S) return errf(p, "seq %u: sample rank %u >= n_samples %u", i, q.sample, S);
        if (i && q.cluster + rc == b->seqs[i - 1].cluster && q.sample < b->seqs[i - 1].sample)
          return errf(p, "seq %u: sample ranks must be non-decreasing inside a cluster", i);
        if (!((b->cluster_presence[(size_t)q.cluster * W + (q.sample >> 5)] >> (q.sample & 31)) & 1u))
          return errf(p, "seq %u: sample %u is not marked present in cluster %u", i, q.sample, q.cluster);
        if (q.base_off & 63u) return errf(p, "seq %u: base_off must be a multiple of 64", i);
        if (q.base_off + q.len > b->n_words * 32ull) return errf(p, "seq %u: bases run past the packed plane", i);
        if (q.strand != 1 && q.strand != -1) return errf(p, "seq %u: strand must be +1/-1", i);
        const bool amb = (q.flags & PF_SEQ_AMBIGUOUS) != 0;
        if (amb) {
          if (!b->amb_codes) return errf(p, "seq %u is ambiguous but amb_codes is NULL", i);
          if (q.amb_off & 31u) return errf(p, "seq %u: amb_off must be a multiple of 32", i);
          if (q.amb_off + q.len > b->n_amb_words * 16ull) return errf(p, "seq %u: symbols run past the 4-bit plane", i);
        }
        const bool target = P.emit_positions && (q.flags & PF_SEQ_TARGET);
        const uint32_t nwin = q.len >= k ? q.len - k + 1 : 0;
        if (!long_k) p.rec += (uint64_t)nwin * mult;
        if (target) p.pos += nwin;
        if (amb || long_k) { p.wrec += (uint64_t)nwin * mult; if (target) p.pwide += nwin; }
        if (amb) {
          p.wide++;
          if (long_k) { p.xrec += (uint64_t)nwin * mult; if (target) p.pxwide += nwin; }
        }
        p.bases += q.len;
      }
    });
    for (auto& p : parts) if (!p.err.empty()) return fail(ctx, PF_ERR_INVALID, "%s", p.err.c_str());
    std::vector<Part> base(n_thr);
    for (uint32_t t = 0; t < n_thr; ++t) {
      base[t].rec = rec; base[t].wrec = wrec; base[t].xrec = xrec; base[t].pos = pos; base[t].pwide = pwide;
      base[t].pxwide = pxwide; base[t].wide = n_wide;
      rec += parts[t].rec; wrec += parts[t].wrec; xrec += parts[t].xrec; pos += parts[t].pos; pwide += parts[t].pwide;
      pxwide += parts[t].pxwide; n_wide += parts[t].wide; bases += parts[t].bases;
    }
    if (rec >= (1ull << 32) - kSortTile || wrec >= (1ull << 32) - kSortTile || xrec >= (1ull << 32) - kSortTile)
      return fail(ctx, PF_ERR_INVALID, "batch holds more than 2^32 k-mer records; split it");
    if (pos >= (1ull << 32)) return fail(ctx, PF_ERR_INVALID, "more than 2^32 positional records; split the batch");
    if (long_k && n_wide) TRY(pin_ensure(ctx, B.h_xpos_slot, (size_t)n_wide * sizeof(uint32_t)));
    uint32_t* hxp = B.h_xpos_slot.as<uint32_t>();
    constexpr uint32_t kUnset = 0xffffffffu;
    for (uint32_t c = 0; c < b->n_clusters; ++c) { nr[c] = {kUnset, kUnset}; wr[c] = {kUnset, kUnset}; xr[c] = {kUnset, kUnset}; }
    run([&](uint32_t t) {
      Part o = base[t];
      const uint32_t i0 = std::min(n, t * per), i1 = std::min(n, i0 + per);
      for (uint32_t i = i0; i < i1; ++i) {
        pf_seq_desc q = b->seqs[i];
        q.cluster -= rc; q.base_off -= rb; q.amb_off -= (q.flags & PF_SEQ_AMBIGUOUS) ? ra : 0;
        const bool amb = (q.flags & PF_SEQ_AMBIGUOUS) != 0;
        const bool target = P.emit_positions && (q.flags & PF_SEQ_TARGET);
        const uint32_t nwin = q.len >= k ? q.len - k + 1 : 0;
        if (i == 0 || q.cluster + rc != b->seqs[i - 1].cluster) {     // first sequence of its cluster
          nr[q.cluster].first = (uint32_t)o.rec;
          wr[q.cluster].first = (uint32_t)o.wrec;
          xr[q.cluster].first = (uint32_t)o.xrec;
        }
        SeqDev& d = hs[i];
        d.base_off = q.base_off; d.amb_off = amb ? q.amb_off : 0; d.len = q.len; d.sample = q.sample;
        d.cluster = q.cluster; d.flags = (target ? 1u : 0u) | (amb ? 2u : 0u);
        d.start = q.start; d.end = q.end; d.offset = q.offset; d.strand = q.strand;
        d.rec_off = (uint32_t)(long_k ? o.xrec : o.rec); d.pos_off = (uint32_t)o.pos; d.wrec_off = (uint32_t)o.wrec;
        d.pwide_off = (uint32_t)o.pwide;
        if (!long_k) o.rec += (uint64_t)nwin * mult;
        if (target) o.pos += nwin;
        if (amb || long_k) { o.wrec += (uint64_t)nwin * mult; if (target) o.pwide += nwin; }
        if (amb) {
          if (long_k) {
            hxp[o.wide] = (uint32_t)o.pxwide;
            o.xrec += (uint64_t)nwin * mult;
            if (target) o.pxwide += nwin;
          }
          hw[o.wide++] = i;
        }
      }
    });
    // clusters without sequences are empty ranges at the start of the next non-empty one
    uint32_t next_n = (uint32_t)rec, next_w = (uint32_t)wrec, next_x = (uint32_t)xrec;
    for (uint32_t c = b->n_clusters; c-- > 0;) {
      if (nr[c].first == kUnset) { nr[c].first = next_n; wr[c].first = next_w; xr[c].first = next_x; }
      nr[c].second = next_n; wr[c].second = next_w; xr[c].second = next_x;
      next_n = nr[c].first; next_w = wr[c].first; next_x = xr[c].first;
    }
  }
  const double t_dbg1 = now_ms();
  TRY(build_clusters(ctx, b, hc, nr.data(), wr.data(), xr.data()));

  const double t_dbg2 = now_ms();
  B.n_seqs = b->n_seqs; B.n_clusters = b->n_clusters; B.n_wide_seqs = n_wide;
  B.n_words = b->n_words; B.n_amb_words = n_wide ? b->n_amb_words : 0; B.n_bases = bases;
  B.n_pos = (uint32_t)pos; B.n_pos_wide = (uint32_t)pwide; B.n_pos_xwide = (uint32_t)pxwide;
  B.nar.n_records = (uint32_t)rec; B.wid.n_records = (uint32_t)wrec; B.xwd.n_records = (uint32_t)xrec;
  TRY(plan_tiles(ctx, B.nar, nr, true));
  TRY(plan_tiles(ctx, B.wid, wr, false));
  // (the 256-bit width exists only for k > 32 batches with N/IUPAC symbols)
  std::vector<WidthState*> widths{&B.nar, &B.wid};
  if (xrec) { TRY(plan_tiles(ctx, B.xwd, xr, false)); widths.push_back(&B.xwd); }
  else B.xwd.n_tiles = 0;

  // ---- device buffers + H2D ------------------------------------------------
  TRY(dev_ensure(ctx, B.d_seqs, std::max<size_t>(1, b->n_seqs) * sizeof(SeqDev)));
  TRY(dev_ensure(ctx, B.d_clusters, std::max<size_t>(1, b->n_clusters) * sizeof(ClusterDev)));
  TRY(dev_ensure(ctx, B.d_presence, std::max<size_t>(1, (size_t)b->n_clusters * W) * 4));
  TRY(dev_ensure(ctx, ctx->d_counters, C_COUNT * 4));
  TRY(pin_ensure(ctx, ctx->h_counters, C_COUNT * 4 + 64 * 4));
  for (WidthState* w : widths) {
    TRY(dev_ensure(ctx, w->tiles, std::max<size_t>(1, w->n_tiles) * sizeof(TileDev)));
    TRY(dev_ensure(ctx, w->seg_start, std::max<size_t>(1, b->n_clusters) * 4));
    TRY(dev_ensure(ctx, w->seg_hist, std::max<size_t>(1, (size_t)b->n_clusters * w->passes * kRadix) * 4));
    TRY(dev_ensure(ctx, w->lookback, std::max<size_t>(1, (size_t)w->n_tiles * kRadix) * 4));
  }
  if (b->n_seqs) CU(cudaMemcpyAsync(B.d_seqs.p, hs, b->n_seqs * sizeof(SeqDev), cudaMemcpyHostToDevice, st));
  if (b->n_clusters) {
    CU(cudaMemcpyAsync(B.d_clusters.p, hc, b->n_clusters * sizeof(ClusterDev), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(B.d_presence.p, b->cluster_presence, (size_t)b->n_clusters * W * 4, cudaMemcpyHostToDevice, st));
  }
  // tile lists are generated on the device from the per-cluster record ranges
  for (WidthState* w : widths) {
    if (b->n_clusters) CU(cudaMemcpyAsync(w->seg_start.p, w->h_seg_start.p, b->n_clusters * 4, cudaMemcpyHostToDevice, st));
    if (w->n_tiles) {
      TRY(dev_ensure(ctx, w->d_tile_base, (size_t)b->n_clusters * 4));
      CU(cudaMemcpyAsync(w->d_tile_base.p, w->h_tiles.p, (size_t)b->n_clusters * 4, cudaMemcpyHostToDevice, st));
      plan_expand_tiles<<<b->n_clusters, 128, 0, st>>>(B.d_clusters.as<ClusterDev>(), b->n_clusters,
                                                       w->d_tile_base.as<uint32_t>(), kSortTile,
                                                       w == &B.xwd ? 2 : w == &B.wid ? 1 : 0, w->tiles.as<TileDev>());
      ctx->launches++;
    }
  }
  B.nar_ranges = nr;
  TRY(plan_local_tiles(ctx, B, st));
  // fused first pass: record index -> sequence lookup tables
  if (b->n_seqs) {
    TRY(dev_ensure(ctx, B.d_seq_rec_off, ((size_t)b->n_seqs + 1) * 4));
    TRY(dev_ensure(ctx, B.d_tile_first_seq, ((size_t)B.nar.n_tiles + 1) * 4));
    plan_seq_rec_off<<<cdiv((uint64_t)b->n_seqs + 1, 256), 256, 0, st>>>(
        B.d_seqs.as<SeqDev>(), b->n_seqs, (uint32_t)rec, B.d_seq_rec_off.as<uint32_t>());
    plan_tile_first_seq<<<cdiv((uint64_t)B.nar.n_tiles + 1, 256), 256, 0, st>>>(
        B.nar.tiles.as<TileDev>(), B.nar.n_tiles, B.d_seq_rec_off.as<uint32_t>(), b->n_seqs,
        B.d_tile_first_seq.as<uint32_t>());
    ctx->launches += 2;
  }
  if (n_wide) {
    const size_t bit_words = (b->n_amb_words + 1) / 2 + 4;
    TRY(dev_ensure(ctx, B.d_amb, (b->n_amb_words + 8) * 8));
    TRY(dev_ensure(ctx, B.d_ambbits, bit_words * 4));
    TRY(dev_ensure(ctx, B.d_wide_seqs, n_wide * 4));
    CU(cudaMemcpyAsync(B.d_amb.p, b->amb_codes, b->n_amb_words * 8, cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync((char*)B.d_amb.p + b->n_amb_words * 8, 0, 8 * 8, st));
    CU(cudaMemcpyAsync(B.d_wide_seqs.p, hw, n_wide * 4, cudaMemcpyHostToDevice, st));
    if (long_k) {
      TRY(dev_ensure(ctx, B.d_xpos_slot, n_wide * 4));
      CU(cudaMemcpyAsync(B.d_xpos_slot.p, B.h_xpos_slot.p, n_wide * 4, cudaMemcpyHostToDevice, st));
    }
    k1_amb_bits<<<cdiv(bit_words, 256), 256, 0, st>>>(B.d_amb.as<uint64_t>(), b->n_amb_words,
                                                       B.d_ambbits.as<uint32_t>(), bit_words);
    ctx->launches++;
  }
  if (ctx->block_mode && b->n_seqs) {
    if (b->n_words >= (1ull << 32)) return fail(ctx, PF_ERR_INVALID, "packed plane holds 2^32 words or more; split the batch");
    TRY(dev_ensure(ctx, B.d_seq_lite, (size_t)b->n_seqs * sizeof(SeqLite)));
    plan_seq_lite<<<cdiv(b->n_seqs, 256), 256, 0, st>>>(B.d_seqs.as<SeqDev>(), b->n_seqs, B.d_seq_lite.as<SeqLite>());
    ctx->launches++;
  }
  CU(cudaEventRecord(B.ev_h2d[1], st));
  if (ctx->block_mode) TRY(plan_blocks(ctx, B, st, false));
  CU(cudaEventRecord(B.ev_up_done, st));
  CU(cudaGetLastError());
  if (dbg_up)
    fprintf(stderr, "[pf] upload %u seqs: head %.3f  seq planning %.3f  clusters %.3f  enqueue %.3f ms\n", b->n_seqs,
            t_dbg0 - t_dbg_in, t_dbg1 - t_dbg0, t_dbg2 - t_dbg1, now_ms() - t_dbg2);
  return PF_OK;
}

// Second half of an upload: wait for the copies and the planning kernels, read n_items back.
int upload_finish(pf_ctx* ctx, BatchState& B, cudaStream_t up) {
  CU(cudaStreamSynchronize(up));
  TRY(lite_finish(ctx, B));
  if (ctx->block_mode) TRY(plan_blocks_finish(ctx, B, up));
  CU(cudaStreamSynchronize(up));
  CU(cudaGetLastError());
  B.have_batch = true;
  return PF_OK;
}
// The same for a slot of the pipelined submit: waits for THAT upload only (later ones may be
// queued behind it on the upload stream) and leaves the last planning kernels to the compute
// stream, which runs the slot's kernels next.
int upload_finish_slot(pf_ctx* ctx, BatchState& B, cudaStream_t compute) {
  CU(cudaEventSynchronize(B.ev_up_done));
  TRY(lite_finish(ctx, B));
  if (ctx->block_mode) TRY(plan_blocks_finish(ctx, B, compute, false));
  CU(cudaGetLastError());
  B.have_batch = true;
  return PF_OK;
}
// A lite slot has to leave the block engine: plan it again on the host (record offsets, tile
// lists) from the device copy of the caller's descriptors; the packed plane is already there.
int replan_full(pf_ctx* ctx) {
  BatchState& B = *ctx;
  if (!B.lite) return PF_OK;
  std::vector<pf_seq_desc> raw(B.n_seqs);
  CU(cudaStreamSynchronize(ctx->stream));
  if (B.n_seqs) CU(cudaMemcpy(raw.data(), B.d_raw.p, (size_t)B.n_seqs * sizeof(pf_seq_desc), cudaMemcpyDeviceToHost));
  for (auto& q : raw) { q.cluster -= B.lite_c0; q.base_off -= B.lite_b0; }
  pf_batch v{};
  v.n_words = B.n_words;
  v.seqs = raw.data(); v.n_seqs = B.n_seqs;
  v.clusters = B.lite_clusters.data(); v.n_clusters = B.n_clusters;
  v.cluster_presence = B.lite_presence.data();
  const SubRange r{0, B.n_seqs, 0, B.n_clusters, 0, B.n_words, 0, 0};
  ctx->lite_ok = false;                     // this input does not suit the block engine: plan on the host from now on
  TRY(upload_async(ctx, B, &v, r, ctx->stream, /*force_full=*/true, /*have_bases=*/true));
  return upload_finish(ctx, B, ctx->stream);
}
}  // namespace

extern "C" int pf_upload(pf_ctx* ctx, const pf_batch* b) {
  if (!ctx) return PF_ERR_INVALID;
  if (!b) return fail(ctx, PF_ERR_INVALID, "pf_upload: null batch");
  CU(cudaSetDevice(ctx->device));
  if (ctx->pipe_pending) return fail(ctx, PF_ERR_STATE, "pf_upload: results of the previous pf_submit were not collected");
  SubRange r{0, b->n_seqs, 0, b->n_clusters, 0, b->n_words, 0, b->n_amb_words};
  TRY(upload_async(ctx, *ctx, b, r, ctx->stream));
  // caller buffers may be pageable: upload_finish makes sure the copies have consumed them
  return upload_finish(ctx, *ctx, ctx->stream);
}
