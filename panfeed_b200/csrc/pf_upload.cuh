// pf_upload.cuh — planning of a batch (device-side: descriptors, offsets, tiles; host-side: MAF
// windows), H2D, pf_upload.
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

// The message for sequence i of the (sub-)batch, which plan_from_raw found to be the first bad one.
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
  if (q.flags & PF_SEQ_AMBIGUOUS) {
    if (!b->amb_codes) return f("seq %u is ambiguous but amb_codes is NULL", i);
    if (q.amb_off & 31u) return f("seq %u: amb_off must be a multiple of 32", i);
    if (q.amb_off + q.len > b->n_amb_words * 16ull) return f("seq %u: symbols run past the 4-bit plane", i);
  }
  return f("seq %u: malformed descriptor", i);
}

// ClusterDev of every cluster of the (sub-)batch: presence popcount, MAF window, filters folded in.
// The record ranges stay zero here; plan_records writes them on the device.
int build_clusters(pf_ctx* ctx, const pf_batch* b, ClusterDev* hc) {
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
    d = ClusterDev{};
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

// Tile list of the local reduce (partition mode): 4096-record tiles for the direct variant, 2048
// for the general one (its exactness guarantee needs <= 2048), from the narrow record ranges.
// local_tiles_count enqueues the counts and their scan; local_tiles_finish, once the total has been
// read back, expands the list.
int local_tiles_count(pf_ctx* ctx, BatchState& B, cudaStream_t st) {
  if (!ctx->partition) return PF_OK;
  const uint32_t nc = B.n_clusters;
  WidthState& w = B.nar;
  B.local_tile = ctx->use_direct ? (uint32_t)kDirectTile : (uint32_t)kLocalTile;
  TRY(dev_ensure(ctx, w.d_ltile_base, ((size_t)nc + 1) * 4));
  if (nc) {
    plan_tile_counts<<<cdiv(nc, 256), 256, 0, st>>>(B.d_clusters.as<ClusterDev>(), nc, B.local_tile, 0,
                                                   w.d_ltile_base.as<uint32_t>());
    ctx->launches++;
  }
  return scan_inplace(ctx, w.d_ltile_base.as<uint32_t>(), nc, &B.d_plan_tot.as<PlanTotals>()->n_ltiles, st,
                      &B.d_bsum_slot);
}
int local_tiles_finish(pf_ctx* ctx, BatchState& B, cudaStream_t st) {
  WidthState& w = B.nar;
  w.n_ltiles = ctx->partition ? B.h_plan_tot.as<PlanTotals>()->n_ltiles : 0;
  if (!w.n_ltiles) return PF_OK;
  TRY(dev_ensure(ctx, w.ltiles, (size_t)w.n_ltiles * sizeof(TileDev)));
  TRY(dev_ensure(ctx, w.tile_first_run, ((size_t)w.n_ltiles + 1) * 4));
  TRY(dev_ensure(ctx, w.lookback, std::max<size_t>((size_t)w.n_tiles * kRadix * 4, (size_t)w.n_ltiles * 8)));
  plan_expand_tiles<<<B.n_clusters, 128, 0, st>>>(B.d_clusters.as<ClusterDev>(), B.n_clusters,
                                                  w.d_ltile_base.as<uint32_t>(), B.local_tile, 0, w.ltiles.as<TileDev>());
  ctx->launches++;
  CU(cudaGetLastError());
  return PF_OK;
}

// Record offsets and tile lists of a batch that runs a record width, on the device, in two halves
// like plan_blocks / plan_blocks_finish.  plan_records enqueues, behind plan_from_raw, the offsets
// of every sequence (SeqDev::rec_off / wrec_off / pos_off / pwide_off, the list of sequences with
// N/IUPAC symbols and their 256-bit positional slots), the record range of every cluster and the
// tile counts; the totals land in PlanTotals.  plan_records_finish, once those have been read
// back, sizes the width buffers and expands the tile lists.
int plan_records(pf_ctx* ctx, BatchState& B, cudaStream_t st) {
  const uint32_t n = B.n_seqs, nc = B.n_clusters;
  const bool long_k = ctx->prm.k > 32;
  const size_t stride = (size_t)n + 1;
  PlanTotals* tot = B.d_plan_tot.as<PlanTotals>();
  TRY(dev_ensure(ctx, B.d_rec_off, kOffFields * stride * 4));
  TRY(dev_ensure(ctx, B.d_wide_seqs, std::max<size_t>(1, n) * 4));
  if (long_k) TRY(dev_ensure(ctx, B.d_xpos_slot, std::max<size_t>(1, n) * 4));
  uint32_t* off = B.d_rec_off.as<uint32_t>();
  if (n) {
    plan_rec_counts<<<cdiv(n, 256), 256, 0, st>>>(B.d_seqs.as<SeqDev>(), n, (int)ctx->prm.k,
                                                 ctx->prm.canonical ? 1u : 2u, long_k, off);
    ctx->launches++;
  }
  for (uint32_t f = 0; f < kOffFields; ++f)
    TRY(scan_inplace(ctx, off + f * stride, n, &tot->seq_tot[f], st, &B.d_bsum_slot));
  if (n) {
    plan_rec_offsets<<<cdiv(n, 256), 256, 0, st>>>(B.d_seqs.as<SeqDev>(), n, long_k, off,
                                                  B.d_wide_seqs.as<uint32_t>(), B.d_xpos_slot.as<uint32_t>());
    ctx->launches++;
  }
  WidthState* widths[3] = {&B.nar, &B.wid, &B.xwd};
  for (WidthState* w : widths) {
    TRY(dev_ensure(ctx, w->seg_start, std::max<size_t>(1, nc) * 4));
    TRY(dev_ensure(ctx, w->d_tile_base, ((size_t)nc + 1) * 4));
  }
  if (nc) {
    plan_cluster_records<<<cdiv(nc, 256), 256, 0, st>>>(B.d_seqs.as<SeqDev>(), n, nc, long_k, off,
                                                       B.d_clusters.as<ClusterDev>(), B.nar.seg_start.as<uint32_t>(),
                                                       B.wid.seg_start.as<uint32_t>(), B.xwd.seg_start.as<uint32_t>(), tot);
    ctx->launches++;
  }
  for (int i = 0; i < 3; ++i) {
    if (nc) {
      plan_tile_counts<<<cdiv(nc, 256), 256, 0, st>>>(B.d_clusters.as<ClusterDev>(), nc, (uint32_t)kSortTile, i,
                                                     widths[i]->d_tile_base.as<uint32_t>());
      ctx->launches++;
    }
    TRY(scan_inplace(ctx, widths[i]->d_tile_base.as<uint32_t>(), nc, &tot->n_tiles[i], st, &B.d_bsum_slot));
  }
  TRY(local_tiles_count(ctx, B, st));
  CU(cudaGetLastError());
  B.records_planned = true;
  return PF_OK;
}
int plan_records_finish(pf_ctx* ctx, BatchState& B, cudaStream_t st) {
  const PlanTotals& t = *B.h_plan_tot.as<PlanTotals>();
  const uint32_t n = B.n_seqs, nc = B.n_clusters;
  const bool long_k = ctx->prm.k > 32;
  B.nar.n_records = long_k ? 0u : t.seq_tot[kOffRec];
  B.wid.n_records = t.seq_tot[kOffWrec];
  B.xwd.n_records = long_k ? t.seq_tot[kOffRec] : 0u;
  B.n_pos_wide = t.seq_tot[kOffPwide];
  B.n_wide_seqs = t.seq_tot[kOffWide];
  B.n_pos_xwide = t.seq_tot[kOffPxwide];
  WidthState* widths[3] = {&B.nar, &B.wid, &B.xwd};
  for (int i = 0; i < 3; ++i) {
    WidthState& w = *widths[i];
    // (the 256-bit width exists only for k > 32 batches with N/IUPAC symbols)
    if (i == 2 && !w.n_records) { w.n_tiles = 0; continue; }
    if (t.max_seg[i] >= (1u << 30))
      return fail(ctx, PF_ERR_INVALID, "a cluster has %u k-mer records; the limit per cluster is 2^30", t.max_seg[i]);
    w.n_tiles = t.n_tiles[i];
    w.max_seg = t.max_seg[i];
    w.sort_bits = auto_sort_bits(ctx, w.max_seg, i == 0);
    w.passes = w.sort_bits / 8;
    TRY(dev_ensure(ctx, w.tiles, std::max<size_t>(1, w.n_tiles) * sizeof(TileDev)));
    TRY(dev_ensure(ctx, w.seg_hist, std::max<size_t>(1, (size_t)nc * w.passes * kRadix) * 4));
    TRY(dev_ensure(ctx, w.lookback, std::max<size_t>(1, (size_t)w.n_tiles * kRadix) * 4));
    if (w.n_tiles) {
      plan_expand_tiles<<<nc, 128, 0, st>>>(B.d_clusters.as<ClusterDev>(), nc, w.d_tile_base.as<uint32_t>(),
                                            kSortTile, i, w.tiles.as<TileDev>());
      ctx->launches++;
    }
  }
  TRY(local_tiles_finish(ctx, B, st));
  // fused first pass: record index -> sequence lookup tables
  if (n) {
    TRY(dev_ensure(ctx, B.d_seq_rec_off, ((size_t)n + 1) * 4));
    TRY(dev_ensure(ctx, B.d_tile_first_seq, ((size_t)B.nar.n_tiles + 1) * 4));
    plan_seq_rec_off<<<cdiv((uint64_t)n + 1, 256), 256, 0, st>>>(B.d_seqs.as<SeqDev>(), n, B.nar.n_records,
                                                                 B.d_seq_rec_off.as<uint32_t>());
    plan_tile_first_seq<<<cdiv((uint64_t)B.nar.n_tiles + 1, 256), 256, 0, st>>>(
        B.nar.tiles.as<TileDev>(), B.nar.n_tiles, B.d_seq_rec_off.as<uint32_t>(), n, B.d_tile_first_seq.as<uint32_t>());
    ctx->launches += 2;
  }
  CU(cudaGetLastError());
  return PF_OK;
}
// The same for a slot that was planned for the block engine only and now runs the record engine
// (pf_execute, after a fall-back): both halves, with one read-back in between.
int plan_records_now(pf_ctx* ctx, BatchState& B, cudaStream_t st) {
  TRY(plan_records(ctx, B, st));
  mirror_counters<<<1, 32, 0, st>>>(B.h_plan_tot.as<uint32_t>(), B.d_plan_tot.as<uint32_t>(), 32);
  CU(cudaStreamSynchronize(st));
  return plan_records_finish(ctx, B, st);
}

// Validate + plan + H2D of the sub-range into the given batch slot, all asynchronous on `st` (the
// caller's buffers must stay valid until `st` has passed).  The host copies the planes and the
// caller's descriptors as they are and builds the per-cluster MAF windows; plan_from_raw validates
// and builds the per-sequence state on the device, plan_records adds record offsets when the batch
// runs a record width, plan_blocks the block engine's work items.  upload_finish completes it.
int upload_async(pf_ctx* ctx, BatchState& B, const pf_batch* full, const SubRange& r, cudaStream_t st) {
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
  B.have_batch = false;
  B.executed = false;
  B.blocks_planned = B.records_planned = false;
  B.n_items = 0;
  const pf_params& P = ctx->prm;
  const uint32_t W = ctx->W, n = b->n_seqs, nc = b->n_clusters;
  if (n && (!b->seqs || !b->packed_bases)) return fail(ctx, PF_ERR_INVALID, "null seqs/packed_bases");
  if (nc && (!b->clusters || !b->cluster_presence)) return fail(ctx, PF_ERR_INVALID, "null clusters/cluster_presence");
  if (nc == 0 && n) return fail(ctx, PF_ERR_INVALID, "sequences without clusters");
  // (pf_execute of another slot may turn block_mode off while this upload runs: read it once)
  const bool blocks = ctx->block_mode;
  if (blocks && n && b->n_words >= (1ull << 32))
    return fail(ctx, PF_ERR_INVALID, "packed plane holds 2^32 words or more; split the batch");
  B.src = view;
  B.src_c0 = r.c0; B.src_b0 = r.w0 * 32ull; B.src_a0 = r.a0 * 16ull;
  const bool amb_plane = b->amb_codes && b->n_amb_words;

  static const bool dbg_up = getenv("PF_DEBUG_PIPE") != nullptr;
  auto now_ms = []() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t_dbg0 = now_ms();
  const size_t slack_words = 80;
  TRY(dev_ensure(ctx, B.d_bases, (b->n_words + slack_words) * 8));
  CU(cudaEventRecord(B.ev_h2d[0], st));
  if (b->n_words) CU(cudaMemcpyAsync(B.d_bases.p, b->packed_bases, b->n_words * 8, cudaMemcpyHostToDevice, st));
  CU(cudaMemsetAsync((char*)B.d_bases.p + b->n_words * 8, 0, slack_words * 8, st));
  // descriptors: straight from the caller's array if it is pinned, else through the slot's pinned
  // staging buffer (a plain copy on the worker threads; a pageable cudaMemcpyAsync would block)
  TRY(dev_ensure(ctx, B.d_raw, std::max<size_t>(1, n) * sizeof(pf_seq_desc)));
  if (n) {
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
  }
  const double t_dbg1 = now_ms();
  // clusters
  TRY(pin_ensure(ctx, B.h_clusters, std::max<size_t>(1, nc) * sizeof(ClusterDev)));
  TRY(build_clusters(ctx, b, B.h_clusters.as<ClusterDev>()));
  const double t_dbg2 = now_ms();
  TRY(dev_ensure(ctx, B.d_seqs, std::max<size_t>(1, n) * sizeof(SeqDev)));
  TRY(dev_ensure(ctx, B.d_seq_lite, std::max<size_t>(1, n) * sizeof(SeqLite)));
  TRY(dev_ensure(ctx, B.d_clusters, std::max<size_t>(1, nc) * sizeof(ClusterDev)));
  TRY(dev_ensure(ctx, B.d_presence, std::max<size_t>(1, (size_t)nc * W) * 4));
  TRY(dev_ensure(ctx, ctx->d_counters, C_COUNT * 4));
  TRY(pin_ensure(ctx, ctx->h_counters, C_COUNT * 4));
  TRY(dev_ensure(ctx, B.d_plan_tot, sizeof(PlanTotals)));
  TRY(pin_ensure(ctx, B.h_plan_tot, sizeof(PlanTotals)));
  if (nc) {
    CU(cudaMemcpyAsync(B.d_clusters.p, B.h_clusters.p, (size_t)nc * sizeof(ClusterDev), cudaMemcpyHostToDevice, st));
    // (the presence words go through a pageable host copy, consumed before cudaMemcpyAsync
    //  returns: straight from a pinned caller array, this small copy lengthened the pipelined
    //  upload of config #2 by ~8 us per sub-batch on a B200)
    const std::vector<uint32_t> presence(b->cluster_presence, b->cluster_presence + (size_t)nc * W);
    CU(cudaMemcpyAsync(B.d_presence.p, presence.data(), (size_t)nc * W * 4, cudaMemcpyHostToDevice, st));
  }
  CU(cudaMemsetAsync(B.d_plan_tot.p, 0, sizeof(PlanTotals), st));
  CU(cudaMemsetAsync(&B.d_plan_tot.as<PlanTotals>()->err, 0xff, 8, st));
  if (n) {
    plan_from_raw<<<cdiv(n, 256), 256, 0, st>>>(B.d_raw.as<pf_seq_desc>(), n, r.c0, B.src_b0, B.src_a0, nc,
                                                 P.n_samples, W, B.d_presence.as<uint32_t>(), b->n_words * 32ull,
                                                 b->amb_codes != nullptr, b->n_amb_words * 16ull, (int)P.k,
                                                 P.emit_positions, B.d_seqs.as<SeqDev>(), B.d_seq_lite.as<SeqLite>(),
                                                 B.d_plan_tot.as<PlanTotals>());
    ctx->launches++;
  }
  if (amb_plane) {
    const size_t bit_words = (b->n_amb_words + 1) / 2 + 4;
    TRY(dev_ensure(ctx, B.d_amb, (b->n_amb_words + 8) * 8));
    TRY(dev_ensure(ctx, B.d_ambbits, bit_words * 4));
    CU(cudaMemcpyAsync(B.d_amb.p, b->amb_codes, b->n_amb_words * 8, cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync((char*)B.d_amb.p + b->n_amb_words * 8, 0, 8 * 8, st));
    k1_amb_bits<<<cdiv(bit_words, 256), 256, 0, st>>>(B.d_amb.as<uint64_t>(), b->n_amb_words,
                                                       B.d_ambbits.as<uint32_t>(), bit_words);
    ctx->launches++;
  }
  B.n_seqs = n; B.n_clusters = nc; B.n_wide_seqs = 0;
  B.n_words = b->n_words; B.n_amb_words = amb_plane ? b->n_amb_words : 0;
  B.n_bases = 0; B.n_pos = 0; B.n_pos_wide = 0; B.n_pos_xwide = 0;   // totals: upload_finish*
  for (WidthState* w : {&B.nar, &B.wid, &B.xwd}) {
    w->n_records = 0; w->n_tiles = 0; w->max_seg = 0; w->sort_bits = 8; w->passes = 1;
  }
  B.nar.n_ltiles = 0;
  // record offsets only for a batch that runs a record width: the record engine, the wide records
  // of sequences with N/IUPAC symbols, the 21-byte positional records.  A block-engine batch that
  // falls back to the record engine gets them in pf_execute.
  if (!blocks || amb_plane || P.emit_positions == 1u) TRY(plan_records(ctx, B, st));
  mirror_counters<<<1, 32, 0, st>>>(B.h_plan_tot.as<uint32_t>(), B.d_plan_tot.as<uint32_t>(), 32);
  CU(cudaEventRecord(B.ev_h2d[1], st));
  if (blocks) {
    TRY(plan_blocks(ctx, B, st, false));
    B.blocks_planned = true;
  }
  CU(cudaEventRecord(B.ev_up_done, st));
  CU(cudaGetLastError());
  if (dbg_up)
    fprintf(stderr, "[pf] upload %u seqs: head %.3f  descriptors %.3f  clusters %.3f  enqueue %.3f ms\n", n,
            t_dbg0 - t_dbg_in, t_dbg1 - t_dbg0, t_dbg2 - t_dbg1, now_ms() - t_dbg2);
  return PF_OK;
}

// After the stream has passed the upload: errors and totals of plan_from_raw, then the host halves
// of the record and block plans
int upload_check(pf_ctx* ctx, BatchState& B, cudaStream_t st) {
  const PlanTotals& t = *B.h_plan_tot.as<PlanTotals>();
  if (t.err != ~0ull) {
    const uint32_t i = (uint32_t)(t.err >> 32);
    if (i < B.n_seqs) return fail(ctx, PF_ERR_INVALID, "%s", describe_bad_seq(ctx, &B.src, i, B.src_c0, B.src_b0, B.src_a0).c_str());
    return fail(ctx, PF_ERR_INVALID, "seq %u: malformed descriptor (check %u)", i, (uint32_t)t.err);
  }
  // (every record width holds at most windows x strands records)
  const uint64_t mult = ctx->prm.canonical ? 1u : 2u;
  if (t.windows * mult >= (1ull << 32) - kSortTile) return fail(ctx, PF_ERR_INVALID, "batch holds more than 2^32 k-mer records; split it");
  if (t.pos_windows >= (1ull << 32)) return fail(ctx, PF_ERR_INVALID, "more than 2^32 positional records; split the batch");
  B.n_bases = t.bases;
  B.nar.n_records = ctx->prm.k > 32 ? 0u : (uint32_t)(t.windows * mult);
  B.n_pos = (uint32_t)t.pos_windows;
  if (B.records_planned) TRY(plan_records_finish(ctx, B, st));
  return PF_OK;
}

// Second half of an upload: wait for the copies and the planning kernels, read n_items back.
int upload_finish(pf_ctx* ctx, BatchState& B, cudaStream_t up) {
  CU(cudaStreamSynchronize(up));
  TRY(upload_check(ctx, B, up));
  if (B.blocks_planned) TRY(plan_blocks_finish(ctx, B, up));
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
  TRY(upload_check(ctx, B, compute));
  if (B.blocks_planned) TRY(plan_blocks_finish(ctx, B, compute, false));
  CU(cudaGetLastError());
  B.have_batch = true;
  return PF_OK;
}
}  // namespace

extern "C" int pf_upload(pf_ctx* ctx, const pf_batch* b) {
  if (!ctx) return PF_ERR_INVALID;
  if (!b) return fail(ctx, PF_ERR_INVALID, "pf_upload: null batch");
  CU(cudaSetDevice(ctx->device));
  if (ctx->pipe_pending) return fail(ctx, PF_ERR_STATE, "pf_upload: results of the previous pf_submit were not collected");
  ctx->assoc.batch_ready = false;
  SubRange r{0, b->n_seqs, 0, b->n_clusters, 0, b->n_words, 0, b->n_amb_words};
  TRY(upload_async(ctx, *ctx, b, r, ctx->stream));
  // caller buffers may be pageable: upload_finish makes sure the copies have consumed them
  return upload_finish(ctx, *ctx, ctx->stream);
}
