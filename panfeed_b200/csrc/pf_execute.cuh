// pf_execute.cuh — stage launchers and pf_execute: the kernel sequence of one resident batch.
// Part of libpanfeed_b200.so's single translation unit: included once, in order, by pf_api.cu.

namespace {

template <typename KeyT>
int hist_width(pf_ctx* ctx, WidthState& w, bool fused = false) {
  if (w.n_records == 0) return PF_OK;
  cudaStream_t st = ctx->stream;
  const int shift0 = KeyTraits<KeyT>::kBits - w.sort_bits;
  const uint32_t n_seg = ctx->n_clusters;
  CU(cudaMemsetAsync(w.seg_hist.p, 0, (size_t)n_seg * w.passes * kRadix * 4, st));
  if (fused) {
    const uint32_t chunks = cdiv(ctx->n_seqs, kHistSeqsPerChunk);
    const uint32_t grid = std::min<uint32_t>(cdiv(chunks, kK1Warps), 148 * 8);
    if (ctx->prm.canonical)
      k1_histogram_fused<true><<<grid, kK1Warps * 32, 0, st>>>(
          ctx->d_bases.as<uint64_t>(), ctx->d_ambbits.as<uint32_t>(), ctx->d_seqs.as<SeqDev>(), ctx->n_seqs,
          (int)ctx->prm.k, w.passes, shift0, w.seg_hist.as<uint32_t>());
    else
      k1_histogram_fused<false><<<grid, kK1Warps * 32, 0, st>>>(
          ctx->d_bases.as<uint64_t>(), ctx->d_ambbits.as<uint32_t>(), ctx->d_seqs.as<SeqDev>(), ctx->n_seqs,
          (int)ctx->prm.k, w.passes, shift0, w.seg_hist.as<uint32_t>());
    const uint32_t rows = n_seg * w.passes;
    k2_scan_histogram<<<cdiv(rows, 8), 256, 0, st>>>(w.seg_hist.as<uint32_t>(), w.seg_start.as<uint32_t>(), rows, w.passes);
    ctx->launches += 2;
    CU(cudaGetLastError());
    return PF_OK;
  }
  const uint32_t hist_ctas = std::min<uint32_t>(w.n_tiles, 148 * 8);
  const uint32_t per = cdiv(w.n_tiles, hist_ctas);
  k2_histogram<KeyT><<<cdiv(w.n_tiles, per), 256, 0, st>>>(w.keys[0].as<KeyT>(), w.tiles.as<TileDev>(),
                                                           w.n_tiles, per, w.passes, shift0,
                                                           w.seg_hist.as<uint32_t>());
  const uint32_t rows = n_seg * w.passes;
  k2_scan_histogram<<<cdiv(rows, 8), 256, 0, st>>>(w.seg_hist.as<uint32_t>(), w.seg_start.as<uint32_t>(), rows, w.passes);
  ctx->launches += 2;
  CU(cudaGetLastError());
  return PF_OK;
}

template <typename KeyT>
int passes_width(pf_ctx* ctx, WidthState& w, int ticket_idx, bool unstable = false, bool fused = false) {
  if (w.n_records == 0) { w.final_buf = 0; return PF_OK; }
  cudaStream_t st = ctx->stream;
  const int shift0 = KeyTraits<KeyT>::kBits - w.sort_bits;
  uint32_t* counters = ctx->d_counters.as<uint32_t>();
  int src = 0;
  for (int p = 0; p < w.passes; ++p) {
    const bool atomic_pass = (fused || unstable) && p == 0;
    if (atomic_pass) {
      const size_t hist_bytes = (size_t)ctx->n_clusters * w.passes * kRadix * 4;
      TRY(dev_ensure(ctx, w.cursors, std::max<size_t>(hist_bytes, 4)));
      CU(cudaMemcpyAsync(w.cursors.p, w.seg_hist.p, hist_bytes, cudaMemcpyDeviceToDevice, st));
    } else {
      CU(cudaMemsetAsync(w.lookback.p, 0, (size_t)w.n_tiles * kRadix * 4, st));
      CU(cudaMemsetAsync(counters + ticket_idx, 0, 4, st));
    }
    if (fused && p == 0) {
      if (ctx->prm.canonical)
        k2_extract_scatter<true><<<w.n_tiles, kSortThreads, sizeof(ScatterSmem<uint64_t>), st>>>(
            ctx->d_bases.as<uint64_t>(), ctx->d_ambbits.as<uint32_t>(), ctx->d_seqs.as<SeqDev>(),
            ctx->d_seq_rec_off.as<uint32_t>(), ctx->n_seqs, ctx->d_tile_first_seq.as<uint32_t>(), (int)ctx->prm.k,
            w.keys[src ^ 1].template as<uint64_t>(), w.vals[src ^ 1].template as<uint32_t>(), w.tiles.template as<TileDev>(),
            w.n_tiles, w.cursors.template as<uint32_t>(), w.passes, shift0);
      else
        k2_extract_scatter<false><<<w.n_tiles, kSortThreads, sizeof(ScatterSmem<uint64_t>), st>>>(
            ctx->d_bases.as<uint64_t>(), ctx->d_ambbits.as<uint32_t>(), ctx->d_seqs.as<SeqDev>(),
            ctx->d_seq_rec_off.as<uint32_t>(), ctx->n_seqs, ctx->d_tile_first_seq.as<uint32_t>(), (int)ctx->prm.k,
            w.keys[src ^ 1].template as<uint64_t>(), w.vals[src ^ 1].template as<uint32_t>(), w.tiles.template as<TileDev>(),
            w.n_tiles, w.cursors.template as<uint32_t>(), w.passes, shift0);
    } else if (unstable && p == 0)   // LSD: only the first pass may ignore the incoming order
      k2_scatter_pass<KeyT><<<w.n_tiles, kSortThreads, sizeof(ScatterSmem<KeyT>), st>>>(
          w.keys[src].as<KeyT>(), w.vals[src].as<uint32_t>(), w.keys[src ^ 1].as<KeyT>(),
          w.vals[src ^ 1].as<uint32_t>(), w.tiles.as<TileDev>(), w.n_tiles, w.cursors.as<uint32_t>(), p,
          w.passes, shift0 + 8 * p);
    else
      k2_onesweep_pass<KeyT><<<w.n_tiles, kSortThreads, sizeof(SortSmem<KeyT>), st>>>(
          w.keys[src].as<KeyT>(), w.vals[src].as<uint32_t>(), w.keys[src ^ 1].as<KeyT>(),
          w.vals[src ^ 1].as<uint32_t>(), w.tiles.as<TileDev>(), w.n_tiles, w.seg_hist.as<uint32_t>(), p,
          w.passes, shift0 + 8 * p, w.lookback.as<uint32_t>(), counters + ticket_idx, counters + C_ERR);
    ctx->launches++;
    src ^= 1;
  }
  w.final_buf = src;
  CU(cudaGetLastError());
  return PF_OK;
}

template <typename KeyT>
int mark_width(pf_ctx* ctx, WidthState& w, int ticket_idx, int runs_idx, bool local_tiles) {
  if (w.n_records == 0) return PF_OK;
  cudaStream_t st = ctx->stream;
  uint32_t* counters = ctx->d_counters.as<uint32_t>();
  const int other = w.final_buf ^ 1;
  // the idle ping-pong buffers hold the run lists: keys[other] = run_start | run_seg, vals[other] = nrows
  uint32_t* run_start = w.keys[other].as<uint32_t>();
  uint32_t* run_seg = run_start + ((size_t)w.n_records + 1);
  const uint32_t nt = local_tiles ? w.n_ltiles : w.n_tiles;
  CU(cudaMemsetAsync(w.lookback.p, 0, (size_t)nt * 8, st));
  CU(cudaMemsetAsync(counters + ticket_idx, 0, 4, st));
  if (local_tiles && ctx->local_tile == (uint32_t)kDirectTile)
    k3_mark_runs<KeyT, kDirectTile / kSortThreads><<<nt, kSortThreads, 0, st>>>(
        w.keys[w.final_buf].as<KeyT>(), w.ltiles.as<TileDev>(), nt, w.sort_bits, run_start, run_seg,
        w.tile_first_run.as<uint32_t>(), w.lookback.as<uint64_t>(), counters + ticket_idx,
        counters + runs_idx, counters + C_ERR);
  else if (local_tiles)
    k3_mark_runs<KeyT, kLocalItems><<<nt, kSortThreads, 0, st>>>(
        w.keys[w.final_buf].as<KeyT>(), w.ltiles.as<TileDev>(), nt, w.sort_bits, run_start, run_seg,
        w.tile_first_run.as<uint32_t>(), w.lookback.as<uint64_t>(), counters + ticket_idx,
        counters + runs_idx, counters + C_ERR);
  else
    k3_mark_runs<KeyT, kSortItems><<<nt, kSortThreads, 0, st>>>(
        w.keys[w.final_buf].as<KeyT>(), w.tiles.as<TileDev>(), nt, w.sort_bits, run_start, run_seg,
        nullptr, w.lookback.as<uint64_t>(), counters + ticket_idx, counters + runs_idx, counters + C_ERR);
  ctx->launches++;
  CU(cudaGetLastError());
  return PF_OK;
}

int scan_inplace(pf_ctx* ctx, uint32_t* data, uint32_t n, uint32_t* total_dev, cudaStream_t st, DevBuf* scratch) {
  if (!st) st = ctx->stream;
  DevBuf& bsum = scratch ? *scratch : ctx->d_bsum;
  const uint32_t nb = std::max(1u, cdiv(n, kScanBlock));
  TRY(dev_ensure(ctx, bsum, ((size_t)nb + 1) * 4));
  scan_block_sums<<<nb, 256, 0, st>>>(data, n, bsum.as<uint32_t>());
  scan_of_sums<<<1, 1024, 0, st>>>(bsum.as<uint32_t>(), nb, total_dev);
  scan_apply<<<nb, 256, 0, st>>>(data, n, bsum.as<uint32_t>(), nb);
  ctx->launches += 3;
  CU(cudaGetLastError());
  return PF_OK;
}

// n_unique (COUNT pass, may be null): += the distinct live keys of the runs
template <typename KeyT, bool EMIT>
int runs_width(pf_ctx* ctx, WidthState& w, RowOut out, uint32_t* n_unique = nullptr) {
  if (w.n_runs == 0) return PF_OK;
  cudaStream_t st = ctx->stream;
  const int other = w.final_buf ^ 1;
  uint32_t* run_start = w.keys[other].as<uint32_t>();
  uint32_t* run_seg = run_start + ((size_t)w.n_records + 1);
  uint32_t* nrows = w.vals[other].as<uint32_t>();
  const size_t smem = (size_t)8 * ctx->W * 4;
  const uint32_t grid = std::min<uint32_t>(cdiv(w.n_runs, 8), kGridPersist * 2);
  k3_runs<KeyT, EMIT><<<grid, 256, smem, st>>>(w.keys[w.final_buf].as<KeyT>(), w.vals[w.final_buf].as<uint32_t>(),
                                               run_start, run_seg, w.n_runs, w.n_records,
                                               ctx->d_clusters.as<ClusterDev>(), nrows, out, n_unique);
  ctx->launches++;
  CU(cudaGetLastError());
  return PF_OK;
}

// Ensure the table of a pattern space can take `extra` more patterns at <= 50 % load.
int table_reserve(pf_ctx* ctx, PatternSpace& s, uint64_t extra) {
  cudaStream_t st = ctx->stream;
  const uint64_t need = (s.n + extra) * 2 + 16;
  if (need >= (1ull << 31)) return fail(ctx, PF_ERR_NOMEM, "pattern table would exceed 2^31 slots");
  TRY(pool_ensure(ctx, s.pool, std::max<size_t>(1, (s.n + extra)) * s.key_words * 4));
  if (need <= s.table_size) return PF_OK;
  uint32_t size = std::max<uint32_t>(1024, s.table_size);
  while (size < need) size *= 2;
  DevBuf nt;
  TRY(dev_ensure(ctx, nt, (size_t)size * 4));
  CU(cudaMemsetAsync(nt.p, 0xff, (size_t)size * 4, st));
  if (s.n) {
    k4_rehash<<<std::min<uint32_t>(cdiv(s.n, 8), kGridPersist), 256, 0, st>>>(
        s.pool.as<uint32_t>(), (uint32_t)s.n, s.key_words, nt.as<uint32_t>(), size - 1);
    ctx->launches++;
  }
  CU(cudaStreamSynchronize(st));
  if (s.table.p) CU(cudaFree(s.table.p));
  s.table = nt;
  s.table_size = size;
  return PF_OK;
}

// Dedup n candidate keys against a pattern space; ids to `ids_out`, number of
// new patterns to counters[new_idx] (device).
int dedup(pf_ctx* ctx, PatternSpace& s, const uint32_t* cand, uint32_t n, DevBuf& rep, DevBuf& slot_of,
          DevBuf& winner, uint32_t* ids_out, int new_idx) {
  cudaStream_t st = ctx->stream;
  uint32_t* counters = ctx->d_counters.as<uint32_t>();
  if (n == 0) { CU(cudaMemsetAsync(counters + new_idx, 0, 4, st)); return PF_OK; }
  TRY(table_reserve(ctx, s, n));
  TRY(dev_ensure(ctx, rep, (size_t)n * 4));
  TRY(dev_ensure(ctx, slot_of, (size_t)n * 4));
  TRY(dev_ensure(ctx, winner, ((size_t)n + 1) * 4));
  // lanes per row: at most 4 words per lane
  const int L = s.key_words <= 16 ? 4 : s.key_words <= 32 ? 8 : s.key_words <= 64 ? 16 : 32;
  const uint32_t grid = std::min<uint32_t>(cdiv(n, 256 / L), kGridPersist * 4);
#define PF_K4(LL)                                                                                      \
  do {                                                                                                 \
    k4_probe<LL><<<grid, 256, 0, st>>>(cand, n, s.key_words, s.pool.as<uint32_t>(), s.table.as<uint32_t>(), \
                                       s.table_size - 1, rep.as<uint32_t>(), slot_of.as<uint32_t>(),   \
                                       winner.as<uint32_t>());                                         \
    ctx->launches++;                                                                                   \
    TRY(scan_inplace(ctx, winner.as<uint32_t>(), n, counters + new_idx));                              \
    k4_commit<LL><<<grid, 256, 0, st>>>(cand, n, s.key_words, s.pool.as<uint32_t>(), (uint32_t)s.n,     \
                                        s.table.as<uint32_t>(), rep.as<uint32_t>(), slot_of.as<uint32_t>(), \
                                        winner.as<uint32_t>(), ids_out);                               \
    ctx->launches++;                                                                                   \
  } while (0)
  if (L == 4) PF_K4(4); else if (L == 8) PF_K4(8); else if (L == 16) PF_K4(16); else PF_K4(32);
#undef PF_K4
  CU(cudaGetLastError());
  return PF_OK;
}

// A previous pf_execute that was never collected: fold its new-pattern count in.
int finalize_pending(pf_ctx* ctx) {
  if (!ctx->kp_pending) return PF_OK;
  CU(cudaStreamSynchronize(ctx->stream));
  // (a row prefetch of results nobody collected may still be draining on the copy stream: it is
  //  not waited for — the next prefetch queues behind it on that stream, pf_collect syncs it)
  ctx->kp.n = ctx->kp_pending_base + *ctx->kp_pending_count;
  ctx->kp_pending = false;
  return PF_OK;
}

void fill_timings(pf_ctx* ctx, const BatchState* slot = nullptr) {
  const BatchState& B = slot ? *slot : *ctx;
  pf_stats& s = ctx->stats;
  auto ms = [](cudaEvent_t a, cudaEvent_t b) { float m = 0; if (cudaEventElapsedTime(&m, a, b) != cudaSuccess) { cudaGetLastError(); m = 0; } return m; };
  s.ms_h2d = ms(B.ev_h2d[0], B.ev_h2d[1]);
  s.ms_extract = ms(B.ev[EV_START], B.ev[EV_EXTRACT]);
  s.ms_hist = ms(B.ev[EV_EXTRACT], B.ev[EV_HIST]);
  s.ms_sort = ms(B.ev[EV_HIST], B.ev[EV_SORT]);
  s.ms_mark = ms(B.ev[EV_SORT], B.ev[EV_MARK]);
  s.ms_count = ms(B.ev[EV_MARK], B.ev[EV_COUNTED]);
  s.ms_reduce = ms(B.ev[EV_COUNTED], B.ev[EV_REDUCE]);
  s.ms_dedup = ms(B.ev[EV_REDUCE], B.ev[EV_DEDUP]);
  s.ms_total = ms(B.ev[EV_START], B.ev[EV_END]);
  s.sort_passes = (uint32_t)ctx->nar.passes;
  s.engine = ctx->used_block ? 2u : (ctx->partition ? 0u : 1u);
  s.block_windows = ctx->block_windows;
  s.block_slots = ctx->blk_slots;
  s.partial_rows = ctx->used_block ? ctx->partials_last : 0;
  s.sub_batches = ctx->pipe_subs;
}

int check_device_error(pf_ctx* ctx) {
  const uint32_t e = ctx->h_counters.as<uint32_t>()[C_ERR];
  if (e) return fail(ctx, PF_ERR_INTERNAL, "device watchdog: look-back chain stalled (code %u)", e);
  return PF_OK;
}

}  // namespace

namespace {

int ensure_rows(pf_ctx* ctx, uint64_t rows, uint64_t narrow_rows, bool keep) {
  TRY(dev_ensure(ctx, ctx->d_row_cluster, std::max<size_t>(1, rows) * 4, keep));
  TRY(dev_ensure(ctx, ctx->d_row_count, std::max<size_t>(1, rows) * 4, keep));
  TRY(dev_ensure(ctx, ctx->d_row_pattern, std::max<size_t>(1, rows) * 4, keep));
  TRY(dev_ensure(ctx, ctx->d_row_kmer, std::max<size_t>(1, narrow_rows) * 8, keep));
  TRY(dev_ensure(ctx, ctx->d_cand, std::max<size_t>(1, rows) * ctx->Wk * 4, keep));
  return PF_OK;
}

int launch_k1(pf_ctx* ctx) {
  cudaStream_t st = ctx->stream;
  const pf_params& P = ctx->prm;
  WidthState& N = ctx->nar;
  WidthState& Wd = ctx->wid;
  PosOut po{ctx->d_pos_kmer.as<uint64_t>(), ctx->d_pos_seq.as<uint32_t>(), ctx->d_pos_cstart.as<int32_t>(),
            ctx->d_pos_gstart.as<int32_t>(), ctx->d_pos_flags.as<uint8_t>()};
  const bool compact = ctx->prm.emit_positions == 2u;
  if (compact && ctx->n_pos && P.canonical && ctx->n_seqs && P.k <= 32) {
    // compact positional form: one bit per window of the target sequences, nothing else
    const uint32_t grid = std::min<uint32_t>(cdiv(ctx->n_seqs, kK1Warps), 148 * 8);
    k1_strand_bits<<<grid, kK1Warps * 32, 0, st>>>(ctx->d_bases.as<uint64_t>(), ctx->d_seqs.as<SeqDev>(), ctx->n_seqs,
                                                   (int)P.k, ctx->d_pos_bits.as<uint32_t>());
    ctx->launches++;
  }
  if (compact) po = PosOut{nullptr, nullptr, nullptr, nullptr, nullptr};   // k1_extract: no positional records
  if (ctx->n_seqs && N.n_records && !(ctx->fused && (ctx->n_pos == 0 || compact))) {
    const uint32_t grid = std::min<uint32_t>(cdiv(ctx->n_seqs, kK1Warps), 148 * 8);
#define PF_K1(CANON, REC)                                                                              \
    k1_extract<CANON, REC><<<grid, kK1Warps * 32, 0, st>>>(ctx->d_bases.as<uint64_t>(), ctx->d_ambbits.as<uint32_t>(), \
                                                      ctx->d_seqs.as<SeqDev>(), ctx->n_seqs, (int)P.k,  \
                                                      N.keys[0].as<uint64_t>(), N.vals[0].as<uint32_t>(), po)
    if (ctx->fused) { if (P.canonical) PF_K1(true, false); else PF_K1(false, false); }
    else { if (P.canonical) PF_K1(true, true); else PF_K1(false, true); }
#undef PF_K1
    ctx->launches++;
  }
  if (P.k > 32 && ctx->n_seqs && Wd.n_records) {
    // two-word k-mers: records, positional records (or the used_strand plane) of every window
    const uint32_t grid = std::min<uint32_t>(cdiv(ctx->n_seqs, kK1Warps), 148 * 8);
    uint32_t* bits = compact && ctx->n_pos && P.canonical ? ctx->d_pos_bits.as<uint32_t>() : nullptr;
    if (P.canonical)
      k1_extract_long<true><<<grid, kK1Warps * 32, 0, st>>>(ctx->d_bases.as<uint64_t>(), ctx->d_ambbits.as<uint32_t>(),
                                                            ctx->d_seqs.as<SeqDev>(), ctx->n_seqs,
                                                            (int)P.k, Wd.keys[0].as<Key128>(), Wd.vals[0].as<uint32_t>(), po,
                                                            ctx->d_pos_wide.as<uint64_t>(), bits);
    else
      k1_extract_long<false><<<grid, kK1Warps * 32, 0, st>>>(ctx->d_bases.as<uint64_t>(), ctx->d_ambbits.as<uint32_t>(),
                                                             ctx->d_seqs.as<SeqDev>(), ctx->n_seqs,
                                                             (int)P.k, Wd.keys[0].as<Key128>(), Wd.vals[0].as<uint32_t>(), po,
                                                             ctx->d_pos_wide.as<uint64_t>(), nullptr);
    ctx->launches++;
    WidthState& X = ctx->xwd;
    if (ctx->n_wide_seqs && X.n_records) {
      // windows holding N/IUPAC symbols: 256-bit records, and their positional records / strand
      // bits corrected behind k1_extract_long (same stream)
      const uint32_t xg = std::min<uint32_t>(cdiv(ctx->n_wide_seqs, 8), 148 * 8);
      uint64_t* pk = compact ? nullptr : ctx->d_pos_kmer.as<uint64_t>();
      uint64_t* px = compact ? nullptr : ctx->d_pos_xwide.as<uint64_t>();
      if (P.canonical)
        k1_extract_wide<true, Key256><<<xg, 256, 0, st>>>(ctx->d_amb.as<uint64_t>(), ctx->d_seqs.as<SeqDev>(),
                                                          ctx->d_wide_seqs.as<uint32_t>(), ctx->n_wide_seqs, (int)P.k,
                                                          X.keys[0].as<Key256>(), X.vals[0].as<uint32_t>(), px,
                                                          ctx->d_pos_flags.as<uint8_t>(), bits, pk,
                                                          ctx->d_xpos_slot.as<uint32_t>());
      else
        k1_extract_wide<false, Key256><<<xg, 256, 0, st>>>(ctx->d_amb.as<uint64_t>(), ctx->d_seqs.as<SeqDev>(),
                                                           ctx->d_wide_seqs.as<uint32_t>(), ctx->n_wide_seqs, (int)P.k,
                                                           X.keys[0].as<Key256>(), X.vals[0].as<uint32_t>(), px,
                                                           ctx->d_pos_flags.as<uint8_t>(), nullptr, pk,
                                                           ctx->d_xpos_slot.as<uint32_t>());
      ctx->launches++;
    }
  } else if (ctx->n_wide_seqs && Wd.n_records) {
    const uint32_t grid = std::min<uint32_t>(cdiv(ctx->n_wide_seqs, 8), 148 * 8);
    if (P.canonical)
      k1_extract_wide<true, Key128><<<grid, 256, 0, st>>>(ctx->d_amb.as<uint64_t>(), ctx->d_seqs.as<SeqDev>(),
                                                          ctx->d_wide_seqs.as<uint32_t>(), ctx->n_wide_seqs, (int)P.k,
                                                          Wd.keys[0].as<Key128>(), Wd.vals[0].as<uint32_t>(),
                                                          ctx->d_pos_wide.as<uint64_t>(), ctx->d_pos_flags.as<uint8_t>(),
                                                          compact && ctx->n_pos ? ctx->d_pos_bits.as<uint32_t>() : nullptr);
    else
      k1_extract_wide<false, Key128><<<grid, 256, 0, st>>>(ctx->d_amb.as<uint64_t>(), ctx->d_seqs.as<SeqDev>(),
                                                           ctx->d_wide_seqs.as<uint32_t>(), ctx->n_wide_seqs, (int)P.k,
                                                           Wd.keys[0].as<Key128>(), Wd.vals[0].as<uint32_t>(),
                                                           compact ? nullptr : ctx->d_pos_wide.as<uint64_t>(),
                                                           ctx->d_pos_flags.as<uint8_t>(), nullptr);
    ctx->launches++;
  }
  CU(cudaGetLastError());
  return PF_OK;
}

int launch_local(pf_ctx* ctx, RowOut ro, uint32_t n_rescue = 0) {
  WidthState& N = ctx->nar;
  if (N.n_records == 0) return PF_OK;
  cudaStream_t st = ctx->stream;
  uint32_t* counters = ctx->d_counters.as<uint32_t>();
  const int other = N.final_buf ^ 1;
  const uint32_t* run_start = ctx->runs_from_hist ? N.seg_hist.as<uint32_t>() : N.keys[other].as<uint32_t>();
  const uint32_t* run_seg = ctx->runs_from_hist ? nullptr : N.keys[other].as<uint32_t>() + ((size_t)N.n_records + 1);
  uint32_t* rescue = N.vals[other].as<uint32_t>();       // idle in partition mode
  const uint32_t cap = (uint32_t)std::min<uint64_t>(ctx->row_cap, 0x7fffffffu);
  if (n_rescue) {
    // second launch of the direct variant: one CTA per run of the tiles that overflowed;
    // rows/unique counters keep accumulating
    k3_local_direct<<<n_rescue, kLocalThreads, sizeof(DirectSmem), st>>>(
        N.keys[N.final_buf].as<uint64_t>(), N.vals[N.final_buf].as<uint32_t>(), N.ltiles.as<TileDev>(),
        N.n_ltiles, N.tile_first_run.as<uint32_t>(), run_start, N.n_records,
        ctx->d_clusters.as<ClusterDev>(), ro, cap, counters + C_LOCAL, rescue, rescue, run_seg);
    ctx->launches++;
    CU(cudaGetLastError());
    return PF_OK;
  }
  CU(cudaMemsetAsync(counters + C_LOCAL, 0, 5 * 4, st));
  if (ctx->use_direct)
    k3_local_direct<<<N.n_ltiles, kLocalThreads, sizeof(DirectSmem), st>>>(
        N.keys[N.final_buf].as<uint64_t>(), N.vals[N.final_buf].as<uint32_t>(), N.ltiles.as<TileDev>(),
        N.n_ltiles, N.tile_first_run.as<uint32_t>(), run_start, N.n_records,
        ctx->d_clusters.as<ClusterDev>(), ro, cap, counters + C_LOCAL, rescue, nullptr, run_seg);
  else
    k3_local<<<N.n_ltiles, kLocalThreads, sizeof(LocalSmem), st>>>(
        N.keys[N.final_buf].as<uint64_t>(), N.vals[N.final_buf].as<uint32_t>(), N.ltiles.as<TileDev>(),
        N.n_ltiles, N.tile_first_run.as<uint32_t>(), run_start, N.n_records,
        ctx->d_clusters.as<ClusterDev>(), ro, cap, counters + C_LOCAL);
  ctx->launches++;
  CU(cudaGetLastError());
  return PF_OK;
}

// ---- block aggregation: work items = (cluster, position block) -----------------------
// (re)computes the per-cluster block counts for ctx->block_windows; syncs to learn n_items
int plan_blocks(pf_ctx* ctx, BatchState& B, cudaStream_t st, bool sync) {
  const uint32_t nc = B.n_clusters;
  B.n_items = 0;
  if (nc == 0 || B.n_seqs == 0) return PF_OK;
  TRY(dev_ensure(ctx, B.d_cblk, (size_t)nc * sizeof(ClusterBlk)));
  TRY(dev_ensure(ctx, B.d_item_base, ((size_t)nc + 1) * 4));
  TRY(dev_ensure(ctx, B.d_plan_total, 16));
  TRY(pin_ensure(ctx, B.h_plan, 16));
  plan_cluster_blocks<<<cdiv((uint64_t)nc * 32, 256), 256, 0, st>>>(
      B.d_seqs.as<SeqDev>(), B.n_seqs, nc, (int)ctx->prm.k, ctx->block_windows,
      B.d_cblk.as<ClusterBlk>(), B.d_item_base.as<uint32_t>());
  TRY(scan_inplace(ctx, B.d_item_base.as<uint32_t>(), nc, B.d_plan_total.as<uint32_t>(), st, &B.d_bsum_slot));
  if (ctx->n_slices > 1) {
    TRY(dev_ensure(ctx, B.d_slice_seq, (size_t)nc * (ctx->n_slices + 1) * 4));
    plan_cluster_slices<<<cdiv((uint64_t)nc * 32, 256), 256, 0, st>>>(
        B.d_seqs.as<SeqDev>(), B.d_cblk.as<ClusterBlk>(), nc, ctx->n_slices, ctx->slice_samples,
        B.d_slice_seq.as<uint32_t>());
  }
  // n_items is read back through pinned memory (no copy engine); plan_blocks_finish takes it
  mirror_counters<<<1, 32, 0, st>>>(B.h_plan.as<uint32_t>(), B.d_plan_total.as<uint32_t>(), 1);
  CU(cudaGetLastError());
  if (sync) return plan_blocks_finish(ctx, B, st);
  return PF_OK;
}
// after the stream has passed plan_blocks: the item -> cluster map
int plan_blocks_finish(pf_ctx* ctx, BatchState& B, cudaStream_t st, bool sync) {
  const uint32_t nc = B.n_clusters;
  if (nc == 0 || B.n_seqs == 0) return PF_OK;
  if (sync) CU(cudaStreamSynchronize(st));     // (else the caller has waited for plan_blocks)
  B.n_items = B.h_plan.as<uint32_t>()[0];
  TRY(dev_ensure(ctx, B.d_item_cluster, std::max<size_t>(1, B.n_items) * 4));
  plan_expand_owner<<<cdiv((uint64_t)nc * 32, 256), 256, 0, st>>>(B.d_item_base.as<uint32_t>(), nc,
                                                                  B.d_item_cluster.as<uint32_t>());
  const uint64_t n_ka = (uint64_t)B.n_items * ctx->n_slices;
  if (n_ka >= (1ull << 31)) return fail(ctx, PF_ERR_INVALID, "too many (cluster, run, slice) work items; split the batch");
  TRY(dev_ensure(ctx, B.d_item_desc, std::max<size_t>(1, n_ka) * 16));
  if (n_ka)
    plan_item_desc<<<cdiv(n_ka, 256), 256, 0, st>>>(
        B.d_item_base.as<uint32_t>(), B.d_item_cluster.as<uint32_t>(), B.d_cblk.as<ClusterBlk>(),
        ctx->n_slices > 1 ? B.d_slice_seq.as<uint32_t>() : nullptr, B.n_items, ctx->n_slices,
        (uint32_t)kBlkRun, B.d_item_desc.as<uint4>());
  CU(cudaGetLastError());
  return PF_OK;
}

BlkPlan block_plan(const pf_ctx* ctx) {
  BlkPlan bp;
  bp.item_base = ctx->d_item_base.as<uint32_t>();
  bp.item_cluster = ctx->d_item_cluster.as<uint32_t>();
  bp.cblk = ctx->d_cblk.as<ClusterBlk>();
  bp.n_clusters = ctx->n_clusters;
  bp.block_windows = ctx->block_windows;
  bp.slots = ctx->blk_slots;
  bp.cap = ctx->blk_cap;
  bp.cslots = ctx->blk_cslots;
  bp.W = ctx->Ws;
  bp.WP = (ctx->Ws + 3u) & ~3u;
  bp.n_slices = ctx->n_slices;
  bp.slice_samples = ctx->slice_samples;
  bp.slice_seq = ctx->n_slices > 1 ? ctx->d_slice_seq.as<uint32_t>() : nullptr;
  bp.item_desc = ctx->d_item_desc.as<uint4>();
  bp.n_run_items = ctx->n_items;
  return bp;
}

// items == nullptr: all (cluster, block) items with the context's table size, in segments of
// consecutive runs; else the listed items (a rescue launch, one CTA and one run per item) with
// `slots` slots.  Items that overflow are appended to `rescue_out`.
int launch_block_aggregate(pf_ctx* ctx, const uint32_t* items, uint32_t n, uint32_t slots, uint32_t cap,
                           uint32_t cslots, uint32_t* rescue_out) {
  if (n == 0) return PF_OK;
  cudaStream_t st = ctx->stream;
  BlkPlan bp = block_plan(ctx);
  bp.slots = slots;
  bp.cap = cap;
  bp.cslots = cslots;
  const uint32_t cap32 = (uint32_t)std::min<uint64_t>(ctx->partial_cap, 0xfffffff0u);
  uint32_t* counters = ctx->d_counters.as<uint32_t>() + C_LOCAL;
  const uint32_t smem = blkA_smem_bytes(slots, cap, cslots, ctx->Ws);
  auto kernel = ctx->prm.canonical ? kA_block_aggregate<true> : kA_block_aggregate<false>;
  uint32_t grid = n, n_segs = n, seg_runs = 1;
  if (!items) {
    // a grid of resident CTAs takes segments from counters[LC_SEGMENT] (zeroed with the other
    // C_LOCAL words before kA).  Longer segments share more of the per-run set-up, but the GPU
    // must stay full: segments are halved while there are fewer than 4 per resident CTA.
    int sms = 0, dev = 0, per_sm = 0;
    CU(cudaGetDevice(&dev));
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kBlkThreads, smem));
    const uint32_t resident = (uint32_t)std::max(1, sms * per_sm);
    seg_runs = ctx->ka_seg_runs;
    if (seg_runs == 0) {
      seg_runs = 16;
      while (seg_runs > 1 && (uint64_t)cdiv(ctx->n_items, seg_runs) * ctx->n_slices < 4ull * resident) seg_runs /= 2;
    }
    n_segs = cdiv(ctx->n_items, seg_runs) * ctx->n_slices;
    grid = std::min(n_segs, resident);
  }
  kernel<<<grid, kBlkThreads, smem, st>>>(
      ctx->d_bases.as<uint64_t>(), ctx->d_ambbits.as<uint32_t>(), ctx->d_seq_lite.as<SeqLite>(), bp,
      (int)ctx->prm.k, ctx->d_slab_keys.as<uint64_t>(), ctx->d_slab_rows.as<uint32_t>(),
      ctx->d_slab_base.as<uint32_t>(), ctx->d_slab_count.as<uint32_t>(), ctx->d_slab_cnt.as<uint32_t>(),
      cap32, counters, items, n_segs, seg_runs, rescue_out);
  ctx->launches++;
  CU(cudaGetLastError());
  return PF_OK;
}

// kB1 + kB3 (kB1, kB4, kB5 with sample slices) over the `n_partials` partial rows kA left
int launch_block_merge(pf_ctx* ctx, RowOut ro, uint32_t n_partials) {
  if (ctx->n_items == 0 || n_partials == 0) return PF_OK;
  cudaStream_t st = ctx->stream;
  const uint32_t nc = ctx->n_clusters, ns = ctx->n_slices;
  const uint32_t n_cs = nc * ns;                    // (cluster, slice) merge tables
  const uint32_t n_it = ctx->n_items * ns;          // kA work items
  uint32_t* counters = ctx->d_counters.as<uint32_t>();
  const uint32_t WP = (ctx->Ws + 3u) & ~3u;
  // per-(cluster, slice) tables: 2 slots per partial row (+2; PF_MERGE_EIGHTHS / 8), offsets by a scan
  static const uint32_t eighths = []() { const char* e = getenv("PF_MERGE_EIGHTHS"); const int v = e ? atoi(e) : 0;
                                         return (v >= 9 && v <= 32) ? (uint32_t)v : 16u; }();
  TRY(dev_ensure(ctx, ctx->d_group_base, ((size_t)n_cs + 1) * 4));
  if (ns > 1) {
    TRY(dev_ensure(ctx, ctx->d_table2_base, ((size_t)nc + 1) * 4));
    CU(cudaMemsetAsync(ctx->d_table2_base.p, 0, ((size_t)nc + 1) * 4, st));
  }
  plan_merge_tables<<<cdiv((uint64_t)n_cs * 32, 256), 256, 0, st>>>(
      ctx->d_item_base.as<uint32_t>(), nc, ns, ctx->d_slab_count.as<uint32_t>(), eighths,
      ctx->d_group_base.as<uint32_t>(), ns > 1 ? ctx->d_table2_base.as<uint32_t>() : nullptr);
  ctx->launches++;
  TRY(scan_inplace(ctx, ctx->d_group_base.as<uint32_t>(), n_cs, ctx->d_plan_total.as<uint32_t>() + 1));
  const uint64_t n_slots = ((uint64_t)n_partials * eighths + 7) / 8 + 3ull * n_cs + 16;   // >= sum of ceil(p e / 8) + 2
  if (n_slots >= (1ull << 32)) return fail(ctx, PF_ERR_INVALID, "too many partial rows for one batch; split it");
  TRY(dev_ensure(ctx, ctx->d_mtable, n_slots * sizeof(MergeEntry)));
  TRY(dev_ensure(ctx, ctx->d_spill, std::max<size_t>(1, n_cs)));
  CU(cudaMemsetAsync(counters + C_LOCAL + LC_RESCUE, 0, 4, st));     // kB1 counts the folded rows there
  // shared-memory merge per (cluster, slice); clusters too large for it clear their region of the
  // global table (nothing else does) and are merged there by kB1_insert
  kB1_local<<<n_cs, kMergeLocalThreads, merge_local_smem_bytes(ctx->merge_slots), st>>>(
      ctx->d_slab_keys.as<uint64_t>(), ctx->d_slab_rows.as<uint32_t>(), ctx->d_slab_cnt.as<uint32_t>(),
      ctx->d_slab_base.as<uint32_t>(), ctx->d_slab_count.as<uint32_t>(), ctx->d_item_base.as<uint32_t>(), ns,
      ctx->d_group_base.as<uint32_t>(), ctx->d_mtable.as<MergeEntry>(),
      nullptr, WP, counters + C_LOCAL, ctx->merge_slots,
      ctx->d_spill.as<uint8_t>(), ctx->merge_fp_mask);
  ctx->launches++;
  const uint32_t g0 = cdiv((uint64_t)n_it * 32, 256);
  kB1_insert<<<g0, 256, 0, st>>>(ctx->d_slab_keys.as<uint64_t>(), ctx->d_slab_rows.as<uint32_t>(),
                                 ctx->d_slab_cnt.as<uint32_t>(), ctx->d_slab_base.as<uint32_t>(),
                                 ctx->d_slab_count.as<uint32_t>(), ctx->d_item_cluster.as<uint32_t>(), n_it, ns,
                                 ctx->d_group_base.as<uint32_t>(), ctx->d_mtable.as<MergeEntry>(),
                                 nullptr, WP, counters + C_LOCAL,
                                 ctx->d_spill.as<uint8_t>());
  const uint32_t cap = (uint32_t)std::min<uint64_t>(ctx->row_cap, 0x7fffffffu);
  if (ns == 1) {
    kB3_emit<<<g0, 256, 0, st>>>(ctx->d_slab_keys.as<uint64_t>(), ctx->d_slab_rows.as<uint32_t>(),
                                 ctx->d_slab_base.as<uint32_t>(), ctx->d_slab_count.as<uint32_t>(),
                                 ctx->d_item_cluster.as<uint32_t>(), ctx->n_items, ctx->d_slab_cnt.as<uint32_t>(),
                                 ctx->d_clusters.as<ClusterDev>(), ro, cap, counters + C_LOCAL, ctx->W, WP);
    ctx->launches += 2;
    CU(cudaGetLastError());
    return PF_OK;
  }
  // ---- sample slices: sum the per-slice counts of a k-mer, filter on the sum, assemble the survivors ----
  plan_table2_ctas<<<cdiv(nc, 256), 256, 0, st>>>(ctx->d_table2_base.as<uint32_t>(), nc);
  TRY(scan_inplace(ctx, ctx->d_table2_base.as<uint32_t>(), nc, ctx->d_plan_total.as<uint32_t>() + 2));
  const uint64_t max_ctas = ((uint64_t)n_partials + n_partials / 2) / 256 + 2ull * nc + 2;
  TRY(dev_ensure(ctx, ctx->d_table2, max_ctas * 256 * sizeof(LinkEntry)));
  TRY(dev_ensure(ctx, ctx->d_cta_cluster, max_ctas * 4));
  CU(cudaMemsetAsync(ctx->d_table2.p, 0xff, max_ctas * 256 * sizeof(LinkEntry), st));
  TRY(dev_ensure(ctx, ctx->d_home_bits, max_ctas * 32));      // one bit per slot
  CU(cudaMemsetAsync(ctx->d_home_bits.p, 0, max_ctas * 32, st));
  plan_expand_owner<<<cdiv((uint64_t)nc * 32, 256), 256, 0, st>>>(ctx->d_table2_base.as<uint32_t>(), nc,
                                                                  ctx->d_cta_cluster.as<uint32_t>());
  kB4_link<<<g0, 256, 0, st>>>(ctx->d_slab_keys.as<uint64_t>(), ctx->d_slab_rows.as<uint32_t>(),
                               ctx->d_slab_base.as<uint32_t>(), ctx->d_slab_count.as<uint32_t>(),
                               ctx->d_item_cluster.as<uint32_t>(), n_it, ns, ctx->d_slab_cnt.as<uint32_t>(),
                               ctx->d_table2_base.as<uint32_t>(), ctx->d_table2.as<LinkEntry>(), WP);
  // grid of kB5 = CTAs of all cross-slice tables: one small read-back
  TRY(pin_ensure(ctx, ctx->h_plan, 16));
  mirror_counters<<<1, 32, 0, st>>>(ctx->h_plan.as<uint32_t>() + 2, ctx->d_plan_total.as<uint32_t>() + 2, 1);
  CU(cudaStreamSynchronize(st));
  const uint32_t n_ctas = ctx->h_plan.as<uint32_t>()[2];
  if (n_ctas > max_ctas) return fail(ctx, PF_ERR_INTERNAL, "cross-slice table larger than planned");
  if (n_ctas) {
    kB5_emit<<<n_ctas, 256, 0, st>>>(ctx->d_table2.as<LinkEntry>(), ctx->d_cta_cluster.as<uint32_t>(),
                                     ctx->d_table2_base.as<uint32_t>(), ctx->d_home_bits.as<uint32_t>(),
                                     ctx->d_clusters.as<ClusterDev>(), ro, cap, counters + C_LOCAL, ctx->W);
    kB6_scatter<<<g0, 256, 0, st>>>(ctx->d_slab_keys.as<uint64_t>(), ctx->d_slab_rows.as<uint32_t>(),
                                    ctx->d_slab_base.as<uint32_t>(), ctx->d_slab_count.as<uint32_t>(),
                                    ctx->d_item_cluster.as<uint32_t>(), n_it, ns, ctx->d_slab_cnt.as<uint32_t>(),
                                    ctx->d_table2_base.as<uint32_t>(), ctx->d_table2.as<LinkEntry>(),
                                    ctx->d_home_bits.as<uint32_t>(), ro, ctx->W, ctx->Ws, WP);
  }
  ctx->launches += 8;
  CU(cudaGetLastError());
  return PF_OK;
}

// partition mode, one pass: no key read is needed to find the prefix-runs
int tiles_from_hist(pf_ctx* ctx) {
  WidthState& N = ctx->nar;
  if (N.n_records == 0) return PF_OK;
  k3_tiles_from_hist<<<cdiv((uint64_t)N.n_ltiles + 1, 256), 256, 0, ctx->stream>>>(
      N.ltiles.as<TileDev>(), N.n_ltiles, N.seg_hist.as<uint32_t>(), ctx->n_clusters,
      N.tile_first_run.as<uint32_t>());
  ctx->launches++;
  CU(cudaGetLastError());
  return PF_OK;
}

}  // namespace

extern "C" int pf_execute(pf_ctx* ctx) {
  if (!ctx) return PF_ERR_INVALID;
  if (!ctx->have_batch) return fail(ctx, PF_ERR_STATE, "pf_execute: no batch uploaded");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const uint32_t launches0 = ctx->launches;
  WidthState& N = ctx->nar;
  WidthState& Wd = ctx->wid;
  WidthState& X = ctx->xwd;      // k > 32, windows with N/IUPAC symbols (empty otherwise)
  uint32_t* counters = ctx->d_counters.as<uint32_t>();
  uint32_t* hcnt = ctx->h_counters.as<uint32_t>();
  ctx->executed = false;
  ctx->cp_base = ctx->cp.n;
  const bool part = ctx->partition;

  // record buffers (ping-pong); the idle one later holds the run lists, so give
  // it room for n+1 run starts + n run segments (8n+4 bytes <= 8n+16)
  bool blk = ctx->block_mode && part && N.n_records > 0 && ctx->n_items > 0;
  const uint32_t n_ka_items = ctx->n_items * ctx->n_slices;
  auto ensure_records = [&]() -> int {     // the record path needs the narrow ping-pong buffers
    for (int i = 0; i < 2; ++i) {
      TRY(dev_ensure(ctx, N.keys[i], ((size_t)N.n_records + 2) * 8));
      TRY(dev_ensure(ctx, N.vals[i], ((size_t)N.n_records + 2) * 4));
    }
    return PF_OK;
  };
  if (!blk) TRY(ensure_records());
  for (int i = 0; i < 2; ++i) {
    TRY(dev_ensure(ctx, Wd.keys[i], ((size_t)Wd.n_records + 2) * 16));
    TRY(dev_ensure(ctx, Wd.vals[i], ((size_t)Wd.n_records + 2) * 4));
    if (X.n_records) {
      TRY(dev_ensure(ctx, X.keys[i], ((size_t)X.n_records + 2) * 32));
      TRY(dev_ensure(ctx, X.vals[i], ((size_t)X.n_records + 2) * 4));
    }
  }
  const bool compact_pos = ctx->prm.emit_positions == 2u;
  if (ctx->n_pos && compact_pos) {
    if (ctx->prm.canonical) TRY(dev_ensure(ctx, ctx->d_pos_bits, (size_t)ctx->n_words * 4 + 16));
  } else if (ctx->n_pos) {
    TRY(dev_ensure(ctx, ctx->d_pos_kmer, (size_t)ctx->n_pos * 8));
    TRY(dev_ensure(ctx, ctx->d_pos_seq, (size_t)ctx->n_pos * 4));
    TRY(dev_ensure(ctx, ctx->d_pos_cstart, (size_t)ctx->n_pos * 4));
    TRY(dev_ensure(ctx, ctx->d_pos_gstart, (size_t)ctx->n_pos * 4));
    TRY(dev_ensure(ctx, ctx->d_pos_flags, (size_t)ctx->n_pos));
  }
  if (ctx->n_pos_wide && !compact_pos) TRY(dev_ensure(ctx, ctx->d_pos_wide, (size_t)ctx->n_pos_wide * 16));
  if (ctx->n_pos_xwide && !compact_pos) TRY(dev_ensure(ctx, ctx->d_pos_xwide, (size_t)ctx->n_pos_xwide * 32));
  TRY(dev_ensure(ctx, ctx->d_cl_pattern, std::max<size_t>(1, ctx->n_clusters) * 4));
  if (part) {
    uint64_t want_rows = std::max<uint64_t>(65536, (uint64_t)(ctx->row_ratio * 1.3 * (double)N.n_records) + 4096);
    if (!ctx->row_ratio_learned) {
      // the first batch's estimate is a guess: it must not take more than a quarter of the free
      // memory for the candidate bitsets (50,000 samples: 6 kB per row); a guess that turns out too
      // small is corrected by the row-overflow retry below
      size_t free_b = 0, total_b = 0;
      if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess)
        want_rows = std::min<uint64_t>(want_rows, std::max<uint64_t>(65536, free_b / 4 / ((size_t)ctx->Wk * 4 + 24)));
    }
    ctx->row_cap = std::max<uint64_t>(ctx->row_cap, want_rows);
    TRY(ensure_rows(ctx, ctx->row_cap, ctx->row_cap, false));
  }

  if (debug_time()) g_stage_tick = pf_now_ms();
  STAGE("buffers ensured");
  CU(cudaMemsetAsync(counters, 0, C_COUNT * 4, st));
  CU(cudaEventRecord(ctx->ev[EV_START], st));

  // ---- cluster rows (int64 namespace) first: their ids are the NaN-plane word
  //      of k-mer pattern keys in cluster-absent mode ------------------------------
  TRY(dedup(ctx, ctx->cp, ctx->d_presence.as<uint32_t>(), ctx->n_clusters, ctx->d_cl_rep, ctx->d_cl_slot,
            ctx->d_cl_winner, ctx->d_cl_pattern.as<uint32_t>(), C_NEW_CP));
  STAGE("k4 cluster rows");

  RowOut ro{};
  ro.key_words = ctx->Wk; ro.pattern_words = ctx->W;
  ro.cluster_pattern = ctx->d_cl_pattern.as<uint32_t>();

  const uint64_t n_windows = N.n_records / (ctx->prm.canonical ? 1u : 2u);
  ctx->used_block = false;
  for (int attempt = 0;; ++attempt) {
    if (blk) {
      // ---- block aggregation: kA (K1+K2+K3 grouping, no records) + kB (merge, filter, rows) ----
      if (attempt > 12) return fail(ctx, PF_ERR_INTERNAL, "block aggregation did not converge");
      ctx->fused = true;                    // K1 proper only emits positional records
      TRY(launch_k1(ctx));
      STAGE("k1_extract");
      CU(cudaEventRecord(ctx->ev[EV_EXTRACT], st));
      TRY(hist_width<Key128>(ctx, Wd));
      CU(cudaEventRecord(ctx->ev[EV_HIST], st));
      ctx->partial_cap = std::max<uint64_t>(ctx->partial_cap, std::max<uint64_t>(
          65536, (uint64_t)(ctx->partial_ratio * 1.3 * (double)n_windows) + 4096));
      ctx->partial_cap = std::min<uint64_t>(ctx->partial_cap, 0xfffffff0ull);
      const uint32_t WP = (ctx->Ws + 3u) & ~3u;
      TRY(dev_ensure(ctx, ctx->d_slab_base, std::max<size_t>(1, n_ka_items) * 4));
      TRY(dev_ensure(ctx, ctx->d_slab_count, std::max<size_t>(1, n_ka_items) * 4));
      TRY(dev_ensure(ctx, ctx->d_rescue[0], std::max<size_t>(1, n_ka_items) * 4));
      TRY(dev_ensure(ctx, ctx->d_rescue[1], std::max<size_t>(1, n_ka_items) * 4));
      TRY(dev_ensure(ctx, ctx->d_slab_keys, ctx->partial_cap * 8));
      TRY(dev_ensure(ctx, ctx->d_slab_cnt, ctx->partial_cap * 4));
      TRY(dev_ensure(ctx, ctx->d_slab_rows, ctx->partial_cap * WP * 4));
      CU(cudaMemsetAsync(counters + C_LOCAL, 0, LC_COUNT * 4, st));
      TRY(launch_block_aggregate(ctx, nullptr, n_ka_items, ctx->blk_slots, ctx->blk_cap, ctx->blk_cslots,
                                 ctx->d_rescue[0].as<uint32_t>()));
      STAGE("kA_block_aggregate");
      TRY(passes_width<Key128>(ctx, Wd, C_TICKET_W));
      TRY(mark_width<Key128>(ctx, Wd, C_TICKET_MARK_W, C_RUNS_W, false));
      // blocks holding more distinct k-mers than the table takes are rerun with a table twice
      // the size, then four times, ...; past the largest table the batch takes the record path
      mirror_counters<<<1, 32, 0, st>>>(hcnt, counters, C_COUNT);
      CU(cudaStreamSynchronize(st));
      TRY(check_device_error(ctx));
      bool too_big = false;
      static const bool dbg = getenv("PF_DEBUG_BLOCK") != nullptr;
      if (dbg)
        fprintf(stderr, "[pf] kA: items %u slots %u cap %u cslots %u -> overflow %u rescue %u partials %u (one-sample %u) "
                "part_ovf %u\n", ctx->n_items, ctx->blk_slots, ctx->blk_cap, ctx->blk_cslots,
                hcnt[C_LOCAL + LC_TABLE_OVERFLOW], hcnt[C_LOCAL + LC_RESCUE], hcnt[C_LOCAL + LC_PARTIALS],
                hcnt[C_LOCAL + LC_SINGLES], hcnt[C_LOCAL + LC_PARTIAL_OVERFLOW]);
      {
        uint32_t slots = ctx->blk_slots, cap = ctx->blk_cap, cslots = ctx->blk_cslots;
        int cur = 0;
        const uint32_t first_rescue = hcnt[C_LOCAL + LC_RESCUE];
        while (hcnt[C_LOCAL + LC_TABLE_OVERFLOW] == 1u) {
          const uint32_t n_resc = hcnt[C_LOCAL + LC_RESCUE];
          // twice the key slots, as many rows as then fit (the chunk table stays: a full one only
          // sends runs down the direct path)
          uint32_t slots2 = slots * 2u, cap2 = 0;
          if (slots2 <= 8192u && blkA_smem_bytes(slots2, 0u, cslots, ctx->Ws) < kBlkMaxSmem) {
            const uint32_t per_row = 10u + (ctx->Ws | 1u) * 4u;   // rkey, rslot, bitset
            const uint32_t fit = (kBlkMaxSmem - blkA_smem_bytes(slots2, 0u, cslots, ctx->Ws)) / per_row;
            cap2 = std::min<uint32_t>(std::min<uint32_t>(fit, slots2 * 13u / 16u),
                                      std::max<uint32_t>(cap * 2u, slots2 * 5u / 8u));
          }
          if (cap2 <= cap) {        // no more rows with more slots: try all the rows the current slots allow
            slots2 = slots;
            const uint32_t per_row = 10u + (ctx->Ws | 1u) * 4u;   // rkey, rslot, bitset
            const uint32_t fit = (kBlkMaxSmem - blkA_smem_bytes(slots, 0u, cslots, ctx->Ws)) / per_row;
            cap2 = std::min<uint32_t>(fit, slots * 13u / 16u);
          }
          if (cap2 <= cap) { too_big = true; break; }
          slots = slots2;
          cap = cap2;
          CU(cudaMemsetAsync(counters + C_LOCAL + LC_TABLE_OVERFLOW, 0, 4, st));
          CU(cudaMemsetAsync(counters + C_LOCAL + LC_RESCUE, 0, 4, st));
          TRY(launch_block_aggregate(ctx, ctx->d_rescue[cur].as<uint32_t>(), n_resc, slots, cap, cslots,
                                     ctx->d_rescue[cur ^ 1].as<uint32_t>()));
          cur ^= 1;
          mirror_counters<<<1, 32, 0, st>>>(hcnt, counters, C_COUNT);
          CU(cudaStreamSynchronize(st));
          if (dbg)
            fprintf(stderr, "[pf] kA rescue: %u items slots %u cap %u cslots %u -> overflow %u rescue %u partials %u "
                    "(one-sample %u)\n", n_resc, slots, cap, cslots, hcnt[C_LOCAL + LC_TABLE_OVERFLOW],
                    hcnt[C_LOCAL + LC_RESCUE], hcnt[C_LOCAL + LC_PARTIALS], hcnt[C_LOCAL + LC_SINGLES]);
        }
        // many rescued blocks: start the next batches with more rows (and key slots to match)
        if (!too_big && first_rescue > n_ka_items / 8u) {
          uint32_t ns = ctx->blk_slots, ncap = ctx->blk_cap + ctx->blk_cap / 2;
          while (ncap > ns * 13u / 16u) ns *= 2;
          if (ns <= 8192u && blkA_smem_bytes(ns, ncap, ctx->blk_cslots, ctx->Ws) <= kBlkMaxSmem) {
            ctx->blk_slots = ns;
            ctx->blk_cap = ncap;
          }
        }
      }
      CU(cudaEventRecord(ctx->ev[EV_SORT], st));
      CU(cudaEventRecord(ctx->ev[EV_MARK], st));
      if (too_big) {
        // a position block holds more distinct k-mers than the largest table: shorter blocks,
        // then the record path (for this batch; for good after the second time)
        if (ctx->block_windows > (uint32_t)kBlkRun) {
          ctx->block_windows /= 2;
          TRY(plan_blocks(ctx, *ctx, st, true));
        } else {
          blk = false;
          if (++ctx->block_fallbacks >= 2) ctx->block_mode = false;
          TRY(replan_full(ctx));            // (a device-planned upload has no record offsets yet)
          TRY(ensure_records());
        }
        continue;
      }
      if (hcnt[C_LOCAL + LC_PARTIAL_OVERFLOW]) {
        ctx->partial_cap = (uint64_t)hcnt[C_LOCAL + LC_PARTIALS] + 4096;
        continue;
      }
      ro.cluster = ctx->d_row_cluster.as<uint32_t>();
      ro.count = ctx->d_row_count.as<uint32_t>();
      ro.cand = ctx->d_cand.as<uint32_t>();
      ro.kmer = ctx->d_row_kmer.as<uint64_t>();
      ro.row_base = 0;
      TRY(launch_block_merge(ctx, ro, hcnt[C_LOCAL + LC_PARTIALS]));
      STAGE("kB_merge");
      mirror_counters<<<1, 32, 0, st>>>(hcnt, counters, C_COUNT);
      CU(cudaStreamSynchronize(st));
      TRY(check_device_error(ctx));
      ctx->rescued_last = 0;
      ctx->cp.n = ctx->cp_base + hcnt[C_NEW_CP];
      N.n_runs = 0;
      Wd.n_runs = Wd.n_records ? hcnt[C_RUNS_W] : 0;
      X.n_runs = 0;
      if (hcnt[C_LOCAL + LC_PARTIAL_OVERFLOW]) {
        ctx->partial_cap = (uint64_t)hcnt[C_LOCAL + LC_PARTIALS] + 4096;
        continue;
      }
      if (hcnt[C_LOCAL + LC_ROW_OVERFLOW]) {
        ctx->row_cap = (uint64_t)hcnt[C_LOCAL + LC_ROWS] + 1024;
        TRY(ensure_rows(ctx, ctx->row_cap, ctx->row_cap, false));
        continue;
      }
      ctx->used_block = true;
      ctx->partials_last = hcnt[C_LOCAL + LC_PARTIALS];
      if (n_windows) ctx->partial_ratio = std::max(1e-4, (double)ctx->partials_last / (double)n_windows);
      break;
    }
    // ---- K1 + K2 -------------------------------------------------------------
    ctx->fused = part && ctx->use_direct && N.passes <= 2 && !(ctx->prm.debug_flags & 1u);
    TRY(launch_k1(ctx));
    STAGE("k1_extract");
    CU(cudaEventRecord(ctx->ev[EV_EXTRACT], st));
    TRY(hist_width<uint64_t>(ctx, N, ctx->fused));
    TRY(hist_width<Key128>(ctx, Wd));
    TRY(hist_width<Key256>(ctx, X));
    STAGE("k2_histogram");
    CU(cudaEventRecord(ctx->ev[EV_HIST], st));
    TRY(passes_width<uint64_t>(ctx, N, C_TICKET_N, part && ctx->use_direct, ctx->fused));
    TRY(passes_width<Key128>(ctx, Wd, C_TICKET_W));
    TRY(passes_width<Key256>(ctx, X, C_TICKET_X));
    STAGE("k2_onesweep_pass");
    CU(cudaEventRecord(ctx->ev[EV_SORT], st));
    // ---- K3: runs -----------------------------------------------------------------
    ctx->runs_from_hist = part && N.passes == 1;
    if (ctx->runs_from_hist) TRY(tiles_from_hist(ctx));
    else TRY(mark_width<uint64_t>(ctx, N, C_TICKET_MARK_N, C_RUNS_N, part));
    STAGE("k3_mark_runs/k3_tiles_from_hist");
    TRY(mark_width<Key128>(ctx, Wd, C_TICKET_MARK_W, C_RUNS_W, false));
    TRY(mark_width<Key256>(ctx, X, C_TICKET_MARK_X, C_RUNS_X, false));
    STAGE("k3_mark_runs<wide>");
    CU(cudaEventRecord(ctx->ev[EV_MARK], st));
    // local reduce (+ rescue launch of the direct variant), then one sync to read the counters
    auto run_local = [&]() -> int {
      if (part) {
        ro.cluster = ctx->d_row_cluster.as<uint32_t>();
        ro.count = ctx->d_row_count.as<uint32_t>();
        ro.cand = ctx->d_cand.as<uint32_t>();
        ro.kmer = ctx->d_row_kmer.as<uint64_t>();
        ro.row_base = 0;
        TRY(launch_local(ctx, ro));
        STAGE("k3_local");
      }
      mirror_counters<<<1, 32, 0, st>>>(hcnt, counters, C_COUNT);
      CU(cudaStreamSynchronize(st));
      TRY(check_device_error(ctx));
      ctx->rescued_last = 0;
      if (part && ctx->use_direct && N.n_records && hcnt[C_LOCAL + LC_RESCUE] &&
          !hcnt[C_LOCAL + LC_TABLE_OVERFLOW]) {
        ctx->rescued_last = hcnt[C_LOCAL + LC_RESCUE];
        TRY(launch_local(ctx, ro, hcnt[C_LOCAL + LC_RESCUE]));
        mirror_counters<<<1, 32, 0, st>>>(hcnt, counters, C_COUNT);
        CU(cudaStreamSynchronize(st));
      }
      return PF_OK;
    };
    TRY(run_local());
    ctx->cp.n = ctx->cp_base + hcnt[C_NEW_CP];
    N.n_runs = N.n_records ? hcnt[C_RUNS_N] : 0;
    Wd.n_runs = Wd.n_records ? hcnt[C_RUNS_W] : 0;
    X.n_runs = X.n_records ? hcnt[C_RUNS_X] : 0;
    if (!part || N.n_records == 0) break;
    if (attempt > 10) return fail(ctx, PF_ERR_INTERNAL, "partition mode did not converge");
    if (hcnt[C_LOCAL + LC_TABLE_OVERFLOW]) {
      // one prefix-run alone holds more distinct k-mers than a CTA can hold: sort 8 more
      // bits (runs get 256x smaller) and redo the batch.  At 64 bits the general variant
      // always fits (<= 2048 + 1 keys per tile); the direct one falls back to it.
      if (N.sort_bits < 64) {
        ctx->extra_bits += 8;
        N.sort_bits = auto_sort_bits(ctx, N.max_seg, true);
        N.passes = N.sort_bits / 8;
        TRY(dev_ensure(ctx, N.seg_hist, std::max<size_t>(1, (size_t)ctx->n_clusters * N.passes * kRadix) * 4));
      } else if (ctx->use_direct) {
        ctx->use_direct = false;
        TRY(plan_local_tiles(ctx, *ctx, st));
        CU(cudaStreamSynchronize(st));
      } else {
        return fail(ctx, PF_ERR_INTERNAL, "local table overflow at 64 sorted bits");
      }
      continue;
    }
    if (hcnt[C_LOCAL + LC_ROW_OVERFLOW]) {
      ctx->row_cap = (uint64_t)hcnt[C_LOCAL + LC_ROWS] + 1024;
      TRY(ensure_rows(ctx, ctx->row_cap, ctx->row_cap, false));
      TRY(run_local());
      if (hcnt[C_LOCAL + LC_ROW_OVERFLOW] || hcnt[C_LOCAL + LC_TABLE_OVERFLOW])
        return fail(ctx, PF_ERR_INTERNAL, "local reduce overflowed twice");
    }
    break;
  }

  if (part) {
    N.n_rows = N.n_records ? hcnt[C_LOCAL + LC_ROWS] : 0;
    ctx->unique_last = N.n_records ? hcnt[C_LOCAL + LC_UNIQUE] : 0;
    if (ctx->used_block && ctx->n_slices == 1)   // distinct k-mers = partial rows - rows folded into an earlier one
      ctx->unique_last = (uint64_t)hcnt[C_LOCAL + LC_PARTIALS] - hcnt[C_LOCAL + LC_RESCUE];
    if (N.n_records) { ctx->row_ratio = std::max(1e-4, (double)N.n_rows / (double)N.n_records); ctx->row_ratio_learned = true; }
  } else {
    TRY((runs_width<uint64_t, false>(ctx, N, ro)));
  }
  // with 256-bit records (k > 32, N/IUPAC symbols) both wide sections hold dead records of the
  // windows the other one owns: their runs are counted by distinct live keys, not one per run
  const bool exact_unique = X.n_records > 0;
  TRY((runs_width<Key128, false>(ctx, Wd, ro, exact_unique ? counters + C_UNIQUE_WX : nullptr)));
  TRY((runs_width<Key256, false>(ctx, X, ro, counters + C_UNIQUE_WX)));
  CU(cudaEventRecord(ctx->ev[EV_COUNTED], st));
  const bool need_scan = (!part && N.n_runs) || Wd.n_runs || X.n_runs;
  if (need_scan) {
    if (!part && N.n_runs)
      TRY(scan_inplace(ctx, N.vals[N.final_buf ^ 1].as<uint32_t>(), N.n_runs, counters + C_ROWS_N));
    if (Wd.n_runs) TRY(scan_inplace(ctx, Wd.vals[Wd.final_buf ^ 1].as<uint32_t>(), Wd.n_runs, counters + C_ROWS_W));
    if (X.n_runs) TRY(scan_inplace(ctx, X.vals[X.final_buf ^ 1].as<uint32_t>(), X.n_runs, counters + C_ROWS_X));
    mirror_counters<<<1, 32, 0, st>>>(hcnt, counters, C_COUNT);
    CU(cudaStreamSynchronize(st));
    if (!part) N.n_rows = N.n_runs ? hcnt[C_ROWS_N] : 0;
    Wd.n_rows = Wd.n_runs ? hcnt[C_ROWS_W] : 0;
    X.n_rows = X.n_runs ? hcnt[C_ROWS_X] : 0;
  } else {
    if (!part) N.n_rows = 0;
    Wd.n_rows = 0;
    X.n_rows = 0;
  }
  if (!part) ctx->unique_last = N.n_runs;
  ctx->unique_last += exact_unique ? hcnt[C_UNIQUE_WX] : Wd.n_runs;
  const uint64_t rows = (uint64_t)N.n_rows + Wd.n_rows + X.n_rows;
  if (rows >= (1ull << 31)) return fail(ctx, PF_ERR_INVALID, "batch yields 2^31 rows or more; split it");

  if (!part || Wd.n_rows || X.n_rows) TRY(ensure_rows(ctx, std::max<uint64_t>(rows, part ? ctx->row_cap : 0),
                                                      std::max<uint64_t>(N.n_rows, part ? ctx->row_cap : 0), part));
  TRY(dev_ensure(ctx, ctx->d_wrow_kmer, std::max<size_t>(1, Wd.n_rows) * 16));
  if (X.n_rows) TRY(dev_ensure(ctx, ctx->d_xrow_kmer, (size_t)X.n_rows * 32));
  ro.cluster = ctx->d_row_cluster.as<uint32_t>();
  ro.count = ctx->d_row_count.as<uint32_t>();
  ro.cand = ctx->d_cand.as<uint32_t>();
  if (!part && N.n_rows) {
    ro.kmer = ctx->d_row_kmer.as<uint64_t>();
    ro.row_base = 0;
    TRY((runs_width<uint64_t, true>(ctx, N, ro)));
  }
  if (Wd.n_rows) {
    ro.kmer = ctx->d_wrow_kmer.as<uint64_t>();
    ro.row_base = N.n_rows;
    TRY((runs_width<Key128, true>(ctx, Wd, ro)));
  }
  if (X.n_rows) {             // after the wide rows: K4 numbers the patterns of all three sections at once
    ro.kmer = ctx->d_xrow_kmer.as<uint64_t>();
    ro.row_base = N.n_rows + Wd.n_rows;
    TRY((runs_width<Key256, true>(ctx, X, ro)));
  }
  CU(cudaEventRecord(ctx->ev[EV_REDUCE], st));

  // the (cluster, k-mer, count) arrays of the rows are final: start their D2H on the copy
  // stream while K4 numbers the patterns
  ctx->rows_prefetched = false;
  if (rows && !ctx->pipe_mode && ctx->prefetch_rows) {
    TRY(pin_ensure(ctx, ctx->r_row_cluster, rows * 4));
    TRY(pin_ensure(ctx, ctx->r_row_count, rows * 4));
    TRY(pin_ensure(ctx, ctx->r_row_kmer, std::max<size_t>(8, (size_t)N.n_rows * 8)));
    TRY(pin_ensure(ctx, ctx->r_wrow_kmer, std::max<size_t>(8, (size_t)Wd.n_rows * 16)));
    CU(cudaEventRecord(ctx->ev_rows, st));
    CU(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_rows, 0));
    CU(cudaMemcpyAsync(ctx->r_row_cluster.p, ctx->d_row_cluster.p, rows * 4, cudaMemcpyDeviceToHost, ctx->copy_stream));
    CU(cudaMemcpyAsync(ctx->r_row_count.p, ctx->d_row_count.p, rows * 4, cudaMemcpyDeviceToHost, ctx->copy_stream));
    if (N.n_rows) CU(cudaMemcpyAsync(ctx->r_row_kmer.p, ctx->d_row_kmer.p, (size_t)N.n_rows * 8, cudaMemcpyDeviceToHost, ctx->copy_stream));
    if (Wd.n_rows) CU(cudaMemcpyAsync(ctx->r_wrow_kmer.p, ctx->d_wrow_kmer.p, (size_t)Wd.n_rows * 16, cudaMemcpyDeviceToHost, ctx->copy_stream));
    if (X.n_rows) {
      TRY(pin_ensure(ctx, ctx->r_xrow_kmer, (size_t)X.n_rows * 32));
      CU(cudaMemcpyAsync(ctx->r_xrow_kmer.p, ctx->d_xrow_kmer.p, (size_t)X.n_rows * 32, cudaMemcpyDeviceToHost, ctx->copy_stream));
    }
    ctx->rows_prefetched = true;
  }

  STAGE("rows emitted");
  // ---- K4 ---------------------------------------------------------------
  // the previous batch's K4 is long over by now (this call has synchronised the stream at least
  // once since): fold its pattern count in, then number this batch's patterns behind it
  TRY(finalize_pending(ctx));
  ctx->kp_base = ctx->kp.n;
  TRY(dedup(ctx, ctx->kp, ctx->d_cand.as<uint32_t>(), (uint32_t)rows, ctx->d_rep, ctx->d_slot_of,
            ctx->d_winner, ctx->d_row_pattern.as<uint32_t>(), C_NEW_KP));
  STAGE("k4 k-mer rows");
  CU(cudaEventRecord(ctx->ev[EV_DEDUP], st));
  TRY(pin_ensure(ctx, ctx->h_done, 16));
  mirror_counters<<<1, 32, 0, st>>>(hcnt, counters, C_COUNT);
  mirror_counters<<<1, 32, 0, st>>>(ctx->h_done.as<uint32_t>(), counters + C_NEW_KP, 1);
  CU(cudaEventRecord(ctx->ev[EV_END], st));
  ctx->kp_pending = true;
  ctx->kp_pending_base = ctx->kp_base;
  ctx->kp_pending_count = ctx->h_done.as<uint32_t>();
  ctx->executed = true;
  ctx->stats.launches = ctx->launches - launches0;
  return PF_OK;
}
