// pf_lifetime.cuh — pf_maf_window and the small exports, pf_create, pf_destroy.
// Part of libpanfeed_b200.so's single translation unit: included once, in order, by pf_api.cu.

extern "C" int pf_maf_window(double maf, uint32_t n, uint32_t* lo, uint32_t* hi) {
  if (!lo || !hi) return PF_ERR_INVALID;
  if (n == 0) { *lo = 0; *hi = 0; return 1; }   // 0/0 = NaN: neither comparison fires
  const uint32_t mid = (uint32_t)(((uint64_t)n + 1) / 2);   // first c with c/n >= 0.5
  // rising part [0, mid): kept counts form a suffix
  uint32_t a = 0, b = mid;                 // first kept in [a, b) or b
  while (a < b) { uint32_t m = a + (b - a) / 2; if (keep_count(maf, m, n)) b = m; else a = m + 1; }
  const uint32_t rise_lo = a;              // == mid if none
  // falling part [mid, n]: kept counts form a prefix
  uint32_t x = mid, y = n + 1;             // first dropped in [x, y) or y
  while (x < y) { uint32_t m = x + (y - x) / 2; if (!keep_count(maf, m, n)) y = m; else x = m + 1; }
  const uint32_t fall_end = x;             // kept: [mid, fall_end)
  const bool rise = rise_lo < mid, fall = fall_end > mid;
  if (!rise && !fall) { *lo = 1; *hi = 0; return 0; }
  *lo = rise ? rise_lo : mid;
  *hi = fall ? fall_end - 1 : mid - 1;
  return 1;
}

extern "C" uint32_t pf_pattern_words(uint32_t n_samples) { return (n_samples + 31u) / 32u; }
extern "C" int pf_abi_version(void) { return PF_ABI_VERSION; }
extern "C" uint32_t pf_struct_size(int which) {
  switch (which) {
    case 0: return (uint32_t)sizeof(pf_params);
    case 1: return (uint32_t)sizeof(pf_seq_desc);
    case 2: return (uint32_t)sizeof(pf_cluster_desc);
    case 3: return (uint32_t)sizeof(pf_batch);
    case 4: return (uint32_t)sizeof(pf_batch_result);
    case 5: return (uint32_t)sizeof(pf_stats);
    case 6: return (uint32_t)sizeof(pf_synth_params);
    case 7: return (uint32_t)sizeof(pf_cut_result);
    case 8: return (uint32_t)sizeof(pf_cut_planes);
    case 9: return (uint32_t)sizeof(pf_comm);
    case 10: return (uint32_t)sizeof(pf_exchange_result);
    case 11: return (uint32_t)sizeof(pf_assoc_result);
    default: return 0;
  }
}
extern "C" const char* pf_last_error(const pf_ctx* ctx) {
  return ctx ? ctx->err.c_str() : g_create_error.c_str();
}
extern "C" uint32_t pf_kmer_pattern_words(const pf_ctx* ctx) { return ctx ? ctx->Wk : 0; }
extern "C" void* pf_stream(pf_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

extern "C" int pf_create(pf_ctx** out, int device, const pf_params* p) {
  pf_ctx* ctx = nullptr;
  if (!out || !p) return fail(nullptr, PF_ERR_INVALID, "pf_create: null argument");
  *out = nullptr;
  if (p->abi_version != PF_ABI_VERSION)
    return fail(nullptr, PF_ERR_INVALID, "pf_create: ABI version %u != %u", p->abi_version, PF_ABI_VERSION);
  if (p->k < 1 || p->k > 64)
    return fail(nullptr, PF_ERR_UNSUPPORTED, "k=%u unsupported: k-mers of 1..64 bases are packed into one or two 64-bit "
                                             "words (1..32: all engines; 33..64: the 128-bit record engine, 256-bit "
                                             "records for windows with N/IUPAC symbols)", p->k);
  if (p->n_samples < 1) return fail(nullptr, PF_ERR_INVALID, "n_samples must be >= 1");
  if (p->sort_bits != 0 && (p->sort_bits % 8 != 0 || p->sort_bits < 8 || p->sort_bits > 64))
    return fail(nullptr, PF_ERR_INVALID, "sort_bits must be 0 or a multiple of 8 in 8..64");
  if (p->mode > 1) return fail(nullptr, PF_ERR_INVALID, "mode must be 0 (partition) or 1 (full sort)");
  if (!(p->maf <= 0.5) || p->maf < 0)
    return fail(nullptr, PF_ERR_INVALID, "--maf should be in [0, 0.5]");
  int n_dev = 0;
  cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || n_dev == 0)
    return fail(nullptr, PF_ERR_CUDA, "no CUDA device: %s (this library has no CPU fallback)",
                e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
  if (device < 0 || device >= n_dev) return fail(nullptr, PF_ERR_INVALID, "device %d out of range", device);
  e = cudaSetDevice(device);
  if (e != cudaSuccess) return fail(nullptr, PF_ERR_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  if (prop.major < 10)
    return fail(nullptr, PF_ERR_UNSUPPORTED, "device is sm_%d%d; this library is built for sm_100a only",
                prop.major, prop.minor);
  ctx = new pf_ctx();
  ctx->prm = *p;
  ctx->device = device;
  ctx->W = pf_pattern_words(p->n_samples);
  ctx->Wk = ctx->W + (p->consider_missing ? 1u : 0u);
  ctx->kp.key_words = ctx->Wk;
  ctx->cp.key_words = ctx->W;
  // partition mode needs (slot:13 | sample:19) pair words and a bitset row that fits the pool
  ctx->partition = (p->mode == 0) && p->n_samples < kLocalMaxSamples && ctx->W <= (uint32_t)kLocalPoolWords;
  if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete ctx;
    return fail(nullptr, PF_ERR_CUDA, "cudaStreamCreate failed");
  }
  cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
  cudaStreamCreateWithFlags(&ctx->up_stream, cudaStreamNonBlocking);
  for (int i = 0; i < 2; ++i) cudaEventCreate(&ctx->ev_pipe[i]);
  for (BatchState* bs : {static_cast<BatchState*>(ctx), &ctx->alt, &ctx->alt2}) {
    cudaEventCreateWithFlags(&bs->ev_up_done, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&bs->ev_exec_end, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&bs->ev_out_done, cudaEventDisableTiming);
    for (auto& ev : bs->ev) cudaEventCreate(&ev);
    for (auto& ev : bs->ev_h2d) cudaEventCreate(&ev);
  }
  if (const char* e = getenv("PF_PREFETCH_ROWS")) ctx->prefetch_rows = atoi(e) != 0;
  if (const char* e = getenv("PF_PIPELINE_SEQS")) {      // 0 disables the pipelined submit
    const long v = atol(e);
    if (v <= 0) ctx->pipe_min_seqs = 0xffffffffu;
    else {
      ctx->pipe_target_seqs = (uint32_t)std::max<long>(1024, v);
      ctx->pipe_min_seqs = ctx->pipe_target_seqs + ctx->pipe_target_seqs / 2;
      ctx->pipe_first_seqs = std::max(1024u, ctx->pipe_target_seqs * 3 / 8);
    }
  }
  if (const char* e = getenv("PF_PIPELINE_FIRST")) { const long v = atol(e); if (v > 0) ctx->pipe_first_seqs = (uint32_t)std::max<long>(1024, v); }
  cudaEventCreateWithFlags(&ctx->ev_rows, cudaEventDisableTiming);
  for (auto& ev : ctx->ev_d2h) cudaEventCreate(&ev);
  // opt in to > 48 KB dynamic shared memory for the sort passes
  cudaFuncSetAttribute(k2_onesweep_pass<uint64_t>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)sizeof(SortSmem<uint64_t>));
  cudaFuncSetAttribute(k2_onesweep_pass<Key128>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)sizeof(SortSmem<Key128>));
  cudaFuncSetAttribute(k2_onesweep_pass<Key256>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)sizeof(SortSmem<Key256>));
  cudaFuncSetAttribute(k2_scatter_pass<uint64_t>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)sizeof(ScatterSmem<uint64_t>));
  cudaFuncSetAttribute(k2_extract_scatter<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)sizeof(ScatterSmem<uint64_t>));
  cudaFuncSetAttribute(k2_extract_scatter<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)sizeof(ScatterSmem<uint64_t>));
  cudaFuncSetAttribute(k3_local, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(LocalSmem));
  cudaFuncSetAttribute(k3_local_direct, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DirectSmem));
  ctx->use_direct = ctx->W <= kDirectMaxWords;
  {
    // block aggregation: debug_flags bit 1 disables it; PF_BLOCK_WINDOWS / PF_BLOCK_SMEM_KB tune it
    ctx->block_mode = ctx->partition && !(p->debug_flags & 2u);
    if (ctx->W > kDirectMaxWords) {            // S > 1024: partial rows per slice of 512 samples
      ctx->slice_samples = 512;
      ctx->n_slices = (p->n_samples + 511u) / 512u;
      ctx->Ws = 16;
      if (ctx->n_slices > 0xffffu) ctx->block_mode = false;
    } else {
      ctx->slice_samples = 32u * ctx->W;
      ctx->n_slices = 1;
      ctx->Ws = ctx->W;
    }
    if (const char* e = getenv("PF_BLOCK_SLICED")) if (atoi(e) == 0 && ctx->n_slices > 1) ctx->block_mode = false;
    if (const char* e = getenv("PF_BLOCK_MODE")) ctx->block_mode = ctx->block_mode && atoi(e) != 0;
    // tables of kA: two k-mer slots per sample of a 16-window run (about one haplotype per 30
    // samples and position), an eighth as many chunk slots; overflowing runs are rerun with the
    // rescue chunk table and twice the key slots
    ctx->block_windows = (uint32_t)kBlkRun;
    // (about one new k-mer per sample and run of 16 windows, plus the haplotypes' own)
    uint32_t slots = 256;
    const uint32_t s_eff = std::min<uint32_t>(p->n_samples, ctx->slice_samples);   // samples a kA block sees
    while (slots < 2u * s_eff && slots < 4096u) slots *= 2;
    if (const char* e = getenv("PF_BLOCK_SLOTS")) {
      const int v = atoi(e);
      if (v >= 64 && v <= 8192 && (v & (v - 1)) == 0) slots = (uint32_t)v;
    }
    uint32_t cap = slots * 13u / 16u;              // a row costs 14 bytes: as many as the key slots allow
    if (const char* e = getenv("PF_BLOCK_CAP")) {
      const int v = atoi(e);
      if (v >= 32 && (uint32_t)v <= slots * 13u / 16u) cap = (uint32_t)v;
    }
    uint32_t cslots = std::max<uint32_t>(64u, slots / 8u);
    if (const char* e = getenv("PF_BLOCK_CSLOTS")) {
      const int v = atoi(e);
      if (v >= 32 && v <= 8192 && (v & (v - 1)) == 0) cslots = (uint32_t)v;
    }
    const bool canon = p->canonical != 0;
    while (slots > 64u && blkA_smem_bytes(slots, cap, cslots, ctx->Ws, canon) > kBlkMaxSmem) {
      slots /= 2; cap /= 2; cslots = std::max<uint32_t>(32u, cslots / 2);
    }
    // a rescue launch gives every sequence of a work item its own chunk (at one sequence per
    // sample), while 2048 key slots and their rows still fit next to the chunk table
    uint32_t rcs = 32u;
    while (blkA_ccap(rcs) < s_eff && rcs < 2048u) rcs *= 2;
    while (rcs > cslots && blkA_smem_bytes(2048u, 1664u, rcs, ctx->Ws, canon) > kBlkMaxSmem) rcs /= 2;
    ctx->blk_rescue_cslots = std::max(rcs, cslots);
    if (const char* e = getenv("PF_KA_SEG_RUNS")) {   // fixed segment length: tests of small batches, sweeps
      const int v = atoi(e);
      if (v >= 1 && v <= 4096) ctx->ka_seg_runs = (uint32_t)v;
    }
    ctx->blk_slots = slots;
    ctx->blk_cap = cap;
    ctx->blk_cslots = cslots;
    if (p->k == 32 && !p->canonical) ctx->block_mode = false;   // all-T k-mer == the empty-slot mark
    if (p->k > 32) ctx->block_mode = false;                      // two-word k-mers: the 128-bit record pipeline
    if (const char* e = getenv("PF_MERGE_SMEM_KB")) {       // 0: every cluster through the global table
      const long kb = atol(e);
      if (kb >= 0 && kb <= 216) ctx->merge_slots = (uint32_t)(kb * 256);
    }
    if (const char* e = getenv("PF_MERGE_FP_BITS")) {
      const long b = atol(e);
      if (b >= 0 && b <= 15) ctx->merge_fp_mask = (1u << b) - 1u;
    }
    cudaFuncSetAttribute(kB1_local, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         (int)merge_local_smem_bytes(ctx->merge_slots));
    if (const char* e = getenv("PF_PATTERN_SMEM_KB")) {     // 0: every row its own K4 candidate
      const long kb = atol(e);
      if (kb >= 0 && kb <= 200) ctx->pattern_smem = (uint32_t)(kb * 1024);
    }
    cudaFuncSetAttribute(kB3_cluster_emit, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->pattern_smem);
    cudaFuncSetAttribute(kA_block_aggregate<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBlkMaxSmem);
    cudaFuncSetAttribute(kA_block_aggregate<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBlkMaxSmem);
  }
  ctx->row_ratio = std::min(1.0 / 48, 16.0 / (double)std::max<uint32_t>(1u, p->n_samples));
  const int k3_smem = (int)(8 * ctx->W * sizeof(uint32_t));
  if (k3_smem > 48 * 1024) {
    cudaFuncSetAttribute(k3_runs<uint64_t, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, k3_smem);
    cudaFuncSetAttribute(k3_runs<uint64_t, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, k3_smem);
    cudaFuncSetAttribute(k3_runs<Key128, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, k3_smem);
    cudaFuncSetAttribute(k3_runs<Key128, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, k3_smem);
    cudaFuncSetAttribute(k3_runs<Key256, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, k3_smem);
    cudaFuncSetAttribute(k3_runs<Key256, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, k3_smem);
  }
  if (k3_smem > 200 * 1024) {
    pf_destroy(ctx);
    return fail(nullptr, PF_ERR_UNSUPPORTED, "n_samples=%u needs %d B of shared memory per CTA", p->n_samples, k3_smem);
  }
  *out = ctx;
  return PF_OK;
}

extern "C" void pf_destroy(pf_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  auto fd = [](DevBuf& b) { if (b.p) cudaFree(b.p); b.p = nullptr; b.cap = 0; };
  auto fp = [](PinBuf& b) { if (b.p) cudaFreeHost(b.p); b.p = nullptr; b.cap = 0; };
  for (BatchState* bs : {static_cast<BatchState*>(ctx), &ctx->alt, &ctx->alt2}) {
    for (cudaEvent_t* e : {&bs->ev_up_done, &bs->ev_exec_end, &bs->ev_out_done, &bs->ev_h2d[0], &bs->ev_h2d[1]})
      if (*e) cudaEventDestroy(*e);
    for (auto& ev : bs->ev) if (ev) cudaEventDestroy(ev);
    for (DevBuf* b : {&bs->d_bases, &bs->d_amb, &bs->d_ambbits, &bs->d_seqs, &bs->d_clusters, &bs->d_wide_seqs,
                      &bs->d_xpos_slot, &bs->d_xrow_kmer, &bs->d_pos_xwide,
                      &bs->d_presence, &bs->d_row_cluster, &bs->d_row_kmer, &bs->d_wrow_kmer, &bs->d_row_count,
                      &bs->d_row_pattern, &bs->d_cl_pattern, &bs->d_pos_kmer, &bs->d_pos_seq, &bs->d_pos_cstart,
                      &bs->d_pos_gstart, &bs->d_pos_flags, &bs->d_pos_wide, &bs->d_pos_bits, &bs->d_seq_rec_off,
                      &bs->d_tile_first_seq, &bs->d_seq_lite, &bs->d_cblk, &bs->d_item_base, &bs->d_item_cluster,
                      &bs->d_plan_total, &bs->d_bsum_slot, &bs->d_slice_seq, &bs->d_item_desc, &bs->d_raw, &bs->d_plan_tot,
                      &bs->d_rec_off})
      fd(*b);
    for (WidthState* w : {&bs->nar, &bs->wid, &bs->xwd}) {
      for (DevBuf* b : {&w->keys[0], &w->keys[1], &w->vals[0], &w->vals[1], &w->tiles, &w->seg_start,
                        &w->seg_hist, &w->lookback, &w->cursors, &w->ltiles, &w->tile_first_run,
                        &w->d_tile_base, &w->d_ltile_base})
        fd(*b);
    }
    for (PinBuf* b : {&bs->h_clusters, &bs->h_plan, &bs->h_done, &bs->h_raw, &bs->h_plan_tot})
      fp(*b);
  }
  for (DevBuf* b : {&ctx->d_counters, &ctx->d_bsum, &ctx->d_cand, &ctx->d_row_cand, &ctx->d_cand_pattern, &ctx->d_rep, &ctx->d_slot_of, &ctx->d_winner,
                    &ctx->d_cl_rep, &ctx->d_cl_slot, &ctx->d_cl_winner, &ctx->d_digests, &ctx->d_slab_base,
                    &ctx->d_slab_count, &ctx->d_slab_keys, &ctx->d_slab_rows, &ctx->d_group_base, &ctx->d_mtable,
                    &ctx->d_rescue[0], &ctx->d_rescue[1], &ctx->d_table2_base, &ctx->d_table2,
                    &ctx->d_home_bits, &ctx->d_cta_cluster, &ctx->d_slab_cnt, &ctx->d_spill})
    fd(*b);
  {
    AssocState& a = ctx->assoc;
    for (DevBuf* b : {&a.d_key, &a.d_val, &a.d_kp, &a.d_cp, &a.d_table, &a.d_row_seen, &a.d_cl_pass, &a.d_cl_assoc,
                      &a.d_win, &a.d_win_assoc, &a.d_prow, &a.d_prow_assoc, &a.d_prow_seen, &a.d_count})
      fd(*b);
    for (PinBuf* b : {&a.h_count, &a.r_win, &a.r_win_assoc, &a.r_cl_pass, &a.r_cl_assoc, &a.r_prow, &a.r_prow_assoc,
                      &a.r_prow_seen})
      fp(*b);
  }
  ctx->grower.join();
  xrun_free(ctx);                      // pf_exchange_run's buffers and peer mappings
  for (PatternSpace* s : {&ctx->kp, &ctx->cp}) pool_free(s->pool);
  for (PatternSpace* s : {&ctx->kp, &ctx->cp})
    for (DevBuf* b : {&s->table, &s->x_owner, &s->x_pos, &s->x_perm, &s->x_counts, &s->x_unique,
                      &s->x_table, &s->x_rep, &s->x_slot, &s->x_winner})
      fd(*b);
  for (PinBuf* b : {&ctx->h_counters, &ctx->r_row_cluster, &ctx->r_row_kmer, &ctx->r_wrow_kmer, &ctx->r_row_count,
                    &ctx->r_row_pattern, &ctx->r_cl_pattern, &ctx->r_new_kp, &ctx->r_new_cp, &ctx->r_pos_kmer,
                    &ctx->r_pos_seq, &ctx->r_pos_cstart, &ctx->r_pos_gstart, &ctx->r_pos_flags, &ctx->r_pos_wide,
                    &ctx->r_wrow_cluster, &ctx->r_wrow_count, &ctx->r_wrow_pattern, &ctx->r_pos_bits,
                    &ctx->r_xrow_kmer, &ctx->r_pos_xwide})
    fp(*b);
  for (auto& ev : ctx->ev_d2h) if (ev) cudaEventDestroy(ev);
  for (auto& e : ctx->dbg_ev) for (auto& x : e) if (x) cudaEventDestroy(x);
  for (int i = 0; i < 2; ++i) if (ctx->ev_pipe[i]) cudaEventDestroy(ctx->ev_pipe[i]);
  if (ctx->ev_rows) cudaEventDestroy(ctx->ev_rows);
  if (ctx->up_stream) cudaStreamDestroy(ctx->up_stream);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}
