// pf_assoc.cuh — pf_assoc_load / pf_assoc_collect: the --associations join of a second pass (K6,
// k6_assoc.cuh).  Part of libpanfeed_b200.so's single translation unit (pf_api.cu).

extern "C" int pf_assoc_load(pf_ctx* ctx, const uint8_t* digests, uint64_t n) {
  if (!ctx || (n && !digests)) return PF_ERR_INVALID;
  if (n >= (1ull << 30)) return fail(ctx, PF_ERR_INVALID, "pf_assoc_load: %llu digests, at most 2^30",
                                     (unsigned long long)n);
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->stream));
  AssocState& a = ctx->assoc;
  // open addressing on the first digest word (MD5 output is uniform), built here once per run: the
  // passing associations are few, every pattern of every batch is then looked up on the device
  uint32_t slots = 64;
  while (slots < 2 * n) slots *= 2;
  std::vector<uint4> key(slots, make_uint4(0, 0, 0, 0));
  std::vector<uint32_t> val(slots, kAssocNone);
  for (uint64_t i = 0; i < n; ++i) {
    uint32_t d[4];
    memcpy(d, digests + 16 * i, 16);
    uint32_t s = d[0] & (slots - 1);
    for (;; s = (s + 1) & (slots - 1)) {
      if (val[s] == kAssocNone) break;
      if (key[s].x == d[0] && key[s].y == d[1] && key[s].z == d[2] && key[s].w == d[3])
        return fail(ctx, PF_ERR_INVALID, "pf_assoc_load: digests %u and %llu are equal", val[s], (unsigned long long)i);
    }
    key[s] = make_uint4(d[0], d[1], d[2], d[3]);
    val[s] = (uint32_t)i;
  }
  TRY(dev_ensure(ctx, a.d_key, (size_t)slots * 16));
  TRY(dev_ensure(ctx, a.d_val, (size_t)slots * 4));
  CU(cudaMemcpy(a.d_key.p, key.data(), (size_t)slots * 16, cudaMemcpyHostToDevice));
  CU(cudaMemcpy(a.d_val.p, val.data(), (size_t)slots * 4, cudaMemcpyHostToDevice));
  a.mask = slots - 1;
  a.loaded = true;
  a.kp_done = a.cp_done = 0;            // every pattern numbered so far is looked up again
  return PF_OK;
}

extern "C" int pf_assoc_collect(pf_ctx* ctx, pf_assoc_result* out) {
  if (!ctx || !out) return PF_ERR_INVALID;
  AssocState& a = ctx->assoc;
  if (!a.loaded) return fail(ctx, PF_ERR_STATE, "pf_assoc_collect: no association table (pf_assoc_load)");
  if (!a.batch_ready) return fail(ctx, PF_ERR_STATE, "pf_assoc_collect: call it after the pf_collect of a batch");
  if (ctx->prm.emit_positions != 2u)
    return fail(ctx, PF_ERR_STATE, "pf_assoc_collect: the context must emit the compact positional form (emit_positions = 2)");
  CU(cudaSetDevice(ctx->device));
  TRY(finalize_pending(ctx));
  cudaStream_t st = ctx->stream;
  const AssocTable t{a.d_key.as<uint4>(), a.d_val.as<uint32_t>(), a.mask};

  // ---- K6a: association row of every pattern not looked up yet, both namespaces ----
  for (int ns = 0; ns < 2; ++ns) {
    PatternSpace& s = ns ? ctx->cp : ctx->kp;
    DevBuf& d = ns ? a.d_cp : a.d_kp;
    uint64_t& done = ns ? a.cp_done : a.kp_done;
    TRY(dev_ensure(ctx, d, std::max<size_t>(1, s.n) * 4, true));
    if (s.n > done) {
      const uint64_t count = s.n - done;
      k6_pattern_assoc<<<cdiv(count, 128), 128, 0, st>>>(s.pool.as<uint32_t>(), (uint32_t)done, (uint32_t)count,
                                                         s.key_words, ctx->W, ctx->prm.n_samples, ns, ctx->cp.pool.as<uint32_t>(),
                                                         t, d.as<uint32_t>());
      ctx->launches++;
      CU(cudaGetLastError());
      done = s.n;
    }
  }

  // ---- K6e / K6b: the clusters' own patterns, the (cluster, k-mer) table of the rows ----
  const uint32_t nc = ctx->n_clusters;
  const uint64_t n_rows = (uint64_t)ctx->nar.n_rows + ctx->wid.n_rows + ctx->xwd.n_rows;
  uint32_t slots = 64;
  while (slots < 2 * n_rows) slots *= 2;
  TRY(dev_ensure(ctx, a.d_cl_pass, std::max<size_t>(1, nc)));
  TRY(dev_ensure(ctx, a.d_cl_assoc, std::max<size_t>(1, nc) * 4));
  TRY(dev_ensure(ctx, a.d_table, (size_t)slots * 4));
  TRY(dev_ensure(ctx, a.d_row_seen, std::max<size_t>(1, n_rows)));
  TRY(dev_ensure(ctx, a.d_prow, std::max<size_t>(1, n_rows) * 4));
  TRY(dev_ensure(ctx, a.d_prow_assoc, std::max<size_t>(1, n_rows) * 4));
  TRY(dev_ensure(ctx, a.d_prow_seen, std::max<size_t>(1, n_rows)));
  const uint64_t n_emit = (uint64_t)ctx->n_pos * (ctx->prm.canonical ? 1 : 2);
  TRY(dev_ensure(ctx, a.d_win, std::max<size_t>(1, n_emit) * 8));
  TRY(dev_ensure(ctx, a.d_win_assoc, std::max<size_t>(1, n_emit) * 4));
  TRY(dev_ensure(ctx, a.d_count, 16));
  CU(cudaMemsetAsync(a.d_count.p, 0, 16, st));
  CU(cudaMemsetAsync(a.d_table.p, 0xff, (size_t)slots * 4, st));
  if (n_rows) CU(cudaMemsetAsync(a.d_row_seen.p, 0, n_rows, st));
  if (nc) {
    k6_cluster_assoc<<<cdiv(nc, 256), 256, 0, st>>>(ctx->d_cl_pattern.as<uint32_t>(), nc, a.d_cp.as<uint32_t>(),
                                                    a.d_cl_assoc.as<uint32_t>(), a.d_cl_pass.as<uint8_t>());
    ctx->launches++;
  }
  AssocRows rows{ctx->d_row_cluster.as<uint32_t>(), ctx->d_row_pattern.as<uint32_t>(), ctx->d_row_kmer.as<uint64_t>(),
                 ctx->d_wrow_kmer.as<uint64_t>(), ctx->d_xrow_kmer.as<uint64_t>(), ctx->nar.n_rows, ctx->wid.n_rows,
                 ctx->xwd.n_rows};
  if (n_rows) {
    k6_row_index<<<cdiv(n_rows, 256), 256, 0, st>>>(rows, a.d_table.as<uint32_t>(), slots - 1, a.d_kp.as<uint32_t>(),
                                                    a.d_cl_pass.as<uint8_t>());
    ctx->launches++;
  }
  // ---- K6c: the windows of the target sequences ----
  uint32_t* cnt = a.d_count.as<uint32_t>();
  if (n_emit && n_rows && ctx->n_seqs) {
    const uint32_t grid = std::min<uint32_t>(cdiv(ctx->n_seqs, kK1Warps), 148 * 8);
    const uint32_t* bits = ctx->prm.canonical ? ctx->d_pos_bits.as<uint32_t>() : nullptr;
#define PF_K6C(CANON)                                                                                           \
    k6_window_join<CANON><<<grid, kK1Warps * 32, 0, st>>>(                                                       \
        ctx->d_bases.as<uint64_t>(), ctx->d_amb.as<uint64_t>(), ctx->d_ambbits.as<uint32_t>(),                  \
        ctx->d_seqs.as<SeqDev>(), ctx->n_seqs, (int)ctx->prm.k, bits, rows, a.d_table.as<uint32_t>(), slots - 1, \
        a.d_kp.as<uint32_t>(), a.d_cl_pass.as<uint8_t>(), a.d_row_seen.as<uint8_t>(), a.d_win.as<uint64_t>(),    \
        a.d_win_assoc.as<uint32_t>(), cnt)
    if (ctx->prm.canonical) PF_K6C(true); else PF_K6C(false);
#undef PF_K6C
    ctx->launches++;
  }
  // ---- K6d: the passing rows, seen or not ----
  if (n_rows) {
    k6_passing_rows<<<cdiv(n_rows, 256), 256, 0, st>>>(ctx->d_row_pattern.as<uint32_t>(), (uint32_t)n_rows,
                                                       a.d_kp.as<uint32_t>(), a.d_row_seen.as<uint8_t>(),
                                                       a.d_prow.as<uint32_t>(), a.d_prow_assoc.as<uint32_t>(),
                                                       a.d_prow_seen.as<uint8_t>(), cnt + 1);
    ctx->launches++;
  }
  CU(cudaGetLastError());
  TRY(pin_ensure(ctx, a.h_count, 16));
  CU(cudaMemcpyAsync(a.h_count.p, cnt, 8, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  const uint32_t n_win = a.h_count.as<uint32_t>()[0], n_prow = a.h_count.as<uint32_t>()[1];
  auto d2h = [&](PinBuf& dst, const void* src, size_t bytes) -> int {
    TRY(pin_ensure(ctx, dst, std::max<size_t>(bytes, 8)));
    if (bytes) CU(cudaMemcpyAsync(dst.p, src, bytes, cudaMemcpyDeviceToHost, st));
    return PF_OK;
  };
  TRY(d2h(a.r_win, a.d_win.p, (size_t)n_win * 8));
  TRY(d2h(a.r_win_assoc, a.d_win_assoc.p, (size_t)n_win * 4));
  TRY(d2h(a.r_cl_pass, a.d_cl_pass.p, nc));
  TRY(d2h(a.r_cl_assoc, a.d_cl_assoc.p, (size_t)nc * 4));
  TRY(d2h(a.r_prow, a.d_prow.p, (size_t)n_prow * 4));
  TRY(d2h(a.r_prow_assoc, a.d_prow_assoc.p, (size_t)n_prow * 4));
  TRY(d2h(a.r_prow_seen, a.d_prow_seen.p, n_prow));
  CU(cudaStreamSynchronize(st));
  memset(out, 0, sizeof *out);
  out->n_windows = n_win;
  out->window = a.r_win.as<uint64_t>();
  out->window_assoc = a.r_win_assoc.as<uint32_t>();
  out->n_clusters = nc;
  out->cluster_pass = a.r_cl_pass.as<uint8_t>();
  out->cluster_assoc = a.r_cl_assoc.as<uint32_t>();
  out->n_rows = n_prow;
  out->row = a.r_prow.as<uint32_t>();
  out->row_assoc = a.r_prow_assoc.as<uint32_t>();
  out->row_seen = a.r_prow_seen.as<uint8_t>();
  return PF_OK;
}
