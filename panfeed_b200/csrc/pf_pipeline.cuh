// pf_pipeline.cuh — pipelined pf_submit (two batch slots), pf_collect, pattern export / ids, stats.
// Part of libpanfeed_b200.so's single translation unit: included once, in order, by pf_api.cu.

namespace {

// grow a pinned result array, keeping the `used` bytes already copied into it
int pin_grow(pf_ctx* ctx, PinBuf& b, size_t need, size_t used) {
  if (need <= b.cap) return PF_OK;
  if (debug_alloc()) fprintf(stderr, "[pf] alloc: pinned result array %zu -> %zu bytes (copy)\n", b.cap, need);
  CU(cudaStreamSynchronize(ctx->copy_stream));     // copies into the old array are in flight
  size_t want = std::max(need, b.cap + b.cap / 2);
  want = (want + 4095) & ~size_t(4095);
  void* np = nullptr;
  CU(cudaMallocHost(&np, want));
  if (b.p && used) memcpy(np, b.p, used);
  if (b.p) CU(cudaFreeHost(b.p));
  b.p = np;
  b.cap = want;
  return PF_OK;
}

// cut a batch into sub-batches of whole clusters with about `target` sequences each
// (`first` for the first one: nothing runs under its upload, so it is kept short; a short LAST
// one does not pay: the D2H of the one before it would no longer be hidden)
std::vector<SubRange> split_batch(const pf_batch* b, uint32_t target_all, uint32_t first) {
  std::vector<SubRange> subs;
  const uint32_t n = b->n_seqs;
  first = std::min(first, target_all);
  uint32_t s0 = 0, c0 = 0;
  while (s0 < n) {
    const uint64_t rem = n - s0;
    uint64_t target = s0 == 0 ? first : target_all;
    if (rem <= target + target / 2) target = rem;     // the tail: all of it
    uint32_t s1 = n, c1 = b->n_clusters;
    if (target < rem) {
      // first sequence of the cluster that holds sequence s0 + target (clusters are sorted)
      const uint32_t c = b->seqs[s0 + target].cluster;
      uint32_t lo = s0, hi = s0 + (uint32_t)target;
      while (lo < hi) {
        const uint32_t mid = lo + (hi - lo) / 2;
        if (b->seqs[mid].cluster < c) lo = mid + 1; else hi = mid;
      }
      if (lo > s0) { s1 = lo; c1 = c; }
      else {            // one cluster longer than the target: take it whole
        lo = s0 + (uint32_t)target; hi = n;
        while (lo < hi) {
          const uint32_t mid = lo + (hi - lo) / 2;
          if (b->seqs[mid].cluster <= c) lo = mid + 1; else hi = mid;
        }
        s1 = lo;
        c1 = s1 < n ? b->seqs[s1].cluster : b->n_clusters;
      }
    }
    SubRange r{};
    r.s0 = s0; r.s1 = s1; r.c0 = c0; r.c1 = std::max(c1, c0);
    r.w0 = b->seqs[s0].base_off >> 5;
    r.w1 = s1 < n ? (b->seqs[s1].base_off >> 5) : b->n_words;
    r.a0 = 0; r.a1 = 0;
    subs.push_back(r);
    s0 = s1;
    c0 = r.c1;
  }
  if (!subs.empty()) subs.back().c1 = b->n_clusters;     // trailing clusters without sequences
  return subs;
}

void pipe_add_timings(pf_ctx* ctx, const BatchState* slot = nullptr) {
  fill_timings(ctx, slot);
  const pf_stats& t = ctx->stats;
  // (the H2D time of a slot is added when its upload is waited for: by now the slot's H2D
  //  events may belong to a later upload)
  const float v[10] = {0.f, t.ms_extract, t.ms_hist, t.ms_sort, t.ms_mark, t.ms_count, t.ms_reduce,
                       t.ms_dedup, 0.f, 0.f};
  for (int i = 0; i < 10; ++i) ctx->pipe_ms[i] += v[i];
  static const bool dbg = getenv("PF_DEBUG_PIPE") != nullptr;
  if (dbg)
    fprintf(stderr, "[pf] sub-batch stages: cluster rows %.3f  kA %.3f  kB %.3f  emit %.3f  k4 %.3f  (hist %.3f mark %.3f) ms\n",
            t.ms_extract, t.ms_sort, t.ms_count, t.ms_reduce, t.ms_dedup, t.ms_hist, t.ms_mark);
}

// D2H of the current slot's results behind everything it executed, appended to the pinned
// result arrays of the pipelined submit
int pipe_enqueue_results(pf_ctx* ctx, const SubRange& r) {
  cudaStream_t st = ctx->stream, cp = ctx->copy_stream;
  WidthState& N = ctx->nar;
  WidthState& Wd = ctx->wid;
  const uint64_t nr = N.n_rows, nw = Wd.n_rows;
  const uint64_t R = ctx->pipe_rows, RW = ctx->pipe_wide_rows;
  TRY(pin_grow(ctx, ctx->r_row_cluster, (R + nr) * 4, R * 4));
  TRY(pin_grow(ctx, ctx->r_row_count, (R + nr) * 4, R * 4));
  TRY(pin_grow(ctx, ctx->r_row_pattern, (R + nr) * 4, R * 4));
  TRY(pin_grow(ctx, ctx->r_row_kmer, (R + nr) * 8, R * 8));
  TRY(pin_grow(ctx, ctx->r_wrow_cluster, std::max<uint64_t>(8, (RW + nw) * 4), RW * 4));
  TRY(pin_grow(ctx, ctx->r_wrow_count, std::max<uint64_t>(8, (RW + nw) * 4), RW * 4));
  TRY(pin_grow(ctx, ctx->r_wrow_pattern, std::max<uint64_t>(8, (RW + nw) * 4), RW * 4));
  TRY(pin_grow(ctx, ctx->r_wrow_kmer, std::max<uint64_t>(8, (RW + nw) * 16), RW * 16));
  const bool compact = ctx->prm.emit_positions == 2u;
  if (ctx->n_pos && !compact) {
    const uint64_t P0 = ctx->pipe_pos, np = ctx->n_pos;
    TRY(pin_grow(ctx, ctx->r_pos_kmer, (P0 + np) * 8, P0 * 8));
    TRY(pin_grow(ctx, ctx->r_pos_seq, (P0 + np) * 4, P0 * 4));
    TRY(pin_grow(ctx, ctx->r_pos_cstart, (P0 + np) * 4, P0 * 4));
    TRY(pin_grow(ctx, ctx->r_pos_gstart, (P0 + np) * 4, P0 * 4));
    TRY(pin_grow(ctx, ctx->r_pos_flags, (P0 + np), P0));
    if (ctx->n_pos_wide)
      TRY(pin_grow(ctx, ctx->r_pos_wide, (ctx->pipe_pos_wide + ctx->n_pos_wide) * 16, ctx->pipe_pos_wide * 16));
    pos_rebase<<<cdiv(ctx->n_pos, 256), 256, 0, st>>>(ctx->d_pos_seq.as<uint32_t>(), ctx->d_pos_kmer.as<uint64_t>(),
                                                      ctx->d_pos_flags.as<uint8_t>(), ctx->n_pos, r.s0,
                                                      ctx->pipe_pos_wide);
    ctx->launches++;
  }
  CU(cudaEventRecord(ctx->ev_rows, st));
  CU(cudaStreamWaitEvent(cp, ctx->ev_rows, 0));
  auto d2h = [&](PinBuf& dst, size_t dst_off, const void* src, size_t bytes) -> int {
    if (bytes) CU(cudaMemcpyAsync((char*)dst.p + dst_off, src, bytes, cudaMemcpyDeviceToHost, cp));
    return PF_OK;
  };
  TRY(d2h(ctx->r_row_cluster, R * 4, ctx->d_row_cluster.p, nr * 4));
  TRY(d2h(ctx->r_row_count, R * 4, ctx->d_row_count.p, nr * 4));
  TRY(d2h(ctx->r_row_pattern, R * 4, ctx->d_row_pattern.p, nr * 4));
  TRY(d2h(ctx->r_row_kmer, R * 8, ctx->d_row_kmer.p, nr * 8));
  TRY(d2h(ctx->r_wrow_cluster, RW * 4, ctx->d_row_cluster.as<uint32_t>() + nr, nw * 4));
  TRY(d2h(ctx->r_wrow_count, RW * 4, ctx->d_row_count.as<uint32_t>() + nr, nw * 4));
  TRY(d2h(ctx->r_wrow_pattern, RW * 4, ctx->d_row_pattern.as<uint32_t>() + nr, nw * 4));
  TRY(d2h(ctx->r_wrow_kmer, RW * 16, ctx->d_wrow_kmer.p, nw * 16));
  TRY(d2h(ctx->r_cl_pattern, (size_t)ctx->pipe_clusters * 4, ctx->d_cl_pattern.p, (size_t)ctx->n_clusters * 4));
  if (ctx->n_pos && compact && ctx->prm.canonical)      // (r_pos_bits covers the whole batch: sized by the submit)
    TRY(d2h(ctx->r_pos_bits, (size_t)r.w0 * 4, ctx->d_pos_bits.p, (size_t)(r.w1 - r.w0) * 4));   // one bit per base: a u32 per packed word
  if (ctx->n_pos && !compact) {
    const uint64_t P0 = ctx->pipe_pos, np = ctx->n_pos;
    TRY(d2h(ctx->r_pos_kmer, P0 * 8, ctx->d_pos_kmer.p, np * 8));
    TRY(d2h(ctx->r_pos_seq, P0 * 4, ctx->d_pos_seq.p, np * 4));
    TRY(d2h(ctx->r_pos_cstart, P0 * 4, ctx->d_pos_cstart.p, np * 4));
    TRY(d2h(ctx->r_pos_gstart, P0 * 4, ctx->d_pos_gstart.p, np * 4));
    TRY(d2h(ctx->r_pos_flags, P0, ctx->d_pos_flags.p, np));
    if (ctx->n_pos_wide)
      TRY(d2h(ctx->r_pos_wide, ctx->pipe_pos_wide * 16, ctx->d_pos_wide.p, (size_t)ctx->n_pos_wide * 16));
  }
  CU(cudaEventRecord(ctx->ev_out_done, cp));
  ctx->pipe_rows += nr;
  ctx->pipe_wide_rows += nw;
  ctx->pipe_pos += ctx->n_pos;
  ctx->pipe_pos_wide += ctx->n_pos_wide;
  ctx->pipe_clusters += ctx->n_clusters;
  pf_stats& s = ctx->stats;
  s.bases += ctx->n_bases;
  s.instances += (uint64_t)N.n_records + Wd.n_records;
  s.unique_kmers += ctx->unique_last;
  s.rows += nr + nw;
  return PF_OK;
}

// D2H (copy stream) of the k-mer patterns numbered since the last call; the compute stream
// must have passed the K4 that appended them
int pipe_copy_new_patterns(pf_ctx* ctx) {
  const uint64_t done = ctx->kp.n, from = ctx->pipe_kp_copied, base = ctx->pipe_kp_base;
  if (done <= from) return PF_OK;
  const size_t row = (size_t)ctx->Wk * 4;
  TRY(pin_grow(ctx, ctx->r_new_kp, (done - base) * row, (from - base) * row));
  CU(cudaMemcpyAsync((char*)ctx->r_new_kp.p + (from - base) * row, ctx->kp.pool.as<uint32_t>() + from * ctx->Wk,
                     (done - from) * row, cudaMemcpyDeviceToHost, ctx->copy_stream));
  ctx->pipe_kp_copied = done;
  return PF_OK;
}

// pf_submit of a large batch: sub-batches of whole clusters flow through three batch slots, so
// that the H2D of sub-batches j+1 and j+2 (up_stream, enqueued by a helper thread) and the D2H
// of sub-batch j-1 (copy_stream) run under the kernels of sub-batch j (stream).  The pattern
// tables are shared, K4 of the sub-batches is ordered by the compute stream, so pattern ids are
// those of one big batch.
//
// Slots: *ctx holds sub-batch j; `nx` the uploaded (or uploading) j+1; `nx2` is where j+2 goes —
// the slot sub-batch j-1 ran in.  After the kernels of j are enqueued, *ctx and *nx swap
// contents (the helper that filled *nx has been joined; the one filling *nx2 is not touched).
int submit_pipelined(pf_ctx* ctx, const pf_batch* b, const std::vector<SubRange>& subs) {
  cudaStream_t st = ctx->stream, up = ctx->up_stream;
  TRY(finalize_pending(ctx));
  ctx->executed = false;
  ctx->alt.executed = false;
  ctx->alt2.executed = false;
  ctx->pipe_rows = ctx->pipe_wide_rows = ctx->pipe_pos = ctx->pipe_pos_wide = 0;
  ctx->pipe_clusters = 0;
  ctx->pipe_kp_base = ctx->kp.n;
  ctx->pipe_kp_copied = ctx->kp.n;
  ctx->pipe_cp_base = ctx->cp.n;
  for (double& m : ctx->pipe_ms) m = 0;
  TRY(pin_ensure(ctx, ctx->r_cl_pattern, std::max<size_t>(8, (size_t)b->n_clusters * 4)));
  ctx->pipe_bit_words = 0;
  if (ctx->prm.emit_positions == 2u && ctx->prm.canonical) {
    TRY(pin_ensure(ctx, ctx->r_pos_bits, std::max<size_t>(8, (size_t)b->n_words * 4)));
    ctx->pipe_bit_words = b->n_words;
  }
  {
    // row arrays: learned rows-per-base ratio, grown on demand
    const uint64_t est = (uint64_t)(ctx->row_ratio * 1.3 * (double)b->n_words * 32.0) + 65536;
    TRY(pin_grow(ctx, ctx->r_row_cluster, est * 4, 0));
    TRY(pin_grow(ctx, ctx->r_row_count, est * 4, 0));
    TRY(pin_grow(ctx, ctx->r_row_pattern, est * 4, 0));
    TRY(pin_grow(ctx, ctx->r_row_kmer, est * 8, 0));
  }
  struct Guard { pf_ctx* c; ~Guard() { c->pipe_mode = false; } } guard{ctx};
  ctx->pipe_mode = true;
  const size_t J = subs.size();
  ctx->pipe_subs = (uint32_t)J;
  static const bool dbg = getenv("PF_DEBUG_PIPE") != nullptr;
  auto now = []() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t_begin = now();
  double t_up = 0, t_ex = 0, t_out = 0, t_fin = 0, t_join = 0;
  CU(cudaEventRecord(ctx->ev_pipe[0], st));
  if (dbg) {                // GPU-side timeline of the sub-batches, printed by pf_collect
    while (ctx->dbg_ev.size() < J) {
      std::array<cudaEvent_t, 5> e{};
      for (auto& x : e) cudaEventCreate(&x);
      ctx->dbg_ev.push_back(e);
    }
    cudaEventRecord(ctx->dbg_ev[0][0], up);
  }
  auto add_h2d = [&]() {
    float m = 0;
    if (cudaEventElapsedTime(&m, ctx->ev_h2d[0], ctx->ev_h2d[1]) == cudaSuccess) ctx->pipe_ms[0] += m;
    else cudaGetLastError();
  };
  TRY(upload_async(ctx, *ctx, b, subs[0], up));
  if (dbg) cudaEventRecord(ctx->dbg_ev[0][1], up);
  TRY(upload_finish_slot(ctx, *ctx, st));
  add_h2d();

  // One upload runs at a time (the context's uploader thread: validation, planning and the
  // enqueue of the copies of ONE sub-batch), next to this thread driving the kernels
  // (pf_execute blocks on its read-backs).  It is joined before the next one starts and before
  // any return.
  struct Helper {
    AsyncWorker& w;
    int rc = PF_OK;
    void join() { w.join(); }
    ~Helper() { w.join(); }
  } helper{ctx->uploader};
  auto start_upload = [&](size_t j, BatchState* slot) -> int {
    // the kernels of the slot's last occupant must be done with its inputs; its result arrays
    // may still be draining, but an upload does not touch those
    if (cudaStreamWaitEvent(up, slot->ev_exec_end, 0) != cudaSuccess) return fail(ctx, PF_ERR_CUDA, "cudaStreamWaitEvent failed");
    helper.rc = PF_OK;
    helper.w.start([&, j, slot]() {
      cudaSetDevice(ctx->device);
      const double t0 = now();
      if (dbg) cudaEventRecord(ctx->dbg_ev[j][0], up);
      helper.rc = upload_async(ctx, *slot, b, subs[j], up);
      if (dbg) cudaEventRecord(ctx->dbg_ev[j][1], up);
      t_up += now() - t0;
    });
    return PF_OK;
  };
  BatchState* nx = &ctx->alt;
  BatchState* nx2 = &ctx->alt2;
  if (J > 1) TRY(start_upload(1, nx));
  // the upload of sub-batch j+1 has been enqueued (its planning is host work of ~1 ms): wait for
  // that, then start the one of j+2 in the slot sub-batch j-1 ran in
  auto next_upload = [&](size_t j) -> int {
    const double t0 = now();
    helper.join();
    t_join += now() - t0;
    if (helper.rc != PF_OK) return helper.rc;
    if (j + 2 < J) TRY(start_upload(j + 2, nx2));
    return PF_OK;
  };
  for (size_t j = 0; j < J; ++j) {
    double t0 = now();
    // (sub-batch 0 does not wait for the planning of sub-batch 1: its kernels go first)
    if (j > 0) TRY(next_upload(j));
    // this slot's previous rows must have left the device before they are overwritten
    CU(cudaStreamWaitEvent(st, ctx->ev_out_done, 0));
    t0 = now();
    if (dbg) cudaEventRecord(ctx->dbg_ev[j][2], st);
    TRY(pf_execute(ctx));
    t_ex += now() - t0;
    CU(cudaEventRecord(ctx->ev_exec_end, st));
    if (dbg) cudaEventRecord(ctx->dbg_ev[j][3], st);
    t0 = now();
    TRY(pipe_enqueue_results(ctx, subs[j]));
    if (dbg) cudaEventRecord(ctx->dbg_ev[j][4], ctx->copy_stream);
    t_out += now() - t0;
    t0 = now();
    // pf_execute folded sub-batch j-1's pattern count in before its own K4: those patterns are
    // final, and so are the stage timestamps of the slot it ran in (now *nx2)
    TRY(pipe_copy_new_patterns(ctx));
    if (j > 0) pipe_add_timings(ctx, nx2);
    if (j == 0) TRY(next_upload(0));
    if (j + 1 < J) {
      ctx->executed = false;
      std::swap(static_cast<BatchState&>(*ctx), *nx);     // *ctx: sub-batch j+1; *nx: free (j's slot)
      std::swap(nx, nx2);                                  // j+2 is (being) uploaded into the new nx
      TRY(upload_finish_slot(ctx, *ctx, st));
      add_h2d();
      t_fin += now() - t0;
    }
  }
  if (dbg)
    fprintf(stderr, "[pf] pipeline: %zu sub-batches, host ms: total %.2f  upload_async %.2f  join %.2f  execute %.2f  enqueue %.2f  finish %.2f\n",
            J, now() - t_begin, t_up, t_join, t_ex, t_out, t_fin);
  CU(cudaEventRecord(ctx->ev_pipe[1], st));
  ctx->pipe_pending = true;
  return PF_OK;
}

}  // namespace

extern "C" int pf_submit(pf_ctx* ctx, const pf_batch* batch) {
  if (!ctx) return PF_ERR_INVALID;
  if (!batch) return fail(ctx, PF_ERR_INVALID, "pf_submit: null batch");
  if (ctx->pipe_pending) return fail(ctx, PF_ERR_STATE, "pf_submit: results of the previous pf_submit were not collected");
  ctx->assoc.batch_ready = false;
  // with an association table the join (pf_assoc_collect) reads the batch's rows and windows on the
  // device after pf_collect: such batches run whole, as batches with N/IUPAC symbols do
  if (batch->n_seqs >= ctx->pipe_min_seqs && batch->n_amb_words == 0 && batch->seqs && batch->n_clusters > 1 &&
      !ctx->assoc.loaded) {
    CU(cudaSetDevice(ctx->device));
    const std::vector<SubRange> subs = split_batch(batch, ctx->pipe_target_seqs, ctx->pipe_first_seqs);
    if (subs.size() > 1) return submit_pipelined(ctx, batch, subs);
  }
  ctx->pipe_subs = 1;
  int r = pf_upload(ctx, batch);
  if (r != PF_OK) return r;
  return pf_execute(ctx);
}

namespace {
int collect_pipelined(pf_ctx* ctx, pf_batch_result* out) {
  cudaStream_t st = ctx->stream;
  CU(cudaStreamSynchronize(st));
  TRY(check_device_error(ctx));
  uint32_t* hcnt = ctx->h_counters.as<uint32_t>();
  ctx->kp.n = ctx->kp_base + hcnt[C_NEW_KP];      // last sub-batch
  ctx->kp_pending = false;
  ctx->executed = false;
  ctx->alt.executed = false;
  ctx->alt2.executed = false;
  ctx->pipe_pending = false;
  pipe_add_timings(ctx);
  const uint64_t new_kp = ctx->kp.n - ctx->pipe_kp_base, new_cp = ctx->cp.n - ctx->pipe_cp_base;
  CU(cudaEventRecord(ctx->ev_d2h[0], st));
  TRY(pipe_copy_new_patterns(ctx));
  if (!ctx->r_new_kp.p) TRY(pin_ensure(ctx, ctx->r_new_kp, 8));
  TRY(pin_ensure(ctx, ctx->r_new_cp, std::max<size_t>(8, new_cp * ctx->W * 4)));
  if (new_cp)
    CU(cudaMemcpyAsync(ctx->r_new_cp.p, ctx->cp.pool.as<uint32_t>() + ctx->pipe_cp_base * ctx->W, new_cp * ctx->W * 4,
                       cudaMemcpyDeviceToHost, st));
  CU(cudaEventRecord(ctx->ev_d2h[1], st));
  CU(cudaStreamSynchronize(st));
  CU(cudaStreamSynchronize(ctx->copy_stream));
  if (getenv("PF_DEBUG_PIPE") && ctx->dbg_ev.size() >= ctx->pipe_subs) {
    CU(cudaStreamSynchronize(ctx->up_stream));
    for (uint32_t j = 0; j < ctx->pipe_subs; ++j) {
      float t[5] = {0, 0, 0, 0, 0};
      for (int i = 0; i < 5; ++i)
        if (cudaEventElapsedTime(&t[i], ctx->ev_pipe[0], ctx->dbg_ev[j][i]) != cudaSuccess) { cudaGetLastError(); t[i] = -1; }
      fprintf(stderr, "[pf] timeline sub %u: upload %.2f..%.2f  kernels %.2f..%.2f  d2h done %.2f ms\n", j, t[0], t[1], t[2],
              t[3], t[4]);
    }
  }
  if (out) {
    memset(out, 0, sizeof *out);
    out->n_rows = ctx->pipe_rows;
    out->row_cluster = ctx->r_row_cluster.as<uint32_t>();
    out->row_kmer = ctx->r_row_kmer.as<uint64_t>();
    out->row_count = ctx->r_row_count.as<uint32_t>();
    out->row_pattern = ctx->r_row_pattern.as<uint32_t>();
    out->n_wide_rows = ctx->pipe_wide_rows;
    out->wide_row_cluster = ctx->r_wrow_cluster.as<uint32_t>();
    out->wide_row_kmer = ctx->r_wrow_kmer.as<uint64_t>();
    out->wide_row_count = ctx->r_wrow_count.as<uint32_t>();
    out->wide_row_pattern = ctx->r_wrow_pattern.as<uint32_t>();
    // (xwide_row_* / pos_xwide_kmer stay empty: batches with N/IUPAC symbols are not pipelined)
    out->n_clusters = ctx->pipe_clusters;
    out->cluster_pattern = ctx->r_cl_pattern.as<uint32_t>();
    out->kmer_pattern_base = ctx->pipe_kp_base;
    out->n_new_kmer_patterns = new_kp;
    out->new_kmer_patterns = ctx->r_new_kp.as<uint32_t>();
    out->cluster_pattern_base = ctx->pipe_cp_base;
    out->n_new_cluster_patterns = new_cp;
    out->new_cluster_patterns = ctx->r_new_cp.as<uint32_t>();
    out->n_pos = ctx->pipe_pos;
    out->pos_kmer = ctx->r_pos_kmer.as<uint64_t>();
    out->pos_seq = ctx->r_pos_seq.as<uint32_t>();
    out->pos_contig_start = ctx->r_pos_cstart.as<int32_t>();
    out->pos_gene_start = ctx->r_pos_gstart.as<int32_t>();
    out->pos_flags = ctx->r_pos_flags.as<uint8_t>();
    out->pos_wide_kmer = ctx->r_pos_wide.as<uint64_t>();
    out->n_pos_wide = ctx->pipe_pos_wide;
    if (ctx->prm.emit_positions == 2u) {
      out->pos_kmer = nullptr; out->pos_seq = nullptr; out->pos_contig_start = nullptr;
      out->pos_gene_start = nullptr; out->pos_flags = nullptr; out->pos_wide_kmer = nullptr;
      out->n_pos_wide = 0;
      if (ctx->pipe_pos && ctx->pipe_bit_words) {
        out->pos_strand_bits = ctx->r_pos_bits.as<uint32_t>();
        out->n_pos_bit_words = ctx->pipe_bit_words;
      }
    }
  }
  pf_stats& s = ctx->stats;
  s.batches++;
  s.kmer_patterns = ctx->kp.n;
  s.cluster_patterns = ctx->cp.n;
  s.total_launches = ctx->launches;
  s.ms_h2d = (float)ctx->pipe_ms[0]; s.ms_extract = (float)ctx->pipe_ms[1]; s.ms_hist = (float)ctx->pipe_ms[2];
  s.ms_sort = (float)ctx->pipe_ms[3]; s.ms_mark = (float)ctx->pipe_ms[4]; s.ms_count = (float)ctx->pipe_ms[5];
  s.ms_reduce = (float)ctx->pipe_ms[6]; s.ms_dedup = (float)ctx->pipe_ms[7];
  float m = 0;
  if (cudaEventElapsedTime(&m, ctx->ev_pipe[0], ctx->ev_pipe[1]) == cudaSuccess) s.ms_total = m;
  if (cudaEventElapsedTime(&m, ctx->ev_d2h[0], ctx->ev_d2h[1]) == cudaSuccess) s.ms_d2h = m;
  return PF_OK;
}
}  // namespace

extern "C" int pf_collect(pf_ctx* ctx, pf_batch_result* out) {
  if (!ctx) return PF_ERR_INVALID;
  if (ctx->pipe_pending) { CU(cudaSetDevice(ctx->device)); return collect_pipelined(ctx, out); }
  if (!ctx->executed) return fail(ctx, PF_ERR_STATE, "pf_collect: nothing executed");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  CU(cudaStreamSynchronize(st));
  uint32_t* hcnt = ctx->h_counters.as<uint32_t>();
  TRY(check_device_error(ctx));
  WidthState& N = ctx->nar;
  WidthState& Wd = ctx->wid;
  WidthState& X = ctx->xwd;
  const uint64_t rows = (uint64_t)N.n_rows + Wd.n_rows + X.n_rows;
  const uint64_t new_kp = hcnt[C_NEW_KP];
  const uint64_t new_cp = ctx->cp.n - ctx->cp_base;
  ctx->kp.n = ctx->kp_base + new_kp;
  ctx->kp_pending = false;
  ctx->executed = false;      // results are handed out once

  CU(cudaEventRecord(ctx->ev_d2h[0], st));
  auto d2h = [&](PinBuf& dst, const void* src, size_t bytes) -> int {
    TRY(pin_ensure(ctx, dst, std::max<size_t>(bytes, 8)));
    if (bytes) CU(cudaMemcpyAsync(dst.p, src, bytes, cudaMemcpyDeviceToHost, st));
    return PF_OK;
  };
  if (!ctx->rows_prefetched) {
    TRY(d2h(ctx->r_row_cluster, ctx->d_row_cluster.p, rows * 4));
    TRY(d2h(ctx->r_row_count, ctx->d_row_count.p, rows * 4));
    TRY(d2h(ctx->r_row_kmer, ctx->d_row_kmer.p, (size_t)N.n_rows * 8));
    TRY(d2h(ctx->r_wrow_kmer, ctx->d_wrow_kmer.p, (size_t)Wd.n_rows * 16));
    if (X.n_rows) TRY(d2h(ctx->r_xrow_kmer, ctx->d_xrow_kmer.p, (size_t)X.n_rows * 32));
  }
  TRY(d2h(ctx->r_row_pattern, ctx->d_row_pattern.p, rows * 4));
  TRY(d2h(ctx->r_cl_pattern, ctx->d_cl_pattern.p, (size_t)ctx->n_clusters * 4));
  TRY(d2h(ctx->r_new_kp, ctx->kp.pool.as<uint32_t>() + ctx->kp_base * ctx->Wk, new_kp * ctx->Wk * 4));
  TRY(d2h(ctx->r_new_cp, ctx->cp.pool.as<uint32_t>() + ctx->cp_base * ctx->W, new_cp * ctx->W * 4));
  const bool compact = ctx->prm.emit_positions == 2u;
  if (ctx->n_pos && compact) {
    if (ctx->prm.canonical) TRY(d2h(ctx->r_pos_bits, ctx->d_pos_bits.p, (size_t)ctx->n_words * 4));
  } else if (ctx->n_pos) {
    TRY(d2h(ctx->r_pos_kmer, ctx->d_pos_kmer.p, (size_t)ctx->n_pos * 8));
    TRY(d2h(ctx->r_pos_seq, ctx->d_pos_seq.p, (size_t)ctx->n_pos * 4));
    TRY(d2h(ctx->r_pos_cstart, ctx->d_pos_cstart.p, (size_t)ctx->n_pos * 4));
    TRY(d2h(ctx->r_pos_gstart, ctx->d_pos_gstart.p, (size_t)ctx->n_pos * 4));
    TRY(d2h(ctx->r_pos_flags, ctx->d_pos_flags.p, (size_t)ctx->n_pos));
  }
  if (ctx->n_pos_wide && !compact) TRY(d2h(ctx->r_pos_wide, ctx->d_pos_wide.p, (size_t)ctx->n_pos_wide * 16));
  if (ctx->n_pos_xwide && !compact) TRY(d2h(ctx->r_pos_xwide, ctx->d_pos_xwide.p, (size_t)ctx->n_pos_xwide * 32));
  CU(cudaEventRecord(ctx->ev_d2h[1], st));
  CU(cudaStreamSynchronize(st));
  if (ctx->rows_prefetched) CU(cudaStreamSynchronize(ctx->copy_stream));
  ctx->rows_prefetched = false;
  ctx->assoc.batch_ready = true;        // its rows and windows stay on the device until the next upload

  if (out) {
    memset(out, 0, sizeof *out);
    out->n_rows = N.n_rows;
    out->row_cluster = ctx->r_row_cluster.as<uint32_t>();
    out->row_kmer = ctx->r_row_kmer.as<uint64_t>();
    out->row_count = ctx->r_row_count.as<uint32_t>();
    out->row_pattern = ctx->r_row_pattern.as<uint32_t>();
    out->n_wide_rows = Wd.n_rows;
    out->wide_row_cluster = out->row_cluster + N.n_rows;
    out->wide_row_kmer = ctx->r_wrow_kmer.as<uint64_t>();
    out->wide_row_count = out->row_count + N.n_rows;
    out->wide_row_pattern = out->row_pattern + N.n_rows;
    out->n_clusters = ctx->n_clusters;
    out->cluster_pattern = ctx->r_cl_pattern.as<uint32_t>();
    out->kmer_pattern_base = ctx->kp_base;
    out->n_new_kmer_patterns = new_kp;
    out->new_kmer_patterns = ctx->r_new_kp.as<uint32_t>();
    out->cluster_pattern_base = ctx->cp_base;
    out->n_new_cluster_patterns = new_cp;
    out->new_cluster_patterns = ctx->r_new_cp.as<uint32_t>();
    out->n_pos = ctx->n_pos;
    out->pos_kmer = ctx->r_pos_kmer.as<uint64_t>();
    out->pos_seq = ctx->r_pos_seq.as<uint32_t>();
    out->pos_contig_start = ctx->r_pos_cstart.as<int32_t>();
    out->pos_gene_start = ctx->r_pos_gstart.as<int32_t>();
    out->pos_flags = ctx->r_pos_flags.as<uint8_t>();
    out->pos_wide_kmer = ctx->r_pos_wide.as<uint64_t>();
    out->n_pos_wide = ctx->n_pos_wide;
    if (X.n_rows) {           // (rows of the 256-bit section follow the wide ones in the row arrays)
      out->n_xwide_rows = X.n_rows;
      out->xwide_row_cluster = out->row_cluster + N.n_rows + Wd.n_rows;
      out->xwide_row_kmer = ctx->r_xrow_kmer.as<uint64_t>();
      out->xwide_row_count = out->row_count + N.n_rows + Wd.n_rows;
      out->xwide_row_pattern = out->row_pattern + N.n_rows + Wd.n_rows;
    }
    if (ctx->n_pos_xwide && !compact) {
      out->pos_xwide_kmer = ctx->r_pos_xwide.as<uint64_t>();
      out->n_pos_xwide = ctx->n_pos_xwide;
    }
    if (compact) {
      out->pos_kmer = nullptr; out->pos_seq = nullptr; out->pos_contig_start = nullptr;
      out->pos_gene_start = nullptr; out->pos_flags = nullptr; out->pos_wide_kmer = nullptr;
      out->n_pos_wide = 0;
      if (ctx->n_pos && ctx->prm.canonical) {
        out->pos_strand_bits = ctx->r_pos_bits.as<uint32_t>();
        out->n_pos_bit_words = ctx->n_words;
      }
    }
  }
  // ---- stats ---------------------------------------------------------------
  pf_stats& s = ctx->stats;
  s.batches++;
  s.bases += ctx->n_bases;
  s.instances += (uint64_t)N.n_records + Wd.n_records + X.n_records;
  s.unique_kmers += ctx->unique_last;
  s.rows += rows;
  s.kmer_patterns = ctx->kp.n;
  s.cluster_patterns = ctx->cp.n;
  s.sort_passes = (uint32_t)N.passes;
  s.total_launches = ctx->launches;
  fill_timings(ctx);
  {
    float m = 0;
    if (cudaEventElapsedTime(&m, ctx->ev_d2h[0], ctx->ev_d2h[1]) == cudaSuccess) s.ms_d2h = m;
  }
  return PF_OK;
}

extern "C" int pf_reset_patterns(pf_ctx* ctx) {
  if (!ctx) return PF_ERR_INVALID;
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->executed = false;
  ctx->kp_pending = false;
  for (PatternSpace* s : {&ctx->kp, &ctx->cp}) {
    s->n = 0;
    s->x_n_unique = 0;
    if (s->table.p) CU(cudaMemsetAsync(s->table.p, 0xff, (size_t)s->table_size * 4, ctx->stream));
  }
  ctx->kp_base = ctx->cp_base = 0;
  ctx->stats.kmer_patterns = ctx->stats.cluster_patterns = 0;
  ctx->assoc.kp_done = ctx->assoc.cp_done = 0;
  CU(cudaStreamSynchronize(ctx->stream));
  return PF_OK;
}

extern "C" int pf_patterns_export(pf_ctx* ctx, int cluster_namespace, uint64_t first, uint64_t count,
                                  uint32_t* host_out) {
  if (!ctx || !host_out) return PF_ERR_INVALID;
  TRY(finalize_pending(ctx));
  PatternSpace& s = cluster_namespace ? ctx->cp : ctx->kp;
  if (first + count > s.n) return fail(ctx, PF_ERR_INVALID, "pattern range [%llu,%llu) beyond %llu",
                                       (unsigned long long)first, (unsigned long long)(first + count),
                                       (unsigned long long)s.n);
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->stream));
  if (count)
    CU(cudaMemcpy(host_out, s.pool.as<uint32_t>() + first * s.key_words, count * s.key_words * 4,
                  cudaMemcpyDeviceToHost));
  return PF_OK;
}

extern "C" int pf_pattern_ids(pf_ctx* ctx, int cluster_namespace, uint64_t first, uint64_t count,
                              uint8_t* host_digests) {
  if (!ctx || (count && !host_digests)) return PF_ERR_INVALID;
  CU(cudaSetDevice(ctx->device));
  TRY(finalize_pending(ctx));
  PatternSpace& s = cluster_namespace ? ctx->cp : ctx->kp;
  if (first + count > s.n) return fail(ctx, PF_ERR_INVALID, "pattern range [%llu,%llu) beyond %llu",
                                       (unsigned long long)first, (unsigned long long)(first + count),
                                       (unsigned long long)s.n);
  if (count == 0) return PF_OK;
  TRY(dev_ensure(ctx, ctx->d_digests, count * 16));
  k5_md5_ids<<<cdiv(count, 128), 128, 0, ctx->stream>>>(
      s.pool.as<uint32_t>(), (uint32_t)first, (uint32_t)count, s.key_words, ctx->W, ctx->prm.n_samples,
      cluster_namespace ? 1 : 0, ctx->cp.pool.as<uint32_t>(), ctx->d_digests.as<uint8_t>());
  ctx->launches++;
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(host_digests, ctx->d_digests.p, count * 16, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return PF_OK;
}

extern "C" int pf_stats_get(pf_ctx* ctx, pf_stats* out) {
  if (!ctx || !out) return PF_ERR_INVALID;
  if (ctx->executed) {
    TRY(finalize_pending(ctx));
    CU(cudaStreamSynchronize(ctx->stream));
    fill_timings(ctx);
  }
  ctx->stats.kmer_patterns = ctx->kp.n;
  ctx->stats.cluster_patterns = ctx->cp.n;
  *out = ctx->stats;
  out->total_launches = ctx->launches;
  return PF_OK;
}
