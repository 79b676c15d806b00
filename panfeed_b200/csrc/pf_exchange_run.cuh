// pf_exchange_run.cuh — pf_exchange_run / pf_exchange_release: the multi-GPU pattern exchange of
// pf_exchange.cuh in one call, over collectives the caller provides (pf_comm), and pf_comm_local,
// a communicator for the threads of one process.  The kernels are those of pf_exchange.cuh
// (x_classify, x_scatter, x_pack, the K4 dedup of exchange_dedup, x_unpack); the only new device
// code is the scan of the unique counts.
// Part of libpanfeed_b200.so's single translation unit: included once, in order, by pf_api.cu.

namespace pf {
// owner_base[r] = sum of n_unique[r'] over r' < r  (one warp: world <= 32)
__global__ void x_owner_base(const uint32_t* __restrict__ n_unique, uint32_t world, uint32_t* __restrict__ owner_base) {
  const uint32_t r = threadIdx.x;
  const uint32_t v = r < world ? n_unique[r] : 0u;
  uint32_t inc = v;
#pragma unroll
  for (uint32_t d = 1; d < 32; d <<= 1) {
    const uint32_t t = __shfl_up_sync(kFull, inc, d);
    if (r >= d) inc += t;
  }
  if (r < world) owner_base[r] = inc - v;
}
}  // namespace pf

namespace {

constexpr uint32_t kXMaxWorld = 32;              // XDest holds 32 destinations
constexpr uint32_t kXMagic = 0x50465852u;        // "PFXR"
constexpr uint32_t kXSlackRows = 1024;           // a receive buffer grows to need * 5/4 + this

enum : uint32_t { XR_NO_PEER = 1, XR_A2A = 2, XR_CM = 4 };

// What every rank all-gathers before the keys move (fixed size: the receive side always has room
// for kXMaxWorld records, so that a rank with a wrong `world` cannot overrun it).  Namespace index
// as in the ABI: 0 = k-mer, 1 = cluster.
struct XRec {
  uint32_t magic, world, rank, flags;
  uint64_t host, pid;
  int32_t device;
  uint32_t buf_ok[2];            // the receive buffer exists (growth did not fail)
  uint32_t ipc_ok[2];            // ... and has a CUDA IPC handle
  uint32_t pad;
  uint64_t cap[2];               // receive capacity in rows
  uint64_t ptr[2];               // raw device pointer of the receive buffer
  uint8_t handle[2][64];
  uint32_t counts[2][kXMaxWorld];   // bucket sizes to every owner (copied on the device from x_counts)
};

struct XPeer {
  bool used = false, ipc = false;
  unsigned char handle[64];
  void* ptr = nullptr;
};

struct XNs {
  // peer memory: this rank's receive buffer, [cap rows x key words | cap unique indices]
  DevBuf recv;
  uint64_t cap = 0;
  bool buf_ok = true, ipc_ok = false;
  unsigned char handle[64] = {};
  XPeer peer[kXMaxWorld];
  bool seen = false;             // peer buffers mapped at least once
  // all-to-all transport
  DevBuf send, a2a_recv, uniq;
  // both
  DevBuf returned, l2g, writer;
  uint64_t n_local = 0, bytes_sent = 0;
};

struct XRunState {
  XNs ns[2];
  bool peer_failed = false;      // a call fell back to the all-to-all: so do later ones
  DevBuf d_rec;                  // [1 + kXMaxWorld] records: mine, then every rank's
  DevBuf d_small;                // per namespace: n_unique, all n_unique[32], owner_base[32]; then ok word, ok[32]
  PinBuf h_rec;                  // [1 + kXMaxWorld] records
  PinBuf h_small;                // all n_unique of both namespaces [2][32], ok words [32]
  uint64_t host_id = 0;
};

constexpr size_t kXSmallNs = 1 + 2 * kXMaxWorld;     // words per namespace in d_small
inline uint32_t* xs_nu(XRunState& x, int ns) { return x.d_small.as<uint32_t>() + ns * kXSmallNs; }
inline uint32_t* xs_all_nu(XRunState& x, int ns) { return xs_nu(x, ns) + 1; }
inline uint32_t* xs_base(XRunState& x, int ns) { return xs_nu(x, ns) + 1 + kXMaxWorld; }
inline uint32_t* xs_ok(XRunState& x) { return x.d_small.as<uint32_t>() + 2 * kXSmallNs; }

uint64_t host_identity() {
  // the boot id tells hosts apart (a hostname may repeat across containers); the hostname if absent
  char buf[256] = {};
  size_t n = 0;
  if (FILE* f = fopen("/proc/sys/kernel/random/boot_id", "r")) { n = fread(buf, 1, sizeof buf - 1, f); fclose(f); }
  if (n == 0) { gethostname(buf, sizeof buf - 1); n = strlen(buf); }
  uint64_t h = 1469598103934665603ull;                // FNV-1a
  for (size_t i = 0; i < n; ++i) { h ^= (unsigned char)buf[i]; h *= 1099511628211ull; }
  return h;
}

int xr_state(pf_ctx* ctx, XRunState*& out) {
  if (!ctx->xrun) {
    ctx->xrun = new XRunState();
    ctx->xrun->host_id = host_identity();
  }
  XRunState& x = *ctx->xrun;
  TRY(dev_ensure(ctx, x.d_rec, (1 + kXMaxWorld) * sizeof(XRec)));
  TRY(dev_ensure(ctx, x.d_small, (2 * kXSmallNs + 1 + kXMaxWorld) * 4));
  TRY(pin_ensure(ctx, x.h_rec, (1 + kXMaxWorld) * sizeof(XRec)));
  TRY(pin_ensure(ctx, x.h_small, 3 * kXMaxWorld * 4));
  out = &x;
  return PF_OK;
}

int xr_collective_failed(pf_ctx* ctx, const char* what, int rc) {
  return fail(ctx, PF_ERR_STATE, "pf_exchange_run: the communicator's %s returned %d", what, rc);
}

int xr_gather(pf_ctx* ctx, const pf_comm* c, const void* send, void* recv, uint64_t bytes) {
  const int rc = c->all_gather(send, recv, bytes, (void*)ctx->stream, c->user);
  return rc ? xr_collective_failed(ctx, "all_gather", rc) : PF_OK;
}

int xr_a2a(pf_ctx* ctx, const pf_comm* c, const void* send, const uint64_t* sb, void* recv, const uint64_t* rb) {
  const int rc = c->all_to_all_v(send, sb, recv, rb, (void*)ctx->stream, c->user);
  return rc ? xr_collective_failed(ctx, "all_to_all_v", rc) : PF_OK;
}

// every rank's `ok`, ANDed (a host sync); with ok = true it is a barrier of the host threads
int xr_all_ok(pf_ctx* ctx, const pf_comm* c, XRunState& x, bool ok, bool& all) {
  uint32_t* h = x.h_small.as<uint32_t>() + 2 * kXMaxWorld;
  uint32_t* d = xs_ok(x);
  CU(cudaMemsetAsync(d + 1, 0, kXMaxWorld * 4, ctx->stream));
  CU(cudaMemsetAsync(d, ok ? 1 : 0, 1, ctx->stream));
  CU(cudaMemsetAsync((char*)d + 1, 0, 3, ctx->stream));
  TRY(xr_gather(ctx, c, d, d + 1, 4));
  CU(cudaMemcpyAsync(h, d + 1, c->world * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  all = true;
  for (uint32_t r = 0; r < c->world; ++r) all = all && h[r] == 1;
  return PF_OK;
}

void xr_close_peer(pf_ctx* ctx, XPeer& p) {
  if (p.used && p.ipc && p.ptr) { cudaSetDevice(ctx->device); if (cudaIpcCloseMemHandle(p.ptr) != cudaSuccess) cudaGetLastError(); }
  p = XPeer();
}

// this rank's receive buffer of a namespace holds at least `rows` rows (+ their unique indices)
void xr_grow(pf_ctx* ctx, XNs& n, uint32_t key_words, uint64_t rows) {
  const size_t row = (size_t)(key_words + 1) * 4;
  if (n.recv.p && n.cap >= rows) return;
  cudaStreamSynchronize(ctx->stream);
  if (n.recv.p) { cudaFree(n.recv.p); n.recv = DevBuf(); n.cap = 0; }      // (contents are scratch)
  n.buf_ok = n.ipc_ok = false;
  void* p = nullptr;
  if (cudaMalloc(&p, std::max<size_t>(row, rows * row)) != cudaSuccess) { cudaGetLastError(); return; }
  n.recv.p = p;
  n.recv.cap = std::max<size_t>(row, rows * row);
  n.cap = n.recv.cap / row;
  n.buf_ok = true;
  cudaIpcMemHandle_t h;
  if (cudaIpcGetMemHandle(&h, p) == cudaSuccess) { memcpy(n.handle, &h, 64); n.ipc_ok = true; }
  else cudaGetLastError();                 // (peers in this process do not need it)
}

// fill and all-gather the records (one host sync); nss: the namespaces of this step
int xr_records(pf_ctx* ctx, const pf_comm* c, XRunState& x, uint32_t flags, const int* nss, int n_ns,
               const XRec*& all) {
  const uint32_t world = c->world;
  XRec* mine = x.h_rec.as<XRec>();
  memset(mine, 0, sizeof(XRec));
  mine->magic = kXMagic;
  mine->world = world;
  mine->rank = c->rank;
  mine->flags = ((flags & PF_EXCHANGE_NO_PEER) ? XR_NO_PEER : 0u) | (c->all_to_all_v ? XR_A2A : 0u) |
                (ctx->prm.consider_missing ? XR_CM : 0u);
  mine->host = x.host_id;
  mine->pid = (uint64_t)getpid();
  mine->device = ctx->device;
  for (int ns = 0; ns < 2; ++ns) {
    const XNs& n = x.ns[ns];
    mine->buf_ok[ns] = n.buf_ok;
    mine->ipc_ok[ns] = n.ipc_ok;
    mine->cap[ns] = n.cap;
    mine->ptr[ns] = (uint64_t)(uintptr_t)n.recv.p;
    memcpy(mine->handle[ns], n.handle, 64);
  }
  XRec* d = x.d_rec.as<XRec>();
  cudaStream_t st = ctx->stream;
  CU(cudaMemcpyAsync(d, mine, sizeof(XRec), cudaMemcpyHostToDevice, st));
  for (int i = 0; i < n_ns; ++i) {       // bucket sizes straight from the classify kernels
    PatternSpace& s = nss[i] ? ctx->cp : ctx->kp;
    CU(cudaMemcpyAsync(d->counts[nss[i]], s.x_counts.p, world * 4, cudaMemcpyDeviceToDevice, st));
  }
  CU(cudaMemsetAsync(d + 1, 0, kXMaxWorld * sizeof(XRec), st));
  TRY(xr_gather(ctx, c, d, d + 1, sizeof(XRec)));
  CU(cudaMemcpyAsync(mine + 1, d + 1, kXMaxWorld * sizeof(XRec), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  all = mine + 1;
  // every rank sees the same records: all of them return here alike
  for (uint32_t r = 0; r < kXMaxWorld; ++r) {
    const XRec& q = all[r];
    const bool agree = r < world ? (q.magic == kXMagic && q.world == world && q.rank == r &&
                                    (q.flags & XR_CM) == (mine->flags & XR_CM))
                                 : q.magic == 0;
    if (!agree)
      return fail(ctx, PF_ERR_INVALID, "pf_exchange_run: the ranks disagree on the communicator or the "
                                       "consider_missing setting (rank %u, world %u, record %u)", c->rank, world, r);
  }
  return PF_OK;
}

// peer memory: receive buffers large enough on every rank, the peers' buffers mapped; ok = this
// rank could use every buffer.  opening: mappings were (re)made, the caller agrees on ok.
int xr_peer_setup(pf_ctx* ctx, const pf_comm* c, XRunState& x, uint32_t flags, const int* nss, int n_ns,
                  const XRec*& all, bool& ok, bool& opening) {
  const uint32_t world = c->world, rank = c->rank;
  bool grow_any = false;
  opening = false;
  for (int i = 0; i < n_ns; ++i) {
    const int ns = nss[i];
    opening = opening || !x.ns[ns].seen;
    for (uint32_t o = 0; o < world; ++o) {
      uint64_t need = 0;
      for (uint32_t r = 0; r < world; ++r) need += all[r].counts[ns][o];
      if (need > all[o].cap[ns] || !all[o].buf_ok[ns]) grow_any = true;
    }
  }
  if (grow_any) {
    // mappings of buffers about to be freed go first; their owners wait for that (barrier)
    uint64_t need_mine[2] = {0, 0};
    bool grow_rank[2][kXMaxWorld] = {};
    for (int i = 0; i < n_ns; ++i) {
      const int ns = nss[i];
      for (uint32_t o = 0; o < world; ++o) {
        uint64_t need = 0;
        for (uint32_t r = 0; r < world; ++r) need += all[r].counts[ns][o];
        grow_rank[ns][o] = need > all[o].cap[ns] || !all[o].buf_ok[ns];
        if (o == rank) need_mine[ns] = need;
        if (grow_rank[ns][o] && o != rank) xr_close_peer(ctx, x.ns[ns].peer[o]);
      }
    }
    CU(cudaStreamSynchronize(ctx->stream));
    bool all_ok = true;
    TRY(xr_all_ok(ctx, c, x, true, all_ok));                  // barrier
    for (int i = 0; i < n_ns; ++i) {
      const int ns = nss[i];
      if (grow_rank[ns][rank])
        xr_grow(ctx, x.ns[ns], (ns ? ctx->cp : ctx->kp).key_words, need_mine[ns] + need_mine[ns] / 4 + kXSlackRows);
    }
    TRY(xr_records(ctx, c, x, flags, nss, n_ns, all));
    opening = true;
  }
  ok = true;
  int can = 0;
  for (int i = 0; i < n_ns; ++i) {
    const int ns = nss[i];
    XNs& n = x.ns[ns];
    ok = ok && n.buf_ok;
    for (uint32_t r = 0; r < world; ++r) {
      if (r == rank) continue;
      const XRec& q = all[r];
      XPeer& p = n.peer[r];
      if (!q.buf_ok[ns]) { ok = false; continue; }
      const bool same_process = q.host == x.host_id && q.pid == (uint64_t)getpid();
      if (same_process) {
        if (q.device != ctx->device) {
          if (cudaDeviceCanAccessPeer(&can, ctx->device, q.device) != cudaSuccess || !can) { cudaGetLastError(); ok = false; continue; }
          const cudaError_t e = cudaDeviceEnablePeerAccess(q.device, 0);
          if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); ok = false; continue; }
          cudaGetLastError();                                   // (clears "already enabled")
        }
        p.used = true; p.ipc = false; p.ptr = (void*)(uintptr_t)q.ptr[ns];
        continue;
      }
      if (p.used && p.ipc && memcmp(p.handle, q.handle[ns], 64) == 0) continue;     // cached mapping
      xr_close_peer(ctx, p);
      if (!q.ipc_ok[ns]) { ok = false; continue; }
      cudaIpcMemHandle_t h;
      memcpy(&h, q.handle[ns], 64);
      void* mapped = nullptr;
      if (cudaIpcOpenMemHandle(&mapped, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); ok = false; continue; }
      p.used = true; p.ipc = true; p.ptr = mapped;
      memcpy(p.handle, q.handle[ns], 64);
    }
    if (!n.seen) opening = true;
    n.seen = true;
  }
  return PF_OK;
}

// owner side + ids back + unpack of one namespace, either transport; recv: the received keys
int xr_finish(pf_ctx* ctx, const pf_comm* c, XRunState& x, int ns, uint32_t flags, const XRec* all, bool peer,
              const uint32_t* recv, uint64_t n_recv, uint32_t* uniq) {
  const uint32_t world = c->world, rank = c->rank;
  PatternSpace& s = ns ? ctx->cp : ctx->kp;
  XNs& n = x.ns[ns];
  cudaStream_t st = ctx->stream;
  const uint32_t nl = (uint32_t)n.n_local;
  TRY(exchange_dedup(ctx, s, recv, n_recv, uniq, xs_nu(x, ns), (flags & PF_EXCHANGE_KEEP_UNIQUE) != 0));
  // every owner's unique count; on the peer path also the barrier before the indices are read back
  TRY(xr_gather(ctx, c, xs_nu(x, ns), xs_all_nu(x, ns), 4));
  x_owner_base<<<1, 32, 0, st>>>(xs_all_nu(x, ns), world, xs_base(x, ns));
  ctx->launches++;
  CU(cudaGetLastError());
  TRY(dev_ensure(ctx, n.returned, std::max<size_t>(1, nl) * 4));
  uint32_t* returned = n.returned.as<uint32_t>();
  if (peer) {
    // this rank's bucket in owner o's buffer: rows [row0, row0 + count) of its unique indices
    uint64_t send0 = 0;
    for (uint32_t o = 0; o < world; ++o) {
      const uint64_t cnt = all[rank].counts[ns][o];
      uint64_t row0 = 0;
      for (uint32_t r = 0; r < rank; ++r) row0 += all[r].counts[ns][o];
      if (cnt) {
        const uint32_t* base = o == rank ? n.recv.as<uint32_t>() : static_cast<const uint32_t*>(n.peer[o].ptr);
        const uint32_t* src = base + all[o].cap[ns] * s.key_words + row0;
        CU(cudaMemcpyAsync(returned + send0, src, cnt * 4, cudaMemcpyDefault, st));
      }
      send0 += cnt;
    }
  } else {
    uint64_t sb[kXMaxWorld], rb[kXMaxWorld];
    for (uint32_t r = 0; r < world; ++r) { sb[r] = (uint64_t)all[r].counts[ns][rank] * 4; rb[r] = (uint64_t)all[rank].counts[ns][r] * 4; }
    TRY(xr_a2a(ctx, c, uniq, sb, returned, rb));
  }
  TRY(dev_ensure(ctx, n.l2g, std::max<size_t>(1, nl) * 4));
  uint8_t* writer = nullptr;
  if (flags & PF_EXCHANGE_WRITER) { TRY(dev_ensure(ctx, n.writer, std::max<size_t>(1, nl))); writer = n.writer.as<uint8_t>(); }
  if (nl) {
    x_unpack<<<cdiv(nl, 256), 256, 0, st>>>(returned, s.x_perm.as<uint32_t>(), s.x_owner.as<uint32_t>(), xs_base(x, ns),
                                            nl, n.l2g.as<uint32_t>(), writer);
    ctx->launches++;
    CU(cudaGetLastError());
  }
  return PF_OK;
}

// one step: the namespaces nss (both at once, or one), k-mer keys rewritten with mask_remap
int xr_step(pf_ctx* ctx, const pf_comm* c, XRunState& x, uint32_t flags, const int* nss, int n_ns,
            const uint32_t* mask_remap) {
  const uint32_t world = c->world, rank = c->rank;
  cudaStream_t st = ctx->stream;
  for (int i = 0; i < n_ns; ++i) {
    const int ns = nss[i];
    PatternSpace& s = ns ? ctx->cp : ctx->kp;
    if (s.n >= (1ull << 31)) return fail(ctx, PF_ERR_INVALID, "too many local patterns for the exchange");
    x.ns[ns].n_local = s.n;
    x.ns[ns].bytes_sent = s.n * s.key_words * 4;
    TRY(exchange_classify(ctx, s, world, ns ? nullptr : mask_remap));
    if (!x.ns[ns].recv.p && !(flags & PF_EXCHANGE_NO_PEER) && !x.peer_failed)
      xr_grow(ctx, x.ns[ns], s.key_words, 1);
  }
  const XRec* all = nullptr;
  TRY(xr_records(ctx, c, x, flags, nss, n_ns, all));
  bool any_no_peer = false, all_a2a = true;
  for (uint32_t r = 0; r < world; ++r) {
    any_no_peer = any_no_peer || (all[r].flags & XR_NO_PEER);
    all_a2a = all_a2a && (all[r].flags & XR_A2A);
  }
  bool peer = !any_no_peer && !x.peer_failed;
  if (peer) {
    bool ok = true, opening = false;
    TRY(xr_peer_setup(ctx, c, x, flags, nss, n_ns, all, ok, opening));
    if (opening) {
      bool agreed = true;
      TRY(xr_all_ok(ctx, c, x, ok, agreed));
      if (!agreed) { x.peer_failed = true; peer = false; }
    } else if (!ok) {
      return fail(ctx, PF_ERR_STATE, "pattern exchange: a cached peer mapping went away");
    }
  }
  if (!peer && !all_a2a)          // every rank sees the same records and the same agreement
    return fail(ctx, PF_ERR_UNSUPPORTED, "pattern exchange: %s and a rank has no all_to_all_v",
                any_no_peer ? "the all-to-all transport was asked for" : "peer memory is not available");
  for (int i = 0; i < n_ns; ++i) {
    const int ns = nss[i];
    PatternSpace& s = ns ? ctx->cp : ctx->kp;
    XNs& n = x.ns[ns];
    const uint32_t nl = (uint32_t)n.n_local;
    const uint32_t* remap = ns ? nullptr : mask_remap;
    uint64_t n_recv = 0, send0[kXMaxWorld];
    for (uint32_t r = 0; r < world; ++r) n_recv += all[r].counts[ns][rank];
    for (uint32_t o = 0, run = 0; o < world; ++o) { send0[o] = run; run += all[rank].counts[ns][o]; }
    if (peer) {
      if (nl) {
        XDest d{};
        for (uint32_t o = 0; o < world; ++o) {
          uint64_t row0 = 0;
          for (uint32_t r = 0; r < rank; ++r) row0 += all[r].counts[ns][o];
          d.ptr[o] = static_cast<uint32_t*>(o == rank ? n.recv.p : n.peer[o].ptr);
          d.row0[o] = (uint32_t)row0;
          d.send0[o] = (uint32_t)send0[o];
        }
        xr_launch_by_width(s.key_words, [&](auto LL) {
          constexpr int L = decltype(LL)::value;
          x_scatter<L><<<std::min<uint32_t>(cdiv(nl, 256 / L), kGridPersist * 4), 256, 0, st>>>(
              s.pool.as<uint32_t>(), nl, s.key_words, remap, s.x_owner.as<uint32_t>(), s.x_pos.as<uint32_t>(), d,
              s.x_perm.as<uint32_t>());
        });
        ctx->launches++;
        CU(cudaGetLastError());
      }
      // every rank's scatter has completed before an owner reads its buffer
      TRY(xr_gather(ctx, c, xs_ok(x), xs_ok(x) + 1, 4));
      uint32_t* recv = n.recv.as<uint32_t>();
      TRY(xr_finish(ctx, c, x, ns, flags, all, true, recv, n_recv, recv + n.cap * s.key_words));
    } else {
      TRY(dev_ensure(ctx, n.send, std::max<size_t>(1, nl) * s.key_words * 4));
      TRY(dev_ensure(ctx, n.a2a_recv, std::max<uint64_t>(1, n_recv) * s.key_words * 4));
      TRY(dev_ensure(ctx, n.uniq, std::max<uint64_t>(1, n_recv) * 4));
      if (nl) {
        xr_launch_by_width(s.key_words, [&](auto LL) {
          constexpr int L = decltype(LL)::value;
          x_pack<L><<<std::min<uint32_t>(cdiv(nl, 256 / L), kGridPersist * 4), 256, 0, st>>>(
              s.pool.as<uint32_t>(), nl, s.key_words, remap, s.x_owner.as<uint32_t>(), s.x_pos.as<uint32_t>(),
              s.x_counts.as<uint32_t>() + world, n.send.as<uint32_t>(), s.x_perm.as<uint32_t>());
        });
        ctx->launches++;
        CU(cudaGetLastError());
      }
      uint64_t sb[kXMaxWorld], rb[kXMaxWorld];
      for (uint32_t r = 0; r < world; ++r) {
        sb[r] = (uint64_t)all[rank].counts[ns][r] * s.key_words * 4;
        rb[r] = (uint64_t)all[r].counts[ns][rank] * s.key_words * 4;
      }
      TRY(xr_a2a(ctx, c, n.send.p, sb, n.a2a_recv.p, rb));
      TRY(xr_finish(ctx, c, x, ns, flags, all, false, n.a2a_recv.as<uint32_t>(), n_recv, n.uniq.as<uint32_t>()));
    }
  }
  return PF_OK;
}

void xrun_free(pf_ctx* ctx) {
  if (!ctx->xrun) return;
  XRunState& x = *ctx->xrun;
  auto fd = [](DevBuf& b) { if (b.p) cudaFree(b.p); b.p = nullptr; b.cap = 0; };
  auto fp = [](PinBuf& b) { if (b.p) cudaFreeHost(b.p); b.p = nullptr; b.cap = 0; };
  for (XNs& n : x.ns) {
    for (XPeer& p : n.peer) xr_close_peer(ctx, p);
    for (DevBuf* b : {&n.recv, &n.send, &n.a2a_recv, &n.uniq, &n.returned, &n.l2g, &n.writer}) fd(*b);
  }
  fd(x.d_rec); fd(x.d_small);
  fp(x.h_rec); fp(x.h_small);
  delete ctx->xrun;
  ctx->xrun = nullptr;
}

}  // namespace

extern "C" int pf_exchange_run(pf_ctx* ctx, const pf_comm* comm, uint32_t flags, pf_exchange_result* out) {
  if (!ctx || !comm || !out || !comm->all_gather) return ctx ? fail(ctx, PF_ERR_INVALID, "pf_exchange_run: null argument") : PF_ERR_INVALID;
  if (comm->world == 0 || comm->world > kXMaxWorld || comm->rank >= comm->world)
    return fail(ctx, PF_ERR_INVALID, "pf_exchange_run: rank %u of world %u (1..%u ranks)", comm->rank, comm->world, kXMaxWorld);
  if (flags & ~(uint32_t)(PF_EXCHANGE_WRITER | PF_EXCHANGE_KEEP_UNIQUE | PF_EXCHANGE_NO_PEER))
    return fail(ctx, PF_ERR_INVALID, "pf_exchange_run: unknown flags 0x%x", flags);
  memset(out, 0, sizeof *out);
  CU(cudaSetDevice(ctx->device));
  TRY(finalize_pending(ctx));
  XRunState* xp = nullptr;
  TRY(xr_state(ctx, xp));
  XRunState& x = *xp;
  if (ctx->prm.consider_missing) {
    // k-mer keys end with the GLOBAL id of the cluster pattern giving their NaN plane: the cluster
    // namespace is numbered first
    const int cl[1] = {1}, km[1] = {0};
    TRY(xr_step(ctx, comm, x, flags, cl, 1, nullptr));
    TRY(xr_step(ctx, comm, x, flags, km, 1, x.ns[1].l2g.as<uint32_t>()));
  } else {
    const int both[2] = {1, 0};
    TRY(xr_step(ctx, comm, x, flags, both, 2, nullptr));
  }
  // the final counts: the one sync after the keys moved
  uint32_t* h = x.h_small.as<uint32_t>();
  for (int ns = 0; ns < 2; ++ns)
    CU(cudaMemcpyAsync(h + ns * kXMaxWorld, xs_all_nu(x, ns), comm->world * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  for (int ns = 0; ns < 2; ++ns) {
    pf_exchange_ns& o = ns ? out->cluster : out->kmer;
    const XNs& n = x.ns[ns];
    const uint32_t* c = h + ns * kXMaxWorld;
    o.n_local = n.n_local;
    o.bytes_sent = n.bytes_sent;
    for (uint32_t r = 0; r < comm->world; ++r) {
      o.n_global += c[r];
      if (r < comm->rank) o.owned_base += c[r];
    }
    o.n_owned = c[comm->rank];
    (ns ? ctx->cp : ctx->kp).x_n_unique = o.n_owned;       // for pf_exchange_unique_export
    o.local_to_global = n.l2g.as<uint32_t>();
    o.writer = (flags & PF_EXCHANGE_WRITER) ? n.writer.as<uint8_t>() : nullptr;
  }
  return PF_OK;
}

extern "C" int pf_exchange_release(pf_ctx* ctx, const pf_comm* comm) {
  if (!ctx || !comm || !comm->all_gather) return PF_ERR_INVALID;
  if (comm->world == 0 || comm->world > kXMaxWorld || comm->rank >= comm->world)
    return fail(ctx, PF_ERR_INVALID, "pf_exchange_release: rank %u of world %u", comm->rank, comm->world);
  CU(cudaSetDevice(ctx->device));
  XRunState* xp = nullptr;
  TRY(xr_state(ctx, xp));
  for (XNs& n : xp->ns) {
    for (XPeer& p : n.peer) xr_close_peer(ctx, p);
    n.seen = false;
  }
  // every rank has unmapped before any rank goes on to free the buffers the others had mapped
  CU(cudaStreamSynchronize(ctx->stream));
  bool all = true;
  return xr_all_ok(ctx, comm, *xp, true, all);
}

// ---------------------------------------------------------------------------
// pf_comm_local: collectives between the host threads of one process.  Each collective:
//   1. every rank records an event on its stream behind the data it sends,
//   2. the host threads meet at a barrier,
//   3. every stream waits for the peers' events and copies the peers' segments into its own
//      receive buffer (cudaMemcpyAsync, cudaMemcpyPeerAsync between devices),
//   4. a second event + barrier: every stream waits until all copies out of its send buffer are
//      done, so the sender may reuse it as soon as its own stream moves on.
// The two barriers also order the reuse of the events and the published pointers.
// ---------------------------------------------------------------------------
struct pf_comm_local {
  struct Rank {
    pf_comm_local* g = nullptr;
    uint32_t rank = 0;
    int device = -1;
    cudaEvent_t ready = nullptr, done = nullptr;
    cudaStream_t stream = nullptr;
    const void* send = nullptr;
    std::vector<uint64_t> send_bytes;
  };
  uint32_t world = 0;
  std::mutex mu;
  std::condition_variable cv;
  uint32_t arrived = 0;
  uint64_t generation = 0;
  bool aborted = false;
  std::vector<Rank> ranks;
};

namespace {

int local_barrier(pf_comm_local* g) {
  std::unique_lock<std::mutex> lk(g->mu);
  if (g->aborted) return -1;
  const uint64_t gen = g->generation;
  if (++g->arrived == g->world) {
    g->arrived = 0;
    ++g->generation;
    g->cv.notify_all();
    return 0;
  }
  g->cv.wait(lk, [&] { return g->generation != gen || g->aborted; });
  return g->generation != gen ? 0 : -1;
}

int local_events(pf_comm_local::Rank& me) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return -1;
  if (me.ready && me.device == dev) return 0;
  if (me.ready) { cudaEventDestroy(me.ready); cudaEventDestroy(me.done); me.ready = me.done = nullptr; }
  if (cudaEventCreateWithFlags(&me.ready, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&me.done, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); return -1; }
  me.device = dev;
  return 0;
}

// steps 1-2 of a collective: publish this rank's send side, meet the others
int local_enter(pf_comm_local::Rank& me, const void* send, const uint64_t* send_bytes, void* stream) {
  if (local_events(me)) return -1;
  me.stream = static_cast<cudaStream_t>(stream);
  me.send = send;
  if (send_bytes) me.send_bytes.assign(send_bytes, send_bytes + me.g->world);
  if (cudaEventRecord(me.ready, me.stream) != cudaSuccess) { cudaGetLastError(); return -1; }
  return local_barrier(me.g);
}

int local_copy(const pf_comm_local::Rank& me, const pf_comm_local::Rank& q, void* dst, const void* src, uint64_t bytes) {
  if (!bytes) return 0;
  const cudaError_t e = q.device == me.device
      ? cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, me.stream)
      : cudaMemcpyPeerAsync(dst, me.device, src, q.device, bytes, me.stream);
  if (e != cudaSuccess) { cudaGetLastError(); return -1; }
  return 0;
}

// step 4: the senders' buffers stay untouched until every copy out of them is done
int local_leave(pf_comm_local::Rank& me, int rc) {
  if (cudaEventRecord(me.done, me.stream) != cudaSuccess) { cudaGetLastError(); rc = -1; }
  if (local_barrier(me.g)) return -1;
  for (const pf_comm_local::Rank& q : me.g->ranks)
    if (&q != &me && cudaStreamWaitEvent(me.stream, q.done, 0) != cudaSuccess) { cudaGetLastError(); rc = -1; }
  return rc;
}

int local_all_gather(const void* send, void* recv, uint64_t bytes, void* stream, void* user) {
  auto& me = *static_cast<pf_comm_local::Rank*>(user);
  if (local_enter(me, send, nullptr, stream)) return -1;
  int rc = 0;
  for (const pf_comm_local::Rank& q : me.g->ranks) {
    if (&q != &me && cudaStreamWaitEvent(me.stream, q.ready, 0) != cudaSuccess) { cudaGetLastError(); rc = -1; continue; }
    if (local_copy(me, q, static_cast<char*>(recv) + q.rank * bytes, q.send, bytes)) rc = -1;
  }
  return local_leave(me, rc);
}

int local_all_to_all_v(const void* send, const uint64_t* send_bytes, void* recv, const uint64_t* recv_bytes,
                       void* stream, void* user) {
  auto& me = *static_cast<pf_comm_local::Rank*>(user);
  if (local_enter(me, send, send_bytes, stream)) return -1;
  int rc = 0;
  uint64_t at = 0;
  for (const pf_comm_local::Rank& q : me.g->ranks) {
    // q's segment for this rank sits behind its segments for the ranks before
    uint64_t from = 0;
    for (uint32_t j = 0; j < me.rank; ++j) from += q.send_bytes[j];
    const uint64_t n = q.send_bytes[me.rank];
    if (n != recv_bytes[q.rank]) rc = -1;                 // the ranks disagree on the split sizes
    else if (&q != &me && cudaStreamWaitEvent(me.stream, q.ready, 0) != cudaSuccess) { cudaGetLastError(); rc = -1; }
    else if (local_copy(me, q, static_cast<char*>(recv) + at, static_cast<const char*>(q.send) + from, n)) rc = -1;
    at += recv_bytes[q.rank];
  }
  return local_leave(me, rc);
}

}  // namespace

extern "C" int pf_comm_local_create(uint32_t world, pf_comm_local** out) {
  if (!out || world == 0 || world > kXMaxWorld) return PF_ERR_INVALID;
  pf_comm_local* g = new (std::nothrow) pf_comm_local();
  if (!g) return PF_ERR_NOMEM;
  g->world = world;
  g->ranks.resize(world);
  for (uint32_t r = 0; r < world; ++r) { g->ranks[r].g = g; g->ranks[r].rank = r; }
  *out = g;
  return PF_OK;
}

extern "C" int pf_comm_local_get(pf_comm_local* g, uint32_t rank, pf_comm* out) {
  if (!g || !out || rank >= g->world) return PF_ERR_INVALID;
  out->rank = rank;
  out->world = g->world;
  out->user = &g->ranks[rank];
  out->all_gather = local_all_gather;
  out->all_to_all_v = local_all_to_all_v;
  return PF_OK;
}

extern "C" void pf_comm_local_abort(pf_comm_local* g) {
  if (!g) return;
  std::lock_guard<std::mutex> lk(g->mu);
  g->aborted = true;
  g->cv.notify_all();
}

extern "C" void pf_comm_local_destroy(pf_comm_local* g) {
  if (!g) return;
  for (pf_comm_local::Rank& r : g->ranks) {
    if (r.ready) cudaEventDestroy(r.ready);
    if (r.done) cudaEventDestroy(r.done);
  }
  delete g;
}
