// pf_exchange.cuh — multi-GPU pattern exchange kernels, the classify and owner-side dedup steps
// pf_exchange_run.cuh sequences, and the export of the owner's unique keys.
// Part of libpanfeed_b200.so's single translation unit: included once, in order, by pf_api.cu.

// ---------------------------------------------------------------------------
// multi-GPU exchange (SURVEY.md §8(e))
// ---------------------------------------------------------------------------
namespace pf {

// owner of every local pattern + its position inside the owner's bucket.  L lanes hash one
// key (as in K4: short keys would leave most of a warp idle), a warp handles 32 consecutive
// patterns and hands out their bucket positions with ONE atomic per distinct owner — a counter
// per rank shared by millions of patterns would serialise in L2.
template <int L>
__global__ void __launch_bounds__(256)
x_classify(const uint32_t* __restrict__ pool, uint32_t n, uint32_t key_words,
           const uint32_t* __restrict__ mask_remap, uint32_t world, uint32_t* __restrict__ owner,
           uint32_t* __restrict__ pos, uint32_t* __restrict__ counts) {
  const uint32_t lane = lane_id(), gl = lane & (L - 1), g = lane / L;
  constexpr uint32_t G = 32 / L;                   // patterns hashed at once by a warp
  const uint32_t total_warps = gridDim.x * (blockDim.x >> 5);
  for (uint32_t e0 = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 32u; e0 < n; e0 += total_warps * 32u) {
    uint32_t my_owner = 0xffffffffu;
    const uint32_t cnt = min(32u, n - e0);
    for (uint32_t p0 = 0; p0 < 32u; p0 += G) {     // (uniform trip count: the shuffles need all lanes)
      const uint32_t p = p0 + g;
      uint64_t h = 0;
      if (p < cnt) {
        const uint32_t* key = pool + (size_t)(e0 + p) * key_words;
        for (uint32_t w = gl; w < key_words; w += L) {
          uint32_t v = key[w];
          if (mask_remap && w == key_words - 1) v = mask_remap[v];
          h += word_hash(v, w);
        }
      }
#pragma unroll
      for (int m = L / 2; m >= 1; m >>= 1) h += __shfl_xor_sync(kFull, h, m);
      h = fmix64(h);
      const uint32_t o = (uint32_t)((h >> 32) % world);
      // lane p of the warp keeps pattern p's owner: it sits in group p - p0, any lane of it
      const uint32_t got = __shfl_sync(kFull, o, (lane - p0) * L);
      if (lane >= p0 && lane < p0 + G && lane < cnt) my_owner = got;
    }
    const uint32_t m = __match_any_sync(kFull, my_owner);
    if (lane < cnt) {
      const int leader = __ffs(m) - 1;
      uint32_t base = 0;
      if ((int)lane == leader) base = atomicAdd(&counts[my_owner], (uint32_t)__popc(m));
      base = __shfl_sync(m, base, leader);
      owner[e0 + lane] = my_owner;
      pos[e0 + lane] = base + __popc(m & lanemask_lt());
    }
  }
}

// exclusive offsets of the `world` buckets behind the counts (counts[world .. 2 world))
__global__ void x_offsets(uint32_t* __restrict__ counts, uint32_t world) {
  if (threadIdx.x == 0) {
    uint32_t run = 0;
    for (uint32_t r = 0; r < world; ++r) { counts[world + r] = run; run += counts[r]; }
  }
}

template <int L>
__global__ void __launch_bounds__(256)
x_pack(const uint32_t* __restrict__ pool, uint32_t n, uint32_t key_words,
       const uint32_t* __restrict__ mask_remap, const uint32_t* __restrict__ owner,
       const uint32_t* __restrict__ pos, const uint32_t* __restrict__ offsets,
       uint32_t* __restrict__ send, uint32_t* __restrict__ perm) {
  const uint32_t gl = lane_id() & (L - 1);
  const uint32_t total = gridDim.x * (blockDim.x / L);
  for (uint32_t e = blockIdx.x * (blockDim.x / L) + threadIdx.x / L; e < n; e += total) {
    const uint32_t dst = offsets[owner[e]] + pos[e];
    const uint32_t* key = pool + (size_t)e * key_words;
    uint32_t* out = send + (size_t)dst * key_words;
    for (uint32_t w = gl; w < key_words; w += L) {
      uint32_t v = key[w];
      if (mask_remap && w == key_words - 1) v = mask_remap[v];
      out[w] = v;
    }
    if (gl == 0) perm[e] = dst;
  }
}

// The same move without the send buffer and the all-to-all: every key goes straight to its
// place in the OWNER's receive buffer, which this rank has mapped (CUDA IPC, NVLink peer
// stores).  row0[o]: first row of this rank's bucket inside owner o's buffer; send0[o]: the
// bucket's first position in this rank's send order (what x_pack calls offsets).
struct XDest {
  uint32_t* ptr[32];
  uint32_t row0[32];
  uint32_t send0[32];
};
template <int L>
__global__ void __launch_bounds__(256)
x_scatter(const uint32_t* __restrict__ pool, uint32_t n, uint32_t key_words,
          const uint32_t* __restrict__ mask_remap, const uint32_t* __restrict__ owner,
          const uint32_t* __restrict__ pos, const XDest d, uint32_t* __restrict__ perm) {
  __shared__ uint32_t* s_ptr[32];
  __shared__ uint32_t s_row0[32], s_send0[32];
  if (threadIdx.x < 32) { s_ptr[threadIdx.x] = d.ptr[threadIdx.x]; s_row0[threadIdx.x] = d.row0[threadIdx.x]; s_send0[threadIdx.x] = d.send0[threadIdx.x]; }
  __syncthreads();
  const uint32_t gl = lane_id() & (L - 1);
  const uint32_t total = gridDim.x * (blockDim.x / L);
  for (uint32_t e = blockIdx.x * (blockDim.x / L) + threadIdx.x / L; e < n; e += total) {
    const uint32_t o = owner[e], p = pos[e];
    const uint32_t* key = pool + (size_t)e * key_words;
    uint32_t* out = s_ptr[o] + ((size_t)s_row0[o] + p) * key_words;
    for (uint32_t w = gl; w < key_words; w += L) {
      uint32_t v = key[w];
      if (mask_remap && w == key_words - 1) v = mask_remap[v];
      out[w] = v;
    }
    if (gl == 0) perm[e] = s_send0[o] + p;
  }
}

// unique index of every received key + compacted unique keys
template <int L>
__global__ void __launch_bounds__(256)
x_finish(const uint32_t* __restrict__ recv, uint32_t n, uint32_t key_words,
         const uint32_t* __restrict__ rep, const uint32_t* __restrict__ winner_rank,
         uint32_t* __restrict__ unique_index, uint32_t* __restrict__ unique_keys) {
  const uint32_t gl = lane_id() & (L - 1);
  const uint32_t total = gridDim.x * (blockDim.x / L);
  for (uint32_t e = blockIdx.x * (blockDim.x / L) + threadIdx.x / L; e < n; e += total) {
    const uint32_t q = rep[e] & ~kTentative;         // every rep is tentative here (empty pool)
    const uint32_t u = winner_rank[q];
    // bit 31: this copy is the representative of its pattern - its sender writes the pattern row
    if (gl == 0) unique_index[e] = u | (q == e ? 0x80000000u : 0u);
    if (q == e && unique_keys) {
      const uint32_t* src = recv + (size_t)e * key_words;
      uint32_t* dst = unique_keys + (size_t)u * key_words;
      for (uint32_t w = gl; w < key_words; w += L) dst[w] = src[w];
    }
  }
}

// returned[]: the owner's unique index (bit 31 = writer flag) of every pattern, in send order;
// owner_base[r] (may be null): global id of rank r's first unique pattern
__global__ void x_unpack(const uint32_t* __restrict__ returned, const uint32_t* __restrict__ perm,
                         const uint32_t* __restrict__ owner, const uint32_t* __restrict__ owner_base,
                         uint32_t n, uint32_t* __restrict__ local_to_global, uint8_t* __restrict__ writer) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t v = returned[perm[i]];
  local_to_global[i] = (v & 0x7fffffffu) + (owner_base ? owner_base[owner[i]] : 0u);
  if (writer) writer[i] = (uint8_t)(v >> 31);
}

}  // namespace pf

namespace {
// One instantiation per lanes-per-key L: short keys would leave most of a warp idle (as in K4).
template <typename F>
void xr_launch_by_width(uint32_t key_words, F&& f) {
  const int L = key_words <= 16 ? 4 : key_words <= 32 ? 8 : key_words <= 64 ? 16 : 32;
  if (L == 4) f(std::integral_constant<int, 4>());
  else if (L == 8) f(std::integral_constant<int, 8>());
  else if (L == 16) f(std::integral_constant<int, 16>());
  else f(std::integral_constant<int, 32>());
}

// owners, bucket positions, bucket sizes (x_counts[0, world)) and bucket offsets
// (x_counts[world, 2 world)) of the local patterns of one namespace, on the stream
int exchange_classify(pf_ctx* ctx, PatternSpace& s, uint32_t world, const uint32_t* mask_remap_dev) {
  cudaStream_t st = ctx->stream;
  const uint32_t n = (uint32_t)s.n;
  TRY(dev_ensure(ctx, s.x_owner, std::max<size_t>(1, n) * 4));
  TRY(dev_ensure(ctx, s.x_pos, std::max<size_t>(1, n) * 4));
  TRY(dev_ensure(ctx, s.x_perm, std::max<size_t>(1, n) * 4));
  TRY(dev_ensure(ctx, s.x_counts, (size_t)world * 2 * 4));
  CU(cudaMemsetAsync(s.x_counts.p, 0, (size_t)world * 2 * 4, st));
  if (n == 0) return PF_OK;
  xr_launch_by_width(s.key_words, [&](auto LL) {
    constexpr int L = decltype(LL)::value;
    x_classify<L><<<std::min<uint32_t>(cdiv(n, 256), kGridPersist * 2), 256, 0, st>>>(
        s.pool.as<uint32_t>(), n, s.key_words, mask_remap_dev, world, s.x_owner.as<uint32_t>(),
        s.x_pos.as<uint32_t>(), s.x_counts.as<uint32_t>());
  });
  x_offsets<<<1, 32, 0, st>>>(s.x_counts.as<uint32_t>(), world);
  ctx->launches += 2;
  CU(cudaGetLastError());
  return PF_OK;
}

// owner side of one namespace, on the stream: the unique index of every received key (bit 31 set
// on the first copy of a pattern: its sender writes the pattern row) and their number to
// *n_unique_dev; keep_unique: the unique keys stay in s.x_unique for pf_exchange_unique_export
int exchange_dedup(pf_ctx* ctx, PatternSpace& s, const uint32_t* recv, uint64_t n_recv, uint32_t* unique_index,
                   uint32_t* n_unique_dev, bool keep_unique) {
  cudaStream_t st = ctx->stream;
  s.x_n_unique = 0;                   // (pf_exchange_run sets it once the count is on the host)
  if (n_recv == 0) {
    CU(cudaMemsetAsync(n_unique_dev, 0, 4, st));
    return PF_OK;
  }
  if (n_recv >= (1ull << 30)) return fail(ctx, PF_ERR_INVALID, "too many received patterns");
  const uint32_t n = (uint32_t)n_recv;
  uint32_t size = 1024;
  while (size < 2ull * n + 16) size *= 2;
  // scratch kept across calls: no cudaMalloc in the steady state
  TRY(dev_ensure(ctx, s.x_table, (size_t)size * 4));
  TRY(dev_ensure(ctx, s.x_rep, (size_t)n * 4));
  TRY(dev_ensure(ctx, s.x_slot, (size_t)n * 4));
  TRY(dev_ensure(ctx, s.x_winner, ((size_t)n + 1) * 4));
  if (keep_unique) TRY(dev_ensure(ctx, s.x_unique, (size_t)n * s.key_words * 4));
  s.x_have_unique = keep_unique;
  CU(cudaMemsetAsync(s.x_table.p, 0xff, (size_t)size * 4, st));
  xr_launch_by_width(s.key_words, [&](auto LL) {
    constexpr int L = decltype(LL)::value;
    k4_probe<L><<<std::min<uint32_t>(cdiv(n, 256 / L), kGridPersist * 4), 256, 0, st>>>(
        recv, n, s.key_words, nullptr, s.x_table.as<uint32_t>(), size - 1, s.x_rep.as<uint32_t>(),
        s.x_slot.as<uint32_t>(), s.x_winner.as<uint32_t>());
  });
  TRY(scan_inplace(ctx, s.x_winner.as<uint32_t>(), n, n_unique_dev));
  xr_launch_by_width(s.key_words, [&](auto LL) {
    constexpr int L = decltype(LL)::value;
    x_finish<L><<<std::min<uint32_t>(cdiv(n, 256 / L), kGridPersist * 4), 256, 0, st>>>(
        recv, n, s.key_words, s.x_rep.as<uint32_t>(), s.x_winner.as<uint32_t>(), unique_index,
        keep_unique ? s.x_unique.as<uint32_t>() : nullptr);
  });
  ctx->launches += 2;
  CU(cudaGetLastError());
  return PF_OK;
}
}  // namespace

// the owner-side unique keys of the last pf_exchange_run with PF_EXCHANGE_KEEP_UNIQUE
extern "C" int pf_exchange_unique_count(pf_ctx* ctx, int cluster_namespace, uint64_t* n_unique_host) {
  if (!ctx || !n_unique_host) return PF_ERR_INVALID;
  *n_unique_host = (cluster_namespace ? ctx->cp : ctx->kp).x_n_unique;
  return PF_OK;
}

extern "C" int pf_exchange_unique_export(pf_ctx* ctx, int cluster_namespace, uint32_t* host_out) {
  if (!ctx) return PF_ERR_INVALID;
  PatternSpace& s = cluster_namespace ? ctx->cp : ctx->kp;
  const uint64_t n = s.x_n_unique;
  if (n == 0) return PF_OK;
  if (!host_out) return PF_ERR_INVALID;
  if (!s.x_have_unique) return fail(ctx, PF_ERR_STATE, "pf_exchange_run was not asked to keep the unique keys");
  CU(cudaSetDevice(ctx->device));
  CU(cudaMemcpy(host_out, s.x_unique.p, n * s.key_words * 4, cudaMemcpyDeviceToHost));
  return PF_OK;
}
