// Graph ingestion and per-edge operand staging for libbotgat (sm_100a).
// Replaces DGLGraph construction, `create_formats_()` and the degree queries of
// the reference (src/no-sampling/run.py:133-148, src/ogbn-proteins/gat.py:64-66,
// src/no-sampling/models.py:478,501,551) plus dgl.to_bidirected /
// remove_self_loop / add_self_loop.  Integer work, bit-exact by construction:
// stable LSD radix sort (CUB) keyed on the row id with the edge id as payload.
#include <cub/cub.cuh>

#include <atomic>
#include <cstdarg>
#include <cstring>

#include "common.cuh"

namespace botgat {

static thread_local char g_err[512] = "";
std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// ---------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------
__global__ void k_narrow_and_check(int64_t n, const int64_t* __restrict__ a, int64_t bound, int32_t* __restrict__ out,
                                   int32_t* __restrict__ iota, int* __restrict__ bad) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t v = a[i];
    const bool oob = v < 0 || v >= bound;
    if (oob) *bad = 1;
    // an out-of-range id is reported after the build (graph_create reads `bad` back); until then it must not index
    // anything: the histogram, the sort and the gathers below all use these narrowed ids
    out[i] = oob ? 0 : (int32_t)v;
    if (iota) iota[i] = (int32_t)i;
  }
}

__global__ void k_histogram(int64_t n, const int32_t* __restrict__ keys, int32_t* __restrict__ counts) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    atomicAdd(counts + keys[i], 1);  // integer adds commute: result is exact and order-independent
}

__global__ void k_gather_i32(int64_t n, const int32_t* __restrict__ table, const int32_t* __restrict__ idx,
                             int32_t* __restrict__ out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = table[idx[i]];
}

// stats[0] = max degree, stats[1] = number of zero-degree rows
__global__ void k_deg_stats(int64_t n, const int32_t* __restrict__ deg, int* __restrict__ stats) {
  int mx = 0, zeros = 0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int d = deg[i];
    mx = max(mx, d);
    zeros += d == 0;
  }
  for (int o = 16; o > 0; o >>= 1) {
    mx = max(mx, __shfl_xor_sync(kFull, mx, o));
    zeros += __shfl_xor_sync(kFull, zeros, o);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMax(stats, mx);
    atomicAdd(stats + 1, zeros);
  }
}

static inline int grid_for(int64_t n, int block = 256) {
  int64_t b = (n + block - 1) / block;
  return (int)std::max<int64_t>(1, std::min<int64_t>(b, 148 * 32));
}

// *flag = 1 unless eid[p] == p everywhere
__global__ void k_check_identity(int64_t n, const int32_t* __restrict__ eid, int* __restrict__ flag) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    if (eid[i] != (int32_t)i) *flag = 1;
}

// tile key of every out-CSR position: (source block, destination block), source-block-major; one warp per row
__global__ void k_tile_keys(int n_src, const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                            int rows_per_s, int rows_per_d, int tiles_d, int32_t* __restrict__ keys,
                            int32_t* __restrict__ iota) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  for (int r = warp; r < n_src; r += nwarps) {
    const int ts = r / rows_per_s;
    for (int p = indptr[r] + lane; p < indptr[r + 1]; p += 32) {
      keys[p] = ts * tiles_d + indices[p] / rows_per_d;
      iota[p] = p;
    }
  }
}

static int bits_for(int64_t n) {
  int b = 1;
  while ((1ll << b) < n) ++b;
  return b;
}

// Stable sort of (key -> eid) and the CSR arrays that follow from it.
static int build_csr(int64_t n_rows, int64_t n_edges, const int32_t* key, const int32_t* other, const int32_t* iota,
                     int32_t* key_sorted_tmp, int32_t* indptr, int32_t* indices, int32_t* eid, int32_t* deg,
                     cudaStream_t st) {
  if (n_edges > 0) {
    size_t tmp_bytes = 0;
    BG_CHECK(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, key, key_sorted_tmp, iota, eid, (int)n_edges, 0,
                                             bits_for(n_rows), st));
    void* tmp = nullptr;
    BG_CHECK(cudaMallocAsync(&tmp, tmp_bytes, st));
    BG_CHECK(cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, key, key_sorted_tmp, iota, eid, (int)n_edges, 0,
                                             bits_for(n_rows), st)); BG_LAUNCHED(1);
    BG_CHECK(cudaFreeAsync(tmp, st));
    k_gather_i32<<<grid_for(n_edges), 256, 0, st>>>(n_edges, other, eid, indices); BG_LAUNCHED(1);
    BG_CHECK(cudaGetLastError());
  }
  BG_CHECK(cudaMemsetAsync(deg, 0, sizeof(int32_t) * (n_rows + 1), st));  // deg has n_rows+1 slots (scan input)
  if (n_edges > 0) {
    k_histogram<<<grid_for(n_edges), 256, 0, st>>>(n_edges, key, deg); BG_LAUNCHED(1);
    BG_CHECK(cudaGetLastError());
  }
  {
    size_t tmp_bytes = 0;
    BG_CHECK(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, deg, indptr, (int)(n_rows + 1), st));
    void* tmp = nullptr;
    BG_CHECK(cudaMallocAsync(&tmp, tmp_bytes, st));
    BG_CHECK(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, deg, indptr, (int)(n_rows + 1), st)); BG_LAUNCHED(1);
    BG_CHECK(cudaFreeAsync(tmp, st));
  }
  return 0;
}

}  // namespace botgat

using namespace botgat;

extern "C" int botgat_abi_version(void) { return BOTGAT_ABI_VERSION; }
extern "C" const char* botgat_last_error(void) { return g_err; }
extern "C" int64_t botgat_launch_count(void) { return (int64_t)g_launches.load(); }

// The structure arrays come from the device's stream-ordered pool (cudaMallocAsync): mini-batch blocks are created and
// destroyed every step, and cudaMalloc / cudaFree would synchronise the device each time.
static void configure_pool(int device) {
  static std::atomic<unsigned> done{0};
  const unsigned bit = 1u << (device & 31);
  if (done.fetch_or(bit) & bit) return;
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, device) != cudaSuccess) return;
  uint64_t thr = 0;
  // keep freed blocks cached (up to 2 GiB) unless the application already chose a threshold
  if (cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr) == cudaSuccess && thr == 0) {
    thr = 2ull << 30;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
  }
}

static void destroy_impl(botgat_graph* g, bool async, cudaStream_t st) {
  if (!g) return;
  DeviceGuard guard(g->device);
  void* ptrs[] = {g->in_indptr, g->in_indices, g->in_eid, g->out_indptr, g->out_indices, g->out_eid, g->in_deg, g->out_deg};
  for (void* q : ptrs) {
    if (!q) continue;
    // cudaFree of pool memory synchronises, then releases; it is also the fallback if the stream is unusable
    if (!async || cudaFreeAsync(q, st) != cudaSuccess) { cudaGetLastError(); cudaFree(q); }
  }
  if (g->out_tile_order && (!async || cudaFreeAsync(g->out_tile_order, st) != cudaSuccess)) { cudaGetLastError(); cudaFree(g->out_tile_order); }
  free_segments(&g->seg_in, async, st); free_segments(&g->seg_out, async, st);
  delete g;
}

extern "C" void botgat_graph_destroy(botgat_graph* g) { destroy_impl(g, false, nullptr); }
extern "C" void botgat_graph_destroy_async(botgat_graph* g, void* stream) { destroy_impl(g, true, (cudaStream_t)stream); }

extern "C" int botgat_graph_create(int64_t n_src, int64_t n_dst, int64_t n_edges, const int64_t* src,
                                   const int64_t* dst, int device, void* stream, botgat_graph** out) {
  BG_REQUIRE(out, "graph_create: null out");
  *out = nullptr;
  BG_REQUIRE(n_src >= 0 && n_dst >= 0 && n_edges >= 0, "graph_create: negative size");
  BG_REQUIRE(n_edges < (1ll << 31) - 1 && n_src < (1ll << 31) - 1 && n_dst < (1ll << 31) - 1,
             "graph_create: sizes must be < 2^31-1 (int32 structure arrays)");
  BG_REQUIRE(n_edges == 0 || (src && dst), "graph_create: null src/dst");
  DeviceGuard guard(device);
  cudaStream_t st = (cudaStream_t)stream;

  botgat_graph* g = new botgat_graph();
  g->device = device; g->n_src = n_src; g->n_dst = n_dst; g->n_edges = n_edges;
  cudaDeviceGetAttribute(&g->sm_count, cudaDevAttrMultiProcessorCount, device);
  struct Cleanup {
    botgat_graph*& g;
    bool armed = true;
    ~Cleanup() { if (armed) { botgat_graph_destroy(g); } }
  } cleanup{g};

  configure_pool(device);
  const size_t eb = sizeof(int32_t) * (size_t)std::max<int64_t>(n_edges, 1);
  BG_CHECK(cudaMallocAsync(&g->in_indptr, sizeof(int32_t) * (n_dst + 1), st));
  BG_CHECK(cudaMallocAsync(&g->out_indptr, sizeof(int32_t) * (n_src + 1), st));
  BG_CHECK(cudaMallocAsync(&g->in_indices, eb, st)); BG_CHECK(cudaMallocAsync(&g->in_eid, eb, st));
  BG_CHECK(cudaMallocAsync(&g->out_indices, eb, st)); BG_CHECK(cudaMallocAsync(&g->out_eid, eb, st));
  BG_CHECK(cudaMallocAsync(&g->in_deg, sizeof(int32_t) * (n_dst + 1), st));
  BG_CHECK(cudaMallocAsync(&g->out_deg, sizeof(int32_t) * (n_src + 1), st));

  int32_t *src32 = nullptr, *dst32 = nullptr, *iota = nullptr, *ktmp = nullptr;
  int* flags = nullptr;  // [bad, max_in, zero_in, max_out, zero_out, in_eid is not the identity]
  BG_CHECK(cudaMallocAsync(&src32, eb, st)); BG_CHECK(cudaMallocAsync(&dst32, eb, st));
  BG_CHECK(cudaMallocAsync(&iota, eb, st)); BG_CHECK(cudaMallocAsync(&ktmp, eb, st));
  BG_CHECK(cudaMallocAsync(&flags, sizeof(int) * 6, st));
  BG_CHECK(cudaMemsetAsync(flags, 0, sizeof(int) * 6, st));
  if (n_edges > 0) {
    k_narrow_and_check<<<grid_for(n_edges), 256, 0, st>>>(n_edges, src, n_src, src32, iota, flags); BG_LAUNCHED(1);
    k_narrow_and_check<<<grid_for(n_edges), 256, 0, st>>>(n_edges, dst, n_dst, dst32, nullptr, flags); BG_LAUNCHED(1);
    BG_CHECK(cudaGetLastError());
  }
  int rc = build_csr(n_dst, n_edges, dst32, src32, iota, ktmp, g->in_indptr, g->in_indices, g->in_eid, g->in_deg, st);
  if (rc) return rc;
  rc = build_csr(n_src, n_edges, src32, dst32, iota, ktmp, g->out_indptr, g->out_indices, g->out_eid, g->out_deg, st);
  if (rc) return rc;
  if (n_dst > 0) k_deg_stats<<<grid_for(n_dst), 256, 0, st>>>(n_dst, g->in_deg, flags + 1); BG_LAUNCHED(1);
  if (n_src > 0) k_deg_stats<<<grid_for(n_src), 256, 0, st>>>(n_src, g->out_deg, flags + 3); BG_LAUNCHED(1);
  if (n_edges > 0) k_check_identity<<<grid_for(n_edges), 256, 0, st>>>(n_edges, g->in_eid, flags + 5); BG_LAUNCHED(1);
  BG_CHECK(cudaGetLastError());
  int h[6];
  BG_CHECK(cudaMemcpyAsync(h, flags, sizeof(h), cudaMemcpyDeviceToHost, st));
  BG_CHECK(cudaFreeAsync(src32, st)); BG_CHECK(cudaFreeAsync(dst32, st));
  BG_CHECK(cudaFreeAsync(flags, st));
  BG_CHECK(cudaStreamSynchronize(st));
  if (h[0] != 0) { cudaFreeAsync(iota, st); cudaFreeAsync(ktmp, st); }
  BG_REQUIRE(h[0] == 0, "graph_create: node id out of range [0,n_src) / [0,n_dst)");
  g->max_in_deg = h[1]; g->has_zero_in_degree = h[2] > 0; g->max_out_deg = h[3];
  g->in_eid_identity = h[5] == 0;
  // Cache-blocked out-CSR traversal for the in <-> out record transposes (edge_ops.cu).  Worth it only when both
  // sides of a (source block x destination block) tile are RUNS inside their CSR rows — which needs sorted neighbour
  // lists (the canonical numbering) and enough neighbours per row and block.
  {
    int ts = 1, td = 1;
    const char* force = env_str("BOTGAT_TILES");  // "ts,td" (tests / sweeps); "0" = off
    if (force) {
      if (sscanf(force, "%d,%d", &ts, &td) != 2) ts = td = 1;
    } else if (g->in_eid_identity && n_edges >= (1 << 22) && n_src > 0 && n_dst > 0) {
      const double avg_in = (double)n_edges / n_dst, avg_out = (double)n_edges / n_src;
      const int cap_s = std::max(1, (int)(avg_in / 16)), cap_d = std::max(1, (int)(avg_out / 16));  // runs >= 16 records
      const double need = (double)n_edges * 32.0 / ((double)env_int("BOTGAT_TILE_MB", 20) * (1 << 20));  // tiles wanted
      int want = 1;
      while ((double)want * want < need) ++want;
      ts = std::min(want, cap_s); td = std::min(want, cap_d);
      while ((double)ts * td < need && ts < cap_s) ++ts;
      while ((double)ts * td < need && td < cap_d) ++td;
      if ((double)ts * td < need * 0.5) ts = td = 1;  // rows too short to block this graph down to the L2: plain order
    }
    ts = std::max(1, std::min(ts, 64)); td = std::max(1, std::min(td, 64));
    if (ts * td > 1 && n_edges > 0 && n_src > 0 && n_dst > 0) {
      const int rows_per_s = (int)((n_src + ts - 1) / ts), rows_per_d = (int)((n_dst + td - 1) / td);
      BG_CHECK(cudaMallocAsync(&g->out_tile_order, eb, st));
      k_tile_keys<<<grid_for(n_src * 32), 256, 0, st>>>((int)n_src, g->out_indptr, g->out_indices, rows_per_s, rows_per_d,
                                                       td, ktmp, iota); BG_LAUNCHED(1);
      int32_t* ksorted = nullptr;
      BG_CHECK(cudaMallocAsync(&ksorted, eb, st));
      size_t tmp_bytes = 0;
      const int kbits = bits_for((int64_t)ts * td);
      BG_CHECK(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, ktmp, ksorted, iota, g->out_tile_order, (int)n_edges, 0, kbits, st));
      void* tmp = nullptr;
      BG_CHECK(cudaMallocAsync(&tmp, tmp_bytes, st));
      BG_CHECK(cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, ktmp, ksorted, iota, g->out_tile_order, (int)n_edges, 0, kbits, st)); BG_LAUNCHED(1);
      BG_CHECK(cudaFreeAsync(tmp, st)); BG_CHECK(cudaFreeAsync(ksorted, st));
      g->tiles_s = ts; g->tiles_d = td;
    }
  }
  BG_CHECK(cudaFreeAsync(iota, st)); BG_CHECK(cudaFreeAsync(ktmp, st));
  // heavy rows: split into segments (no-op for graphs whose longest row fits one segment)
  rc = build_segments((int)n_dst, g->in_indptr, g->in_deg, g->max_in_deg, &g->seg_in, st);
  if (rc) return rc;
  rc = build_segments((int)n_src, g->out_indptr, g->out_deg, g->max_out_deg, &g->seg_out, st);
  if (rc) return rc;
  cleanup.armed = false;
  *out = g;
  return 0;
}

extern "C" int botgat_graph_get(const botgat_graph* g, int which, void** dev_ptr, int64_t* len) {
  BG_REQUIRE(g && dev_ptr && len, "graph_get: null argument");
  switch (which) {
    case BOTGAT_IN_INDPTR: *dev_ptr = g->in_indptr; *len = g->n_dst + 1; break;
    case BOTGAT_IN_INDICES: *dev_ptr = g->in_indices; *len = g->n_edges; break;
    case BOTGAT_IN_EID: *dev_ptr = g->in_eid; *len = g->n_edges; break;
    case BOTGAT_OUT_INDPTR: *dev_ptr = g->out_indptr; *len = g->n_src + 1; break;
    case BOTGAT_OUT_INDICES: *dev_ptr = g->out_indices; *len = g->n_edges; break;
    case BOTGAT_OUT_EID: *dev_ptr = g->out_eid; *len = g->n_edges; break;
    case BOTGAT_IN_DEG: *dev_ptr = g->in_deg; *len = g->n_dst; break;
    case BOTGAT_OUT_DEG: *dev_ptr = g->out_deg; *len = g->n_src; break;
    default: set_error("graph_get: unknown array %d", which); return -1;
  }
  return 0;
}

extern "C" int botgat_graph_get_info(const botgat_graph* g, botgat_graph_info* info) {
  BG_REQUIRE(g && info, "graph_get_info: null argument");
  info->n_src = g->n_src; info->n_dst = g->n_dst; info->n_edges = g->n_edges;
  info->max_in_deg = g->max_in_deg; info->max_out_deg = g->max_out_deg;
  info->has_zero_in_degree = g->has_zero_in_degree; info->device = g->device;
  info->n_slots_in = g->seg_in.n_slots; info->n_slots_out = g->seg_out.n_slots;
  info->in_eid_identity = g->in_eid_identity; info->tiles_src = g->tiles_s; info->tiles_dst = g->tiles_d;
  info->n_seg_in = g->seg_in.n_items; info->n_seg_out = g->seg_out.n_items; info->reserved_ = 0;
  return 0;
}

// ---------------------------------------------------------------------------
// COO preprocessing
// ---------------------------------------------------------------------------
namespace botgat {

__global__ void k_pack_bidirected(int64_t n, const int64_t* __restrict__ src, const int64_t* __restrict__ dst,
                                  int64_t n_nodes, uint64_t* __restrict__ keys, int* __restrict__ bad) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t s = src[i], d = dst[i];
    if (s < 0 || s >= n_nodes || d < 0 || d >= n_nodes) *bad = 1;
    keys[i] = (uint64_t)s * (uint64_t)n_nodes + (uint64_t)d;
    keys[n + i] = (uint64_t)d * (uint64_t)n_nodes + (uint64_t)s;
  }
}
__global__ void k_unpack(int64_t n, const uint64_t* __restrict__ keys, int64_t n_nodes, int64_t* __restrict__ src,
                         int64_t* __restrict__ dst) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    src[i] = (int64_t)(keys[i] / (uint64_t)n_nodes);
    dst[i] = (int64_t)(keys[i] % (uint64_t)n_nodes);
  }
}
__global__ void k_flag_not_loop(int64_t n, const int64_t* __restrict__ src, const int64_t* __restrict__ dst,
                                uint8_t* __restrict__ flag) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    flag[i] = src[i] != dst[i];
}
__global__ void k_iota64(int64_t n, int64_t* __restrict__ a, int64_t* __restrict__ b) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    a[i] = i;
    b[i] = i;
  }
}

}  // namespace botgat

extern "C" int botgat_coo_to_bidirected(int64_t n_nodes, int64_t n_edges, const int64_t* src, const int64_t* dst,
                                        int64_t* out_src, int64_t* out_dst, int64_t* n_out, int device, void* stream) {
  BG_REQUIRE(n_out, "to_bidirected: null n_out");
  *n_out = 0;
  if (n_edges == 0) return 0;
  BG_REQUIRE(src && dst && out_src && out_dst, "to_bidirected: null pointer");
  BG_REQUIRE(2 * n_edges < (1ll << 31) - 1, "to_bidirected: too many edges");
  DeviceGuard guard(device);
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t n2 = 2 * n_edges;
  uint64_t *keys = nullptr, *sorted = nullptr, *uniq = nullptr;
  int64_t* d_count = nullptr;
  int* bad = nullptr;
  BG_CHECK(cudaMallocAsync(&keys, sizeof(uint64_t) * n2, st));
  BG_CHECK(cudaMallocAsync(&sorted, sizeof(uint64_t) * n2, st));
  BG_CHECK(cudaMallocAsync(&uniq, sizeof(uint64_t) * n2, st));
  BG_CHECK(cudaMallocAsync(&d_count, sizeof(int64_t), st));
  BG_CHECK(cudaMallocAsync(&bad, sizeof(int), st));
  BG_CHECK(cudaMemsetAsync(bad, 0, sizeof(int), st));
  k_pack_bidirected<<<grid_for(n_edges), 256, 0, st>>>(n_edges, src, dst, n_nodes, keys, bad); BG_LAUNCHED(1);
  BG_CHECK(cudaGetLastError());
  const int bits = std::min(64, 2 * bits_for(n_nodes) + 1);
  size_t tb = 0, tb2 = 0;
  BG_CHECK(cub::DeviceRadixSort::SortKeys(nullptr, tb, keys, sorted, (int)n2, 0, bits, st));
  BG_CHECK(cub::DeviceSelect::Unique(nullptr, tb2, sorted, uniq, d_count, (int)n2, st));
  void* tmp = nullptr;
  BG_CHECK(cudaMallocAsync(&tmp, std::max(tb, tb2), st));
  BG_CHECK(cub::DeviceRadixSort::SortKeys(tmp, tb, keys, sorted, (int)n2, 0, bits, st)); BG_LAUNCHED(1);
  BG_CHECK(cub::DeviceSelect::Unique(tmp, tb2, sorted, uniq, d_count, (int)n2, st)); BG_LAUNCHED(1);
  int64_t cnt = 0;
  int hbad = 0;
  BG_CHECK(cudaMemcpyAsync(&cnt, d_count, sizeof(cnt), cudaMemcpyDeviceToHost, st));
  BG_CHECK(cudaMemcpyAsync(&hbad, bad, sizeof(hbad), cudaMemcpyDeviceToHost, st));
  BG_CHECK(cudaStreamSynchronize(st));
  if (!hbad && cnt > 0) {
    k_unpack<<<grid_for(cnt), 256, 0, st>>>(cnt, uniq, n_nodes, out_src, out_dst); BG_LAUNCHED(1);
    BG_CHECK(cudaGetLastError());
  }
  BG_CHECK(cudaFreeAsync(tmp, st)); BG_CHECK(cudaFreeAsync(keys, st)); BG_CHECK(cudaFreeAsync(sorted, st));
  BG_CHECK(cudaFreeAsync(uniq, st)); BG_CHECK(cudaFreeAsync(d_count, st)); BG_CHECK(cudaFreeAsync(bad, st));
  BG_CHECK(cudaStreamSynchronize(st));
  BG_REQUIRE(!hbad, "to_bidirected: node id out of range");
  *n_out = cnt;
  return 0;
}

extern "C" int botgat_coo_remove_self_loop(int64_t n_edges, const int64_t* src, const int64_t* dst, int64_t* out_src,
                                           int64_t* out_dst, int64_t* n_out, int device, void* stream) {
  BG_REQUIRE(n_out, "remove_self_loop: null n_out");
  *n_out = 0;
  if (n_edges == 0) return 0;
  BG_REQUIRE(src && dst && out_src && out_dst, "remove_self_loop: null pointer");
  BG_REQUIRE(n_edges < (1ll << 31) - 1, "remove_self_loop: too many edges");
  DeviceGuard guard(device);
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* flag = nullptr;
  int64_t* d_count = nullptr;
  BG_CHECK(cudaMallocAsync(&flag, n_edges, st));
  BG_CHECK(cudaMallocAsync(&d_count, sizeof(int64_t), st));
  k_flag_not_loop<<<grid_for(n_edges), 256, 0, st>>>(n_edges, src, dst, flag); BG_LAUNCHED(1);
  BG_CHECK(cudaGetLastError());
  size_t tb = 0;
  BG_CHECK(cub::DeviceSelect::Flagged(nullptr, tb, src, flag, out_src, d_count, (int)n_edges, st));
  void* tmp = nullptr;
  BG_CHECK(cudaMallocAsync(&tmp, tb, st));
  BG_CHECK(cub::DeviceSelect::Flagged(tmp, tb, src, flag, out_src, d_count, (int)n_edges, st)); BG_LAUNCHED(1);
  BG_CHECK(cub::DeviceSelect::Flagged(tmp, tb, dst, flag, out_dst, d_count, (int)n_edges, st)); BG_LAUNCHED(1);
  int64_t cnt = 0;
  BG_CHECK(cudaMemcpyAsync(&cnt, d_count, sizeof(cnt), cudaMemcpyDeviceToHost, st));
  BG_CHECK(cudaFreeAsync(tmp, st)); BG_CHECK(cudaFreeAsync(flag, st)); BG_CHECK(cudaFreeAsync(d_count, st));
  BG_CHECK(cudaStreamSynchronize(st));
  *n_out = cnt;
  return 0;
}

extern "C" int botgat_coo_add_self_loop(int64_t n_nodes, int64_t n_edges, const int64_t* src, const int64_t* dst,
                                        int64_t* out_src, int64_t* out_dst, int device, void* stream) {
  BG_REQUIRE(out_src && out_dst, "add_self_loop: null output");
  DeviceGuard guard(device);
  cudaStream_t st = (cudaStream_t)stream;
  if (n_edges > 0) {
    BG_CHECK(cudaMemcpyAsync(out_src, src, sizeof(int64_t) * n_edges, cudaMemcpyDeviceToDevice, st));
    BG_CHECK(cudaMemcpyAsync(out_dst, dst, sizeof(int64_t) * n_edges, cudaMemcpyDeviceToDevice, st));
  }
  if (n_nodes > 0) {
    k_iota64<<<grid_for(n_nodes), 256, 0, st>>>(n_nodes, out_src + n_edges, out_dst + n_edges); BG_LAUNCHED(1);
    BG_CHECK(cudaGetLastError());
  }
  return 0;
}

// ---------------------------------------------------------------------------
// multi-GPU helpers: 1-D partition and halo row packing
// ---------------------------------------------------------------------------
namespace botgat {

__global__ void k_partition_bounds(int n_rows, const int32_t* __restrict__ indptr, int n_parts, int64_t n_edges,
                                   int64_t* __restrict__ bounds) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p > n_parts) return;
  if (p == 0) { bounds[0] = 0; return; }
  if (p == n_parts) { bounds[p] = n_rows; return; }
  const int64_t target = (int64_t)p * n_edges / n_parts;
  int lo = 0, hi = n_rows + 1;  // first index r in [0, n_rows] with indptr[r] >= target
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if ((int64_t)indptr[mid] < target) lo = mid + 1; else hi = mid;
  }
  bounds[p] = min(lo, n_rows);
}

// edges of rows [lo,hi) in edge-id order: flag by dst range, then select
__global__ void k_flag_range(int64_t n_edges, const int32_t* __restrict__ out_indices_by_eid_dst, int64_t lo,
                             int64_t hi, uint8_t* __restrict__ flag) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_edges; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t d = out_indices_by_eid_dst[i];
    flag[i] = d >= lo && d < hi;
  }
}

// dst/src of every edge id, rebuilt from the in-CSR (row of position p is found by the caller's expansion)
__global__ void k_expand_rows(int n_rows, const int32_t* __restrict__ indptr, const int32_t* __restrict__ eid,
                              const int32_t* __restrict__ indices, int32_t* __restrict__ dst_by_eid,
                              int32_t* __restrict__ src_by_eid) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  for (int r = warp; r < n_rows; r += nwarps) {
    for (int p = indptr[r] + lane; p < indptr[r + 1]; p += 32) {
      const int e = eid[p];
      dst_by_eid[e] = r;
      src_by_eid[e] = indices[p];
    }
  }
}

__global__ void k_extract_write(int64_t n, const int32_t* __restrict__ sel_eid, const int32_t* __restrict__ src_by_eid,
                                const int32_t* __restrict__ dst_by_eid, int64_t lo, int64_t* __restrict__ out_eid,
                                int64_t* __restrict__ out_src, int64_t* __restrict__ out_ldst) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int e = sel_eid[i];
    out_eid[i] = e;
    out_src[i] = src_by_eid[e];
    out_ldst[i] = dst_by_eid[e] - lo;
  }
}

__global__ void k_rows_gather(const float* __restrict__ table, int64_t ld, int64_t width, const int64_t* __restrict__ rows,
                              int64_t n_rows, float* __restrict__ out) {
  const int64_t total = n_rows * width;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / width, c = i - r * width;
    out[i] = table[rows[r] * ld + c];
  }
}
__global__ void k_rows_scatter_add(float* __restrict__ table, int64_t ld, int64_t width, const int64_t* __restrict__ rows,
                                   int64_t n_rows, const float* __restrict__ in) {
  const int64_t total = n_rows * width;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / width, c = i - r * width;
    table[rows[r] * ld + c] += in[i];  // rows are unique: no two threads touch one element
  }
}

}  // namespace botgat

extern "C" int botgat_partition_1d(const botgat_graph* g, int32_t n_parts, int64_t* bounds, void* stream) {
  BG_REQUIRE(g && bounds && n_parts >= 1, "partition_1d: bad arguments");
  DeviceGuard guard(g->device);
  cudaStream_t st = (cudaStream_t)stream;
  int64_t* d = nullptr;
  BG_CHECK(cudaMallocAsync(&d, sizeof(int64_t) * (n_parts + 1), st));
  k_partition_bounds<<<(n_parts + 1 + 127) / 128, 128, 0, st>>>((int)g->n_dst, g->in_indptr, n_parts, g->n_edges, d); BG_LAUNCHED(1);
  BG_CHECK(cudaGetLastError());
  BG_CHECK(cudaMemcpyAsync(bounds, d, sizeof(int64_t) * (n_parts + 1), cudaMemcpyDeviceToHost, st));
  BG_CHECK(cudaFreeAsync(d, st));
  BG_CHECK(cudaStreamSynchronize(st));
  for (int p = 1; p <= n_parts; ++p)
    if (bounds[p] < bounds[p - 1]) bounds[p] = bounds[p - 1];
  return 0;
}

extern "C" int botgat_partition_extract(const botgat_graph* g, int64_t lo, int64_t hi, int64_t* out_eid,
                                        int64_t* out_src, int64_t* out_ldst, int64_t* n_local, void* stream) {
  BG_REQUIRE(g && n_local, "partition_extract: bad arguments");
  BG_REQUIRE(0 <= lo && lo <= hi && hi <= g->n_dst, "partition_extract: bad range [%lld,%lld)", (long long)lo, (long long)hi);
  DeviceGuard guard(g->device);
  cudaStream_t st = (cudaStream_t)stream;
  // rows [lo,hi) own the contiguous in-CSR span [indptr[lo], indptr[hi])
  int32_t span[2] = {0, 0};
  BG_CHECK(cudaMemcpyAsync(&span[0], g->in_indptr + lo, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  BG_CHECK(cudaMemcpyAsync(&span[1], g->in_indptr + hi, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  BG_CHECK(cudaStreamSynchronize(st));
  const int64_t cnt = (int64_t)span[1] - span[0];
  *n_local = cnt;
  if (!out_eid || cnt == 0) return 0;
  BG_REQUIRE(out_src && out_ldst, "partition_extract: null output");
  // edge-id order inside the range: sort the span's edge ids (they are unique)
  int32_t *sel = nullptr, *dst_by_eid = nullptr, *src_by_eid = nullptr;
  BG_CHECK(cudaMallocAsync(&sel, sizeof(int32_t) * cnt, st));
  BG_CHECK(cudaMallocAsync(&dst_by_eid, sizeof(int32_t) * g->n_edges, st));
  BG_CHECK(cudaMallocAsync(&src_by_eid, sizeof(int32_t) * g->n_edges, st));
  size_t tb = 0;
  BG_CHECK(cub::DeviceRadixSort::SortKeys(nullptr, tb, g->in_eid + span[0], sel, (int)cnt, 0, bits_for(g->n_edges), st));
  void* tmp = nullptr;
  BG_CHECK(cudaMallocAsync(&tmp, tb, st));
  BG_CHECK(cub::DeviceRadixSort::SortKeys(tmp, tb, g->in_eid + span[0], sel, (int)cnt, 0, bits_for(g->n_edges), st)); BG_LAUNCHED(1);
  k_expand_rows<<<grid_for(g->n_dst * 32), 256, 0, st>>>((int)g->n_dst, g->in_indptr, g->in_eid, g->in_indices,
                                                        dst_by_eid, src_by_eid); BG_LAUNCHED(1);
  k_extract_write<<<grid_for(cnt), 256, 0, st>>>(cnt, sel, src_by_eid, dst_by_eid, lo, out_eid, out_src, out_ldst); BG_LAUNCHED(1);
  BG_CHECK(cudaGetLastError());
  BG_CHECK(cudaFreeAsync(tmp, st)); BG_CHECK(cudaFreeAsync(sel, st));
  BG_CHECK(cudaFreeAsync(dst_by_eid, st)); BG_CHECK(cudaFreeAsync(src_by_eid, st));
  BG_CHECK(cudaStreamSynchronize(st));
  return 0;
}

extern "C" int botgat_rows_gather(const float* table, int64_t ld, int64_t width, const int64_t* rows, int64_t n_rows,
                                  float* out, void* stream) {
  if (n_rows == 0 || width == 0) return 0;
  BG_REQUIRE(table && rows && out, "rows_gather: null pointer");
  k_rows_gather<<<grid_for(n_rows * width), 256, 0, (cudaStream_t)stream>>>(table, ld, width, rows, n_rows, out); BG_LAUNCHED(1);
  BG_CHECK(cudaGetLastError());
  return 0;
}

extern "C" int botgat_rows_scatter_add(float* table, int64_t ld, int64_t width, const int64_t* rows, int64_t n_rows,
                                       const float* in, void* stream) {
  if (n_rows == 0 || width == 0) return 0;
  BG_REQUIRE(table && rows && in, "rows_scatter_add: null pointer");
  k_rows_scatter_add<<<grid_for(n_rows * width), 256, 0, (cudaStream_t)stream>>>(table, ld, width, rows, n_rows, in); BG_LAUNCHED(1);
  BG_CHECK(cudaGetLastError());
  return 0;
}
