// Per-edge operand staging for libbotgat (sm_100a).
//
// Edge tensors arrive in edge-id order (DGL `edata`: `attn_edge_fc(feat_edge)` of
// src/ogbn-proteins/models.py:131, the edge-drop keep set of models.py:137-139, the attention-dropout mask
// of models.py:141/143); the gather kernels stream them in CSR order, head-major.  These kernels are the
// permutation between the two: one random (4*H)-byte record access per edge on the edge-id side, fully
// coalesced on the CSR side.  They are DRAM-random-access bound, so what matters is bytes fetched per
// record: records are read/written with the widest aligned vector the row stride allows (a row stride of
// 8 floats makes every H<=8 record exactly one 32-byte sector), and loads carry an L2 prefetch-size hint.
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/transform_iterator.h>

#include "common.cuh"

namespace botgat {

static int env_pf() {
  return (int)env_int("BOTGAT_PF", 0);  // L2 prefetch-size hints measured neutral on B200 (profiles/r01_sweeps.md)
}

template <int PF> __device__ __forceinline__ float4 ld_rec4(const float* p) {
  float4 r;
  if constexpr (PF == 64)
    asm("ld.global.nc.L2::64B.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  else if constexpr (PF == 128)
    asm("ld.global.nc.L2::128B.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  else if constexpr (PF == 256)
    asm("ld.global.nc.L2::256B.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  else
    r = __ldg(reinterpret_cast<const float4*>(p));
  return r;
}
template <int PF> __device__ __forceinline__ float2 ld_rec2(const float* p) {
  float2 r;
  if constexpr (PF == 64) asm("ld.global.nc.L2::64B.v2.f32 {%0,%1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
  else if constexpr (PF == 128) asm("ld.global.nc.L2::128B.v2.f32 {%0,%1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
  else if constexpr (PF == 256) asm("ld.global.nc.L2::256B.v2.f32 {%0,%1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
  else r = __ldg(reinterpret_cast<const float2*>(p));
  return r;
}
template <int PF> __device__ __forceinline__ float ld_rec1(const float* p) {
  float r;
  if constexpr (PF == 64) asm("ld.global.nc.L2::64B.f32 %0, [%1];" : "=f"(r) : "l"(p));
  else if constexpr (PF == 128) asm("ld.global.nc.L2::128B.f32 %0, [%1];" : "=f"(r) : "l"(p));
  else if constexpr (PF == 256) asm("ld.global.nc.L2::256B.f32 %0, [%1];" : "=f"(r) : "l"(p));
  else r = __ldg(p);
  return r;
}

constexpr int kHMax = 8;  // heads handled per record pass (records wider than this take several passes)

// read H <= kHMax floats of one record; VEC = 4, 2 or 1 floats per load (alignment established by the host)
template <int VEC, int PF> __device__ __forceinline__ void load_record(const float* rec, int H, float (&v)[kHMax]) {
  if constexpr (VEC == 4) {
#pragma unroll
    for (int q = 0; q < kHMax / 4; ++q) {
      if (q * 4 < H) {
        const float4 t = ld_rec4<PF>(rec + q * 4);
        v[q * 4] = t.x; v[q * 4 + 1] = t.y; v[q * 4 + 2] = t.z; v[q * 4 + 3] = t.w;
      }
    }
  } else if constexpr (VEC == 2) {
#pragma unroll
    for (int q = 0; q < kHMax / 2; ++q) {
      if (q * 2 < H) {
        const float2 t = ld_rec2<PF>(rec + q * 2);
        v[q * 2] = t.x; v[q * 2 + 1] = t.y;
      }
    }
  } else {
#pragma unroll
    for (int q = 0; q < kHMax; ++q)
      if (q < H) v[q] = ld_rec1<PF>(rec + q);
  }
}
template <int VEC> __device__ __forceinline__ void store_record(float* rec, int H, const float (&v)[kHMax]) {
  if constexpr (VEC == 4) {
#pragma unroll
    for (int q = 0; q < kHMax / 4; ++q)
      if (q * 4 < H) *reinterpret_cast<float4*>(rec + q * 4) = make_float4(v[q * 4], v[q * 4 + 1], v[q * 4 + 2], v[q * 4 + 3]);
  } else if constexpr (VEC == 2) {
#pragma unroll
    for (int q = 0; q < kHMax / 2; ++q)
      if (q * 2 < H) *reinterpret_cast<float2*>(rec + q * 2) = make_float2(v[q * 2], v[q * 2 + 1]);
  } else {
#pragma unroll
    for (int q = 0; q < kHMax; ++q)
      if (q < H) rec[q] = v[q];
  }
}

// widest vector (floats) usable for records at `p` with row stride `ld`, given that a vector load may run past
// H up to the next multiple of the vector width (so that multiple must still fit inside the row stride)
static int record_vec(const void* p, int64_t ld, int H) {
  auto fits = [&](int w) { return ld % w == 0 && ((uintptr_t)p % (4 * w)) == 0 && ((H + w - 1) / w) * w <= ld; };
  return fits(4) ? 4 : (fits(2) ? 2 : 1);
}

// ---------------------------------------------------------------------------
// stage: edge-id order -> CSR order, head-major.  One thread per CSR position, heads [h0, h0+Hn).
// ---------------------------------------------------------------------------
// keep bytes -> bits.  The staging pass looks the keep flag up by edge id (random): as bytes that is a second random
// DRAM access per edge (+0.29 ms at E = 39.6 M), as bits the whole mask (E/8 bytes, 4.9 MB) is L2-resident.
__global__ void k_pack_keep(int64_t n_edges, const uint8_t* __restrict__ keep, uint32_t* __restrict__ bits) {
  const int64_t n_round = (n_edges + 31) & ~(int64_t)31;  // whole warps reach the ballot
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n_round; e += (int64_t)gridDim.x * blockDim.x) {
    const unsigned b = __ballot_sync(0xffffffffu, e < n_edges && __ldg(keep + e) != 0);
    if ((threadIdx.x & 31) == 0) bits[e >> 5] = b;
  }
}

// The kept positions of one CSR order (botgat_edge_subset.kept / base): bit p&31 of word p>>5 is the kept flag of
// position p, base[w] the number of kept positions before word w.  At 1/8 byte + 1/8 byte per edge both stay L2-resident,
// so the compacted position of p costs two cached loads instead of a stream of 4 bytes per edge.
struct KeptMap {
  const uint32_t* bits;  // null: no subset
  const int32_t* base;
  // kept positions before x (x in [0, n_edges])
  __device__ __forceinline__ int64_t rank(int64_t x) const {
    return __ldg(base + (x >> 5)) + __popc(__ldg(bits + (x >> 5)) & ((1u << (x & 31)) - 1u));
  }
  __device__ __forceinline__ bool kept(int64_t p) const { return (__ldg(bits + (p >> 5)) >> (p & 31)) & 1u; }
};

// `order` (optional): the CSR positions in the order they are to be visited — the cache-blocked traversal of the
// out-CSR (common.cuh `out_tile_order`).  With the canonical edge numbering a (source block x destination block)
// tile is a set of RUNS on both sides: consecutive threads still write consecutive CSR positions, and the records
// they read lie inside a few-MB window of the edge-ordered array that the L2 holds until every 128-byte line
// (4 records) has been used — instead of one DRAM line fill per 32-byte record.
// `km` (optional): the kept positions of botgat_edge_subset.  A kept position p is written to its rank (runs stay runs)
// together with its adjacency entry (`sub_indices` / `sub_eid`, when given); a dropped one is skipped.
template <int VEC, int PF>
__global__ void k_edge_stage(int64_t n_edges, int h0, int Hn, const int32_t* __restrict__ eid,
                             const int32_t* __restrict__ order,
                             const float* __restrict__ src, int64_t ld, const uint8_t* __restrict__ keep,
                             const uint32_t* __restrict__ keep_bits, float* __restrict__ dst,
                             const KeptMap km, const int32_t* __restrict__ indices,
                             int32_t* __restrict__ sub_indices, int32_t* __restrict__ sub_eid) {
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n_edges; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = order ? __ldg(order + t) : t;
    int64_t q = p;  // destination position
    if (km.bits) {
      if (!km.kept(p)) continue;
      q = km.rank(p);
    }
    const int64_t e = __ldg(eid + p);
    float v[kHMax];
#pragma unroll
    for (int c = 0; c < kHMax; ++c) v[c] = 0.f;
    if (src) load_record<VEC, PF>(src + e * ld + h0, Hn, v);
    const bool dropped = keep_bits ? !((__ldg(keep_bits + (e >> 5)) >> (e & 31)) & 1u) : (keep && !__ldg(keep + e));
#pragma unroll
    for (int c = 0; c < kHMax; ++c)
      if (c < Hn) dst[(int64_t)(h0 + c) * n_edges + q] = dropped ? -INFINITY : v[c];
    if (sub_indices) {
      sub_indices[q] = __ldg(indices + p);
      if (sub_eid) sub_eid[q] = (int32_t)e;
    }
  }
}

// unstage: CSR order, head-major -> edge-id order records.  Columns [h0+Hn, h0+Hw) of the record are row padding
// and receive zeros.  With `km` (kept positions) gz is compacted: a kept position p reads the column of its rank, a
// dropped edge's record is all zeros.
template <int VEC>
__global__ void k_edge_unstage(int64_t n_edges, int h0, int Hn, int Hw, const int32_t* __restrict__ eid,
                               const int32_t* __restrict__ order, const KeptMap km,
                               const float* __restrict__ gz, float* __restrict__ dst, int64_t ld) {
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n_edges; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = order ? __ldg(order + t) : t;
    const int64_t e = __ldg(eid + p);
    int64_t q = p;
    bool kept = true;
    if (km.bits) {
      kept = km.kept(p);
      q = km.rank(p);
    }
    float v[kHMax];
#pragma unroll
    for (int c = 0; c < kHMax; ++c) v[c] = (c < Hn && kept) ? __ldg(gz + (int64_t)(h0 + c) * n_edges + q) : 0.f;
    store_record<VEC>(dst + e * ld + h0, Hw, v);
  }
}

// kept flags in CSR position order as bits, one word per 32 positions (n_words = n_edges/32 + 1: the last word also
// covers position n_edges, which is never kept)
__global__ void k_kept_bits(int64_t n_edges, int64_t n_words, const int32_t* __restrict__ eid, const uint8_t* __restrict__ keep,
                            const uint32_t* __restrict__ keep_bits, uint32_t* __restrict__ bits) {
  for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < n_words * 32; p += (int64_t)gridDim.x * blockDim.x) {
    bool k = false;
    if (p < n_edges) {
      const int64_t e = eid ? __ldg(eid + p) : p;  // null eid: the position is the edge id
      k = keep_bits ? ((__ldg(keep_bits + (e >> 5)) >> (e & 31)) & 1u) : __ldg(keep + e) != 0;
    }
    const unsigned b = __ballot_sync(0xffffffffu, k);
    if ((threadIdx.x & 31) == 0) bits[p >> 5] = b;
  }
}

struct WordCount {
  const uint32_t* bits;
  __device__ int operator()(int64_t w) const { return __popc(__ldg(bits + w)); }
};

// indptr' = rank(indptr) and the row segments [rank(beg), rank(end))
__global__ void k_subset_bounds(int n_rows, const int32_t* __restrict__ indptr, int n_seg, const int32_t* __restrict__ seg_beg,
                                const int32_t* __restrict__ seg_end, const KeptMap km,
                                int32_t* __restrict__ sub_indptr, int32_t* __restrict__ sub_beg, int32_t* __restrict__ sub_end) {
  const int n = max(n_rows + 1, n_seg);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    if (i <= n_rows) sub_indptr[i] = (int32_t)km.rank(__ldg(indptr + i));
    if (i < n_seg) {
      sub_beg[i] = (int32_t)km.rank(__ldg(seg_beg + i));
      sub_end[i] = (int32_t)km.rank(__ldg(seg_end + i));
    }
  }
}

// grad_er[v,h] = sum over in-edges k of grad_ee[k,h]: one warp per work item (a destination row, or one segment
// of a heavy row whose partial sums go to a scratch slot), lanes stride its edges
template <int VEC, int PF>
__global__ void __launch_bounds__(256)
k_edge_reduce_dst(int n_items, int H, int h0, int Hn, const int32_t* __restrict__ indptr, const int32_t* __restrict__ eid,
                  const int32_t* __restrict__ seg_row, const int32_t* __restrict__ seg_beg,
                  const int32_t* __restrict__ seg_end, const int32_t* __restrict__ seg_slot,
                  const float* __restrict__ grad_ee, int64_t ld, float* __restrict__ grad_er, float* __restrict__ scratch) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item = blockIdx.x * 8 + warp;
  if (item >= n_items) return;
  const int v = seg_row ? seg_row[item] : item;
  const int beg = seg_row ? seg_beg[item] : indptr[v], end = seg_row ? seg_end[item] : indptr[v + 1];
  const int slot = seg_row ? seg_slot[item] : -1;
  float s[kHMax];
#pragma unroll
  for (int q = 0; q < kHMax; ++q) s[q] = 0.f;
  for (int pos = beg + lane; pos < end; pos += 32) {
    float r[kHMax];
#pragma unroll
    for (int q = 0; q < kHMax; ++q) r[q] = 0.f;
    load_record<VEC, PF>(grad_ee + (int64_t)__ldg(eid + pos) * ld + h0, Hn, r);
#pragma unroll
    for (int q = 0; q < kHMax; ++q) s[q] += r[q];
  }
#pragma unroll
  for (int q = 0; q < kHMax; ++q) {
    if (q < Hn) {
      const float t = warp_sum(s[q]);
      if (lane == 0) {
        if (slot >= 0) scratch[(int64_t)slot * H + h0 + q] = t;
        else grad_er[(int64_t)v * H + h0 + q] = t;
      }
    }
  }
}

__global__ void k_edge_reduce_combine(int n_split, int H, const int32_t* __restrict__ split_rows,
                                      const int32_t* __restrict__ split_first, const float* __restrict__ scratch,
                                      float* __restrict__ grad_er) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_split * H) return;
  const int i = t / H, h = t - i * H;
  float a = 0.f;
  for (int s = split_first[i]; s < split_first[i + 1]; ++s) a += scratch[(int64_t)s * H + h];
  grad_er[(int64_t)split_rows[i] * H + h] = a;
}

static inline int grid_for(int64_t n, int block = 256) {
  int64_t b = (n + block - 1) / block;
  return (int)std::max<int64_t>(1, std::min<int64_t>(b, 148 * 32));
}

#define BG_PF_SWITCH(CALL)                        \
  switch (pf) {                                   \
    case 64: { constexpr int PF = 64; CALL; break; }   \
    case 128: { constexpr int PF = 128; CALL; break; } \
    case 256: { constexpr int PF = 256; CALL; break; } \
    default: { constexpr int PF = 0; CALL; break; }    \
  }

// Keep flags looked up by edge id at random are packed into bits first (L2-resident); the scratch words come from and
// return to the stream-ordered pool.  Not for the in-order of a canonically numbered graph (its byte lookups are
// coalesced), and not for keep alone: the byte lookup is cheaper than pack + bit lookup there (measured).
struct KeepBits {
  uint32_t* p = nullptr;
  cudaStream_t st = nullptr;
  ~KeepBits() { if (p) cudaFreeAsync(p, st); }
};
static int pack_keep_bits(const botgat_graph* g, const int32_t* eid, const uint8_t* keep, bool with_records, cudaStream_t st,
                          KeepBits* kb) {
  const bool coalesced = eid == g->in_eid && g->in_eid_identity;
  if (!keep || !with_records || g->n_edges < (1 << 20) || coalesced) return 0;
  kb->st = st;
  BG_CHECK(cudaMallocAsync(&kb->p, sizeof(uint32_t) * (size_t)((g->n_edges + 31) / 32), st));
  k_pack_keep<<<grid_for(g->n_edges), 256, 0, st>>>(g->n_edges, keep, kb->p);
  BG_LAUNCHED(1);
  return 0;
}

// the kept adjacency of one CSR order (botgat_edge_subset) except its indices / eid, which the staging pass writes
static int build_subset(const botgat_graph* g, int order, const uint8_t* keep, const uint32_t* keep_bits,
                        botgat_edge_subset* s, cudaStream_t st) {
  const bool in = order == BOTGAT_ORDER_IN;
  const int32_t* eid = in ? g->in_eid : g->out_eid;
  const botgat_graph::SegTable& seg = in ? g->seg_in : g->seg_out;
  const int n_rows = (int)(in ? g->n_dst : g->n_src);
  const int n_seg = seg.n_items;
  const int64_t n_words = g->n_edges / 32 + 1;
  k_kept_bits<<<grid_for(n_words * 32), 256, 0, st>>>(g->n_edges, n_words, in && g->in_eid_identity ? nullptr : eid, keep,
                                                      keep_bits, s->kept);
  BG_LAUNCHED(1);
  auto counts = thrust::make_transform_iterator(thrust::counting_iterator<int64_t>(0), WordCount{s->kept});
  size_t tb = 0;
  BG_CHECK(cub::DeviceScan::ExclusiveSum(nullptr, tb, counts, s->base, (int)n_words, st));
  void* tmp = nullptr;
  BG_CHECK(cudaMallocAsync(&tmp, tb, st));
  const cudaError_t scan = cub::DeviceScan::ExclusiveSum(tmp, tb, counts, s->base, (int)n_words, st);
  BG_LAUNCHED(1);
  BG_CHECK(cudaFreeAsync(tmp, st));
  BG_CHECK(scan);
  const KeptMap km{s->kept, s->base};
  k_subset_bounds<<<grid_for(std::max(n_rows + 1, n_seg)), 256, 0, st>>>(n_rows, in ? g->in_indptr : g->out_indptr, n_seg,
                                                                        seg.beg, seg.end, km, s->indptr, s->seg_beg,
                                                                        s->seg_end);
  BG_LAUNCHED(1);
  BG_CHECK(cudaGetLastError());
  return 0;
}

// `sub` (optional): write compacted through its kept positions; the adjacency entries go with the first head block
static int stage_one(const botgat_graph* g, const int32_t* eid, const int32_t* order, int H, const float* src, int64_t ld,
                     const uint8_t* keep, float* dst, const botgat_edge_subset* sub, const int32_t* indices,
                     cudaStream_t st) {
  const int pf = env_pf();
  KeepBits kb;
  if (int rc = pack_keep_bits(g, eid, keep, src != nullptr, st, &kb)) return rc;
  const uint32_t* keep_bits = kb.p;
  const KeptMap km{sub ? sub->kept : nullptr, sub ? sub->base : nullptr};
  for (int h0 = 0; h0 < H; h0 += kHMax) {
    const int Hn = std::min(kHMax, H - h0);
    const int vec = src ? record_vec(src + h0, ld, Hn) : 1;
    int32_t* sub_indices = sub && indices && h0 == 0 ? sub->indices : nullptr;
    int32_t* sub_eid = sub_indices ? sub->eid : nullptr;
    // cache-blocked traversal: ONE position per thread and no grid-stride loop, so that the blocks resident at any
    // time cover one contiguous window of the visiting order (a grid-stride loop would interleave ~30 far-apart
    // windows, i.e. ~30 tiles, and the L2 would hold none of them)
    const int grid = order ? (int)((g->n_edges + 255) / 256) : grid_for(g->n_edges);
#define BG_ST(VEC) BG_PF_SWITCH((k_edge_stage<VEC, PF><<<grid, 256, 0, st>>>(g->n_edges, h0, Hn, eid, order, src, ld, keep, keep_bits, dst, km, indices, sub_indices, sub_eid)))
    if (vec == 4) { BG_ST(4) } else if (vec == 2) { BG_ST(2) } else { BG_ST(1) }
#undef BG_ST
    BG_LAUNCHED(1);
    BG_CHECK(cudaGetLastError());
  }
  return 0;
}

}  // namespace botgat

using namespace botgat;

extern "C" int botgat_edge_stage(const botgat_graph* g, int order, int32_t H, const float* ee, int64_t ld_ee,
                                 const uint8_t* keep, const float* attn_mul, int64_t ld_am, float* eb, float* am,
                                 botgat_edge_subset* subset, void* stream) {
  BG_REQUIRE(g && H > 0, "edge_stage: bad arguments");
  BG_REQUIRE(order == BOTGAT_ORDER_IN || order == BOTGAT_ORDER_OUT, "edge_stage: bad order %d", order);
  BG_REQUIRE((eb != nullptr) == (ee != nullptr || keep != nullptr), "edge_stage: eb must be given iff ee or keep is");
  BG_REQUIRE((am != nullptr) == (attn_mul != nullptr), "edge_stage: am must be given iff attn_mul is");
  BG_REQUIRE(!ee || ld_ee >= H, "edge_stage: ld_ee < H");
  BG_REQUIRE(!attn_mul || ld_am >= H, "edge_stage: ld_am < H");
  BG_REQUIRE(!subset || keep, "edge_stage: the kept-edge subset needs keep");
  const bool split = (order == BOTGAT_ORDER_IN ? g->seg_in : g->seg_out).n_items > 0;
  BG_REQUIRE(!subset || (subset->kept && subset->base && subset->indptr && subset->indices &&
                         (!split || (subset->seg_beg && subset->seg_end))),
             "edge_stage: subset needs kept, base, indptr, indices and, for a CSR with split rows, seg_beg / seg_end");
  DeviceGuard guard(g->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (g->n_edges == 0) {
    if (subset)  // every row is empty
      BG_CHECK(cudaMemsetAsync(subset->indptr, 0, sizeof(int32_t) * (size_t)((order == BOTGAT_ORDER_IN ? g->n_dst : g->n_src) + 1), st));
    return 0;
  }
  if (!eb && !am) return 0;
  const int32_t* eid = order == BOTGAT_ORDER_IN ? g->in_eid : g->out_eid;
  const int32_t* visit = order == BOTGAT_ORDER_OUT ? g->out_tile_order : nullptr;
  if (subset) {
    KeepBits kb;
    int rc = pack_keep_bits(g, eid, keep, ee != nullptr, st, &kb);
    if (!rc) rc = build_subset(g, order, keep, kb.p, subset, st);
    if (rc) return rc;
  }
  const int32_t* indices = order == BOTGAT_ORDER_IN ? g->in_indices : g->out_indices;
  if (eb) {
    int rc = stage_one(g, eid, visit, ee ? H : 1, ee, ld_ee, subset ? nullptr : keep, eb, subset, indices, st);
    if (rc) return rc;
  }
  if (am) {
    int rc = stage_one(g, eid, visit, H, attn_mul, ld_am, nullptr, am, subset, nullptr, st);
    if (rc) return rc;
  }
  return 0;
}

extern "C" int botgat_edge_unstage(const botgat_graph* g, int order, int32_t H, const float* gz, float* grad_ee,
                                   int64_t ld_gee, const botgat_edge_subset* subset, void* stream) {
  BG_REQUIRE(g && H > 0, "edge_unstage: bad arguments");
  BG_REQUIRE(order == BOTGAT_ORDER_IN || order == BOTGAT_ORDER_OUT, "edge_unstage: bad order %d", order);
  if (g->n_edges == 0) return 0;
  BG_REQUIRE(gz && grad_ee, "edge_unstage: null gz/grad_ee");
  BG_REQUIRE(ld_gee >= H, "edge_unstage: ld_gee < H");
  BG_REQUIRE(!subset || (subset->kept && subset->base), "edge_unstage: subset without kept / base");
  DeviceGuard guard(g->device);
  cudaStream_t st = (cudaStream_t)stream;
  const int32_t* eid = order == BOTGAT_ORDER_IN ? g->in_eid : g->out_eid;
  const int32_t* visit = order == BOTGAT_ORDER_OUT ? g->out_tile_order : nullptr;
  const KeptMap km{subset ? subset->kept : nullptr, subset ? subset->base : nullptr};
  for (int h0 = 0; h0 < ld_gee; h0 += kHMax) {
    const int Hn = std::max(0, std::min(kHMax, H - h0));              // heads in this pass
    const int Hw = (int)std::min<int64_t>(kHMax, ld_gee - h0);        // floats written (heads + zeroed padding)
    const int vec = record_vec(grad_ee + h0, ld_gee, Hw);
    const int grid = visit ? (int)((g->n_edges + 255) / 256) : grid_for(g->n_edges);  // see stage_one
    if (vec == 4) k_edge_unstage<4><<<grid, 256, 0, st>>>(g->n_edges, h0, Hn, Hw, eid, visit, km, gz, grad_ee, ld_gee);
    else if (vec == 2) k_edge_unstage<2><<<grid, 256, 0, st>>>(g->n_edges, h0, Hn, Hw, eid, visit, km, gz, grad_ee, ld_gee);
    else k_edge_unstage<1><<<grid, 256, 0, st>>>(g->n_edges, h0, Hn, Hw, eid, visit, km, gz, grad_ee, ld_gee);
    BG_LAUNCHED(1);
    BG_CHECK(cudaGetLastError());
  }
  return 0;
}

extern "C" int botgat_edge_reduce_dst(const botgat_graph* g, int32_t H, const float* grad_ee, int64_t ld_gee,
                                      float* grad_er, float* scratch, void* stream) {
  BG_REQUIRE(g && H > 0 && grad_er, "edge_reduce_dst: bad arguments");
  BG_REQUIRE(grad_ee || g->n_edges == 0, "edge_reduce_dst: null grad_ee");
  BG_REQUIRE(ld_gee >= H || g->n_edges == 0, "edge_reduce_dst: ld_gee < H");
  if (g->n_dst == 0) return 0;
  DeviceGuard guard(g->device);
  cudaStream_t st = (cudaStream_t)stream;
  const int pf = env_pf();
  const botgat_graph::SegTable& seg = g->seg_in;
  const bool split = seg.n_items > 0;
  BG_REQUIRE(!split || seg.n_slots == 0 || scratch, "edge_reduce_dst: this graph has split rows; scratch (n_slots_in*H floats) is required");
  const int n_items = split ? seg.n_items : (int)g->n_dst;
  const int32_t *sr = split ? seg.row : nullptr, *sb = seg.beg, *se = seg.end, *ss = seg.slot;
  const int grid = (n_items + 7) / 8;
  for (int h0 = 0; h0 < H; h0 += kHMax) {
    const int Hn = std::min(kHMax, H - h0);
    const int vec = g->n_edges ? record_vec(grad_ee + h0, ld_gee, Hn) : 1;
#define BG_RD(VEC) BG_PF_SWITCH((k_edge_reduce_dst<VEC, PF><<<grid, 256, 0, st>>>(n_items, H, h0, Hn, g->in_indptr, g->in_eid, sr, sb, se, ss, grad_ee, ld_gee, grad_er, scratch)))
    if (vec == 4) { BG_RD(4) } else if (vec == 2) { BG_RD(2) } else { BG_RD(1) }
#undef BG_RD
    BG_LAUNCHED(1);
    BG_CHECK(cudaGetLastError());
  }
  if (split && seg.n_split > 0) {
    const int n = seg.n_split * H;
    k_edge_reduce_combine<<<(n + 255) / 256, 256, 0, st>>>(seg.n_split, H, seg.split_rows, seg.split_first, scratch, grad_er);
    BG_LAUNCHED(1);
    BG_CHECK(cudaGetLastError());
  }
  return 0;
}
