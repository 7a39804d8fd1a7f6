// Shared host/device helpers for libbotgat (sm_100a only).
#pragma once

#include <atomic>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <type_traits>

#include "botgat.h"

namespace botgat {

void set_error(const char* fmt, ...);
// host (plan.cu): environment variables; an unset or empty one reads as null / `dflt`
const char* env_str(const char* name);
int64_t env_int(const char* name, int64_t dflt);
extern std::atomic<long long> g_launches;  // kernels launched by this library (botgat_launch_count)
#define BG_LAUNCHED(n) (::botgat::g_launches.fetch_add(n, std::memory_order_relaxed))

#define BG_CHECK(expr)                                                                  \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess) {                                                            \
      ::botgat::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return -2;                                                                        \
    }                                                                                   \
  } while (0)

#define BG_REQUIRE(cond, ...)            \
  do {                                   \
    if (!(cond)) {                       \
      ::botgat::set_error(__VA_ARGS__);  \
      return -1;                         \
    }                                    \
  } while (0)

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (dev != prev) cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    int cur;
    cudaGetDevice(&cur);
    if (cur != prev && prev >= 0) cudaSetDevice(prev);
  }
};

// Grid of a grid-stride streaming kernel: whole waves of resident blocks (occupancy x SM count), never more
// blocks than there is work for.  A partial last wave costs a full wave's time on these bandwidth-bound loops.
template <typename K>
static inline int resident_grid(K kernel, int block_threads, int64_t blocks_of_work) {
  int dev = 0, sms = 148, per_sm = 1;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, block_threads, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
  const int64_t resident = (int64_t)sms * per_sm;
  return (int)(blocks_of_work < 1 ? 1 : (blocks_of_work < resident ? blocks_of_work : resident));
}

}  // namespace botgat

// The opaque graph handle.  Immutable after create.
struct botgat_graph {
  int device = 0;
  int sm_count = 148;
  int64_t n_src = 0, n_dst = 0, n_edges = 0;
  int64_t max_in_deg = 0, max_out_deg = 0;
  int has_zero_in_degree = 0;
  int32_t *in_indptr = nullptr, *in_indices = nullptr, *in_eid = nullptr;
  int32_t *out_indptr = nullptr, *out_indices = nullptr, *out_eid = nullptr;
  int32_t *in_deg = nullptr, *out_deg = nullptr;
  // Canonical edge numbering: in_eid[p] == p for every p (the COO came sorted by destination), so edge-ordered
  // operands ARE in in-CSR order and, with the COO sorted by (dst, src), both CSRs have sorted neighbour lists.
  int in_eid_identity = 0;
  // Cache-blocked traversal of the out-CSR for the in <-> out transposes of per-edge records (edge_ops.cu): the
  // out-CSR positions grouped by (source block, destination block), tiles_s x tiles_d blocks; nullptr = plain order.
  int32_t* out_tile_order = nullptr;
  int tiles_s = 1, tiles_d = 1;
  // Row splitting for heavy-tailed degree distributions.  When a CSR has a row longer than the segment length,
  // its work items are SEGMENTS (at most seg_len neighbours of one row) instead of rows: a heavy row is spread over
  // several warps whose partial results go to scratch slots and are merged by a combine kernel.  Empty = no split.
  struct SegTable {
    int n_items = 0;   // segments (>= rows)
    int n_slots = 0;   // segments that are only part of a row (each owns one scratch slot)
    int n_split = 0;   // rows that are split
    int32_t *row = nullptr, *beg = nullptr, *end = nullptr, *slot = nullptr;  // per item
    int32_t *split_rows = nullptr, *split_first = nullptr;                    // per split row (+1 sentinel)
  } seg_in, seg_out;
};

namespace botgat {

#ifndef BG_WPB
#define BG_WPB 4
#endif
constexpr int kWarpsPerBlock = BG_WPB;
constexpr unsigned kFull = 0xffffffffu;

// ---------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------
// -inf (a dropped edge, a lane past the row end) must stay -inf for every slope >= 0: -inf * 0 would be NaN
__device__ __forceinline__ float leaky_relu(float z, float slope) {
  return z > 0.f ? z : (z == -INFINITY ? -INFINITY : z * slope);
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(kFull, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}

// Philox4x32-10 keyed on (seed), counter (eid, head>>2); component head&3.
// Used for the in-kernel ("fast") attention dropout; reproducible from
// (seed, edge id, head) so forward and both backward passes agree.
__device__ __forceinline__ uint32_t philox_u32(uint64_t seed, uint32_t eid, uint32_t head) {
  uint32_t c0 = eid, c1 = head >> 2, c2 = 0x9E3779B9u, c3 = 0xBB67AE85u;
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  uint32_t sel = head & 3u;
  return sel == 0 ? c0 : sel == 1 ? c1 : sel == 2 ? c2 : c3;
}
// multiplier 0 or 1/(1-p); keep iff u >= p with u = (x >> 8) * 2^-24
__device__ __forceinline__ float philox_dropout_mul(uint64_t seed, uint32_t eid, uint32_t head, float p, float inv_keep) {
  float u = (float)(philox_u32(seed, eid, head) >> 8) * (1.0f / 16777216.0f);
  return u >= p ? inv_keep : 0.f;
}

// ---------------------------------------------------------------------------
// VW-wide vectors (VW = 4, 2, 1 floats) with read-only global loads
// ---------------------------------------------------------------------------
template <int VW> struct Vec;
template <> struct Vec<4> {
  float4 v;
  __device__ __forceinline__ void load(const float* p) { v = __ldg(reinterpret_cast<const float4*>(p)); }
  // predicated load straight into the live registers: the value is KEPT when on == 0 (no select, no copy)
  __device__ __forceinline__ void load_if(const float* p, unsigned on) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %5, 0;\n\t@q ld.global.nc.v4.f32 {%0,%1,%2,%3}, [%4];\n\t}"
                 : "+f"(v.x), "+f"(v.y), "+f"(v.z), "+f"(v.w) : "l"(p), "r"(on));
  }
  __device__ __forceinline__ void store(float* p) const { *reinterpret_cast<float4*>(p) = v; }
  __device__ __forceinline__ void zero() { v = make_float4(0.f, 0.f, 0.f, 0.f); }
  __device__ __forceinline__ void fma(float w, const Vec& o) {
    v.x = fmaf(w, o.v.x, v.x); v.y = fmaf(w, o.v.y, v.y); v.z = fmaf(w, o.v.z, v.z); v.w = fmaf(w, o.v.w, v.w);
  }
  __device__ __forceinline__ float dot(const Vec& o, float acc) const {
    acc = fmaf(v.x, o.v.x, acc); acc = fmaf(v.y, o.v.y, acc); acc = fmaf(v.z, o.v.z, acc); acc = fmaf(v.w, o.v.w, acc);
    return acc;
  }
  __device__ __forceinline__ void scale(float s) { v.x *= s; v.y *= s; v.z *= s; v.w *= s; }
  __device__ __forceinline__ void add(const Vec& o) { v.x += o.v.x; v.y += o.v.y; v.z += o.v.z; v.w += o.v.w; }
  __device__ __forceinline__ void mul(const Vec& o) { v.x *= o.v.x; v.y *= o.v.y; v.z *= o.v.z; v.w *= o.v.w; }
  __device__ __forceinline__ void relu() { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
  __device__ __forceinline__ void add_shfl_xor(int o) {
    v.x += __shfl_xor_sync(kFull, v.x, o); v.y += __shfl_xor_sync(kFull, v.y, o);
    v.z += __shfl_xor_sync(kFull, v.z, o); v.w += __shfl_xor_sync(kFull, v.w, o);
  }
};
template <> struct Vec<2> {
  float2 v;
  __device__ __forceinline__ void load(const float* p) { v = __ldg(reinterpret_cast<const float2*>(p)); }
  __device__ __forceinline__ void load_if(const float* p, unsigned on) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %3, 0;\n\t@q ld.global.nc.v2.f32 {%0,%1}, [%2];\n\t}"
                 : "+f"(v.x), "+f"(v.y) : "l"(p), "r"(on));
  }
  __device__ __forceinline__ void store(float* p) const { *reinterpret_cast<float2*>(p) = v; }
  __device__ __forceinline__ void zero() { v = make_float2(0.f, 0.f); }
  __device__ __forceinline__ void fma(float w, const Vec& o) { v.x = fmaf(w, o.v.x, v.x); v.y = fmaf(w, o.v.y, v.y); }
  __device__ __forceinline__ float dot(const Vec& o, float acc) const {
    acc = fmaf(v.x, o.v.x, acc); acc = fmaf(v.y, o.v.y, acc);
    return acc;
  }
  __device__ __forceinline__ void scale(float s) { v.x *= s; v.y *= s; }
  __device__ __forceinline__ void add(const Vec& o) { v.x += o.v.x; v.y += o.v.y; }
  __device__ __forceinline__ void mul(const Vec& o) { v.x *= o.v.x; v.y *= o.v.y; }
  __device__ __forceinline__ void relu() { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); }
  __device__ __forceinline__ void add_shfl_xor(int o) {
    v.x += __shfl_xor_sync(kFull, v.x, o); v.y += __shfl_xor_sync(kFull, v.y, o);
  }
};
template <> struct Vec<1> {
  float v;
  __device__ __forceinline__ void load(const float* p) { v = __ldg(p); }
  __device__ __forceinline__ void load_if(const float* p, unsigned on) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %2, 0;\n\t@q ld.global.nc.f32 %0, [%1];\n\t}"
                 : "+f"(v) : "l"(p), "r"(on));
  }
  __device__ __forceinline__ void store(float* p) const { *p = v; }
  __device__ __forceinline__ void zero() { v = 0.f; }
  __device__ __forceinline__ void fma(float w, const Vec& o) { v = fmaf(w, o.v, v); }
  __device__ __forceinline__ float dot(const Vec& o, float acc) const { return fmaf(v, o.v, acc); }
  __device__ __forceinline__ void scale(float s) { v *= s; }
  __device__ __forceinline__ void add(const Vec& o) { v += o.v; }
  __device__ __forceinline__ void mul(const Vec& o) { v *= o.v; }
  __device__ __forceinline__ void relu() { v = fmaxf(v, 0.f); }
  __device__ __forceinline__ void add_shfl_xor(int o) { v += __shfl_xor_sync(kFull, v, o); }
};

// ---------------------------------------------------------------------------
// Work decomposition shared by the forward and the backward gather pass.
//
// A work item is (head h, column part cp, CSR row r) and is owned by one warp.
// Items are ordered head-major, then column part, then row, so that all warps
// resident at one time gather from the same (N x part_cols) slab of the feature
// table — a slab is sized to stay L2-resident (DESIGN.md "Slabs").
//
// Inside the warp, a group of G = 1<<gshift lanes serves one neighbour; lane j of
// the group owns vectors (i*G + j - o), i = 0..VPL-1, of the slab row (VW floats
// each), so one warp instruction covers 32/G neighbours.  G is chosen so that one
// group reads one 128-byte line per instruction, and `o` (lanes) shifts the
// mapping so that each instruction's piece is line-ALIGNED even when the slab
// starts mid-line (odd heads at D=80): an L1 wavefront then carries a full line.
// ---------------------------------------------------------------------------
struct Tiling {
  int vw;         // floats per vector (4, 2 or 1)
  int vpl;        // vector slots per lane
  int gshift;     // log2(lanes per neighbour)
  int col_parts;  // parts per head
  int part_cols;  // floats per part (last part may be shorter)
  int omask;      // lane-offset mask: o = (first vector index of the slab) & omask; 0 = no alignment shift
};

// host (segments.cu): build / free the segment table of one CSR; a no-op when no row exceeds the segment length
int build_segments(int n_rows, const int32_t* indptr, const int32_t* deg, int64_t max_deg, botgat_graph::SegTable* t,
                   cudaStream_t st);
void free_segments(botgat_graph::SegTable* t, bool async, cudaStream_t st);

// steps (of 32/G neighbours each) whose row loads a lane keeps in flight together.
// Measured on B200 (profiles/r01_*): at D=80 (3 slots) two steps at 3 blocks/SM beat four steps at 2 blocks/SM.
#ifdef BG_NS
__host__ __device__ constexpr int steps_in_flight(int vpl) { return BG_NS; }
#else
__host__ __device__ constexpr int steps_in_flight(int vpl) { return vpl <= 1 ? 4 : vpl <= 2 ? 3 : vpl <= 4 ? 2 : 1; }
#endif

// Resident blocks per SM the gather kernels are compiled for (= their register cap: 65536 / (128 threads x blocks)).
// The narrow instantiations run at the occupancy the sweeps chose (profiles/r01_sweeps.md: forward 6 blocks, backward
// src pass 4); the wide ones (>= 4 / 5 vector slots per lane: D >= 128 at 8 lanes per neighbour, the arxiv D = 250
// path) get the registers their accumulators need instead of spilling them (round 1: up to 628 bytes of local loads
// per thread in gat_fwd_kernel<4,5,8>).  -DBG_MINB / -DBG_MINB_BWD override the narrow figure for sweeps.
#ifndef BG_MINB
#define BG_MINB 6
#endif
#ifndef BG_MINB_BWD
#define BG_MINB_BWD 4
#endif
#ifndef BG_MINB4
#define BG_MINB4 5
#endif
__host__ __device__ constexpr int fwd_min_blocks(int vpl) { return vpl <= 3 ? BG_MINB : vpl == 4 ? (BG_MINB < BG_MINB4 ? BG_MINB : BG_MINB4) : vpl <= 6 ? 4 : 3; }
__host__ __device__ constexpr int bwd_min_blocks(int vpl) { return vpl <= 3 ? BG_MINB_BWD : vpl <= 5 ? (BG_MINB_BWD < 3 ? BG_MINB_BWD : 3) : 2; }

// (vector width, log2 lanes per neighbour, slots per lane) combinations the gather kernels are instantiated
// for; choose_tiling() only returns members of this set.
#define BG_VPL_SMALL(X, VW, GSH) X(VW, GSH, 1) X(VW, GSH, 2)
#define BG_VPL_FULL(X, VW, GSH) X(VW, GSH, 1) X(VW, GSH, 2) X(VW, GSH, 3) X(VW, GSH, 4) X(VW, GSH, 5) X(VW, GSH, 6) X(VW, GSH, 7) X(VW, GSH, 8)
#define BG_VPL_BIG(X, VW, GSH) X(VW, GSH, 5) X(VW, GSH, 6) X(VW, GSH, 7) X(VW, GSH, 8)
#define BG_COMBOS(X)                                                                                        \
  BG_VPL_SMALL(X, 4, 0) BG_VPL_SMALL(X, 4, 1) BG_VPL_SMALL(X, 4, 2) BG_VPL_FULL(X, 4, 3) BG_VPL_BIG(X, 4, 4)   \
  BG_VPL_BIG(X, 4, 5)                                                                                       \
  BG_VPL_SMALL(X, 2, 0) BG_VPL_SMALL(X, 2, 1) BG_VPL_SMALL(X, 2, 2) BG_VPL_SMALL(X, 2, 3) BG_VPL_FULL(X, 2, 4) \
  BG_VPL_BIG(X, 2, 5)                                                                                       \
  BG_VPL_SMALL(X, 1, 0) BG_VPL_SMALL(X, 1, 1) BG_VPL_SMALL(X, 1, 2) BG_VPL_SMALL(X, 1, 3) BG_VPL_SMALL(X, 1, 4) \
  BG_VPL_FULL(X, 1, 5)

// Calls f(VW, GSH, VPL), each a std::integral_constant, for the instantiated combination equal to (vw, gsh, vpl);
// false when there is none.
template <class F>
inline bool with_combo(int vw, int gsh, int vpl, F&& f) {
#define BG_X(VW, GSH, VPL)                                                                                          \
  if (vw == VW && gsh == GSH && vpl == VPL)                                                                         \
    return f(std::integral_constant<int, VW>(), std::integral_constant<int, GSH>(), std::integral_constant<int, VPL>()), true;
  BG_COMBOS(BG_X)
#undef BG_X
  return false;
}

}  // namespace botgat
