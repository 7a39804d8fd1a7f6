// Backward src pass with TMA-staged rows (sm_100a).  Same math and operand conventions as gat_bwd_src_kernel
// (gat_bwd.cu; the adjoint of src/no-sampling/models.py:523-555 / src/ogbn-proteins/models.py:125-156 on the
// reversed graph), different data movement:
//
//   * the g'[v] rows of a source row's out-neighbours are fetched by the tensor-memory accelerator,
//     `cp.async.bulk.tensor.2d ... tile::gather4` (SASS UTMALDG.2D.GATHER4: FOUR table rows per request), into a
//     double-buffered shared-memory ring of 32-row chunks, completion on an mbarrier.  No registers hold rows in
//     flight and no load-address arithmetic is issued, so the next chunk travels while the FMA chains of the
//     current one run (the LDG kernel spends 47 % of its stall samples on its own loads, profiles/r02_src_ldg_*).
//   * one warp per block: every shared-memory address is a compile-time constant and the head width is a template
//     argument, so a row vector is ONE LDS.128 with an immediate offset.
//   * lanes-per-neighbour is chosen so that D/4 vectors divide evenly (G = 4 at D = 80: no idle slots, where the
//     LDG kernel needs G = 8 to read whole 128-byte lines), and both FMA streams (acc += w*x and <ft[u], x>) are
//     packed `fma.rn.f32x2` (FFMA2) on the 64-bit halves of the LDS.128 results.
#include <cuda.h>  // CUtensorMap (types only: the encoder is fetched through cudaGetDriverEntryPoint)

#include <type_traits>

#include "common.cuh"
#include "params.cuh"

namespace botgat {

#ifndef BG_TMA_MINB
#define BG_TMA_MINB 12  // register cap only (<= 168); residency is set by the 2 x 32 x D x 4 bytes of ring per warp
#endif
constexpr int kTmaStages = 2;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint64_t pack2(float a, float b) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ void unpack2(uint64_t v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ void fma2(uint64_t& d, uint64_t a, uint64_t b) { asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(d) : "l"(a), "l"(b)); }
__device__ __forceinline__ float sum2(uint64_t a, uint64_t b) {
  uint64_t t;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(t) : "l"(a), "l"(b));
  float lo, hi;
  unpack2(t, lo, hi);
  return lo + hi;
}
__device__ __forceinline__ void lds128(uint32_t addr, uint64_t& a, uint64_t& b) {
  asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "r"(addr));
}

// DV = D / 4 (float4 vectors per head row), G = 1 << GSH lanes per neighbour (4 or 8).
// MODE selects the operand set at compile time, so that the optional-operand tests (and, in mode 1, the edge-id stream)
// fold away — ~50 of the ~420 instructions per 32-edge chunk:
//   1  the common staged backward: logit term `eb` and `gz` in out-CSR order, nothing else
//   2  nothing addressed by edge id: optional `eb` / `am` / `gz` in out-CSR order, optional in-kernel Philox dropout
//   0  everything (operands by edge id: ee, keep, attn_mul, gz_e)
template <int DV, int GSH, int MODE>
__global__ void __launch_bounds__(32, BG_TMA_MINB) gat_bwd_src_tma_kernel(const BwdParams p, const __grid_constant__ CUtensorMap tmap) {
  constexpr int G = 1 << GSH;           // lanes per neighbour = steps per 32-neighbour chunk
  constexpr int RPS = 32 >> GSH;        // neighbour rows per step (a multiple of the 4 rows of one request)
  constexpr int VPL = (DV + G - 1) / G; // float4 slots per lane
  constexpr int ROWB = DV * 16;         // bytes of one staged row
  constexpr int STAGEB = 32 * ROWB;
  constexpr int D = DV * 4;
  constexpr bool kRagged = VPL * G != DV;  // the last slot is owned by only some lanes of a group
  constexpr bool kStaged = MODE == 1, kNoEid = MODE != 0;
  static_assert(RPS >= 4 && G >= 2, "a step must cover whole gather4 requests");
  __shared__ __align__(128) unsigned char ring[kTmaStages * STAGEB];
  __shared__ __align__(8) uint64_t bars[kTmaStages];
  const int lane = threadIdx.x;
  uint32_t ring0 = smem_u32(ring), bar0 = smem_u32(bars);
  // opaque from here on: otherwise every use re-derives the window address (S2UR CgaCtaId + ULEA) on the uniform path
  asm volatile("" : "+r"(ring0), "+r"(bar0));
  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < kTmaStages; ++s) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0 + 8 * s));
  }
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncwarp();

  const int hl = blockIdx.x / p.n_items;
  const int item = blockIdx.x - hl * p.n_items;
  const int h = hl + p.h_begin;
  // heavy rows are split into segments (segments.cu): a work item is then a segment whose partial result goes to a slot
  const int row = p.seg_row ? p.seg_row[item] : item;
  const int slot = p.seg_row ? p.seg_slot[item] : -1;
  const int grp = lane >> GSH, l = lane & (G - 1);
  const bool act_last = l + (VPL - 1) * G < DV;
  // byte offset of this lane's slot 0 inside a stage; the last slot of a lane that does not own it re-reads slot 0
  // (finite values against fu = 0 and an accumulator that is never stored)
  const uint32_t lane_off = (uint32_t)(grp * ROWB + l * 16);
  const uint32_t last_off = lane_off + ((!kRagged || act_last) ? (uint32_t)((VPL - 1) * G * 16) : 0u);

  const int beg = p.seg_row ? p.seg_beg[item] : p.indptr[row];
  const int end = p.seg_row ? p.seg_end[item] : p.indptr[row + 1];
  const float slope = p.slope;
  const float csu = p.cs ? p.cs[row] : 1.f;
  const float el_u = p.el[(int64_t)row * p.H + h];
  uint64_t fu[VPL][2], acc[VPL][2];
  {
    const float4* f = reinterpret_cast<const float4*>(p.ft + (int64_t)row * p.ld_ft + h * D) + l;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (i < VPL - 1 || act_last) v = __ldg(f + i * G);
      fu[i][0] = pack2(v.x * csu, v.y * csu);
      fu[i][1] = pack2(v.z * csu, v.w * csu);
      acc[i][0] = acc[i][1] = 0ull;  // the bit pattern of (0.f, 0.f)
    }
  }
  const float4* __restrict__ drec_h = p.drec + (int64_t)h * p.n_dst;  // head-major records (BwdParams::drec)
  const float* __restrict__ eb_h = (kStaged || p.eb) ? p.eb + (int64_t)(p.Hb == 1 ? 0 : h) * p.n_edges : nullptr;
  const float* __restrict__ am_h = (!kStaged && p.am) ? p.am + (int64_t)h * p.n_edges : nullptr;
  float* __restrict__ gz_h = (kStaged || p.gz) ? p.gz + (int64_t)h * p.n_edges : nullptr;
  const float* __restrict__ ee_h = (!kNoEid && p.ee) ? p.ee + h : nullptr;
  const float* __restrict__ amul_h = (!kNoEid && p.amul_e) ? p.amul_e + h : nullptr;
  const uint8_t* __restrict__ keep = kNoEid ? nullptr : p.keep;
  float* __restrict__ gze_h = (!kNoEid && p.gz_e) ? p.gz_e + h : nullptr;
  const int H = p.H;
  const bool philox = !kStaged && (p.am == nullptr) && (kNoEid || p.amul_e == nullptr) && p.attn_p > 0.f;
  const bool need_eid = !kStaged && (ee_h || amul_h || keep || philox || gze_h);
  float gel_lane = 0.f;
  const int col0 = h * D;

  auto load_index = [&](int base, int& v) {
    const int pos = base + lane;
    v = 0;  // past the row end: row 0, a valid row (its weight is 0)
    if (pos < end) v = __ldg(p.indices + pos);
  };
  auto load_eid = [&](int base, int& k) {
    const int pos = base + lane;
    k = 0;
    if (need_eid && pos < end) k = __ldg(p.eid + pos);
  };
  auto load_operands = [&](int base, int v, int k, SrcOps& o) {
    const int pos = base + lane;
    o.rec = make_float4(0.f, 0.f, 0.f, 0.f);
    o.eb = -INFINITY;  // lanes past the row end behave like dropped edges: alpha = 0
    o.amul = 1.f; o.ame = 1.f; o.amp = 1.f;
    o.ee = 0.f;
    o.kp = 1;
    if (pos < end) {
      o.rec = __ldg(drec_h + v);
      if constexpr (kStaged) {
        o.eb = __ldg(eb_h + pos);
        return;
      }
      o.eb = eb_h ? __ldg(eb_h + pos) : 0.f;
      if (am_h) o.amul = __ldg(am_h + pos);
      if constexpr (!kNoEid) {
        if (ee_h) o.ee = __ldg(ee_h + (int64_t)k * H);
        if (keep) o.kp = __ldg(keep + k);
        if (amul_h) o.ame = __ldg(amul_h + (int64_t)k * H);
      }
      if (philox) o.amp = philox_dropout_mul(p.seed, (uint32_t)k, (uint32_t)h, p.attn_p, p.inv_keep);
    }
  };
  // Fetch the chunk starting at `base` (lane j holds the row id of neighbour base + j) into stage `s`.  Requests
  // cover whole steps, so that every row a step reads has been written by this chunk's requests.
  auto issue = [&](int base, int vtx, uint32_t s) {
    const int cnt = min(32, end - base);
    const int rows = (cnt + RPS - 1) & ~(RPS - 1);
    const uint32_t bar = bar0 + 8 * s;
    if (lane == 0) asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(rows * ROWB) : "memory");
    const int b = (lane & 7) * 4;
    const int r0 = __shfl_sync(kFull, vtx, b), r1 = __shfl_sync(kFull, vtx, b + 1);
    const int r2 = __shfl_sync(kFull, vtx, b + 2), r3 = __shfl_sync(kFull, vtx, b + 3);
    if (lane * 4 < rows)
      asm volatile(
          "cp.async.bulk.tensor.2d.shared::cta.global.tile::gather4.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];" ::
              "r"(ring0 + s * STAGEB + lane * (4 * ROWB)), "l"(&tmap), "r"(col0), "r"(r0), "r"(r1), "r"(r2), "r"(r3), "r"(bar)
          : "memory");
  };

  float w_lane = 0.f;
  float part[G];
  uint32_t it = 0;  // chunk counter: stage = it & 1, barrier phase parity = (it >> 1) & 1
  // one step: RPS neighbours, one per lane group
  auto step = [&](uint32_t a0, uint32_t a1, int st) {
    uint64_t x[VPL][2];
    const float w = __shfl_sync(kFull, w_lane, st * RPS + grp);
#pragma unroll
    for (int i = 0; i < VPL; ++i) lds128(((kRagged && i == VPL - 1) ? a1 : a0 + i * (G * 16)) + st * (RPS * ROWB), x[i][0], x[i][1]);
    const uint64_t w2 = pack2(w, w);
    uint64_t da = 0ull, db = 0ull;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      fma2(acc[i][0], w2, x[i][0]);
      fma2(acc[i][1], w2, x[i][1]);
      fma2(da, fu[i][0], x[i][0]);  // fu is 0 on a slot this lane does not own
      fma2(db, fu[i][1], x[i][1]);
    }
    part[st] = sum2(da, db);
  };

  int vtx0, vtx1, vtx2, vtx3 = 0, k0, k1, k2 = 0;
  load_index(beg, vtx0);
  load_index(beg + 32, vtx1);
  load_index(beg + 64, vtx2);
  load_eid(beg, k0);
  load_eid(beg + 32, k1);
  if (beg < end) issue(beg, vtx0, 0);
  if (beg + 32 < end) issue(beg + 32, vtx1, 1);
  SrcOps o0, o1;
  load_operands(beg, vtx0, k0, o0);

  for (int base = beg; base < end; base += 32, ++it) {
    const int cnt = min(32, end - base);
    load_index(base + 96, vtx3);
    load_eid(base + 64, k2);
    load_operands(base + 32, vtx1, k1, o1);

    // lane = neighbour: recompute the attention weight of this edge
    const float z = el_u + o0.rec.x + o0.logit_term();
    const float s = leaky_relu(z, slope);
    const float alpha = (s == -INFINITY) ? 0.f : __expf(s - o0.rec.y) * o0.rec.z;
    const float dz = z > 0.f ? 1.f : slope;
    const float am0 = o0.multiplier();
    w_lane = alpha * am0;

    const uint32_t stg = it & 1u;
    {
      const uint32_t bar = bar0 + 8 * stg, parity = (it >> 1) & 1u;
      asm volatile(
          "{\n\t.reg .pred q;\n\tLAB_WAIT:\n\tmbarrier.try_wait.parity.shared::cta.b64 q, [%0], %1;\n\t@q bra DONE;\n\tbra LAB_WAIT;\n\tDONE:\n\t}" ::"r"(bar),
          "r"(parity)
          : "memory");
    }
    const uint32_t a0 = ring0 + stg * STAGEB + lane_off, a1 = ring0 + stg * STAGEB + last_off;
    if (cnt == 32) {
#pragma unroll
      for (int st = 0; st < G; ++st) step(a0, a1, st);
    } else {
#pragma unroll
      for (int st = 0; st < G; ++st) {
        part[st] = 0.f;
        if (st * RPS < cnt) step(a0, a1, st);
      }
    }
    __syncwarp();  // every lane is done with the stage before it is refilled
    if (base + 64 < end) issue(base + 64, vtx2, stg);

    // Packed butterfly over the G lanes of a group: at every level a lane hands half of its live partial dots to its
    // partner.  Afterwards lane (grp, l) holds the dot of step l, neighbour grp of the step; one indexed shuffle
    // hands every neighbour's dot to the lane that owns the neighbour.
    int k = G;
#pragma unroll
    for (int o = G >> 1; o > 0; o >>= 1) {
      const bool upper = (lane & o) != 0;
#pragma unroll
      for (int i = 0; i < G / 2; ++i) {
        if (i < k / 2) {
          const float send = upper ? part[i] : part[i + k / 2];
          const float keepv = upper ? part[i + k / 2] : part[i];
          part[i] = keepv + __shfl_xor_sync(kFull, send, o);
        }
      }
      k >>= 1;
    }
    const float d_lane = __shfl_sync(kFull, part[0], (lane & (RPS - 1)) * G + lane / RPS);
    // d_lane = <src_scale*ft[u], g'[v]>; softmax + leaky_relu adjoint (App. A.3)
    const float gz = alpha * (d_lane * am0 - o0.rec.w) * dz;
    if ((kStaged || gz_h) && lane < cnt) gz_h[base + lane] = gz;
    if (!kNoEid && gze_h && lane < cnt) gze_h[(int64_t)k0 * H] = gz;
    gel_lane += gz;
    vtx0 = vtx1; vtx1 = vtx2; vtx2 = vtx3; k0 = k1; k1 = k2; o0 = o1;
  }

  float4 r[VPL];
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    unpack2(acc[i][0], r[i].x, r[i].y);
    unpack2(acc[i][1], r[i].z, r[i].w);
#pragma unroll
    for (int o = G; o < 32; o <<= 1) {
      r[i].x += __shfl_xor_sync(kFull, r[i].x, o); r[i].y += __shfl_xor_sync(kFull, r[i].y, o);
      r[i].z += __shfl_xor_sync(kFull, r[i].z, o); r[i].w += __shfl_xor_sync(kFull, r[i].w, o);
    }
  }
  const float gel = warp_sum(gel_lane);
  if (slot >= 0) {
    // segment of a split row: partial grad_el and (unscaled) partial grad_ft go to this segment's scratch slot
    float* sl = p.scratch + (int64_t)slot * bwd_slot_floats(p.H, D);
    if (grp == 0) {
      float4* o = reinterpret_cast<float4*>(sl + (int64_t)h * D) + l;
#pragma unroll
      for (int i = 0; i < VPL; ++i)
        if (i < VPL - 1 || act_last) o[i * G] = r[i];
    }
    if (lane == 0) sl[p.H * D + h] = gel;
    return;
  }
  if (grp == 0) {
    float4* o = reinterpret_cast<float4*>(p.grad_ft + (int64_t)row * p.ld_gft + h * D) + l;
#pragma unroll
    for (int i = 0; i < VPL; ++i)
      if (i < VPL - 1 || act_last) o[i * G] = make_float4(r[i].x * csu, r[i].y * csu, r[i].z * csu, r[i].w * csu);
  }
  if (lane == 0) p.grad_el[(int64_t)row * p.H + h] = gel;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int launch_src_tma(const BwdParams& p, const SrcPlan& plan, cudaStream_t st) {
  static EncodeTiledFn encode = nullptr;
  if (!encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn) {
      cudaGetLastError();
      BG_REQUIRE(false, "backward: driver entry point cuTensorMapEncodeTiled not found");
    }
    encode = (EncodeTiledFn)fn;
  }
  CUtensorMap tmap;
  cuuint64_t gdim[2] = {(cuuint64_t)p.ld_g, (cuuint64_t)p.n_dst};
  cuuint64_t gstride[1] = {(cuuint64_t)p.ld_g * 4};
  cuuint32_t box[2] = {(cuuint32_t)p.D, 1};  // tile::gather4: a box of ONE row, four row coordinates per request
  cuuint32_t estr[2] = {1, 1};
  const CUresult cr = encode(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)p.g, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                             CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  BG_REQUIRE(cr == CUDA_SUCCESS, "backward: cuTensorMapEncodeTiled failed (CUresult %d) for D=%d", (int)cr, p.D);
  const bool launched = with_tma_combo(plan.tma_dv, plan.tma_gsh, [&](auto dv, auto gsh) {
    if (plan.tma_mode == 1)
      gat_bwd_src_tma_kernel<dv.value, gsh.value, 1><<<plan.grid, 32, 0, st>>>(p, tmap);
    else if (plan.tma_mode == 2)
      gat_bwd_src_tma_kernel<dv.value, gsh.value, 2><<<plan.grid, 32, 0, st>>>(p, tmap);
    else
      gat_bwd_src_tma_kernel<dv.value, gsh.value, 0><<<plan.grid, 32, 0, st>>>(p, tmap);
  });
  BG_REQUIRE(launched, "backward: no TMA kernel for D=%d lanes=%d", 4 * plan.tma_dv, 1 << plan.tma_gsh);
  BG_LAUNCHED(1);
  return 0;
}

}  // namespace botgat
