// All-heads-per-row variants of the two gather kernels, for tables that cannot be L2-resident
// (ogbn-products: 2.45 M rows x 1920 B = 4.7 GB; one head's slab alone is 1.18 GB).
//
// The head-major kernels (gat_fwd.cu / gat_bwd.cu / gat_bwd_tma.cu) visit a CSR row once per head so that all resident
// warps gather from one (N x D) slab that lives in L2.  When no slab fits, that order only costs: every pass fetches
// a 4*D-byte piece of the row from DRAM (480 B at a 96-byte phase at the products shape: 18 lines touched for 15
// lines of data, ncu 1.34x the row bytes), re-reads the row's indices and pays the row's dependent load chain H times,
// and keeps only 4*D bytes per neighbour in flight (profiles/r02_o_products_*: 72 % of the stall samples on the
// row loads' scoreboard, DRAM at 50 %).  Here ONE warp owns a row for ALL heads:
//   * a group of G = 32 / pow2ceil(H) lanes owns a head, so a warp instruction reads pieces of ONE neighbour's row
//     (4*H*D contiguous bytes, whole lines) instead of pieces of 32/G different neighbours' rows;
//   * the per-edge scalars (logits, softmax terms) are computed lane = edge for all heads and handed to the head
//     groups through shared memory (one broadcast LDS per neighbour);
//   * the per-head reductions over the 32 edges of a chunk use a packed butterfly whose result for head g lands in
//     the lanes of group g — where the accumulators of that head live;
//   * row loads run through a register ring of U neighbours: a neighbour's vectors are re-issued as soon as they are
//     consumed, so 4*H*D*U bytes per warp are in flight continuously.
// Same math, operand conventions, scratch-slot layout (split rows) and determinism as the head-major kernels.
// Staged per-edge operands only (eb / am / gz in CSR order, in-kernel Philox); the edge-id ("direct") operand mode
// stays on the head-major kernels.
#include "common.cuh"
#include "params.cuh"

namespace botgat {

// neighbours whose row vectors a lane keeps in flight (U x VPL float4 registers)
__host__ __device__ constexpr int rw_in_flight(int vpl) { return vpl <= 2 ? 8 : vpl <= 4 ? 4 : 2; }
__host__ __device__ constexpr int rw_in_flight_bwd(int vpl) { return vpl <= 4 ? 4 : 2; }
__host__ __device__ constexpr int rw_fwd_blocks(int vpl) { return vpl <= 4 ? 4 : 3; }
__host__ __device__ constexpr int rw_bwd_blocks(int vpl) { return vpl <= 4 ? 3 : 2; }

// Reduces HG per-lane values over the 32 lanes of the warp: on return lane group g (= lane >> GSH, G = 1 << GSH lanes)
// holds the reduction of v[g] in every one of its lanes.  HG - 1 + GSH shuffles instead of 5 * HG: at each of the first
// log2(HG) levels a lane hands the half of its live values that its partner keeps.  `v` is clobbered.
template <int GSH, bool kMax>
__device__ __forceinline__ float packed_reduce(float (&v)[32 >> GSH], int lane) {
  constexpr int HG = 32 >> GSH;
  int k = HG;
#pragma unroll
  for (int o = 16; o >= (1 << GSH); o >>= 1) {
    if (k > 1) {
      const bool upper = (lane & o) != 0;
#pragma unroll
      for (int i = 0; i < (HG > 1 ? HG / 2 : 1); ++i) {
        if (i < k / 2) {
          const float send = upper ? v[i] : v[i + k / 2];
          const float keep = upper ? v[i + k / 2] : v[i];
          const float got = __shfl_xor_sync(kFull, send, o);
          v[i] = kMax ? fmaxf(keep, got) : keep + got;
        }
      }
      k >>= 1;
    }
  }
#pragma unroll
  for (int o = (1 << GSH) >> 1; o > 0; o >>= 1) {
    const float got = __shfl_xor_sync(kFull, v[0], o);
    v[0] = kMax ? fmaxf(v[0], got) : v[0] + got;
  }
  return v[0];
}

// attention-dropout multipliers of heads hd0 .. hd0 + HG - 1 of one edge: one Philox block per four heads
template <int HG>
__device__ __forceinline__ void philox_heads(uint64_t seed, uint32_t eid, int hd0, int n, float p, float inv_keep, float (&out)[HG]) {
#pragma unroll
  for (int hh = 0; hh < HG; ++hh) out[hh] = hh < n ? philox_dropout_mul(seed, eid, (uint32_t)(hd0 + hh), p, inv_keep) : 1.f;
}

// ---------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------
template <int GSH, int VPL, bool EP>
__global__ void __launch_bounds__(kWarpsPerBlock * 32, rw_fwd_blocks(VPL)) gat_fwd_rowwise_kernel(const FwdParams p) {
  constexpr int G = 1 << GSH;     // lanes per head
  constexpr int HG = 32 >> GSH;   // head groups per warp (>= heads of this launch)
  constexpr int U = rw_in_flight(VPL);
  __shared__ __align__(16) float wsm_all[kWarpsPerBlock][32 * HG];  // float4 stores
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item = blockIdx.x * kWarpsPerBlock + warp;
  if (item >= p.n_items) return;
  float* wsm = wsm_all[warp];
  const int row = p.seg_row ? p.seg_row[item] : item;
  const int slot = p.seg_row ? p.seg_slot[item] : -1;
  const int grp = lane >> GSH, j = lane & (G - 1);
  const int hc = p.h_count;
  const bool hval = grp < hc;
  const int h = p.h_begin + (hval ? grp : hc - 1);  // idle groups shadow the last head (loads stay in the row)
  const int H = p.H, D = p.D;
  const int nv = D >> 2;

  // One base pointer per lane; slot i sits at the compile-time offset i * G * 16 bytes, only the last slot can be ragged:
  // a lane past the head's end re-reads the head's last vector (same line as a neighbouring lane's: no extra sector)
  // into an accumulator that is never stored.  Idle head groups shadow the last head lane for lane (the coalescer
  // merges them).  Row loads are therefore plain unpredicated LDG.128 (a predicated load into a live register makes
  // ptxas load into a temporary and copy — the copy waits on the load right where it was issued).
  bool act[VPL];
#pragma unroll
  for (int i = 0; i < VPL; ++i) act[i] = hval && (j + i * G) < nv;
  const char* bp = reinterpret_cast<const char*>(p.ft + h * D + j * 4);
  const int last_off = (min(j + (VPL - 1) * G, nv - 1) - j) * 16;
  const unsigned ldb = (unsigned)(p.ld_ft * 4);

  const int beg = p.seg_row ? p.seg_beg[item] : p.indptr[row];
  const int end = p.seg_row ? p.seg_end[item] : p.indptr[row + 1];
  const float slope = p.slope;
  const float* __restrict__ el = p.el + p.h_begin;
  const float* __restrict__ eb = p.eb ? p.eb + (int64_t)(p.Hb == 1 ? 0 : p.h_begin) * p.n_edges : nullptr;
  const int64_t eb_hs = p.Hb == 1 ? 0 : p.n_edges;  // head stride of eb
  const float* __restrict__ am = p.am ? p.am + (int64_t)p.h_begin * p.n_edges : nullptr;
  const float* __restrict__ cs = p.cs;
  const bool philox = (p.am == nullptr) && p.attn_p > 0.f;

  const float* __restrict__ er = p.er ? p.er + (int64_t)row * H + p.h_begin : nullptr;
  float m_own = -INFINITY;  // running max and sum of this group's head (group-uniform)
  float l_own = 0.f;
  Vec<4> acc[VPL], x[U][VPL];
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    acc[i].zero();
#pragma unroll
    for (int s = 0; s < U; ++s) x[s][i].zero();
  }

  auto load_index = [&](int base, int& u, int& k) {
    const int pos = base + lane;
    u = k = 0;
    if (pos < end) {
      u = __ldg(p.indices + pos);
      if (philox) k = __ldg(p.eid + pos);
    }
  };
  int u0, u1, k0, k1;
  load_index(beg, u0, k0);
  load_index(beg + 32, u1, k1);

  for (int base = beg; base < end; base += 32) {
    const int cnt = min(32, end - base);
    const int pos = base + lane;
    const bool valid = pos < end;
    int u2, k2;
    load_index(base + 64, u2, k2);

    // the first U neighbours' rows only need the indices: issue them before the logit operands are even requested
#pragma unroll
    for (int s = 0; s < U; ++s) {
      if (s < cnt) {  // warp-uniform
        const char* r = bp + (size_t)(unsigned)__shfl_sync(kFull, u0, s) * ldb;
#pragma unroll
        for (int i = 0; i < VPL; ++i) x[s][i].load(reinterpret_cast<const float*>(r + (i < VPL - 1 ? i * G * 16 : last_off)));
      }
    }

    // ---- lane = edge: logits of every head, online softmax ----
    float sv[HG], mul[HG];
    {
      const float csv = (valid && cs) ? __ldg(cs + u0) : 1.f;
      float elv[HG], ebv[HG], amv[HG];
#pragma unroll
      for (int hh = 0; hh < HG; ++hh) {
        const bool hv = valid && hh < hc;
        elv[hh] = -INFINITY; ebv[hh] = 0.f; amv[hh] = 1.f;
        if (hv) {
          elv[hh] = __ldg(el + (int64_t)u0 * H + hh);
          if (er) elv[hh] += __ldg(er + hh);
          if (eb) ebv[hh] = __ldg(eb + hh * eb_hs + pos);
          if (am) amv[hh] = __ldg(am + (int64_t)hh * p.n_edges + pos);
        }
      }
      if (philox) {
        float pm[HG];
        philox_heads<HG>(p.seed, (uint32_t)k0, p.h_begin, hc, p.attn_p, p.inv_keep, pm);
#pragma unroll
        for (int hh = 0; hh < HG; ++hh) amv[hh] *= pm[hh];
      }
#pragma unroll
      for (int hh = 0; hh < HG; ++hh) {
        sv[hh] = leaky_relu(elv[hh] + ebv[hh], slope);  // -inf: dropped edge / lane past the row end / idle head
        mul[hh] = amv[hh] * csv;
      }
    }
    float red[HG];
#pragma unroll
    for (int hh = 0; hh < HG; ++hh) red[hh] = sv[hh];
    const float m_new = fmaxf(m_own, packed_reduce<GSH, true>(red, lane));
    if (m_new > m_own) {
      const float f = __expf(m_own - m_new);  // m_own == -inf -> 0, and everything accumulated so far is 0
      l_own *= f;
#pragma unroll
      for (int i = 0; i < VPL; ++i) acc[i].scale(f);
      m_own = m_new;
    }
    float wv[HG];
#pragma unroll
    for (int hh = 0; hh < HG; ++hh) {
      const float mh = __shfl_sync(kFull, m_new, hh << GSH);
      red[hh] = (sv[hh] == -INFINITY) ? 0.f : __expf(sv[hh] - mh);
      wv[hh] = red[hh] * mul[hh];
    }
    l_own += packed_reduce<GSH, false>(red, lane);
    if constexpr (HG % 4 == 0) {
#pragma unroll
      for (int q = 0; q < HG / 4; ++q)
        reinterpret_cast<float4*>(wsm + lane * HG)[q] = make_float4(wv[4 * q], wv[4 * q + 1], wv[4 * q + 2], wv[4 * q + 3]);
    } else {
#pragma unroll
      for (int hh = 0; hh < HG; ++hh) wsm[lane * HG + hh] = wv[hh];
    }
    __syncwarp();

    // ---- group = head: acc += w * row, ring of U neighbours ----
    for (int e = 0; e < cnt; e += U) {
#pragma unroll
      for (int s = 0; s < U; ++s) {
        const float w = (e + s < cnt) ? wsm[(e + s) * HG + grp] : 0.f;
#pragma unroll
        for (int i = 0; i < VPL; ++i) acc[i].fma(w, x[s][i]);
        const int nx = e + s + U;  // re-issue this ring slot
        if (nx < cnt) {            // warp-uniform
          const char* r = bp + (size_t)(unsigned)__shfl_sync(kFull, u0, nx) * ldb;
#pragma unroll
          for (int i = 0; i < VPL; ++i) x[s][i].load(reinterpret_cast<const float*>(r + (i < VPL - 1 ? i * G * 16 : last_off)));
        }
      }
    }
    __syncwarp();
    u0 = u1; u1 = u2; k0 = k1; k1 = k2;
  }

  const float l = l_own;
  if (slot >= 0) {
    // segment of a split row: park (max, sum, unnormalised accumulator) in this segment's scratch slot
    float* sl = p.scratch + (int64_t)slot * fwd_slot_floats(H, D);
#pragma unroll
    for (int i = 0; i < VPL; ++i)
      if (act[i]) acc[i].store(sl + (int64_t)h * D + (j + i * G) * 4);
    if (hval && j == 0) { sl[H * D + h * 2] = m_own; sl[H * D + h * 2 + 1] = l; }
    return;
  }
  float scale = l > 0.f ? 1.f / l : 0.f;
  if (p.ds) scale *= p.ds[row];
  float* o = p.out + (int64_t)row * p.ld_out + h * D;
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    if (act[i]) {
      acc[i].scale(scale);
      if constexpr (EP) p.ep.apply(acc[i], row, (int64_t)h * D + (j + i * G) * 4);
      acc[i].store(o + (j + i * G) * 4);
    }
  }
  if (hval && j == 0) {
    p.row_max[(int64_t)row * H + h] = m_own;
    p.row_sum[(int64_t)row * H + h] = l;
  }
}

// ---------------------------------------------------------------------------
// backward src pass
// ---------------------------------------------------------------------------
template <int GSH, int VPL>
__global__ void __launch_bounds__(kWarpsPerBlock * 32, rw_bwd_blocks(VPL)) gat_bwd_src_rowwise_kernel(const BwdParams p) {
  constexpr int G = 1 << GSH;
  constexpr int HG = 32 >> GSH;
  constexpr int U = rw_in_flight_bwd(VPL) <= G ? rw_in_flight_bwd(VPL) : G;  // the packed dot reduction needs U <= G
  constexpr int LPU = G / U;                                                  // lanes of a group per ring slot after it
  __shared__ __align__(16) float wsm_all[kWarpsPerBlock][32 * HG];  // float4 stores
  __shared__ __align__(16) float dsm_all[kWarpsPerBlock][32 * HG];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item = blockIdx.x * kWarpsPerBlock + warp;
  if (item >= p.n_items) return;
  float* wsm = wsm_all[warp];
  float* dsm = dsm_all[warp];
  const int row = p.seg_row ? p.seg_row[item] : item;
  const int slot = p.seg_row ? p.seg_slot[item] : -1;
  const int grp = lane >> GSH, j = lane & (G - 1);
  const int hc = p.h_count;
  const bool hval = grp < hc;
  const int h = p.h_begin + (hval ? grp : hc - 1);
  const int H = p.H, D = p.D;
  const int nv = D >> 2;

  bool act[VPL];
#pragma unroll
  for (int i = 0; i < VPL; ++i) act[i] = hval && (j + i * G) < nv;
  const char* bp = reinterpret_cast<const char*>(p.g + h * D + j * 4);
  const int last_off = (min(j + (VPL - 1) * G, nv - 1) - j) * 16;  // see the forward
  const unsigned ldb = (unsigned)(p.ld_g * 4);

  const int beg = p.seg_row ? p.seg_beg[item] : p.indptr[row];
  const int end = p.seg_row ? p.seg_end[item] : p.indptr[row + 1];
  const float slope = p.slope;
  const float csu = p.cs ? p.cs[row] : 1.f;
  Vec<4> fu[VPL], acc[VPL], x[U][VPL];
  {
    const float* f = p.ft + (int64_t)row * p.ld_ft + h * D;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      if (act[i]) { fu[i].load(f + (j + i * G) * 4); fu[i].scale(csu); } else fu[i].zero();
      acc[i].zero();
#pragma unroll
      for (int s = 0; s < U; ++s) x[s][i].zero();
    }
  }
  float el_u[HG], gel_lane[HG];
#pragma unroll
  for (int hh = 0; hh < HG; ++hh) {
    el_u[hh] = hh < hc ? p.el[(int64_t)row * H + p.h_begin + hh] : 0.f;
    gel_lane[hh] = 0.f;
  }
  const float4* __restrict__ drec = p.drec + (unsigned)(p.h_begin * p.drec_hs);
  const float* __restrict__ eb = p.eb ? p.eb + (int64_t)(p.Hb == 1 ? 0 : p.h_begin) * p.n_edges : nullptr;
  const int64_t eb_hs = p.Hb == 1 ? 0 : p.n_edges;
  const float* __restrict__ am = p.am ? p.am + (int64_t)p.h_begin * p.n_edges : nullptr;
  float* __restrict__ gz = p.gz ? p.gz + (int64_t)p.h_begin * p.n_edges : nullptr;
  const bool philox = (p.am == nullptr) && p.attn_p > 0.f;

  auto load_index = [&](int base, int& v, int& k) {
    const int pos = base + lane;
    v = k = 0;
    if (pos < end) {
      v = __ldg(p.indices + pos);
      if (philox) k = __ldg(p.eid + pos);
    }
  };
  int v0, v1, k0, k1;
  load_index(beg, v0, k0);
  load_index(beg + 32, v1, k1);

  for (int base = beg; base < end; base += 32) {
    const int cnt = min(32, end - base);
    const int pos = base + lane;
    const bool valid = pos < end;
    int v2, k2;
    load_index(base + 64, v2, k2);

#pragma unroll
    for (int s = 0; s < U; ++s) {
      if (s < cnt) {  // warp-uniform
        const char* r = bp + (size_t)(unsigned)__shfl_sync(kFull, v0, s) * ldb;
#pragma unroll
        for (int i = 0; i < VPL; ++i) x[s][i].load(reinterpret_cast<const float*>(r + (i < VPL - 1 ? i * G * 16 : last_off)));
      }
    }

    // ---- lane = edge: recompute the attention weight of this edge for every head ----
    float ca[HG], cb[HG];  // gz = ca * <src_scale * ft[u], g'[v]> - cb   (softmax + leaky_relu adjoint, App. A.3)
    {
      float4 rec[HG];
      float ebv[HG], amv[HG];
#pragma unroll
      for (int hh = 0; hh < HG; ++hh) {
        const bool hv = valid && hh < hc;
        rec[hh] = make_float4(0.f, 0.f, 0.f, 0.f);
        ebv[hh] = -INFINITY;  // lanes past the row end / idle heads behave like dropped edges: alpha = 0
        amv[hh] = 1.f;
        if (hv) {
          rec[hh] = __ldg(drec + (unsigned)(hh * p.drec_hs + v0 * p.drec_vs));
          ebv[hh] = eb ? __ldg(eb + hh * eb_hs + pos) : 0.f;
          if (am) amv[hh] = __ldg(am + (int64_t)hh * p.n_edges + pos);
        }
      }
      if (philox) {
        float pm[HG];
        philox_heads<HG>(p.seed, (uint32_t)k0, p.h_begin, hc, p.attn_p, p.inv_keep, pm);
#pragma unroll
        for (int hh = 0; hh < HG; ++hh) amv[hh] *= pm[hh];
      }
      float wv[HG];
#pragma unroll
      for (int hh = 0; hh < HG; ++hh) {
        const float z = el_u[hh] + rec[hh].x + ebv[hh];
        const float s = leaky_relu(z, slope);
        const float alpha = (s == -INFINITY) ? 0.f : __expf(s - rec[hh].y) * rec[hh].z;
        const float dz = z > 0.f ? 1.f : slope;
        wv[hh] = alpha * amv[hh];
        ca[hh] = wv[hh] * dz;
        cb[hh] = alpha * rec[hh].w * dz;
      }
      if constexpr (HG % 4 == 0) {
#pragma unroll
        for (int q = 0; q < HG / 4; ++q)
          reinterpret_cast<float4*>(wsm + lane * HG)[q] = make_float4(wv[4 * q], wv[4 * q + 1], wv[4 * q + 2], wv[4 * q + 3]);
      } else {
#pragma unroll
        for (int hh = 0; hh < HG; ++hh) wsm[lane * HG + hh] = wv[hh];
      }
    }
    __syncwarp();

    // ---- group = head: acc += w * g'[v], dot <g'[v], ft[u]> back to the edge's lane through shared memory ----
    for (int e = 0; e < cnt; e += U) {
      float part[U];
#pragma unroll
      for (int s = 0; s < U; ++s) {
        const float w = (e + s < cnt) ? wsm[(e + s) * HG + grp] : 0.f;
        part[s] = 0.f;
#pragma unroll
        for (int i = 0; i < VPL; ++i) {
          acc[i].fma(w, x[s][i]);
          part[s] = x[s][i].dot(fu[i], part[s]);  // fu is 0 on slots this lane does not own
        }
        const int nx = e + s + U;
        if (nx < cnt) {  // warp-uniform
          const char* r = bp + (size_t)(unsigned)__shfl_sync(kFull, v0, nx) * ldb;
#pragma unroll
          for (int i = 0; i < VPL; ++i) x[s][i].load(reinterpret_cast<const float*>(r + (i < VPL - 1 ? i * G * 16 : last_off)));
        }
      }
      // U partial dots per lane -> packed butterfly over the G lanes of the group: slot s's sum ends in lanes
      // [s * LPU, (s + 1) * LPU) of the group
      int k = U;
#pragma unroll
      for (int o = G >> 1; o > 0; o >>= 1) {
        if (k > 1) {
          const bool upper = (lane & o) != 0;
#pragma unroll
          for (int i = 0; i < (U > 1 ? U / 2 : 1); ++i) {
            if (i < k / 2) {
              const float send = upper ? part[i] : part[i + k / 2];
              const float keep = upper ? part[i + k / 2] : part[i];
              part[i] = keep + __shfl_xor_sync(kFull, send, o);
            }
          }
          k >>= 1;
        } else {
          part[0] += __shfl_xor_sync(kFull, part[0], o);
        }
      }
      if ((j & (LPU - 1)) == 0) dsm[(e + j / LPU) * HG + grp] = part[0];  // e + s <= 31
    }
    __syncwarp();

    if (valid) {
#pragma unroll
      for (int hh = 0; hh < HG; ++hh) {
        if (hh < hc) {
          const float gzv = fmaf(ca[hh], dsm[lane * HG + hh], -cb[hh]);
          if (gz) gz[(int64_t)hh * p.n_edges + pos] = gzv;
          gel_lane[hh] += gzv;
        }
      }
    }
    __syncwarp();
    v0 = v1; v1 = v2; k0 = k1; k1 = k2;
  }

  const float gel = packed_reduce<GSH, false>(gel_lane, lane);
  if (slot >= 0) {
    // segment of a split row: partial grad_el and (unscaled) partial grad_ft go to this segment's scratch slot
    float* sl = p.scratch + (int64_t)slot * bwd_slot_floats(H, D);
#pragma unroll
    for (int i = 0; i < VPL; ++i)
      if (act[i]) acc[i].store(sl + (int64_t)h * D + (j + i * G) * 4);
    if (hval && j == 0) sl[H * D + h] = gel;
    return;
  }
  float* o = p.grad_ft + (int64_t)row * p.ld_gft + h * D;
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    if (act[i]) {
      acc[i].scale(csu);
      acc[i].store(o + (j + i * G) * 4);
    }
  }
  if (hval && j == 0) p.grad_el[(int64_t)row * H + h] = gel;
}


// ---------------------------------------------------------------------------
// backward src pass, rows staged by bulk copies
//
// Same pass with the g'[v] rows fetched by the copy engine instead of LDG: one `cp.async.bulk` (UBLKCP) per
// neighbour row — the whole 4*H*D contiguous bytes in ONE request — into a per-warp shared-memory ring of R slots,
// completion on one mbarrier per slot, rows consumed with LDS.128.  The register ring above keeps U = 4 neighbours
// (7.7 KB at the products shape) per warp in flight at 168 registers / 12 warps per SM (92 KB per SM) and leaves DRAM
// at 57 % (profiles/r02_s_rw_summary.txt); here the ring is R = 8 rows per warp in shared memory, no register holds
// a row in flight, and the resident warps are bounded by shared memory instead (13 one-warp blocks x 15 KB).
// One warp per block, as in gat_bwd_tma.cu.  Each lane issues the copy of ITS OWN neighbour (lane = edge), so no
// index shuffles are needed on the issue side.
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t rw_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ float4 rw_lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void rw_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred q;\n\tRW_WAIT:\n\tmbarrier.try_wait.parity.shared::cta.b64 q, [%0], %1;\n\t@q bra RW_DONE;\n\tbra RW_WAIT;\n\tRW_DONE:\n\t}" ::"r"(bar),
      "r"(parity)
      : "memory");
}

template <int GSH, int VPL>
__global__ void __launch_bounds__(32, 10) gat_bwd_src_rowbulk_kernel(const BwdParams p, int slotB) {
  constexpr int G = 1 << GSH;
  constexpr int HG = 32 >> GSH;
  constexpr int U = 4;         // neighbours per packed dot reduction (G >= 4 in every instantiation)
  constexpr int LPU = G / U;
  constexpr int R = kBulkRing;
  extern __shared__ __align__(128) unsigned char ring[];  // R slots of slotB bytes
  __shared__ __align__(8) uint64_t bars[R];
  __shared__ __align__(16) float wsm[32 * HG];
  __shared__ __align__(16) float dsm[32 * HG];
  const int lane = threadIdx.x;
  uint32_t ring0 = rw_smem_u32(ring), bar0 = rw_smem_u32(bars);
  asm volatile("" : "+r"(ring0), "+r"(bar0));
  if (lane < R) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0 + 8 * lane));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncwarp();

  const int item = blockIdx.x;
  const int row = p.seg_row ? p.seg_row[item] : item;
  const int slot = p.seg_row ? p.seg_slot[item] : -1;
  const int grp = lane >> GSH, j = lane & (G - 1);
  const int hc = p.h_count;
  const bool hval = grp < hc;
  const int hl = hval ? grp : hc - 1;  // idle groups shadow the last head (reads stay inside the staged row)
  const int h = p.h_begin + hl;
  const int H = p.H, D = p.D;
  const int nv = D >> 2;
  const uint32_t rowB = (uint32_t)(hc * D * 4);  // staged bytes of one neighbour: the heads of this launch

  bool act[VPL];
#pragma unroll
  for (int i = 0; i < VPL; ++i) act[i] = hval && (j + i * G) < nv;
  const uint32_t lane_off = (uint32_t)((hl * D + j * 4) * 4);
  const uint32_t last_off = lane_off + (uint32_t)((min(j + (VPL - 1) * G, nv - 1) - j) * 16);
  const char* gbase = reinterpret_cast<const char*>(p.g + p.h_begin * D);
  const size_t ldb = (size_t)p.ld_g * 4;

  const int beg = p.seg_row ? p.seg_beg[item] : p.indptr[row];
  const int end = p.seg_row ? p.seg_end[item] : p.indptr[row + 1];
  const float slope = p.slope;
  const float csu = p.cs ? p.cs[row] : 1.f;
  Vec<4> fu[VPL], acc[VPL];
  {
    const float* f = p.ft + (int64_t)row * p.ld_ft + h * D;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      if (act[i]) { fu[i].load(f + (j + i * G) * 4); fu[i].scale(csu); } else fu[i].zero();
      acc[i].zero();
    }
  }
  float gel_lane[HG];
#pragma unroll
  for (int hh = 0; hh < HG; ++hh) gel_lane[hh] = 0.f;
  const float* __restrict__ el_u = p.el + (int64_t)row * H + p.h_begin;
  const float4* __restrict__ drec = p.drec + (unsigned)(p.h_begin * p.drec_hs);
  const float* __restrict__ eb = p.eb ? p.eb + (int64_t)(p.Hb == 1 ? 0 : p.h_begin) * p.n_edges : nullptr;
  const int64_t eb_hs = p.Hb == 1 ? 0 : p.n_edges;
  const float* __restrict__ am = p.am ? p.am + (int64_t)p.h_begin * p.n_edges : nullptr;
  float* __restrict__ gz = p.gz ? p.gz + (int64_t)p.h_begin * p.n_edges : nullptr;
  const bool philox = (p.am == nullptr) && p.attn_p > 0.f;

  auto load_index = [&](int base, int& v, int& k) {
    const int pos = base + lane;
    v = k = 0;
    if (pos < end) {
      v = __ldg(p.indices + pos);
      if (philox) k = __ldg(p.eid + pos);
    }
  };
  // neighbours [lo, hi) of the current chunk (lane = neighbour) go to the ring slots q0 + (lane - lo), ...
  auto issue = [&](int lo, int hi, uint32_t q0, int v) {
    if (lane >= lo && lane < hi) {
      const uint32_t s = (q0 + (uint32_t)(lane - lo)) & (R - 1);
      const uint32_t bar = bar0 + 8 * s;
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(rowB) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(ring0 + s * slotB),
                   "l"(gbase + (size_t)(unsigned)v * ldb), "r"(rowB), "r"(bar)
                   : "memory");
    }
  };
  int v0, v1, k0, k1;
  load_index(beg, v0, k0);
  load_index(beg + 32, v1, k1);
  uint32_t q = 0;  // neighbours issued so far (ring write position); consumed: c (read position, phase = c / R)
  uint32_t c = 0;

  for (int base = beg; base < end; base += 32) {
    const int cnt = min(32, end - base);
    const int pos = base + lane;
    const bool valid = pos < end;
    int v2, k2;
    load_index(base + 64, v2, k2);

    // the ring is empty at a chunk boundary: fill it before the logit operands are even requested
    int issued = min(cnt, R);
    issue(0, issued, q, v0);
    q += (uint32_t)issued;

    // ---- lane = edge: recompute the attention weight of this edge for every head ----
    float ca[HG], cb[HG];  // gz = ca * <src_scale * ft[u], g'[v]> - cb   (softmax + leaky_relu adjoint, App. A.3)
    {
      float4 rec[HG];
      float ebv[HG], amv[HG];
#pragma unroll
      for (int hh = 0; hh < HG; ++hh) {
        const bool hv = valid && hh < hc;
        rec[hh] = make_float4(0.f, 0.f, 0.f, 0.f);
        ebv[hh] = -INFINITY;  // lanes past the row end / idle heads behave like dropped edges: alpha = 0
        amv[hh] = 1.f;
        if (hv) {
          rec[hh] = __ldg(drec + (unsigned)(hh * p.drec_hs + v0 * p.drec_vs));
          ebv[hh] = eb ? __ldg(eb + hh * eb_hs + pos) : 0.f;
          if (am) amv[hh] = __ldg(am + (int64_t)hh * p.n_edges + pos);
        }
      }
      if (philox) {
        float pm[HG];
        philox_heads<HG>(p.seed, (uint32_t)k0, p.h_begin, hc, p.attn_p, p.inv_keep, pm);
#pragma unroll
        for (int hh = 0; hh < HG; ++hh) amv[hh] *= pm[hh];
      }
      float wv[HG];
#pragma unroll
      for (int hh = 0; hh < HG; ++hh) {
        const float z = (hh < hc ? __ldg(el_u + hh) : 0.f) + rec[hh].x + ebv[hh];
        const float s = leaky_relu(z, slope);
        const float alpha = (s == -INFINITY) ? 0.f : __expf(s - rec[hh].y) * rec[hh].z;
        const float dz = z > 0.f ? 1.f : slope;
        wv[hh] = alpha * amv[hh];
        ca[hh] = wv[hh] * dz;
        cb[hh] = alpha * rec[hh].w * dz;
      }
      if constexpr (HG % 4 == 0) {
#pragma unroll
        for (int qd = 0; qd < HG / 4; ++qd)
          reinterpret_cast<float4*>(wsm + lane * HG)[qd] = make_float4(wv[4 * qd], wv[4 * qd + 1], wv[4 * qd + 2], wv[4 * qd + 3]);
      } else {
#pragma unroll
        for (int hh = 0; hh < HG; ++hh) wsm[lane * HG + hh] = wv[hh];
      }
    }
    __syncwarp();

    // ---- group = head: acc += w * g'[v], dot <g'[v], ft[u]> back to the edge's lane through shared memory ----
    for (int e = 0; e < cnt; e += U) {
      float part[U];
#pragma unroll
      for (int s = 0; s < U; ++s) {
        part[s] = 0.f;
        if (e + s < cnt) {  // warp-uniform
          const uint32_t sl = c & (R - 1);
          rw_wait(bar0 + 8 * sl, (c >> kBulkRingLog2) & 1u);
          ++c;
          const uint32_t a = ring0 + sl * slotB;
          const float w = wsm[(e + s) * HG + grp];
#pragma unroll
          for (int i = 0; i < VPL; ++i) {
            Vec<4> x;
            x.v = rw_lds128(a + (i < VPL - 1 ? lane_off + i * G * 16 : last_off));
            acc[i].fma(w, x);
            part[s] = x.dot(fu[i], part[s]);  // fu is 0 on slots this lane does not own
          }
        }
      }
      __syncwarp();  // every lane is done with these U slots before they are refilled
      {
        const int more = min(U, cnt - issued);
        if (more > 0) {
          issue(issued, issued + more, q, v0);
          q += (uint32_t)more;
          issued += more;
        }
      }
      int k = U;
#pragma unroll
      for (int o = G >> 1; o > 0; o >>= 1) {
        if (k > 1) {
          const bool upper = (lane & o) != 0;
#pragma unroll
          for (int i = 0; i < U / 2; ++i) {
            if (i < k / 2) {
              const float send = upper ? part[i] : part[i + k / 2];
              const float keep = upper ? part[i + k / 2] : part[i];
              part[i] = keep + __shfl_xor_sync(kFull, send, o);
            }
          }
          k >>= 1;
        } else {
          part[0] += __shfl_xor_sync(kFull, part[0], o);
        }
      }
      if ((j & (LPU - 1)) == 0) dsm[(e + j / LPU) * HG + grp] = part[0];  // e + s <= 31
    }
    __syncwarp();

    if (valid) {
#pragma unroll
      for (int hh = 0; hh < HG; ++hh) {
        if (hh < hc) {
          const float gzv = fmaf(ca[hh], dsm[lane * HG + hh], -cb[hh]);
          if (gz) gz[(int64_t)hh * p.n_edges + pos] = gzv;
          gel_lane[hh] += gzv;
        }
      }
    }
    __syncwarp();
    v0 = v1; v1 = v2; k0 = k1; k1 = k2;
  }

  const float gel = packed_reduce<GSH, false>(gel_lane, lane);
  if (slot >= 0) {
    float* sl = p.scratch + (int64_t)slot * bwd_slot_floats(H, D);
#pragma unroll
    for (int i = 0; i < VPL; ++i)
      if (act[i]) acc[i].store(sl + (int64_t)h * D + (j + i * G) * 4);
    if (hval && j == 0) sl[H * D + h] = gel;
    return;
  }
  float* o = p.grad_ft + (int64_t)row * p.ld_gft + h * D;
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    if (act[i]) {
      acc[i].scale(csu);
      acc[i].store(o + (j + i * G) * 4);
    }
  }
  if (hval && j == 0) p.grad_el[(int64_t)row * H + h] = gel;
}

// ---------------------------------------------------------------------------
// launch
// ---------------------------------------------------------------------------
int launch_fwd_rowwise(const FwdParams& p, const FwdPlan& plan, cudaStream_t st) {
  const bool launched = with_rw_combo(plan.rw_gsh, plan.rw_vpl, [&](auto gsh, auto vpl) {
    if (p.ep.any())
      gat_fwd_rowwise_kernel<gsh.value, vpl.value, true><<<plan.grid, kWarpsPerBlock * 32, 0, st>>>(p);
    else
      gat_fwd_rowwise_kernel<gsh.value, vpl.value, false><<<plan.grid, kWarpsPerBlock * 32, 0, st>>>(p);
  });
  BG_REQUIRE(launched, "forward: no row-wise kernel for lanes=%d slots=%d", 1 << plan.rw_gsh, plan.rw_vpl);
  BG_LAUNCHED(1);
  return 0;
}

int launch_src_rowwise(const BwdParams& p, const SrcPlan& plan, cudaStream_t st) {
  cudaError_t err = cudaSuccess;
  const bool launched = with_rw_combo(plan.rw_gsh, plan.rw_vpl, [&](auto gsh, auto vpl) {
    if (plan.family == Family::rowwise) {
      gat_bwd_src_rowwise_kernel<gsh.value, vpl.value><<<plan.grid, kWarpsPerBlock * 32, 0, st>>>(p);
      return;
    }
    auto* kernel = gat_bwd_src_rowbulk_kernel<gsh.value, vpl.value>;
    static bool attr_set = false;  // one per instantiation
    if (!attr_set) {
      err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBulkRingMax);
      if (err != cudaSuccess) return;
      cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
      attr_set = true;
    }
    kernel<<<plan.grid, 32, plan.bulk_ring_bytes, st>>>(p, plan.bulk_slot_bytes);
  });
  BG_REQUIRE(launched, "backward: no row-wise kernel for lanes=%d slots=%d", 1 << plan.rw_gsh, plan.rw_vpl);
  if (err != cudaSuccess) cudaGetLastError();  // reported here, not by the next launch
  BG_REQUIRE(err == cudaSuccess, "backward: bulk-copy row-wise kernel: %zu bytes of shared memory refused: %s", kBulkRingMax,
             cudaGetErrorString(err));
  BG_LAUNCHED(1);
  return 0;
}

}  // namespace botgat
