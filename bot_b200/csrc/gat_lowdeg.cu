// Group-per-row variants of the two gather kernels, for LOW-DEGREE graphs (ogbn-arxiv ~15, ogbn-products ~25,
// Cora ~5 in-edges per node, and the per-rank out-CSR of a partitioned graph).
//
// In gat_fwd.cu / gat_bwd.cu one warp owns one CSR row and its 32/G lane groups serve 32/G neighbours of that
// row at a time.  With rows shorter than a 32-neighbour chunk, most of a row's time is its dependent load
// chain (index -> logit operands -> feature rows) plus the cross-group reduction of the epilogue.  Here a
// G-lane GROUP owns a row: a warp works on 32/G consecutive rows at once, chunks are G neighbours long, the
// softmax reductions stay inside the group and no cross-group reduction is needed.  Per step the warp still
// gathers 32/G feature rows (one per group), so the steady-state gather rate is unchanged.
//
// Same math, same operand conventions and the same software pipeline as the warp-per-row kernels.
#include "common.cuh"
#include "params.cuh"

namespace botgat {


template <int G> __device__ __forceinline__ float group_max(float v) {
#pragma unroll
  for (int o = G >> 1; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(kFull, v, o));
  return v;
}
template <int G> __device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int o = G >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}

// ---------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------
template <int VW, int GSH, int VPL, bool EP>
__global__ void __launch_bounds__(kWarpsPerBlock * 32, fwd_min_blocks(VPL)) gat_fwd_lowdeg_kernel(const FwdParams p, int warps_per_slab) {
  constexpr int NS = steps_in_flight(VPL);
  constexpr int G = 1 << GSH;     // lanes per row
  constexpr int RPW = 32 >> GSH;  // rows per warp
  const int lane = threadIdx.x & 31;
  const int gw = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  const int slab = gw / warps_per_slab;
  const int wrow = gw - slab * warps_per_slab;
  if (slab >= p.h_count * p.col_parts) return;
  const int j = lane & (G - 1), gbase = lane & ~(G - 1);
  // a work item is a CSR row or, for a row that exceeds the segment length (segments.cu), one segment of it whose
  // partial result goes to a scratch slot: a heavy row of a sparse graph is shared by many groups instead of one
  const int item = wrow * RPW + (lane >> GSH);
  const bool valid = item < p.n_items;
  const int row = (valid && p.seg_row) ? p.seg_row[item] : item;
  const int slot = (valid && p.seg_row) ? p.seg_slot[item] : -1;
  const int hl = slab / p.col_parts;  // head within this launch's range
  const int h = hl + p.h_begin;
  const int cp = slab - hl * p.col_parts;
  const int c0 = cp * p.part_cols;
  const int nv = (min(p.D - c0, p.part_cols) + VW - 1) / VW;
  const int v0 = j - (((h * p.D + c0) / VW) & p.omask);

  const char* bp[VPL];
  bool act[VPL];
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const int v = v0 + i * G;
    act[i] = v >= 0 && v < nv;
    bp[i] = reinterpret_cast<const char*>(p.ft + h * p.D + c0 + min(max(v, 0), nv - 1) * VW);
  }
  const unsigned ldb = (unsigned)(p.ld_ft * 4);

  const int beg = !valid ? 0 : p.seg_row ? p.seg_beg[item] : p.indptr[row];
  const int end = !valid ? 0 : p.seg_row ? p.seg_end[item] : p.indptr[row + 1];
  const float slope = p.slope;
  const int H = p.H;
  const float er_v = (p.er && valid) ? p.er[(int64_t)row * H + h] : 0.f;
  const float* __restrict__ el_h = p.el + h;
  const float* __restrict__ eb_h = p.eb ? p.eb + (int64_t)(p.Hb == 1 ? 0 : h) * p.n_edges : nullptr;
  const float* __restrict__ am_h = p.am ? p.am + (int64_t)h * p.n_edges : nullptr;
  const float* __restrict__ ee_h = p.ee ? p.ee + h : nullptr;
  const float* __restrict__ amul_h = p.amul_e ? p.amul_e + h : nullptr;
  const uint8_t* __restrict__ keep = p.keep;
  const float* __restrict__ cs = p.cs;
  const bool philox = (p.am == nullptr) && (p.amul_e == nullptr) && p.attn_p > 0.f;
  const bool need_eid = ee_h || amul_h || keep || philox;

  Vec<VW> acc[VPL];
#pragma unroll
  for (int i = 0; i < VPL; ++i) acc[i].zero();
  float m = -INFINITY, l_lane = 0.f;

  struct Ops { float el, eb, cs, am; unsigned keep; };
  auto load_index = [&](int base, int& u, int& k) {
    const int pos = base + j;
    u = k = 0;
    if (pos < end) {
      u = __ldg(p.indices + pos);
      if (need_eid) k = __ldg(p.eid + pos);
    }
  };
  auto load_operands = [&](int base, int u, int k, Ops& o) {
    const int pos = base + j;
    o.el = -INFINITY;
    o.eb = 0.f; o.cs = 1.f; o.am = 1.f; o.keep = 1u;
    if (pos < end) {
      o.el = __ldg(el_h + (int64_t)u * H);
      if (eb_h) o.eb = __ldg(eb_h + pos);
      else if (ee_h) o.eb = __ldg(ee_h + (int64_t)k * H);
      if (keep) o.keep = __ldg(keep + k);
      if (cs) o.cs = __ldg(cs + u);
      if (am_h) o.am = __ldg(am_h + pos);
      else if (amul_h) o.am = __ldg(amul_h + (int64_t)k * H);
      else if (philox) o.am = philox_dropout_mul(p.seed, (uint32_t)k, (uint32_t)h, p.attn_p, p.inv_keep);
    }
  };
  int u0, u1, u2 = 0, k0, k1, k2 = 0;
  load_index(beg, u0, k0);
  load_index(beg + G, u1, k1);
  Ops o0, o1;
  load_operands(beg, u0, k0, o0);

  for (int base = beg; __any_sync(kFull, base < end); base += G) {
    const int cnt = max(0, min(G, end - base));
    load_index(base + 2 * G, u2, k2);
    load_operands(base + G, u1, k1, o1);

    const float z0 = o0.keep ? o0.el + er_v + o0.eb : -INFINITY;
    const float s = leaky_relu(z0, slope);
    const float m_new = fmaxf(m, group_max<G>(s));
    if (__any_sync(kFull, m_new > m)) {
      const float f = m_new > m ? __expf(m - m_new) : 1.f;
      l_lane *= f;
#pragma unroll
      for (int i = 0; i < VPL; ++i) acc[i].scale(f);
      m = m_new;
    }
    const float pexp = (s == -INFINITY) ? 0.f : __expf(s - m);
    l_lane += pexp;
    const float w_lane = pexp * o0.cs * o0.am;

    // every group walks its own chunk; the trip count is the longest chunk in the warp
    const int cmax = __reduce_max_sync(kFull, cnt);
    const int last = gbase + max(cnt - 1, 0);
    for (int t = 0; t < cmax; t += NS) {
      Vec<VW> x[NS][VPL];
      float w[NS];
#pragma unroll
      for (int s_ = 0; s_ < NS; ++s_) {
        const int from = min(gbase + t + s_, last);  // past the group's chunk: re-read its last neighbour, weight 0
        const size_t off = (size_t)(unsigned)__shfl_sync(kFull, u0, from) * ldb;
        const float ww = __shfl_sync(kFull, w_lane, from);
        w[s_] = (t + s_ < cnt) ? ww : 0.f;
#pragma unroll
        for (int i = 0; i < VPL; ++i) x[s_][i].load(reinterpret_cast<const float*>(bp[i] + off));
      }
#pragma unroll
      for (int s_ = 0; s_ < NS; ++s_) {
#pragma unroll
        for (int i = 0; i < VPL; ++i) acc[i].fma(w[s_], x[s_][i]);
      }
    }
    u0 = u1; u1 = u2; k1 = k2; o0 = o1;
  }

  const float l = group_sum<G>(l_lane);
  if (valid && slot >= 0) {
    // segment of a split row: park (max, sum, unnormalised accumulator) in this segment's scratch slot (k_fwd_combine)
    float* sl = p.scratch + (int64_t)slot * fwd_slot_floats(H, p.D);
    float* o = sl + (int64_t)h * p.D + c0 + v0 * VW;
#pragma unroll
    for (int i = 0; i < VPL; ++i)
      if (act[i]) acc[i].store(o + i * G * VW);
    if (cp == 0 && j == 0) { sl[H * p.D + h * 2] = m; sl[H * p.D + h * 2 + 1] = l; }
  } else if (valid) {
    float scale = l > 0.f ? 1.f / l : 0.f;
    if (p.ds) scale *= p.ds[row];
    float* o = p.out + (int64_t)row * p.ld_out + h * p.D + c0 + v0 * VW;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      if (act[i]) {
        acc[i].scale(scale);
        if constexpr (EP) p.ep.apply(acc[i], row, (int64_t)h * p.D + c0 + (v0 + i * G) * VW);
        acc[i].store(o + i * G * VW);
      }
    }
    if (cp == 0 && j == 0) {
      p.row_max[(int64_t)row * H + h] = m;
      p.row_sum[(int64_t)row * H + h] = l;
    }
  }
}

int launch_fwd_lowdeg(const FwdParams& p, const FwdPlan& plan, cudaStream_t st) {
  const Tiling& t = plan.t;
  const bool launched = with_combo(t.vw, t.gshift, t.vpl, [&](auto vw, auto gsh, auto vpl) {
    if (p.ep.any())
      gat_fwd_lowdeg_kernel<vw.value, gsh.value, vpl.value, true><<<plan.grid, kWarpsPerBlock * 32, 0, st>>>(p, plan.warps_per_slab);
    else
      gat_fwd_lowdeg_kernel<vw.value, gsh.value, vpl.value, false><<<plan.grid, kWarpsPerBlock * 32, 0, st>>>(p, plan.warps_per_slab);
  });
  BG_REQUIRE(launched, "forward: no low-degree kernel for vw=%d lanes=%d slots=%d", t.vw, 1 << t.gshift, t.vpl);
  BG_LAUNCHED(1);
  return 0;
}

// ---------------------------------------------------------------------------
// backward src pass
// ---------------------------------------------------------------------------
__host__ __device__ constexpr int lowdeg_steps_bwd(int vpl) { return vpl <= 3 ? 4 : vpl <= 6 ? 2 : 1; }

template <int VW, int GSH, int VPL>
__global__ void __launch_bounds__(kWarpsPerBlock * 32, bwd_min_blocks(VPL))
gat_bwd_src_lowdeg_kernel(const BwdParams p, int warps_per_slab) {
  constexpr int NS = lowdeg_steps_bwd(VPL);
  constexpr int G = 1 << GSH;
  constexpr int RPW = 32 >> GSH;
  constexpr bool kPacked = NS > 1 && NS <= G && (NS & (NS - 1)) == 0;
  const int lane = threadIdx.x & 31;
  const int gw = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  const int hl = gw / warps_per_slab;  // head within this launch's range
  const int wrow = gw - hl * warps_per_slab;
  if (hl >= p.h_count) return;
  const int h = hl + p.h_begin;
  const int j = lane & (G - 1), gbase = lane & ~(G - 1);
  const int item = wrow * RPW + (lane >> GSH);   // a row, or a segment of a split row (see the forward)
  const bool valid = item < p.n_items;
  const int row = (valid && p.seg_row) ? p.seg_row[item] : item;
  const int slot = (valid && p.seg_row) ? p.seg_slot[item] : -1;
  const int v0 = j - (((h * p.D) / VW) & p.omask);

  const int nv = p.D / VW;
  const char* bp[VPL];
  bool act[VPL];
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const int v = v0 + i * G;
    act[i] = v >= 0 && v < nv;
    bp[i] = reinterpret_cast<const char*>(p.g + h * p.D + min(max(v, 0), nv - 1) * VW);
  }
  const unsigned ldb = (unsigned)(p.ld_g * 4);

  const int beg = !valid ? 0 : p.seg_row ? p.seg_beg[item] : p.indptr[row];
  const int end = !valid ? 0 : p.seg_row ? p.seg_end[item] : p.indptr[row + 1];
  const float slope = p.slope;
  const int H = p.H;
  const float csu = (p.cs && valid) ? p.cs[row] : 1.f;
  const float el_u = valid ? p.el[(int64_t)row * H + h] : 0.f;
  Vec<VW> fu[VPL], acc[VPL];
  {
    const float* f = p.ft + (int64_t)(valid ? row : 0) * p.ld_ft + h * p.D + v0 * VW;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      if (act[i] && valid) { fu[i].load(f + i * G * VW); fu[i].scale(csu); } else fu[i].zero();
      acc[i].zero();
    }
  }
  const float4* __restrict__ drec_h = p.drec + (int64_t)h * p.n_dst;  // head-major records (BwdParams::drec)
  const float* __restrict__ eb_h = p.eb ? p.eb + (int64_t)(p.Hb == 1 ? 0 : h) * p.n_edges : nullptr;
  const float* __restrict__ am_h = p.am ? p.am + (int64_t)h * p.n_edges : nullptr;
  float* __restrict__ gz_h = p.gz ? p.gz + (int64_t)h * p.n_edges : nullptr;
  const float* __restrict__ ee_h = p.ee ? p.ee + h : nullptr;
  const float* __restrict__ amul_h = p.amul_e ? p.amul_e + h : nullptr;
  const uint8_t* __restrict__ keep = p.keep;
  float* __restrict__ gze_h = p.gz_e ? p.gz_e + h : nullptr;
  const bool philox = (p.am == nullptr) && (p.amul_e == nullptr) && p.attn_p > 0.f;
  const bool need_eid = ee_h || amul_h || keep || philox || gze_h;
  float gel_lane = 0.f;

  auto load_index = [&](int base, int& v, int& k) {
    const int pos = base + j;
    v = k = 0;
    if (pos < end) {
      v = __ldg(p.indices + pos);
      if (need_eid) k = __ldg(p.eid + pos);
    }
  };
  auto load_operands = [&](int base, int v, int k, SrcOps& o) {
    const int pos = base + j;
    o.rec = make_float4(0.f, 0.f, 0.f, 0.f);
    o.eb = -INFINITY;
    o.amul = 1.f;
    if (pos < end) {
      o.rec = __ldg(drec_h + v);
      o.eb = eb_h ? __ldg(eb_h + pos) : 0.f;
      if (ee_h) o.eb += __ldg(ee_h + (int64_t)k * H);
      if (keep && !__ldg(keep + k)) o.eb = -INFINITY;
      if (am_h) o.amul = __ldg(am_h + pos);
      else if (amul_h) o.amul = __ldg(amul_h + (int64_t)k * H);
      else if (philox) o.amul = philox_dropout_mul(p.seed, (uint32_t)k, (uint32_t)h, p.attn_p, p.inv_keep);
    }
  };
  int vtx0, vtx1, vtx2 = 0, k0, k1, k2 = 0;
  load_index(beg, vtx0, k0);
  load_index(beg + G, vtx1, k1);
  SrcOps o0, o1;
  load_operands(beg, vtx0, k0, o0);

  for (int base = beg; __any_sync(kFull, base < end); base += G) {
    const int cnt = max(0, min(G, end - base));
    load_index(base + 2 * G, vtx2, k2);
    load_operands(base + G, vtx1, k1, o1);

    const float z = el_u + o0.rec.x + o0.eb;
    const float s = leaky_relu(z, slope);
    const float alpha = (s == -INFINITY) ? 0.f : __expf(s - o0.rec.y) * o0.rec.z;
    const float dz = z > 0.f ? 1.f : slope;
    const float w_lane = alpha * o0.amul;
    float d_lane = 0.f;

    const int cmax = __reduce_max_sync(kFull, cnt);
    const int last = gbase + max(cnt - 1, 0);
    for (int t = 0; t < cmax; t += NS) {
      Vec<VW> x[NS][VPL];
      float w[NS], part[NS];
#pragma unroll
      for (int s_ = 0; s_ < NS; ++s_) {
        const int from = min(gbase + t + s_, last);
        const size_t off = (size_t)(unsigned)__shfl_sync(kFull, vtx0, from) * ldb;
        const float ww = __shfl_sync(kFull, w_lane, from);
        w[s_] = (t + s_ < cnt) ? ww : 0.f;
#pragma unroll
        for (int i = 0; i < VPL; ++i) x[s_][i].load(reinterpret_cast<const float*>(bp[i] + off));
      }
#pragma unroll
      for (int s_ = 0; s_ < NS; ++s_) {
        part[s_] = 0.f;
#pragma unroll
        for (int i = 0; i < VPL; ++i) {
          acc[i].fma(w[s_], x[s_][i]);
          part[s_] = x[s_][i].dot(fu[i], part[s_]);
        }
      }
      if constexpr (kPacked) {
        // packed butterfly inside the group (see gat_bwd.cu): step s ends up in lanes [s*G/NS, (s+1)*G/NS)
        int k = NS;
#pragma unroll
        for (int o = G >> 1; o > 0; o >>= 1) {
          if (k > 1) {
            const bool upper = (lane & o) != 0;
#pragma unroll
            for (int i = 0; i < NS / 2; ++i) {
              if (i < k / 2) {
                const float send = upper ? part[i] : part[i + k / 2];
                const float keepv = upper ? part[i + k / 2] : part[i];
                part[i] = keepv + __shfl_xor_sync(kFull, send, o);
              }
            }
            k >>= 1;
          } else {
            part[0] += __shfl_xor_sync(kFull, part[0], o);
          }
        }
        const int tq = j - t;  // this lane owns neighbour j of the chunk; it is step tq of this iteration
        const float got = __shfl_sync(kFull, part[0], (gbase + tq * (G / NS)) & 31);
        if (tq >= 0 && tq < NS) d_lane = got;
      } else {
#pragma unroll
        for (int s_ = 0; s_ < NS; ++s_) {
          const float tot = group_sum<G>(part[s_]);
          if (j == t + s_) d_lane = tot;
        }
      }
    }
    const float gz = alpha * (d_lane * o0.amul - o0.rec.w) * dz;
    if (gz_h && j < cnt) gz_h[base + j] = gz;
    if (gze_h && j < cnt) gze_h[(int64_t)k0 * H] = gz;
    gel_lane += gz;
    vtx0 = vtx1; vtx1 = vtx2; k0 = k1; k1 = k2; o0 = o1;
  }

  const float gel = group_sum<G>(gel_lane);
  if (valid && slot >= 0) {
    // segment of a split row: partial grad_el and (unscaled) partial grad_ft go to the segment's slot (k_bwd_combine)
    float* sl = p.scratch + (int64_t)slot * bwd_slot_floats(H, p.D);
    float* o = sl + (int64_t)h * p.D + v0 * VW;
#pragma unroll
    for (int i = 0; i < VPL; ++i)
      if (act[i]) acc[i].store(o + i * G * VW);
    if (j == 0) sl[H * p.D + h] = gel;
  } else if (valid) {
    float* o = p.grad_ft + (int64_t)row * p.ld_gft + h * p.D + v0 * VW;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      if (act[i]) {
        acc[i].scale(csu);
        acc[i].store(o + i * G * VW);
      }
    }
    if (j == 0) p.grad_el[(int64_t)row * H + h] = gel;
  }
}

int launch_src_lowdeg(const BwdParams& p, const SrcPlan& plan, cudaStream_t st) {
  const Tiling& t = plan.t;
  const bool launched = with_combo(t.vw, t.gshift, t.vpl, [&](auto vw, auto gsh, auto vpl) {
    gat_bwd_src_lowdeg_kernel<vw.value, gsh.value, vpl.value><<<plan.grid, kWarpsPerBlock * 32, 0, st>>>(p, plan.warps_per_slab);
  });
  BG_REQUIRE(launched, "backward: no low-degree kernel for vw=%d lanes=%d slots=%d", t.vw, 1 << t.gshift, t.vpl);
  BG_LAUNCHED(1);
  return 0;
}

}  // namespace botgat
