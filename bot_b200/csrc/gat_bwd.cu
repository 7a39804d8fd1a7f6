// GAT backward for sm_100a (adjoint of gat_fwd.cu; SURVEY.md Appendix A.3).
// Replaces the autograd replay of DGL's GSpMM / GSDDMM / EdgeSoftmax backward
// kernels behind src/no-sampling/models.py:523-555 and
// src/ogbn-proteins/models.py:125-156.
//
//   node phase : t[v,h] = <out[v,h,:], gout[v,h,:]>; packs drec[h][v] =
//                {er, row_max, 1/row_sum, t}; g' = gout * dst_scale
//   src phase  : ONE gather pass over the out-CSR (src-major): grad_ft, grad_el
//                and gz (gradient of the per-edge logit, out-CSR order)
//   edge phase : gz -> grad_ee (edge-id order); grad_er[v] = sum over in-edges
//
// The reference's backward gathers E x H x D twice (SpMM on the reversed graph
// for grad_ft, SDDMM-dot for grad_a).  Here the dot <ft[u], g'[v]> rides on the
// rows the src pass gathers anyway (ft[u] is row-local there), so the second
// gather disappears; what remains E-sized is the 4*H-byte-per-edge gz stream.
//
// Attention weights are recomputed from (el, er, eb, row_max, row_sum); nothing
// E-sized is saved by the forward.  No atomics: every output element is produced
// by exactly one warp in a fixed order, so results are run-to-run deterministic.
#include "common.cuh"
#include "params.cuh"

namespace botgat {


// ---------------------------------------------------------------------------
// node phase: one warp per destination row
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
gat_bwd_node_kernel(int n_dst, int H, int D, int64_t ld, const float* __restrict__ out,
                    const float* __restrict__ gout, const float* __restrict__ er,
                    const float* __restrict__ row_max, const float* __restrict__ row_sum,
                    const float* __restrict__ ds, float4* __restrict__ drec, int drec_hs, int drec_vs,
                    float* __restrict__ gprime) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int v = blockIdx.x * kWarpsPerBlock + warp;
  if (v >= n_dst) return;
  const float* o = out + (int64_t)v * ld;
  const float* g = gout + (int64_t)v * ld;
  const float dsv = ds ? ds[v] : 1.f;
  for (int h = 0; h < H; ++h) {
    float t = 0.f;
    for (int d = lane; d < D; d += 32) {
      const float gv = g[h * D + d];
      t = fmaf(o[h * D + d], gv, t);
      if (gprime) gprime[(int64_t)v * ld + h * D + d] = gv * dsv;
    }
    t = warp_sum(t);
    if (lane == 0) {
      const float l = row_sum[(int64_t)v * H + h];
      drec[(unsigned)(h * drec_hs + v * drec_vs)] =
          make_float4(er ? er[(int64_t)v * H + h] : 0.f, row_max[(int64_t)v * H + h], l > 0.f ? 1.f / l : 0.f, t);
    }
  }
}

// ---------------------------------------------------------------------------
// src phase: one warp per (head, source row u) over the out-CSR
// ---------------------------------------------------------------------------

// 4 blocks x 4 warps (16 warps, <= 128 registers) per SM with 4 steps in flight: the src pass carries ft[u] and the
// dot product besides the accumulators, and prefers registers over occupancy (profiles/r01_sweeps.md)
#ifdef BG_NS_BWD
__host__ __device__ constexpr int steps_in_flight_bwd(int) { return BG_NS_BWD; }
#else
__host__ __device__ constexpr int steps_in_flight_bwd(int vpl) { return vpl <= 3 ? 4 : vpl <= 6 ? 2 : 1; }
#endif

template <int VW, int GSH, int VPL>
__global__ void __launch_bounds__(kWarpsPerBlock * 32, bwd_min_blocks(VPL)) gat_bwd_src_kernel(const BwdParams p) {
  constexpr int NS = steps_in_flight_bwd(VPL);
  constexpr int G = 1 << GSH;
  constexpr int EPS = 32 >> GSH;
  constexpr int GSTRIDE = G * VW;
  constexpr bool kPacked = NS > 1 && NS <= G && (NS & (NS - 1)) == 0;  // packed dot-product reduction usable
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int hl = blockIdx.x / p.blocks_per_slab;  // head within this launch's range
  const int h = hl + p.h_begin;
  const int item = (blockIdx.x - hl * p.blocks_per_slab) * kWarpsPerBlock + warp;
  if (item >= p.n_items) return;
  const int row = p.seg_row ? p.seg_row[item] : item;
  const int slot = p.seg_row ? p.seg_slot[item] : -1;
  const int grp = lane >> GSH;
  const int v0 = (lane & (G - 1)) - (((h * p.D) / VW) & p.omask);

  // per-slot base pointers into g' (bytes); out-of-slab (lane, slot) pairs are clamped onto the nearest
  // vector of the slab (same line, no extra sector) and meet fu = 0 / an accumulator that is never stored
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

  const int beg = p.seg_row ? p.seg_beg[item] : p.indptr[row];
  const int end = p.seg_row ? p.seg_end[item] : p.indptr[row + 1];
  const float slope = p.slope;
  const float csu = p.cs ? p.cs[row] : 1.f;
  const float el_u = p.el[(int64_t)row * p.H + h];
  Vec<VW> fu[VPL], acc[VPL];
  {
    const float* f = p.ft + (int64_t)row * p.ld_ft + h * p.D + v0 * VW;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      if (act[i]) { fu[i].load(f + i * GSTRIDE); fu[i].scale(csu); } else fu[i].zero();
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
  const int H = p.H;
  const bool philox = (p.am == nullptr) && (p.amul_e == nullptr) && p.attn_p > 0.f;
  const bool need_eid = ee_h || amul_h || keep || philox || gze_h;
  float gel_lane = 0.f;

  // 3-stage software pipeline, as in the forward: index (c+2) | records (c+1) | row gathers (c)
  auto load_index = [&](int base, int& v, int& k) {
    const int pos = base + lane;
    v = k = 0;
    if (pos < end) {
      v = __ldg(p.indices + pos);
      if (need_eid) k = __ldg(p.eid + pos);
    }
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
      o.eb = eb_h ? __ldg(eb_h + pos) : 0.f;
      if (ee_h) o.ee = __ldg(ee_h + (int64_t)k * H);
      if (keep) o.kp = __ldg(keep + k);
      if (am_h) o.amul = __ldg(am_h + pos);
      if (amul_h) o.ame = __ldg(amul_h + (int64_t)k * H);
      if (philox) o.amp = philox_dropout_mul(p.seed, (uint32_t)k, (uint32_t)h, p.attn_p, p.inv_keep);
    }
  };
  // one step: the group's neighbour row is in x; acc += w*x, and the dot <x, ft[u]> goes to the owner lane
  auto consume = [&](const Vec<VW>(&x)[VPL], float w, int e_s, float& d_lane) {
    float part = 0.f;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      acc[i].fma(w, x[i]);
      part = x[i].dot(fu[i], part);  // fu is 0 on slots this lane does not own
    }
#pragma unroll
    for (int o = G >> 1; o > 0; o >>= 1) part += __shfl_xor_sync(kFull, part, o);
    const float got = __shfl_sync(kFull, part, ((lane - e_s) << GSH) & 31);
    if (lane >= e_s && lane < e_s + EPS) d_lane = got;
  };

  int vtx0, vtx1, vtx2 = 0, k0, k1, k2 = 0;
  load_index(beg, vtx0, k0);
  load_index(beg + 32, vtx1, k1);
  SrcOps o0, o1;
  load_operands(beg, vtx0, k0, o0);

  for (int base = beg; base < end; base += 32) {
    const int cnt = min(32, end - base);
    load_index(base + 64, vtx2, k2);
    load_operands(base + 32, vtx1, k1, o1);

    // lane = neighbour: recompute the attention weight of this edge
    const float z = el_u + o0.rec.x + o0.logit_term();
    const float s = leaky_relu(z, slope);
    const float alpha = (s == -INFINITY) ? 0.f : __expf(s - o0.rec.y) * o0.rec.z;
    const float dz = z > 0.f ? 1.f : slope;
    const float am0 = o0.multiplier();
    const float w_lane = alpha * am0;
    float d_lane = 0.f;

    int e = 0;
    for (; e + NS * EPS <= cnt; e += NS * EPS) {
      Vec<VW> x[NS][VPL];
      float w[NS];
#pragma unroll
      for (int s_ = 0; s_ < NS; ++s_) {
        const int my = e + s_ * EPS + grp;
        const size_t off = (size_t)(unsigned)__shfl_sync(kFull, vtx0, my) * ldb;
        w[s_] = __shfl_sync(kFull, w_lane, my);
#pragma unroll
        for (int i = 0; i < VPL; ++i) x[s_][i].load(reinterpret_cast<const float*>(bp[i] + off));
      }
      if constexpr (kPacked) {
        // NS partial dots per lane -> one packed butterfly over the G lanes of the group: at every level
        // each lane hands half of its live values to its partner (k/2 shuffles) instead of reducing every
        // value on its own (k shuffles).  Afterwards step s's sum sits in lanes [s*G/NS, (s+1)*G/NS) of
        // the group, and ONE indexed shuffle hands all NS*EPS dots to the lanes that own those neighbours.
        float part[NS];
#pragma unroll
        for (int s_ = 0; s_ < NS; ++s_) {
          part[s_] = 0.f;
#pragma unroll
          for (int i = 0; i < VPL; ++i) {
            acc[i].fma(w[s_], x[s_][i]);
            part[s_] = x[s_][i].dot(fu[i], part[s_]);  // fu is 0 on slots this lane does not own
          }
        }
        int k = NS;
#pragma unroll
        for (int o = G >> 1; o > 0; o >>= 1) {
          if (k > 1) {
            const bool upper = (lane & o) != 0;
#pragma unroll
            for (int i = 0; i < NS / 2; ++i) {
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
        const int t = lane - e;  // which of the NS*EPS neighbours of this iteration the lane owns
        const int from = ((t & (EPS - 1)) << GSH) + (t / EPS) * (G / NS);
        const float got = __shfl_sync(kFull, part[0], from & 31);
        if (t >= 0 && t < NS * EPS) d_lane = got;
      } else {
#pragma unroll
        for (int s_ = 0; s_ < NS; ++s_) consume(x[s_], w[s_], e + s_ * EPS, d_lane);
      }
    }
    for (; e < cnt; e += EPS) {
      // a group past the end re-reads the chunk's last neighbour; its weight is 0 and its dot is not delivered
      const int my = e + grp;
      const int src = min(my, cnt - 1);
      const size_t off = (size_t)(unsigned)__shfl_sync(kFull, vtx0, src) * ldb;
      const float ww = __shfl_sync(kFull, w_lane, src);
      Vec<VW> x[VPL];
#pragma unroll
      for (int i = 0; i < VPL; ++i) x[i].load(reinterpret_cast<const float*>(bp[i] + off));
      consume(x, my < cnt ? ww : 0.f, e, d_lane);
    }
    // d_lane = <src_scale*ft[u], g'[v]>; softmax + leaky_relu adjoint (App. A.3)
    const float gz = alpha * (d_lane * am0 - o0.rec.w) * dz;
    if (gz_h && lane < cnt) gz_h[base + lane] = gz;
    if (gze_h && lane < cnt) gze_h[(int64_t)k0 * H] = gz;
    gel_lane += gz;
    vtx0 = vtx1; vtx1 = vtx2; k0 = k1; k1 = k2; o0 = o1;
  }

#pragma unroll
  for (int o = G; o < 32; o <<= 1) {
#pragma unroll
    for (int i = 0; i < VPL; ++i) acc[i].add_shfl_xor(o);
  }
  const float gel = warp_sum(gel_lane);
  if (slot >= 0) {
    // segment of a split row: partial grad_el and (unscaled) partial grad_ft go to this segment's scratch slot
    float* sl = p.scratch + (int64_t)slot * bwd_slot_floats(H, p.D);
    if (grp == 0) {
      float* o = sl + (int64_t)h * p.D + v0 * VW;
#pragma unroll
      for (int i = 0; i < VPL; ++i)
        if (act[i]) acc[i].store(o + i * GSTRIDE);
    }
    if (lane == 0) sl[H * p.D + h] = gel;
    return;
  }
  if (grp == 0) {
    float* o = p.grad_ft + (int64_t)row * p.ld_gft + h * p.D + v0 * VW;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      if (act[i]) {
        acc[i].scale(csu);
        acc[i].store(o + i * GSTRIDE);
      }
    }
  }
  if (lane == 0) p.grad_el[(int64_t)row * p.H + h] = gel;
}

static int launch_src(const BwdParams& p, const SrcPlan& plan, cudaStream_t st) {
  const Tiling& t = plan.t;
  const bool launched = with_combo(t.vw, t.gshift, t.vpl, [&](auto vw, auto gsh, auto vpl) {
    gat_bwd_src_kernel<vw.value, gsh.value, vpl.value><<<plan.grid, kWarpsPerBlock * 32, 0, st>>>(p);
  });
  BG_REQUIRE(launched, "backward: no kernel for vw=%d lanes=%d slots=%d", t.vw, 1 << t.gshift, t.vpl);
  BG_LAUNCHED(1);
  return 0;
}

}  // namespace botgat

using namespace botgat;

extern "C" int botgat_gat_backward(const botgat_graph* g, const botgat_bwd_args* a, void* stream) {
  BG_REQUIRE(g && a, "backward: null graph/args");
  BG_REQUIRE(a->H > 0 && a->D > 0, "backward: bad H=%d D=%d", a->H, a->D);
  DeviceGuard guard(g->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (g->n_dst == 0 || g->n_src == 0) {
    // no destination rows (an empty row range of the 1-D partition still has n_src > 0 halo sources): every gradient
    // is exactly zero — write the zeros, the caller's buffers are uninitialised and may be reduce-scattered to peers.
    // (Checked before the null-pointer tests below: empty tensors legitimately have null data pointers.)
    const int ph = a->phases ? a->phases : 7;
    if ((ph & 2) && g->n_src > 0) {
      BG_REQUIRE(a->grad_ft && a->grad_el && a->ld_gft >= (int64_t)a->H * a->D, "backward: null grad_ft/grad_el");
      BG_CHECK(cudaMemset2DAsync(a->grad_ft, sizeof(float) * a->ld_gft, 0, sizeof(float) * a->H * a->D, (size_t)g->n_src, st));
      BG_CHECK(cudaMemsetAsync(a->grad_el, 0, sizeof(float) * (size_t)g->n_src * a->H, st));
    }
    if ((ph & 4) && a->grad_er && g->n_dst > 0)
      BG_CHECK(cudaMemsetAsync(a->grad_er, 0, sizeof(float) * (size_t)g->n_dst * a->H, st));
    if ((ph & 4) && a->grad_ee && g->n_edges > 0)
      BG_CHECK(cudaMemsetAsync(a->grad_ee, 0, sizeof(float) * (size_t)g->n_edges * (a->ld_gee > 0 ? a->ld_gee : a->H), st));
    return 0;
  }
  BG_REQUIRE(a->ft && a->el && a->out && a->row_max && a->row_sum && a->gout, "backward: null input");
  BG_REQUIRE(a->drec && a->grad_ft && a->grad_el, "backward: null drec/grad_ft/grad_el");
  BG_REQUIRE(!a->dst_scale || a->gprime, "backward: gprime workspace required with dst_scale");
  BG_REQUIRE(!a->grad_er || a->grad_ee || g->n_edges == 0,
             "backward: grad_er needs the grad_ee buffer (it is reduced from it)");
  BG_REQUIRE(!(a->eb_out && (a->ee || a->keep)), "backward: pass edge logits either staged (eb_out) or by edge id (ee/keep)");
  BG_REQUIRE(!(a->am_out && a->attn_mul), "backward: pass the dropout multiplier either staged or by edge id");
  // with the kept-edge subset the src pass writes gz compacted and phase 4 gives the dropped edges their zeros
  BG_REQUIRE(!a->subset_out || (a->eb_out && (a->gz || !a->grad_ee)),
             "backward: a kept-edge subset goes with eb_out and, for grad_ee, the gz workspace");
  const int64_t HD = (int64_t)a->H * a->D;
  BG_REQUIRE(a->ld_ft >= HD && a->ld_out >= HD && a->ld_gft >= HD, "backward: leading dimension < H*D");
  BG_REQUIRE(a->eb_out ? (a->Hb == 1 || a->Hb == a->H) : true, "backward: Hb must be 1 or H");
  dim3 block(kWarpsPerBlock * 32);
  const int phases = a->phases ? a->phases : 7;
  const int64_t ld_gee = a->ld_gee > 0 ? a->ld_gee : a->H;
  BG_REQUIRE(a->gz || ld_gee == a->H, "backward: a padded grad_ee needs the staged path (gz workspace)");

  BG_REQUIRE(g->n_dst * (int64_t)a->H < (1ll << 31), "backward: n_dst * H must be < 2^31");
  const float* gp = a->dst_scale ? a->gprime : a->gout;
  BwdParams p;
  SrcPlan plan;
  if (phases & 3) {
    // the src pass's plan also fixes the layout the node phase writes the records in
    p.n_dst = (int)g->n_dst; p.n_edges = g->n_edges;
    p.H = a->H; p.D = a->D; p.ld_ft = a->ld_ft; p.ld_g = a->ld_out; p.ld_gft = a->ld_gft;
    p.ft = a->ft; p.el = a->el; p.cs = a->src_scale; p.g = gp; p.drec = (const float4*)a->drec;
    p.Hb = a->Hb; p.slope = a->slope; p.attn_p = a->attn_p; p.inv_keep = 1.f / (1.f - a->attn_p); p.seed = a->seed;
    p.grad_ft = a->grad_ft; p.grad_el = a->grad_el;
    p.ee = a->ee; p.keep = a->keep; p.amul_e = a->attn_mul;
    // grad_ee is written straight in edge-id order by the src pass unless the caller supplies the staged
    // workspace gz (then phase 4 un-stages it)
    p.gz = a->gz; p.gz_e = a->gz ? nullptr : a->grad_ee;
    p.indptr = g->out_indptr; p.indices = g->out_indices; p.eid = g->out_eid;
    p.n_rows = (int)g->n_src; p.eb = a->eb_out; p.am = a->am_out;
    const botgat_graph::SegTable& seg = g->seg_out;
    const bool split = seg.n_items > 0;   // every kernel family works on (row | segment) items
    BG_REQUIRE(!split || seg.n_slots == 0 || a->scratch, "backward: this graph has split rows; scratch is required");
    p.seg_row = split ? seg.row : nullptr; p.seg_beg = seg.beg; p.seg_end = seg.end; p.seg_slot = seg.slot;
    p.n_items = split ? seg.n_items : p.n_rows; p.scratch = a->scratch;
    if (const botgat_edge_subset* s = a->subset_out) {
      // the kept edges only; plan_src still sees the full graph (as the forward's plan does)
      BG_REQUIRE(s->indptr && s->indices && (!split || (s->seg_beg && s->seg_end)), "backward: incomplete kept-edge subset");
      BG_REQUIRE(s->eid || a->am_out || !(a->attn_p > 0.f), "backward: in-kernel attention dropout needs the subset's eid");
      p.indptr = s->indptr; p.indices = s->indices; p.eid = s->eid;
      if (split) { p.seg_beg = s->seg_beg; p.seg_end = s->seg_end; }
    }
    p.blocks_per_slab = (p.n_items + kWarpsPerBlock - 1) / kWarpsPerBlock;
    p.h_begin = a->h_begin;
    p.h_count = a->h_count > 0 ? a->h_count : a->H - a->h_begin;
    BG_REQUIRE(p.h_begin >= 0 && p.h_count > 0 && p.h_begin + p.h_count <= a->H, "backward: bad head range [%d, +%d) of %d", a->h_begin, a->h_count, a->H);
    BG_REQUIRE(!split || p.h_count == a->H, "backward: a graph with split rows needs the full head range");
    const int rc = plan_src(Knobs::read(), p, &plan);
    if (rc) return rc;
    p.omask = plan.t.omask;
    p.drec_hs = plan.records_node_major ? 1 : (int)g->n_dst;
    p.drec_vs = plan.records_node_major ? a->H : 1;
  }
  if (phases & 1) {
    dim3 grid((unsigned)((g->n_dst + kWarpsPerBlock - 1) / kWarpsPerBlock));
    gat_bwd_node_kernel<<<grid, block, 0, st>>>((int)g->n_dst, a->H, a->D, a->ld_out, a->out, a->gout, a->er,
                                                a->row_max, a->row_sum, a->dst_scale, (float4*)a->drec, p.drec_hs, p.drec_vs,
                                                a->dst_scale ? a->gprime : nullptr);
    BG_LAUNCHED(1);
    BG_CHECK(cudaGetLastError());
  }

  if (phases & 2) {
    int rc = plan.family == Family::rowwise || plan.family == Family::rowbulk ? launch_src_rowwise(p, plan, st)
             : plan.family == Family::tma                                     ? launch_src_tma(p, plan, st)
             : plan.family == Family::lowdeg                                  ? launch_src_lowdeg(p, plan, st)
                                                                              : launch_src(p, plan, st);
    if (rc) return rc;
    if (p.seg_row) {
      rc = launch_bwd_combine(g->seg_out, a->H, a->D, a->ld_gft, a->scratch, a->src_scale, a->grad_ft, a->grad_el, st);
      if (rc) return rc;
    }
    BG_CHECK(cudaGetLastError());
  }

  if ((phases & 4) && a->grad_ee && a->gz && g->n_edges > 0) {
    int rc = botgat_edge_unstage(g, BOTGAT_ORDER_OUT, a->H, a->gz, a->grad_ee, ld_gee, a->subset_out, stream);
    if (rc) return rc;
  }
  if ((phases & 4) && a->grad_er) {
    // the reduce's own scratch (n_slots_in * H floats) sits behind the src pass's slots
    float* rscratch = a->scratch ? a->scratch + (int64_t)g->seg_out.n_slots * bwd_slot_floats(a->H, a->D) : nullptr;
    int rc = botgat_edge_reduce_dst(g, a->H, a->grad_ee, ld_gee, a->grad_er, rscratch, stream);
    if (rc) return rc;
  }
  return 0;
}
