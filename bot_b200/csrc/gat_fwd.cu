// Fused GAT forward for sm_100a:
//   per-edge logits (el[src] + er[dst] + eb[edge]) -> leaky_relu -> online
//   per-destination softmax -> attention dropout -> weighted neighbour sum ->
//   degree scaling, in ONE pass over the in-CSR.  No E-sized intermediate is
//   written.  Replaces src/no-sampling/models.py:500-505,523-555 and
//   src/ogbn-proteins/models.py:125-156 of the reference (DGL apply_edges,
//   edge_softmax, update_all and the torch elementwise ops between them).
//
// L2/HBM-bound gather: no tensor cores (the only dense contraction, fc, stays a
// torch matmul).  See common.cuh "Work decomposition" for the item/lane layout.
//
// What the profiles asked for (profiles/r01_*):
//   * lane geometry (VW, G, VPL) is compile-time and every (lane, slot) has its own
//     base pointer, so a row load is one 32x32+64 IMAD plus an UNPREDICATED LDG.128
//     (lanes outside the slab re-read the nearest vector of the same line: no extra
//     sector, and their accumulators are never stored);
//   * the neighbour loop runs full steps without bounds checks and handles the row
//     tail separately;
//   * the per-neighbour scalars run in a 3-stage software pipeline — index of
//     chunk c+2, logit operands of chunk c+1 and the row gathers of chunk c are in
//     flight together, so no load waits on a load issued in the same iteration.
#include "common.cuh"
#include "params.cuh"

namespace botgat {


// 6 blocks x 4 warps (24 warps, <= 80 registers) per SM with 2 steps in flight: the best of the occupancy /
// loads-in-flight sweep on B200 (profiles/r01_sweeps.md)

// EP: the fused layer tail (inference) is compiled into its own instantiation — carried as a run-time option it cost
// the training-path forward 2.9 % at the proteins shape (5.94 vs 5.77 ms, same box, profiles/r02_sweeps.md)
template <int VW, int GSH, int VPL, bool EP>
__global__ void __launch_bounds__(kWarpsPerBlock * 32, fwd_min_blocks(VPL)) gat_fwd_kernel(const FwdParams p) {
  constexpr int NS = steps_in_flight(VPL);
  constexpr int G = 1 << GSH;     // lanes per neighbour
  constexpr int EPS = 32 >> GSH;  // neighbours per warp step
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int slab = blockIdx.x / p.blocks_per_slab;
  const int item = (blockIdx.x - slab * p.blocks_per_slab) * kWarpsPerBlock + warp;
  if (item >= p.n_items) return;
  // work item = a whole row, or one segment of a heavy row (segments.cu)
  const int row = p.seg_row ? p.seg_row[item] : item;
  const int slot = p.seg_row ? p.seg_slot[item] : -1;
  const int hl = slab / p.col_parts;  // head within this launch's range
  const int h = hl + p.h_begin;
  const int cp = slab - hl * p.col_parts;
  const int c0 = cp * p.part_cols;
  const int nv = (min(p.D - c0, p.part_cols) + VW - 1) / VW;  // vectors in this slab row
  const int grp = lane >> GSH;
  // first vector of this lane, shifted so that every slot is 128-byte-line aligned
  const int v0 = (lane & (G - 1)) - (((h * p.D + c0) / VW) & p.omask);

  // per-slot base pointers (bytes).  A (lane, slot) outside the slab is clamped onto the nearest
  // vector inside it; it then loads real data into an accumulator that is never stored.
  const char* bp[VPL];
  bool act[VPL];
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const int v = v0 + i * G;
    act[i] = v >= 0 && v < nv;
    bp[i] = reinterpret_cast<const char*>(p.ft + h * p.D + c0 + min(max(v, 0), nv - 1) * VW);
  }
  const unsigned ldb = (unsigned)(p.ld_ft * 4);

  const int beg = p.seg_row ? p.seg_beg[item] : p.indptr[row];
  const int end = p.seg_row ? p.seg_end[item] : p.indptr[row + 1];
  const float slope = p.slope;
  const int H = p.H;
  const float er_v = p.er ? p.er[(int64_t)row * H + h] : 0.f;
  const float* __restrict__ el_h = p.el + h;
  const float* __restrict__ eb_h = p.eb ? p.eb + (int64_t)(p.Hb == 1 ? 0 : h) * p.n_edges : nullptr;
  const float* __restrict__ am_h = p.am ? p.am + (int64_t)h * p.n_edges : nullptr;
  const float* __restrict__ cs = p.cs;
  const float* __restrict__ ee_h = p.ee ? p.ee + h : nullptr;
  const float* __restrict__ amul_h = p.amul_e ? p.amul_e + h : nullptr;
  const uint8_t* __restrict__ keep = p.keep;
  const bool philox = (p.am == nullptr) && (p.amul_e == nullptr) && p.attn_p > 0.f;
  // direct mode: per-edge operands are indexed by edge id inside the pipeline (random 32-byte sectors from
  // DRAM, which this L2-bound kernel leaves idle) instead of being permuted into CSR order by a staging pass
  const bool need_eid = ee_h || amul_h || keep || philox;

  Vec<VW> acc[VPL];
#pragma unroll
  for (int i = 0; i < VPL; ++i) acc[i].zero();
  float m = -INFINITY;  // running row max (warp-uniform)
  float l_lane = 0.f;   // this lane's share of sum exp(s - m)

  // ---- software pipeline over 32-neighbour chunks ----
  // stage 0: neighbour index; stage 1: logit operands (need the index); stage 2: row gathers
  auto load_index = [&](int base, int& u, int& k) {
    const int pos = base + lane;
    u = k = 0;
    if (pos < end) {
      u = __ldg(p.indices + pos);
      if (need_eid) k = __ldg(p.eid + pos);
    }
  };
  // raw loaded values only: any arithmetic on them here would stall on the load just issued and undo the pipeline
  // Raw operands of one chunk, combined one iteration later.  Every field has ONE producer: a default written
  // before the loads and at most one predicated load.  (With an if / else-if chain ptxas puts the default into the
  // else branch BEHIND the load; that MOV then waits on the scoreboard slot the freshly issued loads share —
  // 12 % of the kernel's stall samples in profiles/r01_g.)
  struct Ops { float el, eb, ee, cs, am, ame, amp; unsigned keep; };
  auto load_operands = [&](int base, int u, int k, Ops& o) {
    const int pos = base + lane;
    o.el = -INFINITY;  // lane past the row end: logit -inf, weight 0
    o.eb = 0.f; o.ee = 0.f; o.cs = 1.f; o.am = 1.f; o.ame = 1.f; o.amp = 1.f; o.keep = 1u;
    if (pos < end) {
      o.el = __ldg(el_h + (int64_t)u * H);
      if (eb_h) o.eb = __ldg(eb_h + pos);
      if (ee_h) o.ee = __ldg(ee_h + (int64_t)k * H);
      if (keep) o.keep = __ldg(keep + k);
      if (cs) o.cs = __ldg(cs + u);
      if (am_h) o.am = __ldg(am_h + pos);
      if (amul_h) o.ame = __ldg(amul_h + (int64_t)k * H);
      if (philox) o.amp = philox_dropout_mul(p.seed, (uint32_t)k, (uint32_t)h, p.attn_p, p.inv_keep);
    }
  };
  int u0, u1, u2 = 0, k0, k1, k2 = 0;
  load_index(beg, u0, k0);
  load_index(beg + 32, u1, k1);
  Ops o0, o1;
  load_operands(beg, u0, k0, o0);

  for (int base = beg; base < end; base += 32) {
    const int cnt = min(32, end - base);
    // issue the next stages' loads first; they are consumed one iteration later
    load_index(base + 64, u2, k2);
    load_operands(base + 32, u1, k1, o1);

    // ---- online softmax on chunk c ----
    const float z0 = o0.keep ? o0.el + er_v + (o0.eb + o0.ee) : -INFINITY;
    const float mul0 = o0.cs * (o0.am * o0.ame * o0.amp);
    const float s = leaky_relu(z0, slope);  // -inf stays -inf (dropped edge / lane past the row end)
    const float m_new = fmaxf(m, warp_max(s));
    if (m_new > m) {
      const float f = __expf(m - m_new);  // m == -inf -> 0, and everything accumulated so far is 0
      l_lane *= f;
#pragma unroll
      for (int i = 0; i < VPL; ++i) acc[i].scale(f);
      m = m_new;
    }
    const float pexp = (s == -INFINITY) ? 0.f : __expf(s - m);
    l_lane += pexp;
    const float w_lane = pexp * mul0;

    // ---- group = neighbour: gather slab rows, acc += w * row ----
    int e = 0;
    // full iterations: NS steps, every group has a neighbour
    for (; e + NS * EPS <= cnt; e += NS * EPS) {
      Vec<VW> x[NS][VPL];
      float w[NS];
#pragma unroll
      for (int s_ = 0; s_ < NS; ++s_) {
        const int my = e + s_ * EPS + grp;
        const size_t off = (size_t)(unsigned)__shfl_sync(kFull, u0, my) * ldb;
        w[s_] = __shfl_sync(kFull, w_lane, my);
#pragma unroll
        for (int i = 0; i < VPL; ++i) x[s_][i].load(reinterpret_cast<const float*>(bp[i] + off));
      }
#pragma unroll
      for (int s_ = 0; s_ < NS; ++s_) {
#pragma unroll
        for (int i = 0; i < VPL; ++i) acc[i].fma(w[s_], x[s_][i]);
      }
    }
    // tail: single steps; a group past the end re-reads the chunk's last neighbour with weight 0
    for (; e < cnt; e += EPS) {
      const int my = e + grp;
      const int src = min(my, cnt - 1);
      const size_t off = (size_t)(unsigned)__shfl_sync(kFull, u0, src) * ldb;
      const float ww = __shfl_sync(kFull, w_lane, src);
      Vec<VW> x[VPL];
#pragma unroll
      for (int i = 0; i < VPL; ++i) x[i].load(reinterpret_cast<const float*>(bp[i] + off));
      const float wt = my < cnt ? ww : 0.f;
#pragma unroll
      for (int i = 0; i < VPL; ++i) acc[i].fma(wt, x[i]);
    }
    u0 = u1; u1 = u2; k1 = k2; o0 = o1;
  }

  // ---- epilogue: combine the groups, normalise, degree-scale, store ----
  const float l = warp_sum(l_lane);
#pragma unroll
  for (int o = G; o < 32; o <<= 1) {
#pragma unroll
    for (int i = 0; i < VPL; ++i) acc[i].add_shfl_xor(o);
  }
  if (slot >= 0) {
    // segment of a split row: park (max, sum, unnormalised accumulator) in this segment's scratch slot
    float* sl = p.scratch + (int64_t)slot * fwd_slot_floats(H, p.D);
    if (grp == 0) {
      float* o = sl + (int64_t)h * p.D + c0 + v0 * VW;
#pragma unroll
      for (int i = 0; i < VPL; ++i)
        if (act[i]) acc[i].store(o + i * G * VW);
    }
    if (cp == 0 && lane == 0) { sl[H * p.D + h * 2] = m; sl[H * p.D + h * 2 + 1] = l; }
    return;
  }
  float scale = l > 0.f ? 1.f / l : 0.f;
  if (p.ds) scale *= p.ds[row];
  if (grp == 0) {
    float* o = p.out + (int64_t)row * p.ld_out + h * p.D + c0 + v0 * VW;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      if (act[i]) {
        acc[i].scale(scale);
        if constexpr (EP) p.ep.apply(acc[i], row, (int64_t)h * p.D + c0 + (v0 + i * G) * VW);
        acc[i].store(o + i * G * VW);
      }
    }
  }
  if (cp == 0 && lane == 0) {
    p.row_max[(int64_t)row * H + h] = m;
    p.row_sum[(int64_t)row * H + h] = l;
  }
}

static int launch_fwd(const FwdParams& p, const FwdPlan& plan, cudaStream_t st) {
  const Tiling& t = plan.t;
  const bool launched = with_combo(t.vw, t.gshift, t.vpl, [&](auto vw, auto gsh, auto vpl) {
    if (p.ep.any())
      gat_fwd_kernel<vw.value, gsh.value, vpl.value, true><<<plan.grid, kWarpsPerBlock * 32, 0, st>>>(p);
    else
      gat_fwd_kernel<vw.value, gsh.value, vpl.value, false><<<plan.grid, kWarpsPerBlock * 32, 0, st>>>(p);
  });
  BG_REQUIRE(launched, "forward: no kernel for vw=%d lanes=%d slots=%d", t.vw, 1 << t.gshift, t.vpl);
  BG_LAUNCHED(1);
  return 0;
}

}  // namespace botgat

using namespace botgat;

extern "C" int botgat_gat_forward(const botgat_graph* g, const botgat_fwd_args* a, void* stream) {
  BG_REQUIRE(g && a, "forward: null graph/args");
  BG_REQUIRE(a->H > 0 && a->D > 0, "forward: bad H=%d D=%d", a->H, a->D);
  if (g->n_dst == 0) return 0;  // nothing to write; empty outputs legitimately have null data pointers
  BG_REQUIRE(a->ft && a->el && a->out && a->row_max && a->row_sum, "forward: null ft/el/out/row_max/row_sum");
  BG_REQUIRE(a->ld_ft >= (int64_t)a->H * a->D && a->ld_out >= (int64_t)a->H * a->D, "forward: leading dimension < H*D");
  BG_REQUIRE(a->ld_ft < (1ll << 30), "forward: ld_ft too large");
  BG_REQUIRE(a->eb ? (a->Hb == 1 || a->Hb == a->H) : true, "forward: Hb must be 1 or H when eb is given (got %d)", a->Hb);
  BG_REQUIRE(!(a->eb && (a->ee || a->keep)), "forward: pass edge logits either staged (eb) or by edge id (ee/keep)");
  BG_REQUIRE(!(a->am && a->attn_mul), "forward: pass the dropout multiplier either staged (am) or by edge id (attn_mul)");
  BG_REQUIRE(a->attn_p >= 0.f && a->attn_p < 1.f, "forward: attn_p must be in [0,1)");
  DeviceGuard guard(g->device);
  cudaStream_t st = (cudaStream_t)stream;

  const int64_t HDf = (int64_t)a->H * a->D;
  BG_REQUIRE(!a->res || a->ld_res >= HDf, "forward: ld_res < H*D");
  BG_REQUIRE(!a->res2 || a->ld_res2 >= HDf, "forward: ld_res2 < H*D");
  BG_REQUIRE(!a->y || a->ld_y >= HDf, "forward: ld_y < H*D");
  BG_REQUIRE(a->y || (!a->ep_scale && !a->ep_shift && !a->ep_relu), "forward: the epilogue's scale / shift / relu need y");
  FwdParams p;
  p.indptr = g->in_indptr; p.indices = g->in_indices; p.eid = g->in_eid;
  p.n_rows = (int)g->n_dst; p.n_src_table = g->n_src; p.n_edges = g->n_edges;
  p.H = a->H; p.D = a->D; p.ld_ft = a->ld_ft; p.ld_out = a->ld_out;
  p.ft = a->ft; p.el = a->el; p.er = a->er; p.eb = a->eb; p.am = a->am;
  p.cs = a->src_scale; p.ds = a->dst_scale; p.Hb = a->Hb;
  p.ee = a->ee; p.keep = a->keep; p.amul_e = a->attn_mul;
  p.slope = a->slope; p.attn_p = a->attn_p; p.inv_keep = 1.f / (1.f - a->attn_p); p.seed = a->seed;
  p.out = a->out; p.row_max = a->row_max; p.row_sum = a->row_sum;
  p.ep.res = a->res; p.ep.ld_res = a->ld_res; p.ep.res2 = a->res2; p.ep.ld_res2 = a->ld_res2;
  p.ep.scale = a->ep_scale; p.ep.shift = a->ep_shift; p.ep.relu = a->ep_relu; p.ep.y = a->y; p.ep.ld_y = a->ld_y;
  const botgat_graph::SegTable& seg = g->seg_in;
  const bool split = seg.n_items > 0;   // both kernel families work on (row | segment) items
  BG_REQUIRE(!split || seg.n_slots == 0 || a->scratch, "forward: this graph has split rows; scratch is required");
  p.seg_row = split ? seg.row : nullptr; p.seg_beg = seg.beg; p.seg_end = seg.end; p.seg_slot = seg.slot;
  p.n_items = split ? seg.n_items : p.n_rows; p.scratch = a->scratch;
  if (const botgat_edge_subset* s = a->subset) {
    // the kept edges only; the plan below still sees the full graph (n_edges, n_rows, the table), so every call picks the
    // kernel it picks without the subset
    BG_REQUIRE(a->eb, "forward: a kept-edge subset goes with the edge logits staged with it (eb)");
    BG_REQUIRE(s->indptr && s->indices && (!split || (s->seg_beg && s->seg_end)), "forward: incomplete kept-edge subset");
    BG_REQUIRE(s->eid || a->am || !(a->attn_p > 0.f), "forward: in-kernel attention dropout needs the subset's eid");
    p.indptr = s->indptr; p.indices = s->indices; p.eid = s->eid;
    if (split) { p.seg_beg = s->seg_beg; p.seg_end = s->seg_end; }
  }
  p.blocks_per_slab = (p.n_items + kWarpsPerBlock - 1) / kWarpsPerBlock;
  p.h_begin = a->h_begin;
  p.h_count = a->h_count > 0 ? a->h_count : a->H - a->h_begin;
  BG_REQUIRE(p.h_begin >= 0 && p.h_count > 0 && p.h_begin + p.h_count <= a->H, "forward: bad head range [%d, +%d) of %d", a->h_begin, a->h_count, a->H);
  BG_REQUIRE(!split || p.h_count == a->H, "forward: a graph with split rows needs the full head range");
  FwdPlan plan;
  int rc = plan_forward(Knobs::read(), p, a->col_parts, &plan);
  if (rc) return rc;
  p.col_parts = plan.t.col_parts; p.part_cols = plan.t.part_cols; p.omask = plan.t.omask;
  rc = plan.family == Family::rowwise ? launch_fwd_rowwise(p, plan, st)
       : plan.family == Family::lowdeg ? launch_fwd_lowdeg(p, plan, st)
                                       : launch_fwd(p, plan, st);
  if (rc) return rc;
  if (split) {
    rc = launch_fwd_combine(seg, a->H, a->D, a->ld_out, a->scratch, a->dst_scale, a->out, a->row_max, a->row_sum, p.ep, st);
    if (rc) return rc;
  }
  BG_CHECK(cudaGetLastError());
  return 0;
}
