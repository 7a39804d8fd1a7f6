// Kernel parameter blocks shared by the warp-per-row and the group-per-row gather kernels.
#pragma once
#include "common.cuh"

namespace botgat {

// Fused layer epilogue of the forward (the elementwise tail of a reference layer in inference: residual adds, the
// eval-mode norm as a per-column scale / shift, ReLU; src/no-sampling/models.py:720-731,
// src/ogbn-proteins/models.py:159-160,253-260), applied where an output vector is still in registers:
//   out[v, c] = dst_scale[v] * agg[v, c] + res[v, c] + res2[v, c]       y[v, c] = act(out[v, c] * scale[c] + shift[c])
struct Epilogue {
  const float *res, *res2;
  int64_t ld_res, ld_res2;
  const float *scale, *shift;  // (H*D) or null (= 1 / 0)
  int relu;
  float* y;
  int64_t ld_y;
  __host__ __device__ bool any() const { return res || res2 || y; }
  // `a` holds dst_scale * agg of columns [col, col + VW) of row `row`; on return it holds `out`
  template <int VW>
  __device__ __forceinline__ void apply(Vec<VW>& a, int64_t row, int64_t col) const {
#ifdef BG_NO_EPILOGUE  // developer A/B builds: what the fused tail costs the training-path forward
    return;
#endif
    Vec<VW> t;
    if (res) { t.load(res + row * ld_res + col); a.add(t); }
    if (res2) { t.load(res2 + row * ld_res2 + col); a.add(t); }
    if (y) {
      Vec<VW> r = a;
      if (scale) { t.load(scale + col); r.mul(t); }
      if (shift) { t.load(shift + col); r.add(t); }
      if (relu) r.relu();
      r.store(y + row * ld_y + col);
    }
  }
};

struct FwdParams {
  const int32_t* indptr;
  const int32_t* indices;
  const int32_t* eid;
  int n_rows;
  int64_t n_src_table;  // rows of the gathered table ft
  int64_t n_edges;
  int H, D;
  int64_t ld_ft, ld_out;
  const float *ft, *el, *er, *eb, *am, *cs, *ds;
  const float *ee, *amul_e;  // edge-id-ordered operands (direct mode)
  const uint8_t* keep;
  int Hb;
  float slope, attn_p, inv_keep;
  uint64_t seed;
  float *out, *row_max, *row_sum;
  Epilogue ep;
  int col_parts, part_cols, omask;
  int blocks_per_slab;
  int h_begin, h_count;  // head range of this launch
  // row splitting (segments.cu): work items are segments when seg_row != nullptr
  const int32_t *seg_row, *seg_beg, *seg_end, *seg_slot;
  int n_items;
  float* scratch;
};

struct BwdParams {
  const int32_t* indptr;
  const int32_t* indices;
  const int32_t* eid;
  int n_rows;  // rows of the out-CSR (= n_src)
  int n_dst;
  int64_t n_edges;
  int H, D;
  int64_t ld_ft, ld_g, ld_gft;
  const float *ft, *el, *eb, *am, *cs;
  const float *ee, *amul_e;  // edge-id-ordered operands (direct mode)
  const uint8_t* keep;
  float* gz_e;         // (n_edges, H) edge-id order (direct mode), written by the src pass
  const float* g;      // g' (n_dst, ld_g)
  const float4* drec;  // per-destination records.  The head-major kernels read them head-major, drec[h * n_dst + v]; the
                       // all-heads-per-row kernels (gat_rowwise.cu) through the strides below, which are node-major
                       // (hs = 1, vs = H: one contiguous 16*H-byte read per edge) when SrcPlan::records_node_major
  int drec_hs, drec_vs;  // 32-bit: n_dst * H < 2^31 is checked at launch
  int Hb;
  float slope, attn_p, inv_keep;
  uint64_t seed;
  float *grad_ft, *grad_el, *gz;
  int omask;
  int blocks_per_slab;
  int h_begin, h_count;  // head range of this launch
  const int32_t *seg_row, *seg_beg, *seg_end, *seg_slot;
  int n_items;
  float* scratch;
};

struct SrcOps {
  float4 rec;  // {er[v], row_max[v], 1/row_sum[v], t[v]}
  // raw loads, combined one pipeline stage later by logit_term(): consuming a load where it is issued would
  // stall the warp there (even a predicated-off FADD waits for its source register)
  // every field has one producer (a default written before the loads + at most one predicated load): an
  // if / else-if chain would leave a default MOV behind the loads that waits on their scoreboard slot
  float eb, ee, amul, ame, amp;
  int kp;
  __device__ __forceinline__ float logit_term() const { return kp ? eb + ee : -INFINITY; }
  __device__ __forceinline__ float multiplier() const { return amul * ame * amp; }
};

// Kernel choice (plan.cu): one host-side planner picks the family, lane geometry and grid of every gather launch; the
// launchers below launch exactly that.  Knobs: run-time overrides of the choice (tests, sweeps), read once per ABI call
// rather than once per process because the tests switch them within one process.
struct Knobs {
  int vw;                                  // BOTGAT_VW = 1 / 2: narrower vectors than the alignment allows
  int g;                                   // BOTGAT_G: lanes per neighbour (a power of two <= 32)
  bool noalign;                            // BOTGAT_NOALIGN: no line-alignment shift
  int64_t slab_mb;                         // BOTGAT_SLAB_MB: L2 budget of one head-major slab (64)
  int64_t lowdeg_fwd, lowdeg_bwd;          // BOTGAT_LOWDEG[_BWD]: average row length below which a group owns a row
  int rowwise_fwd, rowwise_bwd;            // BOTGAT_ROWWISE[_FWD|_BWD]: 0 / 1 force the all-heads-per-row kernels; -1 = by size
  int64_t rowwise_mb_fwd, rowwise_mb_bwd;  // BOTGAT_ROWWISE_MB: table size from which they are always used (96 / 256)
  bool bwd_tma;                            // BOTGAT_BWD_TMA=0 turns the TMA src pass off
  bool rw_bulk;                            // BOTGAT_RW_BULK=0 turns the bulk-copy ring of the row-wise src pass off
  static Knobs read();
};

// host: choose the tiling.  `ld_g`/`pg` describe the GATHERED table (alignment shift is derived from it),
// `ld_o`/`po` the row-local one (only constrains the vector width).
Tiling choose_tiling(const Knobs& k, int H, int D, int64_t ld_g, const void* pg, int64_t ld_o, const void* po,
                     int col_parts_req, int64_t n_rows_table);

// warp: one warp per (head, row), gat_fwd.cu / gat_bwd.cu; lowdeg: a lane group per (head, row), gat_lowdeg.cu; rowwise /
// rowbulk: one warp per row for all heads, rows in a register ring / (src pass) a bulk-copy shared-memory ring,
// gat_rowwise.cu; tma: (src pass) one warp per (head, row) with TMA-staged rows, gat_bwd_tma.cu
enum class Family { warp, lowdeg, rowwise, rowbulk, tma };

struct FwdPlan {
  Family family;       // rowwise, lowdeg or warp
  Tiling t;
  int rw_gsh, rw_vpl;  // rowwise: log2(lanes per head), vector slots per lane
  int warps_per_slab;  // lowdeg
  unsigned grid;       // blocks
};

struct SrcPlan {
  Family family;
  Tiling t;
  int rw_gsh, rw_vpl;             // rowwise / rowbulk
  int bulk_slot_bytes;            // rowbulk: one staged row, padded to 128 bytes
  size_t bulk_ring_bytes;         // rowbulk: dynamic shared memory
  int tma_dv, tma_gsh, tma_mode;  // tma: D / 4, log2(lanes per neighbour), operand mode (gat_bwd_tma.cu)
  int warps_per_slab;             // lowdeg
  unsigned grid;                  // blocks
  bool records_node_major;        // layout the node phase writes the per-destination records in (BwdParams::drec)
};

// `p` is filled except for the tiling fields (col_parts, part_cols, omask), which come from the plan.  0 or < 0 on error.
int plan_forward(const Knobs& k, const FwdParams& p, int col_parts_req, FwdPlan* plan);
int plan_src(const Knobs& k, const BwdParams& p, SrcPlan* plan);

int launch_fwd_lowdeg(const FwdParams& p, const FwdPlan& plan, cudaStream_t st);
int launch_fwd_rowwise(const FwdParams& p, const FwdPlan& plan, cudaStream_t st);
int launch_src_lowdeg(const BwdParams& p, const SrcPlan& plan, cudaStream_t st);
int launch_src_rowwise(const BwdParams& p, const SrcPlan& plan, cudaStream_t st);  // rowwise and rowbulk
int launch_src_tma(const BwdParams& p, const SrcPlan& plan, cudaStream_t st);

// ring of the bulk-copy row-wise src pass: kBulkRing staged rows, at most kBulkRingMax bytes of shared memory
constexpr int kBulkRingLog2 = 3;  // R = 8 slots
constexpr int kBulkRing = 1 << kBulkRingLog2;
constexpr size_t kBulkRingMax = 96 * 1024;

// (log2 lanes per head, slots per lane) the all-heads-per-row kernels are instantiated for: every geometry of 1 - 8
// heads with at most 8 float4 slots
#define BG_RW_VPLS(X, GSH) X(GSH, 1) X(GSH, 2) X(GSH, 3) X(GSH, 4) X(GSH, 5) X(GSH, 6) X(GSH, 7) X(GSH, 8)
#define BG_RW_COMBOS(X) BG_RW_VPLS(X, 2) BG_RW_VPLS(X, 3) BG_RW_VPLS(X, 4) BG_RW_VPLS(X, 5)
template <class F>
inline bool with_rw_combo(int gsh, int vpl, F&& f) {
#define BG_X(GSH, VPL) if (gsh == GSH && vpl == VPL) return f(std::integral_constant<int, GSH>(), std::integral_constant<int, VPL>()), true;
  BG_RW_COMBOS(BG_X)
#undef BG_X
  return false;
}

// (D / 4, log2 lanes per neighbour) the TMA src pass is instantiated for: G = 4 where D/4 divides by 4, else G = 8
#define BG_TMA_COMBOS(X) X(4, 2) X(8, 2) X(12, 2) X(16, 2) X(20, 2) X(24, 2) X(32, 2) X(10, 3) X(30, 3) X(40, 3)
template <class F>
inline bool with_tma_combo(int dv, int gsh, F&& f) {
#define BG_X(DV, GSH) if (dv == DV && gsh == GSH) return f(std::integral_constant<int, DV>(), std::integral_constant<int, GSH>()), true;
  BG_TMA_COMBOS(BG_X)
#undef BG_X
  return false;
}

int segment_length();
// floats per scratch slot (rounded to 4 so that float4 stores into a slot stay aligned)
__host__ __device__ inline int64_t fwd_slot_floats(int H, int D) { return ((int64_t)H * (D + 2) + 3) / 4 * 4; }
__host__ __device__ inline int64_t bwd_slot_floats(int H, int D) { return ((int64_t)H * (D + 1) + 3) / 4 * 4; }
int launch_fwd_combine(const botgat_graph::SegTable& t, int H, int D, int64_t ld_out, const float* scratch,
                       const float* ds, float* out, float* row_max, float* row_sum, const Epilogue& ep, cudaStream_t st);
int launch_bwd_combine(const botgat_graph::SegTable& t, int H, int D, int64_t ld_gft, const float* scratch,
                       const float* cs, float* grad_ft, float* grad_el, cudaStream_t st);

}  // namespace botgat
