// Which gather kernel runs each launch of the forward and of the backward src pass, and with which lane geometry and
// grid.  Pure host code: no CUDA calls, no allocations.  The launchers (gat_fwd.cu, gat_bwd.cu, gat_lowdeg.cu,
// gat_rowwise.cu, gat_bwd_tma.cu) launch what the plan names and decide nothing.
#include <algorithm>
#include <cstdlib>

#include "common.cuh"
#include "params.cuh"

namespace botgat {

const char* env_str(const char* name) {
  const char* s = getenv(name);
  return (s && *s) ? s : nullptr;
}

int64_t env_int(const char* name, int64_t dflt) {
  const char* s = env_str(name);
  return s ? atoll(s) : dflt;
}

static int env_force(const char* name, const char* fallback) {
  const char* s = env_str(name);
  if (!s) s = env_str(fallback);
  return s ? *s != '0' : -1;
}

Knobs Knobs::read() {
  Knobs k;
  k.vw = (int)env_int("BOTGAT_VW", 0);
  k.g = (int)env_int("BOTGAT_G", 0);
  k.noalign = env_int("BOTGAT_NOALIGN", 0) != 0;
  k.slab_mb = env_int("BOTGAT_SLAB_MB", 64);
  k.lowdeg_fwd = env_int("BOTGAT_LOWDEG", 20);
  k.lowdeg_bwd = env_int("BOTGAT_LOWDEG_BWD", env_int("BOTGAT_LOWDEG", 96));
  k.rowwise_fwd = env_force("BOTGAT_ROWWISE_FWD", "BOTGAT_ROWWISE");
  k.rowwise_bwd = env_force("BOTGAT_ROWWISE_BWD", "BOTGAT_ROWWISE");
  k.rowwise_mb_fwd = env_int("BOTGAT_ROWWISE_MB", 96);
  k.rowwise_mb_bwd = env_int("BOTGAT_ROWWISE_MB", 256);
  const char* tma = env_str("BOTGAT_BWD_TMA");
  const char* bulk = env_str("BOTGAT_RW_BULK");
  k.bwd_tma = !(tma && *tma == '0');
  k.rw_bulk = !(bulk && *bulk == '0');
  return k;
}

static int pow2ceil(int x) {
  int p = 1;
  while (p < x) p <<= 1;
  return p;
}

static bool fits_grid(int64_t blocks) { return blocks > 0 && blocks < (1ll << 31); }

Tiling choose_tiling(const Knobs& k, int H, int D, int64_t ld_g, const void* pg, int64_t ld_o, const void* po,
                     int col_parts_req, int64_t n_rows_table) {
  constexpr int kVplCap = 8;
  Tiling t;
  auto ok = [&](int vw) {
    return D % vw == 0 && ld_g % vw == 0 && ld_o % vw == 0 && ((uintptr_t)pg % (vw * 4)) == 0 &&
           ((uintptr_t)po % (vw * 4)) == 0;
  };
  t.vw = ok(4) ? 4 : (ok(2) ? 2 : 1);
  if ((k.vw == 1 || k.vw == 2) && k.vw < t.vw) t.vw = k.vw;
  const int gline = 32 / t.vw;  // lanes that cover one 128-byte line
  // line-alignment shift is possible when every gathered row starts on a line boundary
  bool can_align = (ld_g * 4) % 128 == 0 && ((uintptr_t)pg % 128) == 0 && !k.noalign;
  // a caller that needs the head in one part (the backward src pass) gives up the shift before the shift's extra
  // line would push the head past one pass: 32 * kVplCap vectors instead of one line fewer
  if (col_parts_req == 1 && can_align && D > (32 * kVplCap - gline) * t.vw) can_align = false;
  const int cap_cols = (32 * kVplCap - (can_align ? gline : 0)) * t.vw;  // widest part one warp covers in a pass
  int parts = col_parts_req;
  if (parts <= 0) {
    // auto: keep one (n_rows x part_cols) slab of the gathered table within the L2 budget
    const int64_t budget = k.slab_mb << 20;
    const int64_t head_bytes = n_rows_table * (int64_t)D * 4;
    parts = (int)((head_bytes + budget - 1) / budget);
    if (parts < 1) parts = 1;
    const int max_parts = D / (16 * t.vw) > 0 ? D / (16 * t.vw) : 1;  // keep parts >= 16 vectors wide
    if (parts > max_parts) parts = max_parts;
  }
  auto part_cols_of = [&](int np) {
    int pc = (D + np - 1) / np;
    return ((pc + t.vw - 1) / t.vw) * t.vw;
  };
  while (part_cols_of(parts) > cap_cols) ++parts;
  t.part_cols = part_cols_of(parts);
  t.col_parts = (D + t.part_cols - 1) / t.part_cols;
  const int nv = (t.part_cols + t.vw - 1) / t.vw;
  // lanes per neighbour: one 128-byte line per group and instruction (fewer when the part is narrower),
  // more only when the part needs over kVplCap slots
  int G = std::min(gline, pow2ceil(nv));
  if (k.g >= 1 && k.g <= 32 && (k.g & (k.g - 1)) == 0) G = k.g;
  for (;; G <<= 1) {
    t.gshift = 0;
    while ((1 << t.gshift) < G) ++t.gshift;
    t.omask = can_align ? std::min(G, gline) - 1 : 0;
    // worst-case shift over all (head, part) slab starts
    int omax = 0;
    for (int h = 0; h < H && t.omask; ++h)
      for (int cp = 0; cp < t.col_parts; ++cp) omax = std::max(omax, ((h * D + cp * t.part_cols) / t.vw) & t.omask);
    const int need = (nv + omax + G - 1) / G;
    // smallest instantiated slot count that covers the part at this group size (common.cuh BG_COMBOS)
    t.vpl = -1;
    for (int c = need; c <= kVplCap; ++c)
      if (with_combo(t.vw, t.gshift, c, [](auto, auto, auto) {})) { t.vpl = c; break; }
    if (t.vpl > 0 || G >= 32) break;
  }
  if (t.vpl < 0) t.vpl = kVplCap;  // unreachable: cap_cols guarantees a fit at G = 32
  return t;
}

// Low-degree graphs (average row shorter than `thr` neighbours) use the group-per-row kernels (gat_lowdeg.cu).  The
// thresholds were swept on B200 (profiles/r01_sweeps.md): the forward switches late (20: its chunk overhead is per G
// neighbours instead of per 32), the backward src pass early (96: its per-row prologue / epilogue is heavier, ft[u]
// load and two outputs).
static bool low_degree(int64_t thr, int64_t n_edges, int64_t n_rows) { return n_rows > 0 && n_edges < thr * n_rows; }

// lane geometry of the all-heads-per-row kernels for `heads` heads of width D: log2(lanes per head) and vector slots
// per lane; false = not covered
static bool rowwise_geometry(int heads, int D, int* gsh, int* vpl) {
  if (heads < 1 || heads > 8 || D % 4 != 0) return false;
  int hg = 1;
  while (hg < heads) hg <<= 1;
  int g = 32 / hg, s = 0;
  while ((1 << s) < g) ++s;
  const int need = (D / 4 + g - 1) / g;
  if (need > 8) return false;
  *gsh = s;
  *vpl = need;
  return true;
}

// When the all-heads-per-row kernels are used (swept on B200 with tools/rowwise_crossover.sh, profiles/r02_sweeps.md):
//   * never while a head's slab (one column part of it, forward) fits the L2 budget of the head-major order
//     (BOTGAT_SLAB_MB, 64 MB): proteins / Reddit shapes stay head-major, whatever the degree;
//   * beyond that, always for low-degree graphs (< 96 neighbours per row: 1.6 - 2x at 25 and 60 neighbours per row from a
//     69 MB slab upwards — the head-major order pays the row's dependent load chain once per head and part);
//   * for long rows only once the slab is well past the L2: forward from 96 MB (still 1.25x at 240 neighbours per row
//     and a 137 MB slab), backward src pass from 256 MB (at 137 MB and >= 120 neighbours per row the TMA src pass wins).
// BOTGAT_ROWWISE[_FWD|_BWD]=0 / 1 forces the choice (tests, sweeps); BOTGAT_ROWWISE_MB replaces both "always" sizes.
static bool rowwise_wanted(const Knobs& k, int D, int64_t n_rows_table, int64_t n_edges, int64_t n_csr_rows, bool backward) {
  const int force = backward ? k.rowwise_bwd : k.rowwise_fwd;
  if (force >= 0) return force;
  const int64_t always = (backward ? k.rowwise_mb_bwd : k.rowwise_mb_fwd) << 20;
  const int64_t resident = std::min(k.slab_mb << 20, always);
  // the forward may split a head into column parts of >= 16 vectors (choose_tiling); the src pass gathers whole heads
  const int max_parts = (!backward && D / 64 > 0) ? D / 64 : 1;
  const int64_t part_bytes = n_rows_table * (int64_t)D * 4 / max_parts;
  if (part_bytes <= resident) return false;
  // (rows of a handful of out-edges — the per-rank out-CSR of an 8-way partitioned products graph has 3 — are not what
  // the one-warp-per-row src pass was swept on: they keep the group-per-row kernel unless the table is huge)
  const bool low = n_edges < 96 * n_csr_rows && (!backward || n_edges >= 8 * n_csr_rows);
  return low || part_bytes > always;
}

int plan_forward(const Knobs& k, const FwdParams& p, int col_parts_req, FwdPlan* fp) {
  // the row-local arrays (out, residuals, y, the per-column scale / shift) constrain the vector width together
  const Epilogue& ep = p.ep;
  const int64_t ld_o = p.ld_out | (ep.res ? ep.ld_res : 0) | (ep.res2 ? ep.ld_res2 : 0) | (ep.y ? ep.ld_y : 0);
  const uintptr_t po = (uintptr_t)p.out | (uintptr_t)ep.res | (uintptr_t)ep.res2 | (uintptr_t)ep.y | (uintptr_t)ep.scale |
                       (uintptr_t)ep.shift;
  const Tiling t = choose_tiling(k, p.H, p.D, p.ld_ft, p.ft, ld_o, (const void*)po, col_parts_req, p.n_src_table);
  fp->t = t;
  const int64_t nblocks = (int64_t)p.blocks_per_slab * p.h_count * t.col_parts;
  BG_REQUIRE(nblocks < (1ll << 31), "forward: grid too large");
  // all heads per row: float4 rows and no operand by edge id (the row-wise kernels take staged operands only)
  const int64_t rw_blocks = ((int64_t)p.n_items + kWarpsPerBlock - 1) / kWarpsPerBlock;
  if (t.vw == 4 && !p.ee && !p.keep && !p.amul_e && rowwise_wanted(k, p.D, p.n_src_table, p.n_edges, p.n_rows, false) &&
      rowwise_geometry(p.h_count, p.D, &fp->rw_gsh, &fp->rw_vpl) && fits_grid(rw_blocks)) {
    fp->family = Family::rowwise;
    fp->grid = (unsigned)rw_blocks;
  } else if (low_degree(k.lowdeg_fwd, p.n_edges, p.n_rows)) {
    const int rpw = 32 >> t.gshift;  // rows per warp
    fp->family = Family::lowdeg;
    fp->warps_per_slab = (p.n_items + rpw - 1) / rpw;  // fewer blocks than the warp-per-row grid checked above
    fp->grid = (unsigned)(((int64_t)fp->warps_per_slab * p.h_count * t.col_parts + kWarpsPerBlock - 1) / kWarpsPerBlock);
  } else {
    fp->family = Family::warp;
    fp->grid = (unsigned)nblocks;
  }
  return 0;
}

// all heads per row for the src pass over `heads` heads: float4 rows, no operand by edge id and no gz_e
static bool src_rowwise(const Knobs& k, const BwdParams& p, const Tiling& t, int heads, int* gsh, int* vpl) {
  return t.vw == 4 && !p.ee && !p.keep && !p.amul_e && !p.gz_e && rowwise_wanted(k, p.D, p.n_dst, p.n_edges, p.n_rows, true) &&
         rowwise_geometry(heads, p.D, gsh, vpl) && fits_grid(((int64_t)p.n_items + kWarpsPerBlock - 1) / kWarpsPerBlock);
}

int plan_src(const Knobs& k, const BwdParams& p, SrcPlan* sp) {
  // the gathered table is g' (ld_g); ft and grad_ft are row-local and only constrain the vector width
  const int64_t ld_o = p.ld_ft | p.ld_gft;  // low bits clear iff both are multiples of the vector width
  const uintptr_t po = (uintptr_t)p.ft | (uintptr_t)p.grad_ft;
  const Tiling t = choose_tiling(k, p.H, p.D, p.ld_g, p.g, ld_o, (const void*)po, 1, p.n_dst);
  sp->t = t;
  BG_REQUIRE(t.col_parts == 1, "backward: D=%d too wide for one pass (max %d)", p.D, 32 * 8 * t.vw);
  const int64_t nblocks = (int64_t)p.blocks_per_slab * p.h_count;
  BG_REQUIRE(nblocks < (1ll << 31), "backward: grid too large");

  // Layout of the per-destination records (BwdParams::drec).  The node phase writes them and the src pass reads them,
  // possibly in separate calls: phase 1 for all heads, then phase 2 once per head range.  So the layout is decided
  // from what every call of one backward shares (the graph, the pointers, which operands are given) and the full H:
  // node-major when the all-heads-per-row kernel covers all H heads.  Its coverage only grows as the range narrows,
  // so node-major records are always read by it; head-major records may be read by it too (H = 12 in ranges of 6
  // heads), through drec_hs / drec_vs.
  int gsh, vpl;
  sp->records_node_major = src_rowwise(k, p, t, p.H, &gsh, &vpl);
  const bool rowwise = src_rowwise(k, p, t, p.h_count, &sp->rw_gsh, &sp->rw_vpl);
  BG_REQUIRE(rowwise || !sp->records_node_major, "backward: node-major records without the all-heads-per-row src pass");
  if (rowwise) {
    // rows staged by bulk copies (one-warp blocks, shared-memory ring) unless BOTGAT_RW_BULK=0 or a staged row is too
    // large for a ring of kBulkRing slots; the register-ring kernel otherwise
    sp->bulk_slot_bytes = (int)(((int64_t)p.h_count * p.D * 4 + 127) / 128 * 128);
    sp->bulk_ring_bytes = (size_t)kBulkRing * sp->bulk_slot_bytes;
    const bool bulk = k.rw_bulk && sp->bulk_ring_bytes <= kBulkRingMax && ((uintptr_t)p.g % 16) == 0 && p.ld_g % 4 == 0;
    sp->family = bulk ? Family::rowbulk : Family::rowwise;
    sp->grid = (unsigned)(bulk ? p.n_items : (p.n_items + kWarpsPerBlock - 1) / kWarpsPerBlock);
    return 0;
  }
  const bool lowdeg = low_degree(k.lowdeg_bwd, p.n_edges, p.n_rows);
  // TMA-staged rows: float4 access to ft / grad_ft, a 16-byte aligned table with rows a multiple of 16 bytes, and an
  // instantiated (D / 4, lanes per neighbour): G = 4 where D/4 divides by 4, else G = 8
  const int dv = p.D / 4, tgsh = (dv % 4 == 0 && dv <= 32) ? 2 : 3;
  if (!lowdeg && k.bwd_tma && t.vw == 4 && p.D % 8 == 0 && p.ld_g % 4 == 0 && ((uintptr_t)p.g % 16) == 0 &&
      with_tma_combo(dv, tgsh, [](auto, auto) {}) && fits_grid((int64_t)p.n_items * p.h_count)) {
    const bool no_eid = !p.ee && !p.amul_e && !p.keep && !p.gz_e;
    sp->family = Family::tma;
    sp->tma_dv = dv;
    sp->tma_gsh = tgsh;
    sp->tma_mode = !no_eid ? 0 : (p.eb && p.gz && !p.am && !(p.attn_p > 0.f)) ? 1 : 2;
    sp->grid = (unsigned)((int64_t)p.n_items * p.h_count);
  } else if (lowdeg) {
    const int rpw = 32 >> t.gshift;  // rows per warp
    sp->family = Family::lowdeg;
    sp->warps_per_slab = (p.n_items + rpw - 1) / rpw;  // fewer blocks than the warp-per-row grid checked above
    sp->grid = (unsigned)(((int64_t)sp->warps_per_slab * p.h_count + kWarpsPerBlock - 1) / kWarpsPerBlock);
  } else {
    sp->family = Family::warp;
    sp->grid = (unsigned)nblocks;
  }
  return 0;
}

}  // namespace botgat
