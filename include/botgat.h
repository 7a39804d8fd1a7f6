/*
 * botgat.h — C ABI of the B200-native GAT message-passing engine.
 *
 * Drop-in boundary for the sparse section of BoT's GATConv layers
 * (reference: src/no-sampling/models.py:475-566, src/ogbn-proteins/models.py:87-168,
 * src/ogbn-products/models.py:88-167).  The reference reaches this arithmetic
 * through DGL 0.5 Python calls; each entry point below names the call(s) it
 * replaces.  Plain pointers and sizes only — no torch / C++ types.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer on `device` unless marked HOST;
 *  - every entry point enqueues on `stream` (a cudaStream_t passed as void*) and
 *    returns without synchronising unless stated otherwise;
 *  - return value 0 = success, negative = error; the message is available from
 *    botgat_last_error() (thread-local);
 *  - the caller owns every buffer passed in (inputs, outputs, workspaces); the
 *    library owns only the internals of a botgat_graph.
 *  - node ids / edge ids are int64 at the boundary (DGL's idtype) and int32
 *    inside (all structure arrays returned by botgat_graph_get are int32);
 *    n_edges must be < 2^31.
 */
#ifndef BOTGAT_H_
#define BOTGAT_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default) /* the library is built with -fvisibility=hidden */
#endif

#define BOTGAT_ABI_VERSION 5

typedef struct botgat_graph botgat_graph;

int botgat_abi_version(void);
const char* botgat_last_error(void);
/* number of CUDA kernels this library has launched so far in this process (CUB passes count as one each) */
int64_t botgat_launch_count(void);

/* ------------------------------------------------------------------------
 * Graph ingestion.
 * Replaces DGLGraph construction + `graph.create_formats_()`
 * (src/no-sampling/run.py:146, src/ogbn-proteins/gat.py:66,
 * src/ogbn-products/gat.py:75) and `graph.in_degrees()/out_degrees()`
 * (src/no-sampling/models.py:478,501,551).
 *
 * src/dst: (n_edges) int64 COO in edge-id order.  Builds, on the device,
 *   in-CSR  (rows = dst, CSC in DGL terms): indptr, indices (= src), eid
 *   out-CSR (rows = src):                   indptr, indices (= dst), eid
 * with a stable sort (inside a row, increasing edge id), plus degree tables.
 * Synchronises `stream` once before returning (it reads back two scalars).
 * Node ids outside [0, n_src) / [0, n_dst) are detected BEFORE anything is indexed by them and
 * reported as an error (return < 0, no graph).
 * Memory: the structure arrays come from the device's default stream-ordered pool
 * (cudaMallocAsync).  If the application left that pool's release threshold at its default (0),
 * the first call on a device raises it to 2 GiB so that per-batch blocks recycle their memory;
 * an application-chosen threshold is respected.
 * ---------------------------------------------------------------------- */
int botgat_graph_create(int64_t n_src, int64_t n_dst, int64_t n_edges,
                        const int64_t* src, const int64_t* dst,
                        int device, void* stream, botgat_graph** out);
void botgat_graph_destroy(botgat_graph* g);
/* Same, without synchronising the device: the memory returns to the stream-ordered pool after the work already
 * enqueued on `stream` (every consumer of the graph must have been enqueued there or have finished). */
void botgat_graph_destroy_async(botgat_graph* g, void* stream);

enum {
  BOTGAT_IN_INDPTR = 0,   /* int32 (n_dst+1) */
  BOTGAT_IN_INDICES = 1,  /* int32 (n_edges)  source id of each in-CSR entry */
  BOTGAT_IN_EID = 2,      /* int32 (n_edges)  edge id of each in-CSR entry */
  BOTGAT_OUT_INDPTR = 3,  /* int32 (n_src+1) */
  BOTGAT_OUT_INDICES = 4, /* int32 (n_edges)  destination id of each out-CSR entry */
  BOTGAT_OUT_EID = 5,     /* int32 (n_edges) */
  BOTGAT_IN_DEG = 6,      /* int32 (n_dst) */
  BOTGAT_OUT_DEG = 7      /* int32 (n_src) */
};
/* Expose a structure array (device pointer + element count). */
int botgat_graph_get(const botgat_graph* g, int which, void** dev_ptr, int64_t* len);

typedef struct {
  int64_t n_src, n_dst, n_edges;
  int64_t max_in_deg, max_out_deg;
  int32_t has_zero_in_degree; /* replaces `(graph.in_degrees()==0).any()`, models.py:478 */
  int32_t device;
  /* Heavy rows (longer than the segment length, 2048 neighbours) are split over several warps; each partial
   * segment needs one scratch slot.  With r4(x) = x rounded up to a multiple of 4:
   *   forward scratch  = n_slots_in  * r4(H * (D + 2)) floats
   *   backward scratch = n_slots_out * r4(H * (D + 1)) + n_slots_in * H floats
   * Both are 0 for graphs without heavy rows. */
  int64_t n_slots_in, n_slots_out;
  /* 1 when the library's edge numbering equals the in-CSR position (the COO was given sorted by destination):
   * edge-ordered operands then stream coalesced through botgat_edge_stage(BOTGAT_ORDER_IN) / botgat_edge_reduce_dst */
  int32_t in_eid_identity;
  /* cache-blocked out-CSR traversal used by botgat_edge_stage / botgat_edge_unstage(BOTGAT_ORDER_OUT):
   * tiles_src x tiles_dst node blocks (1 x 1 = plain order) */
  int32_t tiles_src, tiles_dst;
  /* row segments (work items) of the in- / out-CSR when it has split rows, else 0: the length of
   * botgat_edge_subset.seg_beg / seg_end (ABI v5) */
  int32_t n_seg_in, n_seg_out;
  int32_t reserved_;
} botgat_graph_info;
int botgat_graph_get_info(const botgat_graph* g, botgat_graph_info* info /* HOST */);

/* ------------------------------------------------------------------------
 * COO preprocessing on the device.
 * Replaces dgl.to_bidirected / remove_self_loop / add_self_loop
 * (src/no-sampling/run.py:137,143).  Outputs are caller-allocated with the
 * stated capacity; *n_out (HOST) receives the edge count; these calls
 * synchronise `stream`.
 * ---------------------------------------------------------------------- */
/* add reverse edges, dedup, sort by (src,dst).  capacity of out_*: 2*n_edges */
int botgat_coo_to_bidirected(int64_t n_nodes, int64_t n_edges,
                             const int64_t* src, const int64_t* dst,
                             int64_t* out_src, int64_t* out_dst, int64_t* n_out,
                             int device, void* stream);
/* drop (i,i) edges, keep order.  capacity: n_edges */
int botgat_coo_remove_self_loop(int64_t n_edges, const int64_t* src, const int64_t* dst,
                                int64_t* out_src, int64_t* out_dst, int64_t* n_out,
                                int device, void* stream);
/* append (i,i), i = 0..n_nodes-1.  capacity: n_edges + n_nodes.  Does not synchronise. */
int botgat_coo_add_self_loop(int64_t n_nodes, int64_t n_edges,
                             const int64_t* src, const int64_t* dst,
                             int64_t* out_src, int64_t* out_dst,
                             int device, void* stream);

/* ------------------------------------------------------------------------
 * Per-edge operand staging.  Edge tensors arrive in edge-id order
 * (DGL `edata`); the fused kernels stream them in CSR order, head-major.
 * ---------------------------------------------------------------------- */
enum { BOTGAT_ORDER_IN = 0, BOTGAT_ORDER_OUT = 1 };
/*
 * eb[hb][p] = (ee ? ee[eid(p)*ld_ee + hb] : 0), or -inf when keep && !keep[eid(p)]
 * am[h][p]  = attn_mul[eid(p)*ld_am + h]
 *   ee        (n_edges, ld_ee>=H) float or NULL — `attn_edge_fc(feat_edge)`, proteins models.py:131
 *   keep      (n_edges) uint8 or NULL           — edge-drop keep set, models.py:529-532
 *   attn_mul  (n_edges, ld_am>=H) float or NULL — attention-dropout multiplier, models.py:537/544
 *   eb        (Hb,n_edges) out, Hb = H if ee else 1; NULL iff ee==NULL && keep==NULL
 *   am        (H,n_edges) out; NULL iff attn_mul==NULL
 * A row stride of 8 floats (32 bytes) makes every H<=8 record one aligned DRAM sector; the kernels use the
 * widest vector access the stride and alignment allow.
 */
/*
 * Per-step kept adjacency (ABI v5).  Edge drop removes a tenth or more of the edges every step; the gather kernels
 * walk this CSR of the kept edges instead of the graph's, so that a dropped edge costs them nothing.  All arrays are
 * caller-owned and keep their full-graph sizes; E' (the kept count) stays on the device.  For the CSR named by
 * `order` (rows = n_dst for BOTGAT_ORDER_IN, n_src for BOTGAT_ORDER_OUT), with W = n_edges/32 + 1 words and
 * rank(x) = base[x/32] + popcount(kept[x/32] & ((1 << x%32) - 1)), the kept positions before x:
 *   kept     (W) uint32   kept flags in CSR position order: bit p%32 of word p/32 (positions >= n_edges: 0)
 *   base     (W) int32    kept positions before word w (exclusive scan of the words' popcounts)
 *                         a kept position p moves to rank(p)
 *   indptr   (rows+1)     indptr[r] = rank(graph indptr[r])
 *   indices  (n_edges)    the kept entries in CSR order (first E' written)
 *   eid      (n_edges)    their edge ids, or NULL; needed when a kernel reads edge ids (in-kernel attention dropout)
 *   seg_beg, seg_end      (n_seg_in / n_seg_out of botgat_graph_info) the row segments translated through rank, or
 *                         NULL when the CSR has no split rows
 */
typedef struct {
  int32_t* indptr;
  int32_t* indices;
  int32_t* eid;
  uint32_t* kept;
  int32_t* base;
  int32_t* seg_beg;
  int32_t* seg_end;
} botgat_edge_subset;
/* With `subset` (requires keep): also fills the kept adjacency, and eb / am are written compacted, eb[hb][rank(p)] for
 * the kept positions only (no -inf markers; the rows keep their stride n_edges).  NULL: the layout above. */
int botgat_edge_stage(const botgat_graph* g, int order, int32_t H,
                      const float* ee, int64_t ld_ee, const uint8_t* keep,
                      const float* attn_mul, int64_t ld_am,
                      float* eb, float* am, botgat_edge_subset* subset /* HOST struct or NULL */, void* stream);
/* grad_ee[eid(p)*ld_gee + h] = gz[h][p]  (gz head-major in the CSR order named by `order`).  With `subset` (the one
 * botgat_edge_stage filled), gz is compacted: kept p reads gz[h][rank(p)], a dropped edge gets zeros. */
int botgat_edge_unstage(const botgat_graph* g, int order, int32_t H, const float* gz,
                        float* grad_ee, int64_t ld_gee, const botgat_edge_subset* subset /* HOST or NULL */,
                        void* stream);
/* grad_er[v,h] = sum over the in-edges k of v of grad_ee[k*ld_gee + h]   (replaces the copy_e/sum SpMM DGL
 * runs as the backward of u_add_v, SURVEY.md Appendix B) */
int botgat_edge_reduce_dst(const botgat_graph* g, int32_t H, const float* grad_ee, int64_t ld_gee,
                           float* grad_er, float* scratch /* n_slots_in*H floats, NULL if n_slots_in == 0 */,
                           void* stream);

/* ------------------------------------------------------------------------
 * Per-edge logit projection  y[k, 0:H] = x[k, 0:C] @ W^T  (W row-major (H, C); H <= 8, C <= 64, H*C <= 256).
 * Replaces `attn_edge_fc(feat_edge)` (src/ogbn-proteins/models.py:131) and its autograd backward — three
 * skinny cuBLAS GEMMs — by streaming kernels.  y rows have stride ld_y >= H; columns [H, min(ld_y, 8)) are
 * written as zeros (the padded record layout of botgat_edge_stage).  Backward: gx (n, ld_gx) and/or gW (H, C);
 * `partials` is a workspace of botgat_edge_proj_gw_blocks() * H * C floats (fixed-order reduction, no atomics).
 * ---------------------------------------------------------------------- */
int botgat_edge_proj_gw_blocks(void);
int botgat_edge_proj_forward(int64_t n, int32_t C, int32_t H, const float* x, int64_t ld_x, const float* W,
                             float* y, int64_t ld_y, int device, void* stream);
int botgat_edge_proj_backward(int64_t n, int32_t C, int32_t H, const float* x, int64_t ld_x, const float* W,
                              const float* gy, int64_t ld_gy, float* gx /* or NULL */, int64_t ld_gx,
                              float* gW /* or NULL */, float* partials, int device, void* stream);

/* ------------------------------------------------------------------------
 * Edge-drop keep mask: keep[e] = 0 for a uniformly random subset of exactly n_drop edges, 1 elsewhere —
 * the set `perm[:bound]` of `perm = torch.randperm(E); bound = int(E * edge_drop)`
 * (src/no-sampling/models.py:528-532, src/ogbn-proteins/models.py:136-139) drawn as a selection on 64-bit
 * Philox4x32-10 keys instead of a sort of E keys.  Deterministic in (n_edges, n_drop, seed).
 * `workspace`: botgat_edge_drop_workspace_bytes(n_edges) bytes, 256-byte aligned.
 * ---------------------------------------------------------------------- */
int64_t botgat_edge_drop_workspace_bytes(int64_t n_edges);
int botgat_edge_drop_draw(int64_t n_edges, int64_t n_drop, uint64_t seed, uint8_t* keep, void* workspace,
                          int device, void* stream);

/* ------------------------------------------------------------------------
 * Fused per-edge encoder + logit projection  y[k, 0:H] = relu(x[k, 0:C] @ W1^T + b1) @ W2^T
 * (W1 row-major (M, C), b1 (M) or NULL, W2 row-major (H, M); C <= 8, M <= 16, H <= 8 —
 * botgat_edge_mlp_supported()).  Replaces, for one layer, `F.relu(edge_encoder[i](efeat))`
 * (src/ogbn-proteins/models.py:245-247) followed by `attn_edge_fc(feat_edge)` (models.py:131) and the
 * autograd backward of both: the (E, M) embedding is never materialised (the reference keeps one per
 * layer for backward).  Output rows as botgat_edge_proj_forward.  Backward recomputes the hidden units and
 * produces gW1 (M, C), gb1 (M), gW2 (H, M) (each may be NULL); x gets no gradient (raw edge features are data).
 * `partials`: botgat_edge_mlp_workspace_floats(C, M, H) floats (fixed-order reduction, no atomics).
 * ---------------------------------------------------------------------- */
int botgat_edge_mlp_supported(int32_t C, int32_t M, int32_t H);
int64_t botgat_edge_mlp_workspace_floats(int32_t C, int32_t M, int32_t H);
int botgat_edge_mlp_forward(int64_t n, int32_t C, int32_t M, int32_t H, const float* x, int64_t ld_x,
                            const float* W1, const float* b1, const float* W2, float* y, int64_t ld_y,
                            int device, void* stream);
int botgat_edge_mlp_backward(int64_t n, int32_t C, int32_t M, int32_t H, const float* x, int64_t ld_x,
                             const float* W1, const float* b1, const float* W2, const float* gy, int64_t ld_gy,
                             float* gW1, float* gb1, float* gW2, float* partials, int device, void* stream);

/* ------------------------------------------------------------------------
 * Fused forward: logits -> leaky_relu -> online edge-softmax -> attention
 * dropout -> u_mul_e/sum SpMM -> degree scaling, one pass over the in-CSR.
 * Replaces src/no-sampling/models.py:500-505,523-555 and
 * src/ogbn-proteins/models.py:125-156 (DGL apply_edges / edge_softmax /
 * update_all and the torch elementwise ops between them).
 *
 *   out[v,h,:] = dst_scale[v] * sum_k a~[k,h] * src_scale[u_k] * ft[u_k,h,:]
 *   a~ = softmax_v( leaky_relu(el[u]+er[v]+eb[k]) ) * am[k]
 * ---------------------------------------------------------------------- */
typedef struct {
  int32_t H;              /* heads */
  int32_t D;              /* per-head width */
  int64_t ld_ft;          /* row stride of ft, floats (>= H*D) */
  int64_t ld_out;         /* row stride of out, floats */
  const float* ft;        /* (n_src, ld_ft)  projected source features, unscaled */
  const float* el;        /* (n_src, H) */
  const float* er;        /* (n_dst, H) or NULL */
  const float* eb;        /* (Hb, n_edges) in-CSR order, or NULL */
  int32_t Hb;             /* 0, 1 or H */
  int32_t col_parts;      /* split each head's D columns in this many parts; 0 = auto */
  const float* am;        /* (H, n_edges) in-CSR order, or NULL */
  /* the same operands in EDGE-ID order (direct mode, no staging pass; exclusive with eb / am): */
  const float* ee;        /* (n_edges, H) `attn_edge_fc(feat_edge)`, or NULL */
  const uint8_t* keep;    /* (n_edges) edge-drop keep set, or NULL */
  const float* attn_mul;  /* (n_edges, H) attention-dropout multiplier, or NULL */
  const float* src_scale; /* (n_src) or NULL */
  const float* dst_scale; /* (n_dst) or NULL */
  float slope;            /* leaky_relu negative slope */
  float attn_p;           /* in-kernel Philox attention dropout prob (used iff am==NULL && attn_p>0) */
  uint64_t seed;          /* Philox key for the above */
  float* out;             /* (n_dst, ld_out) */
  float* row_max;         /* (n_dst, H)  saved for backward */
  float* row_sum;         /* (n_dst, H)  saved for backward */
  float* scratch;         /* forward scratch (see botgat_graph_info), or NULL when n_slots_in == 0 */
  /* Head range of this launch: heads [h_begin, h_begin + h_count); h_count == 0 = all remaining heads.  All array
   * arguments keep their full-H meaning.  Lets a caller overlap per-head transfers with per-head launches (the
   * kernels work head-major anyway).  Graphs with split rows (n_slots_in > 0) need the full range. */
  int32_t h_begin, h_count;
  /* Fused layer epilogue (ABI v4; all NULL / 0 = off).  The elementwise tail of a reference layer where it needs no
   * batch statistics and no gradient, i.e. inference: the residual adds `rst + dst_fc(feat_dst)`
   * (src/ogbn-proteins/models.py:159-160) and `h += h_last` (:253-254, src/no-sampling/models.py:722-723), the
   * eval-mode norm / bias as a per-column scale and shift (:257, no-sampling :727) and ReLU (:258 / :728), applied
   * while an output vector is still in registers instead of as four more passes over (n_dst, H*D):
   *   out[v,c] = dst_scale[v] * agg[v,c] + res[v,c] + res2[v,c]      y[v,c] = act(out[v,c] * ep_scale[c] + ep_shift[c])
   * `out` then carries the residual sum (the next layer's h_last).  The backward expects the plain aggregate in
   * `out`: training keeps these fields NULL. */
  const float* res;       /* (n_dst, ld_res) or NULL */
  int64_t ld_res;
  const float* res2;      /* (n_dst, ld_res2) or NULL */
  int64_t ld_res2;
  const float* ep_scale;  /* (H*D) or NULL = 1; needs y */
  const float* ep_shift;  /* (H*D) or NULL = 0; needs y */
  float* y;               /* (n_dst, ld_y) or NULL */
  int64_t ld_y;
  int32_t ep_relu;        /* 1: y = max(., 0); needs y */
  int32_t reserved_;
  /* kept in-CSR adjacency from botgat_edge_stage(BOTGAT_ORDER_IN, subset), or NULL = the graph's (ABI v5); eb / am
   * must then be the compacted ones staged with it */
  const botgat_edge_subset* subset;
} botgat_fwd_args;
int botgat_gat_forward(const botgat_graph* g, const botgat_fwd_args* a /* HOST */, void* stream);

/* ------------------------------------------------------------------------
 * Backward (SURVEY.md Appendix A.3).  Replaces the autograd replay of DGL's
 * GSpMM / GSDDMM / EdgeSoftmax backward kernels.  Deterministic (no atomics).
 *   phase 1, node : t[v,h] = <out[v,h,:], gout[v,h,:]>, packs per-dst records
 *                   {er, row_max, 1/row_sum, t}; g' = gout * dst_scale
 *   phase 2, src  : ONE gather pass over the out-CSR (src-major): grad_ft,
 *                   grad_el and, on request, gz = d(loss)/d(edge logit) per
 *                   (edge, head) in out-CSR order.  The attention weights are
 *                   recomputed from (el, er, eb, row_max, row_sum).
 *   phase 4, edge : [gz -> grad_ee (edge-id order) when staged;] grad_er[v] = sum of
 *                   grad_ee over the in-edges of v (in-CSR walk, 4*H-byte records).
 * ---------------------------------------------------------------------- */
typedef struct {
  int32_t H, D;
  int64_t ld_ft, ld_out, ld_gft;
  const float* ft;        /* (n_src, ld_ft) */
  const float* el;        /* (n_src, H) */
  const float* er;        /* (n_dst, H) or NULL */
  const float* eb_out;    /* (Hb, n_edges) out-CSR order or NULL */
  int32_t Hb;
  int32_t phases;         /* bitmask of phases to run (1 node, 2 src, 4 edge); 0 = all (profiling splits them) */
  const float* am_out;    /* (H, n_edges) out-CSR order or NULL */
  const float* ee;        /* edge-id-order operands, as in botgat_fwd_args (exclusive with eb_out / am_out) */
  const uint8_t* keep;
  const float* attn_mul;
  const float* src_scale;
  const float* dst_scale;
  float slope;
  float attn_p;
  uint64_t seed;
  const float* out;       /* (n_dst, ld_out) forward output (post dst_scale) */
  const float* row_max;   /* (n_dst, H) */
  const float* row_sum;   /* (n_dst, H) */
  const float* gout;      /* (n_dst, ld_out) gradient w.r.t. out */
  /* workspaces */
  float* drec;            /* (H, n_dst, 4) */
  float* gprime;          /* (n_dst, ld_out); required iff dst_scale != NULL */
  float* scratch;         /* backward scratch (see botgat_graph_info), or NULL when both slot counts are 0 */
  float* gz;              /* (H, n_edges) or NULL.  NULL: the src pass writes grad_ee directly in edge-id order;
                             given: it writes gz in out-CSR order and phase 4 un-stages it into grad_ee */
  /* outputs */
  float* grad_ft;         /* (n_src, ld_gft) w.r.t. the unscaled ft */
  float* grad_el;         /* (n_src, H) */
  float* grad_ee;         /* (n_edges, ld_gee) edge-id order, or NULL; required when grad_er is requested (its input) */
  int64_t ld_gee;         /* row stride of grad_ee in floats; 0 = H */
  float* grad_er;         /* (n_dst, H) or NULL */
  /* head range of the src phase (phases & 2), as in botgat_fwd_args; the node and edge phases always cover all heads */
  int32_t h_begin, h_count;
  /* kept out-CSR adjacency from botgat_edge_stage(BOTGAT_ORDER_OUT, subset), or NULL = the graph's (ABI v5); eb_out /
   * am_out must be the compacted ones staged with it, gz is written compacted and phase 4 un-stages it through it */
  const botgat_edge_subset* subset_out;
} botgat_bwd_args;
int botgat_gat_backward(const botgat_graph* g, const botgat_bwd_args* a /* HOST */, void* stream);

/* ------------------------------------------------------------------------
 * Multi-GPU: 1-D destination-row partition (no reference implementation —
 * the reference is single-GPU; contract in DESIGN.md).
 * ---------------------------------------------------------------------- */
/* bounds[p] = first row r with in_indptr[r] >= floor(p*E/P); bounds (HOST, n_parts+1). Synchronises. */
int botgat_partition_1d(const botgat_graph* g, int32_t n_parts, int64_t* bounds /* HOST */, void* stream);
/*
 * Local edge set of rows [lo,hi): counts the edges (phase 0: out_* NULL, *n_local set)
 * or writes them (phase 1): global edge id, global src, local dst (= dst-lo), edge-id order.
 * Synchronises.
 */
int botgat_partition_extract(const botgat_graph* g, int64_t lo, int64_t hi,
                             int64_t* out_eid, int64_t* out_src, int64_t* out_ldst,
                             int64_t* n_local /* HOST */, void* stream);
/* Row gather/scatter used by the halo exchange (send-list packing and the transposed add). */
int botgat_rows_gather(const float* table, int64_t ld, int64_t width, const int64_t* rows, int64_t n_rows,
                       float* out /* (n_rows,width) */, void* stream);
int botgat_rows_scatter_add(float* table, int64_t ld, int64_t width, const int64_t* rows, int64_t n_rows,
                            const float* in /* (n_rows,width), rows unique */, void* stream);

/* ------------------------------------------------------------------------
 * Halo exchange through NVLink peer memory (SURVEY.md section 8b `botgat_halo_exchange`; no reference implementation).
 * The exchange of the row-sharded source table [ft | el] of the partitioned layer, one COLUMN RANGE (= head range) at
 * a time, by peer loads from buffers every rank has mapped (CUDA VMM / torch symmetric memory) — so that the transfer
 * of head range k+1 overlaps the gather kernel of head range k and nothing is repacked.  The caller provides the
 * inter-GPU barriers (peers' buffers written before a pull, read before they are overwritten).
 *   world <= 16; peer_tables : HOST array of `world` DEVICE pointers (entry `r` = rank r's buffer, own rank included).
 *   n_blocks : grid size (0 = 592 blocks of 128 threads: small blocks, so that the exchange finds room beside the gather
 *   kernel it overlaps — launch it on a higher-priority stream).
 *
 * Every rank holds a table of world * rows_per_rank rows (row stride ld) with the same layout; rank r's OWN slice
 * [r * rows_per_rank, (r+1) * rows_per_rank) of ITS table is the authoritative copy of its rows (written there directly).
 * botgat_halo_pull (forward, the all-gather): into this rank's table (= peer_tables[rank])
 *   table[r * rows_per_rank + i, col0 : col0 + width] = peer_tables[r][r * rows_per_rank + i, same columns]   for r != rank
 * botgat_halo_pull_reduce (backward, the reduce-scatter; summed in the FIXED order r = 0..world-1, deterministic):
 *   out[i, col0 : col0 + width] = sum_r peer_tables[r][rank * rows_per_rank + i, col0 : col0 + width]
 * ---------------------------------------------------------------------- */
int botgat_halo_pull(int32_t world, int32_t rank, const float* const* peer_tables /* HOST */, int64_t rows_per_rank, int64_t ld,
                     int64_t col0, int64_t width, int32_t n_blocks, void* stream);
int botgat_halo_pull_reduce(int32_t world, int32_t rank, const float* const* peer_tables /* HOST */, int64_t rows_per_rank,
                            int64_t ld_table, int64_t col0, int64_t width, float* out, int64_t ld_out, int32_t n_blocks,
                            void* stream);

/* ------------------------------------------------------------------------
 * Neighbour sampling and block construction on the device.  Replaces
 * dgl.dataloading.MultiLayerNeighborSampler + NodeDataLoader and their CPU worker processes
 * (src/ogbn-proteins/gat.py:177-201, src/ogbn-products/gat.py:202-233), per layer:
 *   frontier = sample_neighbors(g, seeds, fanout): botgat_sample_count, then botgat_sample_neighbors
 *   block    = to_block(frontier, seeds):          botgat_block_compact, then botgat_graph_create
 * Uniform without replacement over the in-edges of each seed; every in-edge when in-degree <= fanout or
 * fanout <= 0; fanout <= 256.  Deterministic in (graph, seeds, fanout, seed).
 *
 * botgat_sample_count: offsets[i] (device, n_seeds+1) = start of seed i's picks, *n_out (HOST) = total;
 *   workspace = botgat_sample_workspace_bytes(n_seeds) bytes; synchronises `stream`.
 * botgat_sample_neighbors: for seed i and its j-th pick, at offsets[i]+j: out_src = source node id in g,
 *   out_dst = i (the block's destination id), out_eid = edge id in g.
 * botgat_block_compact: src_nodes = seeds followed by the sampled sources that are not seeds in ascending id
 *   (capacity n_seeds + n_edges), src_local[e] = position of src_global[e] in src_nodes, *n_src (HOST) = length
 *   of src_nodes; seeds must be unique; workspace = botgat_block_workspace_bytes(n_parent) bytes, 256-byte
 *   aligned; synchronises `stream`.
 * ---------------------------------------------------------------------- */
int64_t botgat_sample_workspace_bytes(int64_t n_seeds);
int botgat_sample_count(const botgat_graph* g, int64_t n_seeds, const int64_t* seeds, int32_t fanout,
                        int64_t* offsets, int64_t* n_out /* HOST */, void* workspace, void* stream);
int botgat_sample_neighbors(const botgat_graph* g, int64_t n_seeds, const int64_t* seeds, int32_t fanout,
                            uint64_t seed, const int64_t* offsets, int64_t* out_src, int64_t* out_dst,
                            int64_t* out_eid, void* stream);
int64_t botgat_block_workspace_bytes(int64_t n_parent);
int botgat_block_compact(int64_t n_parent, int64_t n_seeds, const int64_t* seeds, int64_t n_edges,
                         const int64_t* src_global, int64_t* src_local, int64_t* src_nodes, int64_t* n_src /* HOST */,
                         void* workspace, int device, void* stream);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* BOTGAT_H_ */
