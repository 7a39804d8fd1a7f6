"""``GATFusedFn`` — the autograd seam between BoT's GATConv modules and libbotgat.

One call replaces, for a whole layer, the DGL/torch op sequence of
src/no-sampling/models.py:500-505,523-555 and src/ogbn-proteins/models.py:125-156
(SDDMM -> leaky_relu -> [edge-drop] edge_softmax -> attention dropout -> SpMM ->
degree scaling) and, in backward, the autograd replay of their adjoints.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

from . import _lib
from .graph import Graph, _stream


class KernelTimer:
    """Optional per-ABI-call device timing (CUDA events on the launching stream).
    ``bench.py`` installs one to get the per-kernel durations its roofline needs;
    when installed, the backward passes are issued as three separate ABI calls."""

    def __init__(self):
        self.events = []  # (name, start, end)

    def span(self, name):
        return _Span(self, name)

    def totals(self):
        """{name: (n_calls, total_ms)}; call after torch.cuda.synchronize()."""
        out = {}
        for name, s, e in self.events:
            n, t = out.get(name, (0, 0.0))
            out[name] = (n + 1, t + s.elapsed_time(e))
        return out


class _Span:
    def __init__(self, timer, name):
        self.timer, self.name = timer, name

    def __enter__(self):
        if self.timer is not None:
            self.s = torch.cuda.Event(enable_timing=True)
            self.s.record()

    def __exit__(self, *exc):
        if self.timer is not None:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            self.timer.events.append((self.name, self.s, e))


timer = None  # set to a KernelTimer to record

# How per-edge operands (edge logits, keep set, dropout multiplier) reach the kernels:
#   "staged": permuted into CSR order, head-major, by botgat_edge_stage / botgat_edge_unstage first (default)
#   "direct": indexed by edge id inside the kernels' software pipeline.  Measured 1.8x SLOWER on B200 at the
#             proteins shape (H random 32-byte DRAM sectors per edge instead of one 4*H-byte record per edge
#             in the staging pass); kept for graphs whose edge ids already follow the CSR order.
edge_mode = "staged"


def _span(name):
    return _Span(timer, name)


def _r4(x):
    return (x + 3) // 4 * 4


def _f32c(t, name):
    if t is None:
        return None
    if t.dtype != torch.float32:
        raise TypeError(f"{name}: expected float32, got {t.dtype}")
    if not t.is_cuda:
        raise RuntimeError(f"{name}: bot_b200 has no CPU path — tensor must be on a CUDA device")
    return t.contiguous()


def _rows(t, name, H):
    """(tensor, row stride) of a per-edge operand whose rows may carry padding columns beyond H."""
    if t is None:
        return None, 0
    if t.dtype != torch.float32 or not t.is_cuda:
        raise TypeError(f"{name}: expected a float32 CUDA tensor")
    if t.dim() != 2 or t.shape[1] < H:
        raise ValueError(f"{name}: expected (E, >= {H}), got {tuple(t.shape)}")
    if t.stride(1) != 1 or t.stride(0) < t.shape[1]:
        t = t.contiguous()
    return t, t.stride(0)


def pad_heads(H):
    """Row width (floats) that makes one H-float record an aligned power-of-two block (<= one 32-byte sector
    for H <= 8): random record accesses then never straddle a DRAM sector."""
    w = 1
    while w < H and w < 8:
        w *= 2
    return w if H <= 8 else (H + 3) // 4 * 4


class KeptEdges:
    """The CSR of one step's kept edges in one order (``botgat_edge_subset``), filled by :func:`edge_stage`.  The gather
    kernels walk it instead of the graph's CSR, so that an edge dropped this step costs them no traffic.  Arrays keep
    their full-graph sizes (the kept count stays on the device); ``eid`` only when a kernel reads edge ids."""

    def __init__(self, graph, order, with_eid):
        graph._ensure()
        info, dev, E = graph._info, graph.device, graph.number_of_edges()
        inn = order == _lib.ORDER_IN
        rows = graph.number_of_dst_nodes() if inn else graph.number_of_src_nodes()
        n_seg = info.n_seg_in if inn else info.n_seg_out

        def i32(n):
            return torch.empty(n, dtype=torch.int32, device=dev)

        W = E // 32 + 1   # kept-flag words (botgat_edge_subset.kept / base)
        self.kept = torch.empty(W, dtype=torch.int32, device=dev)   # uint32 bits, held as int32
        self.base, self.indptr, self.indices = i32(W), i32(rows + 1), i32(E)
        self.eid = i32(E) if with_eid else None
        self.seg_beg, self.seg_end = (i32(n_seg), i32(n_seg)) if n_seg else (None, None)
        self.c = _lib.EdgeSubset(*(None if t is None else t.data_ptr() for t in (
            self.indptr, self.indices, self.eid, self.kept, self.base, self.seg_beg, self.seg_end)))

    def ptr(self):
        return C.pointer(self.c)


def edge_stage(graph: Graph, order, H, ee=None, keep=None, attn_mul=None, kept=False, kept_eid=False):
    """Permute per-edge operands from edge-id order to CSR order, head-major
    (``botgat_edge_stage``).  ``ee`` / ``attn_mul`` may be (E, >=H) with padded rows.  With ``kept`` and a ``keep`` mask,
    also builds the adjacency of the kept edges (:class:`KeptEdges`, with edge ids when ``kept_eid``) and stages eb / am
    compacted to it.  Returns (eb, Hb, am, KeptEdges | None)."""
    E = graph.number_of_edges()
    dev = graph.device
    eb = am = None
    Hb = 0
    if ee is not None or keep is not None:
        Hb = H if ee is not None else 1
        eb = torch.empty((Hb, E), dtype=torch.float32, device=dev)
    if attn_mul is not None:
        am = torch.empty((H, E), dtype=torch.float32, device=dev)
    if eb is None and am is None:
        return None, 0, None, None
    sub = KeptEdges(graph, order, kept_eid) if kept and keep is not None else None
    ee, ld_ee = _rows(ee, "ee", H)
    attn_mul, ld_am = _rows(attn_mul, "attn_mul", H)
    with _span("edge_stage"):
        rc = _lib.load().botgat_edge_stage(graph._ensure(), order, H, _lib.ptr(ee), ld_ee, _lib.ptr(keep),
                                           _lib.ptr(attn_mul), ld_am, _lib.ptr(eb), _lib.ptr(am),
                                           sub.ptr() if sub is not None else None, _stream())
    _lib.check(rc, "botgat_edge_stage")
    return eb, Hb, am, sub


def _check_edge_operands(graph, H, ee, keep, attn_mul):
    E = graph.number_of_edges()
    ee, ld_ee = _rows(ee, "ee", H)
    attn_mul, ld_am = _rows(attn_mul, "attn_mul", H)
    if ee is not None and ee.shape[0] != E:
        raise ValueError("ee must have one row per edge")
    if keep is not None:
        keep = keep.to(torch.uint8).contiguous()
        if keep.numel() != E:
            raise ValueError("keep must have one entry per edge")
    return ee, ld_ee, keep, attn_mul, ld_am


def _forward_core(graph, ft2d, H, D, el, er, ee, ld_ee, keep, attn_mul, ld_am, src_scale, dst_scale, slope, attn_p, seed,
                  hooks, will_backward, ep=None):
    """Edge staging + the fused forward kernel.  ``ft2d``: 2-D tensor whose first H*D columns are the projected source
    features (any 16-byte-aligned row stride: a column slice of a wider GEMM output works).  Returns
    (out (N_d,H,D), row_max, row_sum, attn_p actually used).  With a ``keep`` mask the kernels walk the kept edges only
    (:class:`KeptEdges`).
    ``ep``: fused layer epilogue of an inference forward (``botgat_fwd_args.res`` ...): a dict with optional 2-D
    ``res`` / ``res2`` (N_d, >= H*D), ``scale`` / ``shift`` (H*D), ``relu``, ``want_y``; the ``y`` tensor is stored
    back into it."""
    lib = _lib.load()
    h = graph._ensure()
    dev = ft2d.device
    N_d = graph.number_of_dst_nodes()
    staged = edge_mode == "staged"
    philox = attn_mul is None and attn_p > 0   # the in-kernel dropout reads edge ids
    eb_in, Hb, am_in, kept = (edge_stage(graph, _lib.ORDER_IN, H, ee, keep, attn_mul, kept=True, kept_eid=philox)
                              if staged else (None, 0, None, None))
    out = torch.empty((N_d, H, D), dtype=torch.float32, device=dev)
    row_max = torch.empty((N_d, H), dtype=torch.float32, device=dev)
    row_sum = torch.empty((N_d, H), dtype=torch.float32, device=dev)
    a = _lib.FwdArgs()
    a.H, a.D, a.ld_ft, a.ld_out = H, D, ft2d.stride(0), H * D
    a.ft, a.el, a.er = ft2d.data_ptr(), el.data_ptr(), (er.data_ptr() if er is not None else None)
    a.eb, a.Hb, a.col_parts = (eb_in.data_ptr() if eb_in is not None else None), Hb, 0
    a.am = am_in.data_ptr() if am_in is not None else None
    if kept is not None:
        a.subset = kept.ptr()
    if not staged:
        if (ee is not None and ld_ee != H) or (attn_mul is not None and ld_am != H):
            raise ValueError("direct edge mode needs unpadded (E,H) edge operands")
        a.ee = ee.data_ptr() if ee is not None else None
        a.keep = keep.data_ptr() if keep is not None else None
        a.attn_mul = attn_mul.data_ptr() if attn_mul is not None else None
    a.src_scale = src_scale.data_ptr() if src_scale is not None else None
    a.dst_scale = dst_scale.data_ptr() if dst_scale is not None else None
    a.slope, a.attn_p, a.seed = float(slope), float(attn_p if attn_mul is None else 0.0), int(seed)
    a.out, a.row_max, a.row_sum = out.data_ptr(), row_max.data_ptr(), row_sum.data_ptr()
    if ep is not None:
        if will_backward:
            raise RuntimeError("the fused layer epilogue is forward-only (the backward expects the plain aggregate)")
        for key, ld in (("res", "ld_res"), ("res2", "ld_res2")):
            t = ep.get(key)
            if t is not None:
                if t.dim() != 2 or t.shape[0] < N_d or t.shape[1] < H * D or t.stride(1) != 1 or t.dtype != torch.float32:
                    raise ValueError(f"epilogue {key} must be a float32 (>= N_dst, >= H*D) matrix with unit column stride")
                setattr(a, key, t.data_ptr())
                setattr(a, ld, t.stride(0))
        if ep.get("want_y", True):
            y = torch.empty((N_d, H * D), dtype=torch.float32, device=dev)
            ep["y"] = y
            a.y, a.ld_y = y.data_ptr(), H * D
            for key, field in (("scale", "ep_scale"), ("shift", "ep_shift")):
                t = ep.get(key)
                if t is not None:
                    t = ep[key] = _f32c(t, key)
                    if t.numel() != H * D:
                        raise ValueError(f"epilogue {key} must have H*D entries")
                    setattr(a, field, t.data_ptr())
            a.ep_relu = 1 if ep.get("relu") else 0
    scratch = None
    if graph._info.n_slots_in:  # heavy rows are split over several warps (segments.cu)
        scratch = torch.empty(graph._info.n_slots_in * _r4(H * (D + 2)), dtype=torch.float32, device=dev)
        a.scratch = scratch.data_ptr()
    if hooks is not None and hooks.pre_kernel is not None:
        hooks.pre_kernel()  # e.g. wait for an asynchronous halo all-gather that fills ft / el
    chunks = hooks.head_chunks if hooks is not None and hooks.head_chunks else [(0, H)]
    for i, (hb, hc) in enumerate(chunks):   # one launch per head range: a caller can feed ft head by head
        if len(chunks) > 1 and hooks.pre_head is not None:
            hooks.pre_head(i)
        a.h_begin, a.h_count = hb, hc
        with _span("gat_fwd"):
            rc = lib.botgat_gat_forward(h, C.byref(a), _stream())
        _lib.check(rc, "botgat_gat_forward")
    return out, row_max, row_sum, float(a.attn_p)


def _backward_core(graph, cfg, hooks, ft2d, el, er, ee, keep, attn_mul, src_scale, dst_scale, out, row_max, row_sum,
                   gout, grad_ft2d, need_er, need_ee, hook_grad_ft=None):
    """The three backward phases.  ``grad_ft2d``: 2-D tensor whose first H*D columns receive grad_ft (any aligned row
    stride).  Returns (grad_el (N_s,H), grad_er | None, grad_ee | None)."""
    lib = _lib.load()
    h = graph._ensure()
    H, D, staged, slope, attn_p, seed = cfg
    N_s, N_d, E = ft2d.shape[0], out.shape[0], graph.number_of_edges()
    dev = ft2d.device

    def p(t):
        return t.data_ptr() if t is not None else None

    philox = attn_mul is None and attn_p > 0
    eb_out, Hb, am_out, kept = (edge_stage(graph, _lib.ORDER_OUT, H, ee, keep, attn_mul, kept=True, kept_eid=philox)
                                if staged else (None, 0, None, None))
    drec = torch.empty((H, N_d, 4), dtype=torch.float32, device=dev)
    gprime = torch.empty_like(gout) if dst_scale is not None else None
    grad_el = torch.empty((N_s, H), dtype=torch.float32, device=dev)
    grad_er = torch.empty((N_d, H), dtype=torch.float32, device=dev) if need_er else None
    # gz (out-CSR order) -> grad_ee (edge-id order); grad_er is reduced from grad_ee
    gz = grad_ee = None
    if need_er or need_ee:
        gz = torch.empty((H, E), dtype=torch.float32, device=dev) if staged else None
        # same row width as the ee that came in (padding columns receive zeros)
        Hp = ee.shape[1] if (ee is not None and staged) else (pad_heads(H) if staged else H)
        grad_ee = torch.empty((E, Hp), dtype=torch.float32, device=dev)
    a = _lib.BwdArgs()
    a.H, a.D, a.ld_ft, a.ld_out, a.ld_gft = H, D, ft2d.stride(0), H * D, grad_ft2d.stride(0)
    a.ft, a.el, a.er = ft2d.data_ptr(), el.data_ptr(), p(er)
    a.eb_out, a.Hb, a.phases, a.am_out = p(eb_out), Hb, 0, p(am_out)
    if not staged:
        a.ee, a.keep, a.attn_mul = p(ee), p(keep), p(attn_mul)
    a.src_scale, a.dst_scale = p(src_scale), p(dst_scale)
    a.slope, a.attn_p, a.seed = slope, attn_p, seed
    a.out, a.row_max, a.row_sum, a.gout = out.data_ptr(), row_max.data_ptr(), row_sum.data_ptr(), gout.data_ptr()
    a.drec, a.gprime, a.gz = drec.data_ptr(), p(gprime), p(gz)
    if kept is not None:
        a.subset_out = kept.ptr()
    scratch = None
    if graph._info.n_slots_out or graph._info.n_slots_in:
        scratch = torch.empty(graph._info.n_slots_out * _r4(H * (D + 1)) + graph._info.n_slots_in * H,
                              dtype=torch.float32, device=dev)
        a.scratch = scratch.data_ptr()
    a.grad_ft, a.grad_el, a.grad_ee, a.grad_er = grad_ft2d.data_ptr(), grad_el.data_ptr(), p(grad_ee), p(grad_er)
    a.ld_gee = grad_ee.stride(0) if grad_ee is not None else 0
    post_src = hooks.post_src if hooks is not None else None
    chunks = hooks.head_chunks if hooks is not None and hooks.head_chunks else None
    if chunks is not None and (len(chunks) > 1 or getattr(hooks, "force_chunked", False)):
        # src phase head range by head range; the caller's hook ships each range's grad_ft while the next one runs
        a.phases = 1
        _lib.check(lib.botgat_gat_backward(h, C.byref(a), _stream()), "botgat_gat_backward")
        for i, (hb, hc) in enumerate(chunks):
            a.phases, a.h_begin, a.h_count = 2, hb, hc
            with _span("gat_bwd_src"):
                rc = lib.botgat_gat_backward(h, C.byref(a), _stream())
            _lib.check(rc, "botgat_gat_backward")
            if hooks.post_src_head is not None:
                hooks.post_src_head(i, grad_ft2d if hook_grad_ft is None else hook_grad_ft, grad_el)
        a.phases, a.h_begin, a.h_count = 4, 0, 0
        with _span("gat_bwd_edge"):
            rc = lib.botgat_gat_backward(h, C.byref(a), _stream())
        _lib.check(rc, "botgat_gat_backward")
    elif timer is None and post_src is None:
        _lib.check(lib.botgat_gat_backward(h, C.byref(a), _stream()), "botgat_gat_backward")
    elif timer is None:
        a.phases = 3
        _lib.check(lib.botgat_gat_backward(h, C.byref(a), _stream()), "botgat_gat_backward")
        post_src(grad_ft2d if hook_grad_ft is None else hook_grad_ft, grad_el)  # e.g. start the halo reduce-scatter while the edge phase runs
        a.phases = 4
        _lib.check(lib.botgat_gat_backward(h, C.byref(a), _stream()), "botgat_gat_backward")
    else:
        for bit, name in ((1, "gat_bwd_node"), (2, "gat_bwd_src"), (4, "gat_bwd_edge")):
            a.phases = bit
            with _span(name):
                rc = lib.botgat_gat_backward(h, C.byref(a), _stream())
            _lib.check(rc, "botgat_gat_backward")
            if bit == 2 and post_src is not None:
                post_src(grad_ft2d if hook_grad_ft is None else hook_grad_ft, grad_el)
    return grad_el, grad_er, (grad_ee if need_ee else None)


# Widest head the backward src pass covers: one warp row of 32 lanes x 8 float4 vectors (csrc/graph.cu choose_tiling).
# GATFusedFn zero-pads a head too wide for its vector width to a multiple of 4 columns, which gets float4 vectors.
BWD_MAX_D = 1024


class GATFusedFn(torch.autograd.Function):
    """out = dst_scale * sum_k softmax_v(leaky_relu(el[u]+er[v]+ee[k]))*attn_mul[k] * src_scale[u] * ft[u].

    Arguments (tensors float32 on the graph's CUDA device):
      graph      bot_b200.Graph
      ft         (N_s,H,D)  projected source features, unscaled
      el         (N_s,H)    er (N_d,H)|None
      ee         (E,Hp>=H)|None, CANONICAL edge order (``gat_fused`` converts from edge-id order); columns >= H are
                 padding (Hp = 8 keeps every record inside one 32-byte DRAM sector, see ``pad_heads``); the gradient
                 comes back with the same shape
      keep       (E,) bool/uint8 | None   edge-drop keep set (canonical order)
      attn_mul   (E,H) | None   explicit attention-dropout multiplier (canonical order)
      src_scale  (N_s,)|None   dst_scale (N_d,)|None
      slope      leaky_relu slope
      attn_p, seed   in-kernel Philox attention dropout (used when attn_mul is None and attn_p > 0)
    """

    @staticmethod
    def forward(ctx, graph, ft, el, er, ee, keep, attn_mul, src_scale, dst_scale, slope, attn_p, seed, hooks=None):
        if ft.dim() != 3:
            raise ValueError("ft must be (N_src, H, D)")
        ft = _f32c(ft, "ft")
        N_s, H, D = ft.shape
        N_d = graph.number_of_dst_nodes()
        if N_s != graph.number_of_src_nodes():
            raise ValueError(f"ft has {N_s} rows, graph has {graph.number_of_src_nodes()} source nodes")
        el = _f32c(el, "el").view(N_s, H)
        er = None if er is None else _f32c(er, "er").view(N_d, H)
        ee, ld_ee, keep, attn_mul, ld_am = _check_edge_operands(graph, H, ee, keep, attn_mul)
        src_scale, dst_scale = _f32c(src_scale, "src_scale"), _f32c(dst_scale, "dst_scale")
        Dk = D
        if any(ctx.needs_input_grad):
            if D > BWD_MAX_D:
                raise ValueError(f"GAT layer with gradients: head width D={D} exceeds the backward's limit of {BWD_MAX_D} "
                                 "columns per head (inference without gradients has no such limit)")
            vw = 4 if D % 4 == 0 and ft.data_ptr() % 16 == 0 else 2 if D % 2 == 0 and ft.data_ptr() % 8 == 0 else 1
            if D > 256 * vw:
                # the src pass covers a head in one pass of 256 vectors of vw floats; a wider head is zero-padded to a
                # multiple of 4 columns and gets float4 vectors (the padding adds zeros to every sum)
                if hooks is not None:
                    raise ValueError(f"GAT layer with hooks: D={D} > {256 * vw} needs a multiple of 4 and a 16-byte aligned ft")
                Dk = _r4(D)
                ft = torch.cat([ft, ft.new_zeros(N_s, H, Dk - D)], 2)
        with torch.cuda.device(ft.device):
            out, row_max, row_sum, attn_p_used = _forward_core(
                graph, ft.view(N_s, H * Dk), H, Dk, el, er, ee, ld_ee, keep, attn_mul, ld_am, src_scale, dst_scale, slope,
                attn_p, seed, hooks, any(ctx.needs_input_grad))
        ctx.graph = graph
        ctx.hooks = hooks
        ctx.D = D
        ctx.cfg = (H, Dk, edge_mode == "staged", float(slope), attn_p_used, int(seed))
        ctx.save_for_backward(ft, el, er, ee, keep, attn_mul, src_scale, dst_scale, out, row_max, row_sum)
        return out if Dk == D else out[:, :, :D].contiguous()

    @staticmethod
    def backward(ctx, gout):
        ft, el, er, ee, keep, attn_mul, src_scale, dst_scale, out, row_max, row_sum = ctx.saved_tensors
        H, D = ctx.cfg[0], ctx.cfg[1]
        need_er = er is not None and ctx.needs_input_grad[3]
        need_ee = ee is not None and ctx.needs_input_grad[4]
        gout = _f32c(gout, "grad_out")
        if D != ctx.D:     # zero-padded head (see forward)
            gout = torch.cat([gout, gout.new_zeros(gout.shape[0], H, D - ctx.D)], 2)
        elif D > 256 and gout.data_ptr() % 16:
            gout = gout.clone()   # a 16-byte aligned g' keeps float4 vectors (one pass per head)
        grad_ft = torch.empty_like(ft)
        with torch.cuda.device(ft.device):
            grad_el, grad_er, grad_ee = _backward_core(
                ctx.graph, ctx.cfg, ctx.hooks, ft.view(-1, H * D), el, er, ee, keep, attn_mul, src_scale, dst_scale,
                out, row_max, row_sum, gout, grad_ft.view(-1, H * D), need_er, need_ee, hook_grad_ft=grad_ft)
        if D != ctx.D:
            grad_ft = grad_ft[:, :, :ctx.D]
        return (None, grad_ft, grad_el, grad_er, grad_ee, None, None, None, None, None, None, None, None)


def _pad_rows(w, rows):
    """(rows, in) copy of the weight block ``w`` with zero rows appended."""
    if w.shape[0] == rows:
        return w
    return torch.cat([w, w.new_zeros(rows - w.shape[0], w.shape[1])], 0)


class GATConvSampledFn(torch.autograd.Function):
    """The whole sampled-variant layer body (src/ogbn-proteins/models.py:106-160) around the fused kernels with the
    node-side projections folded into two GEMMs (SURVEY.md section 8f rank 2):

        Ys = x_src @ [src_fc ; attn_src_fc]^T                       (N_s, pad32(H*D + H))
        Yd = x_dst @ [dst_fc ; attn_dst_fc]^T + [dst_fc.bias ; 0]   (N_d, pad32(H*D + H))
        rst = gat(ft = Ys[:, :HD], el = Ys[:, HD:HD+H], er = Yd[:, HD:HD+H], ...) + Yd[:, :HD]

    instead of four GEMMs (two of them H columns wide: cuBLAS runs those as split-K kernels plus a reduction, each
    slower than the wide ones) and, in backward, eight.  The kernels read ``ft`` and write ``grad_ft`` in place inside
    the wide buffers (row stride = a multiple of 128 bytes, so gathered rows stay line-aligned); the backward is two
    data-gradient and two weight-gradient GEMMs over the assembled (N, pad32) gradient blocks.

    ``w_src`` = cat(src_fc.weight, attn_src_fc.weight) (HD+H, in); ``w_dst`` = cat(dst_fc.weight[, attn_dst_fc.weight]);
    ``b_dst`` = dst_fc.bias (HD).  ``x_dst`` may be the same tensor as ``x_src`` (homogeneous graph, no input scaling).
    """

    @staticmethod
    def forward(ctx, graph, x_src, x_dst, w_src, w_dst, b_dst, ee, keep, attn_mul, dst_scale, H, D, slope, attn_p, seed,
                src_scale=None):
        # ``src_scale`` (full-graph variant, src/no-sampling/models.py:500-505,517): applied to the gathered rows by
        # the kernels and to el here — the logit and the messages see the SCALED projection, er / the residual do not
        x_src, x_dst = _f32c(x_src, "feat_src"), _f32c(x_dst, "feat_dst")
        N_s, N_d, HD = graph.number_of_src_nodes(), graph.number_of_dst_nodes(), H * D
        if x_src.shape[0] != N_s or x_dst.shape[0] != N_d:
            raise ValueError("feat_src / feat_dst rows do not match the graph")
        has_er = w_dst.shape[0] == HD + H
        P = (HD + H + 31) // 32 * 32
        ws, wd = _pad_rows(w_src, P), _pad_rows(w_dst, P)
        bd = torch.cat([b_dst, b_dst.new_zeros(P - HD)])
        ee, ld_ee, keep, attn_mul, ld_am = _check_edge_operands(graph, H, ee, keep, attn_mul)
        dst_scale, src_scale = _f32c(dst_scale, "dst_scale"), _f32c(src_scale, "src_scale")
        vw = 4 if D % 4 == 0 else 2 if D % 2 == 0 else 1
        if any(ctx.needs_input_grad) and D > min(256 * vw, BWD_MAX_D):
            raise ValueError(f"GAT layer with gradients: head width D={D} exceeds the backward's limit of {256 * vw} columns "
                             f"per head at {vw}-float vectors (at most {BWD_MAX_D}, for D a multiple of 4)")
        with torch.cuda.device(x_src.device):
            Ys = x_src @ ws.t()
            Yd = torch.addmm(bd, x_dst, wd.t())
            el = Ys[:, HD:HD + H].contiguous() if src_scale is None else Ys[:, HD:HD + H] * src_scale.unsqueeze(-1)
            er = Yd[:, HD:HD + H].contiguous() if has_er else None
            out, row_max, row_sum, attn_p_used = _forward_core(
                graph, Ys, H, D, el, er, ee, ld_ee, keep, attn_mul, ld_am, src_scale, dst_scale, slope, attn_p, seed, None,
                any(ctx.needs_input_grad))
            rst = out + Yd[:, :HD].view(N_d, H, D)                                    # models.py:159-160
        ctx.graph, ctx.same_x = graph, x_dst is x_src or x_dst.data_ptr() == x_src.data_ptr() and N_s == N_d
        ctx.cfg = (H, D, edge_mode == "staged", float(slope), attn_p_used, int(seed))
        ctx.dims = (P, has_er, w_src.shape[0], w_dst.shape[0])
        ctx.save_for_backward(x_src, x_dst, ws, wd, Ys, el, er, ee, keep, attn_mul, dst_scale, out, row_max, row_sum, src_scale)
        return rst

    @staticmethod
    def backward(ctx, grst):
        x_src, x_dst, ws, wd, Ys, el, er, ee, keep, attn_mul, dst_scale, out, row_max, row_sum, src_scale = ctx.saved_tensors
        H, D = ctx.cfg[0], ctx.cfg[1]
        P, has_er, rows_s, rows_d = ctx.dims
        HD = H * D
        need = ctx.needs_input_grad
        need_ee = ee is not None and need[6]
        grst = _f32c(grst, "grad_out")
        N_s, N_d = x_src.shape[0], x_dst.shape[0]
        dev = x_src.device
        with torch.cuda.device(dev):
            gYs = torch.empty((N_s, P), dtype=torch.float32, device=dev)
            gYd = torch.empty((N_d, P), dtype=torch.float32, device=dev)
            grad_el, grad_er, grad_ee = _backward_core(
                ctx.graph, ctx.cfg, None, Ys, el, er, ee, keep, attn_mul, src_scale, dst_scale, out, row_max, row_sum,
                grst, gYs, has_er, need_ee)
            gYs[:, HD:HD + H] = grad_el if src_scale is None else grad_el * src_scale.unsqueeze(-1)
            gYs[:, HD + H:].zero_()
            gYd[:, :HD] = grst.view(N_d, HD)
            if has_er:
                gYd[:, HD:HD + H] = grad_er
                gYd[:, HD + H:].zero_()
            else:
                gYd[:, HD:].zero_()
            gw_s = (gYs.t() @ x_src)[:rows_s] if need[3] else None
            gw_d = (gYd.t() @ x_dst)[:rows_d] if need[4] else None
            gb = grst.view(N_d, HD).sum(0) if need[5] else None
            gx_s = gx_d = None
            if ctx.same_x and need[1]:
                gx_s = torch.addmm(gYs @ ws, gYd, wd)       # both projections read the same input
            else:
                gx_s = gYs @ ws if need[1] else None
                gx_d = gYd @ wd if need[2] else None
        return (None, gx_s, gx_d, gw_s, gw_d, gb, grad_ee, None, None, None, None, None, None, None, None, None)


class LayerTail:
    """What a reference model does to a layer's output before the next layer (src/no-sampling/models.py:720-731,
    src/ogbn-proteins/models.py:253-260): ``h = conv(...) [+ h_last]; h_last = h; h = act(norm(h))`` — handed to the layer
    so that, in inference (no gradient, eval-mode norm), the fused forward kernel applies it while the output vectors are
    still in registers instead of four more passes over (N, H*D).

    ``h_last``: (>= N_dst, H*D) or None; ``norm``: ``nn.BatchNorm1d`` in eval mode with running statistics, an
    ``ElementWiseLinear``-like module (``weight`` / ``bias`` vectors or None) or None; ``relu``: apply ReLU."""

    def __init__(self, h_last=None, norm=None, relu=False):
        self.h_last, self.norm, self.relu = h_last, norm, relu

    def usable(self):
        if os.environ.get("BOTGAT_FUSE_TAIL", "1") == "0":   # developer A/B switch (tools/tail_bench.py)
            return False
        n = self.norm
        if isinstance(n, torch.nn.BatchNorm1d):
            return not n.training and n.running_mean is not None
        return n is None or (hasattr(n, "weight") and hasattr(n, "bias"))

    def scale_shift(self):
        n = self.norm
        if n is None:
            return None, None
        if isinstance(n, torch.nn.BatchNorm1d):   # y = (x - mean) / sqrt(var + eps) * gamma + beta
            scale = torch.rsqrt(n.running_var + n.eps)
            if n.weight is not None:
                scale = scale * n.weight
            shift = -n.running_mean * scale
            if n.bias is not None:
                shift = shift + n.bias
            return scale.detach(), shift.detach()
        return (None if n.weight is None else n.weight.detach()), (None if n.bias is None else n.bias.detach())


def gat_fused_inference(graph, ft, el, er, ee, keep, attn_mul, src_scale, dst_scale, slope, tail, res=None):
    """Forward of :func:`gat_fused` (operands in canonical edge order) without autograd and with the layer tail fused into
    the gather kernel's epilogue.  ``res``: the layer's own residual projection (N_dst, H*D) or None.  Returns ``(h, y)``:
    ``h = rst [+ res] [+ tail.h_last]`` (N_dst, H*D) and ``y = act(norm(h))``."""
    with torch.no_grad():
        ft = _f32c(ft, "ft")
        N_s, H, D = ft.shape
        N_d = graph.number_of_dst_nodes()
        el = _f32c(el, "el").view(N_s, H)
        er = None if er is None else _f32c(er, "er").view(N_d, H)
        ee, ld_ee, keep, attn_mul, ld_am = _check_edge_operands(graph, H, ee, keep, attn_mul)
        src_scale, dst_scale = _f32c(src_scale, "src_scale"), _f32c(dst_scale, "dst_scale")
        scale, shift = tail.scale_shift()
        h_last = tail.h_last
        if h_last is not None:
            h_last = _f32c(h_last, "h_last").view(h_last.shape[0], -1)
        if res is not None:
            res = _f32c(res, "res").view(res.shape[0], -1)
        ep = {"res": res, "res2": h_last, "scale": scale, "shift": shift, "relu": tail.relu, "want_y": True}
        with torch.cuda.device(ft.device):
            out, _, _, _ = _forward_core(graph, ft.view(N_s, H * D), H, D, el, er, ee, ld_ee, keep, attn_mul, ld_am, src_scale,
                                            dst_scale, slope, 0.0, 0, None, False, ep=ep)
        return out.view(N_d, H * D), ep["y"]


def gat_conv_inference(graph, x_src, x_dst, w_src, w_dst, b_dst, ee, keep, attn_mul, dst_scale, H, D, slope, tail,
                       src_scale=None):
    """Forward of :class:`GATConvSampledFn` without autograd and with the layer tail fused into the gather kernel's
    epilogue.  Returns ``(h, y)``: ``h = rst + dst_fc(x_dst) [+ tail.h_last]`` (N_dst, H*D) — the next layer's ``h_last``
    — and ``y = act(norm(h))``."""
    with torch.no_grad():
        x_src, x_dst = _f32c(x_src, "feat_src"), _f32c(x_dst, "feat_dst")
        N_s, N_d, HD = graph.number_of_src_nodes(), graph.number_of_dst_nodes(), H * D
        if x_src.shape[0] != N_s or x_dst.shape[0] != N_d:
            raise ValueError("feat_src / feat_dst rows do not match the graph")
        has_er = w_dst.shape[0] == HD + H
        P = (HD + H + 31) // 32 * 32
        ws, wd = _pad_rows(w_src, P), _pad_rows(w_dst, P)
        bd = torch.cat([b_dst, b_dst.new_zeros(P - HD)])
        ee, ld_ee, keep, attn_mul, ld_am = _check_edge_operands(graph, H, ee, keep, attn_mul)
        dst_scale, src_scale = _f32c(dst_scale, "dst_scale"), _f32c(src_scale, "src_scale")
        scale, shift = tail.scale_shift()
        h_last = tail.h_last
        if h_last is not None:
            h_last = _f32c(h_last, "h_last").view(h_last.shape[0], -1)
        ep = {"res2": h_last, "scale": scale, "shift": shift, "relu": tail.relu, "want_y": True}
        with torch.cuda.device(x_src.device):
            Ys = x_src @ ws.t()
            Yd = torch.addmm(bd, x_dst, wd.t())
            ep["res"] = Yd                                                    # models.py:159-160, read in place
            el = Ys[:, HD:HD + H].contiguous() if src_scale is None else Ys[:, HD:HD + H] * src_scale.unsqueeze(-1)
            er = Yd[:, HD:HD + H].contiguous() if has_er else None
            out, _, _, _ = _forward_core(graph, Ys, H, D, el, er, ee, ld_ee, keep, attn_mul, ld_am, src_scale, dst_scale,
                                            slope, 0.0, 0, None, False, ep=ep)
        return out.view(N_d, HD), ep["y"]


class EdgeLogitProj(torch.autograd.Function):
    """``ee = feat_edge @ W^T`` emitted with padded rows (E, pad_heads(H)) — `attn_edge_fc(feat_edge)` of
    src/ogbn-proteins/models.py:131 as streaming kernels (``botgat_edge_proj_*``) instead of three skinny GEMMs."""

    @staticmethod
    def forward(ctx, x, weight):
        lib = _lib.load()
        x = _f32c(x, "feat_edge")
        weight = _f32c(weight, "weight")
        E, Cin = x.shape
        H = weight.shape[0]
        y = torch.empty((E, pad_heads(H)), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            with _span("edge_proj_fwd"):
                rc = lib.botgat_edge_proj_forward(E, Cin, H, x.data_ptr(), x.stride(0), weight.data_ptr(), y.data_ptr(),
                                                  y.stride(0), x.device.index, _stream())
        _lib.check(rc, "botgat_edge_proj_forward")
        ctx.save_for_backward(x, weight)
        return y

    @staticmethod
    def backward(ctx, gy):
        lib = _lib.load()
        x, weight = ctx.saved_tensors
        E, Cin = x.shape
        H = weight.shape[0]
        gy, ld_gy = _rows(gy, "grad_ee", H)
        gx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        gw = torch.empty_like(weight) if ctx.needs_input_grad[1] else None
        partials = torch.empty(lib.botgat_edge_proj_gw_blocks() * H * Cin, dtype=torch.float32, device=x.device) \
            if gw is not None else None
        with torch.cuda.device(x.device):
            with _span("edge_proj_bwd"):
                rc = lib.botgat_edge_proj_backward(E, Cin, H, x.data_ptr(), x.stride(0), weight.data_ptr(), gy.data_ptr(),
                                                   ld_gy, _lib.ptr(gx), gx.stride(0) if gx is not None else 0,
                                                   _lib.ptr(gw), _lib.ptr(partials), x.device.index, _stream())
        _lib.check(rc, "botgat_edge_proj_backward")
        return gx, gw


def edge_logits(feat_edge, weight):
    """Padded per-edge logits (E, pad_heads(H)) from edge features (E, C) and an ``nn.Linear`` weight (H, C).
    Falls back to a torch matmul (a library GEMM, still on the GPU) for shapes the streaming kernels do not cover."""
    H, Cin = weight.shape
    if H <= 8 and Cin <= 64 and H * Cin <= 256 and feat_edge.dim() == 2:
        return EdgeLogitProj.apply(feat_edge, weight)
    pad = pad_heads(H) - H
    w = torch.cat([weight, weight.new_zeros(pad, Cin)], 0) if pad > 0 else weight
    return torch.nn.functional.linear(feat_edge, w)


def edge_drop_keep(n_edges, n_drop, seed, device):
    """uint8 keep mask with exactly ``n_drop`` zeros at uniformly random positions (``botgat_edge_drop_draw``)."""
    lib = _lib.load()
    device = torch.device(device)
    if device.type != "cuda":
        raise RuntimeError("bot_b200.edge_drop_keep: no CPU path")
    keep = torch.empty(n_edges, dtype=torch.uint8, device=device)
    ws = torch.empty(lib.botgat_edge_drop_workspace_bytes(n_edges), dtype=torch.uint8, device=device)
    with torch.cuda.device(device):
        with _span("edge_drop_draw"):
            rc = lib.botgat_edge_drop_draw(n_edges, n_drop, seed, keep.data_ptr(), ws.data_ptr(), device.index
                                           if device.index is not None else torch.cuda.current_device(), _stream())
    _lib.check(rc, "botgat_edge_drop_draw")
    return keep


class EdgeMLPLogits(torch.autograd.Function):
    """``ee = relu(efeat @ W1^T + b1) @ W2^T`` in one pass per direction (``botgat_edge_mlp_*``): the model's per-layer
    ``edge_encoder[i]`` + ReLU (src/ogbn-proteins/models.py:245-247) fused with the layer's ``attn_edge_fc``
    (models.py:131).  The (E, edge_emb) embedding is never materialised; backward recomputes the hidden units."""

    @staticmethod
    def forward(ctx, x, w1, b1, w2):
        lib = _lib.load()
        x, w1, w2 = _f32c(x, "efeat"), _f32c(w1, "edge_encoder.weight"), _f32c(w2, "attn_edge_fc.weight")
        b1 = None if b1 is None else _f32c(b1, "edge_encoder.bias")
        E, Cin = x.shape
        M, H = w1.shape[0], w2.shape[0]
        y = torch.empty((E, pad_heads(H)), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            with _span("edge_mlp_fwd"):
                rc = lib.botgat_edge_mlp_forward(E, Cin, M, H, x.data_ptr(), x.stride(0), w1.data_ptr(), _lib.ptr(b1),
                                                 w2.data_ptr(), y.data_ptr(), y.stride(0), x.device.index, _stream())
        _lib.check(rc, "botgat_edge_mlp_forward")
        ctx.save_for_backward(x, w1, b1, w2)
        return y

    @staticmethod
    def backward(ctx, gy):
        lib = _lib.load()
        x, w1, b1, w2 = ctx.saved_tensors
        if ctx.needs_input_grad[0]:
            raise RuntimeError("EdgeMLPLogits: raw edge features get no gradient (use edge_logits on the embedding instead)")
        E, Cin = x.shape
        M, H = w1.shape[0], w2.shape[0]
        gy, ld_gy = _rows(gy, "grad_ee", H)
        gw1 = torch.empty_like(w1) if ctx.needs_input_grad[1] else None
        gb1 = torch.empty_like(b1) if b1 is not None and ctx.needs_input_grad[2] else None
        gw2 = torch.empty_like(w2) if ctx.needs_input_grad[3] else None
        ws = torch.empty(lib.botgat_edge_mlp_workspace_floats(Cin, M, H), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            with _span("edge_mlp_bwd"):
                rc = lib.botgat_edge_mlp_backward(E, Cin, M, H, x.data_ptr(), x.stride(0), w1.data_ptr(), _lib.ptr(b1),
                                                  w2.data_ptr(), gy.data_ptr(), ld_gy, _lib.ptr(gw1), _lib.ptr(gb1),
                                                  _lib.ptr(gw2), ws.data_ptr(), x.device.index, _stream())
        _lib.check(rc, "botgat_edge_mlp_backward")
        return None, gw1, gb1, gw2


class EdgeEmbedding:
    """``relu(encoder(efeat))`` not yet computed.  The model wrappers pass it to ``GATConv.forward`` as ``feat_edge``;
    the layer turns it into its logits with one fused kernel (:class:`EdgeMLPLogits`) when the shapes allow
    (C <= 8 raw features, edge_emb <= 16, H <= 8 and ``efeat`` not requiring grad), else materialises it."""

    def __init__(self, efeat, encoder, canonical=False):
        # ``canonical``: rows of ``efeat`` are in the graph's canonical edge order (``graph.edata.canonical(key)``)
        # rather than edge-id order; the logits then come out canonical too and the layer skips the permutation
        self.efeat, self.encoder, self.canonical = efeat, encoder, canonical

    def materialize(self):
        return torch.relu(self.encoder(self.efeat))

    def logits(self, attn_edge_fc_weight):
        x, enc = self.efeat, self.encoder
        H = attn_edge_fc_weight.shape[0]
        if (x.dim() == 2 and x.is_cuda and not x.requires_grad and os.environ.get("BOTGAT_NO_EDGE_MLP", "0") != "1"
                and _lib.load().botgat_edge_mlp_supported(x.shape[1], enc.weight.shape[0], H)):
            return EdgeMLPLogits.apply(x, enc.weight, enc.bias, attn_edge_fc_weight)
        return edge_logits(self.materialize(), attn_edge_fc_weight)


class Deferred:
    """A tensor whose producer (e.g. a host-to-device copy) runs on another stream.  ``GATConv.forward`` accepts it
    in place of ``feat_edge`` and waits for it only where the edge features are first needed, so the copy
    overlaps the node-side projections and the edge-drop draw."""

    def __init__(self, tensor, event, requires_grad=False):
        self.tensor, self.event, self.requires_grad = tensor, event, requires_grad

    def wait(self):
        cur = torch.cuda.current_stream()
        cur.wait_event(self.event)
        self.tensor.record_stream(cur)
        return self.tensor.requires_grad_(True) if self.requires_grad else self.tensor


class Hooks:
    """Optional call-backs of :class:`GATFusedFn` used by the partitioned layer to overlap its collectives:
    ``pre_kernel()`` runs after edge staging, right before the forward gather kernel is launched;
    ``post_src(grad_ft, grad_el)`` runs in backward after the src pass, before the edge phase."""

    def __init__(self, pre_kernel=None, post_src=None, head_chunks=None, pre_head=None, post_src_head=None):
        self.pre_kernel, self.post_src = pre_kernel, post_src
        # optional head pipelining: ``head_chunks`` = [(h_begin, h_count), ...]; ``pre_head(i)`` runs before the forward
        # launch of chunk i, ``post_src_head(i, grad_ft, grad_el)`` after the backward src launch of chunk i
        self.head_chunks, self.pre_head, self.post_src_head = head_chunks, pre_head, post_src_head


class _ToCanonical(torch.autograd.Function):
    """Rows of a per-edge tensor from edge-id order to the graph's canonical order (and the gradient back)."""

    @staticmethod
    def forward(ctx, t, graph):
        ctx.graph = graph
        return t.index_select(0, graph.edge_perm())

    @staticmethod
    def backward(ctx, g):
        return g.index_select(0, ctx.graph.canonical_edge_ids()), None


def to_canonical(graph, t):
    """Per-edge tensor (E, ...) in edge-id order -> the graph's canonical order (``Graph`` docstring); differentiable.
    A no-op for graphs whose two orders coincide (the sampler's blocks, COOs given sorted by (dst, src))."""
    if t is None or graph.edge_perm() is None:
        return t
    if t.shape[0] != graph.number_of_edges():
        raise ValueError("per-edge operand must have one row per edge")
    return _ToCanonical.apply(t, graph)


def gat_fused(graph, ft, el, er=None, ee=None, keep=None, attn_mul=None, src_scale=None, dst_scale=None,
              slope=0.2, attn_p=0.0, seed=0, hooks=None, edge_order="eid"):
    """Functional form of :class:`GATFusedFn` (accepts the reference's trailing-1 shapes, e.g. el (N,H,1)).

    ``edge_order``: order of the rows of ``ee`` / ``keep`` / ``attn_mul``.  "eid" (default) = edge-id order, DGL's
    ``edata`` semantics — permuted to the canonical order here, one random pass per operand and step; "canonical" =
    already in the graph's canonical order (``graph.edata.canonical(key)``, what the edge-logit producers emit from
    canonical features, what ``edge_drop_keep`` draws): no permutation.  The gradient of ``ee`` comes back in the order
    it was given in.  The in-kernel attention dropout is keyed on the canonical edge number
    (``graph.canonical_edge_ids()``)."""
    H = ft.shape[1]
    el = el.reshape(-1, H)
    er = None if er is None else er.reshape(-1, H)
    if ee is not None and ee.dim() == 3:
        ee = ee.reshape(ee.shape[0], -1)
    if attn_mul is not None and attn_mul.dim() == 3:
        attn_mul = attn_mul.reshape(attn_mul.shape[0], -1)
    if edge_order == "eid":
        ee, keep, attn_mul = to_canonical(graph, ee), to_canonical(graph, keep), to_canonical(graph, attn_mul)
    elif edge_order != "canonical":
        raise ValueError(f"edge_order must be 'eid' or 'canonical', got {edge_order!r}")
    return GATFusedFn.apply(graph, ft, el, er, ee, keep, attn_mul, src_scale, dst_scale, slope, attn_p, seed, hooks)
