"""Multi-GPU path: 1-D destination-row partition + halo exchange (one process per GPU).

The reference is single-GPU (SURVEY.md section 2c: no distributed code at all), so this
module has no reference counterpart; its contract is "partitioned result == single-GPU
result" and the partition maps are bit-exact against ``oracle/graph_ref.py``.

* Destination rows are split into P contiguous ranges balanced on EDGE count
  (``partition_bounds``: bounds[p] = first row r with in_indptr[r] >= floor(p*E/P)).
* Rank p owns the nodes of its range, both as destinations and as the home of their
  source rows ``[ft | el]``.  Per layer and direction there is exactly one exchange:
  forward  — gather the source rows the local edges reference (halo),
  backward — the transposed collective, adding partial ``grad_ft/grad_el`` back at the owners.
* Two exchange plans, both autograd-aware and both plain ``torch.distributed`` collectives
  (NCCL over NVLink/NVSwitch on GPUs; gloo in the CPU tests):
  "dense"  — ``all_gather_into_tensor`` of the whole row-sharded table (equal-sized padded
             shards) / ``reduce_scatter_tensor`` back.  Optimal when the halo is ~everything,
             which is the case for uniformly random edges.
  "sparse" — ``all_to_all_single`` of only the referenced rows / the same in reverse with an
             ``index_add_`` at the owner.  For graphs with locality.
  The map construction is device-agnostic torch code so that it runs under gloo on CPU; the
  per-rank compute is ``bot_b200.functional.gat_fused`` on the local block graph (CUDA only).
"""
from __future__ import annotations

import os

import torch
import torch.distributed as dist

from .graph import Graph


def partition_bounds(dst, n_nodes, n_parts):
    """Edge-balanced contiguous row ranges; identical to ``oracle.graph_ref.partition_bounds``."""
    counts = torch.bincount(dst, minlength=n_nodes)
    indptr = torch.zeros(n_nodes + 1, dtype=torch.int64, device=dst.device)
    indptr[1:] = torch.cumsum(counts, 0)
    e = int(dst.numel())
    targets = torch.tensor([(p * e) // n_parts for p in range(1, n_parts)], dtype=torch.int64, device=dst.device)
    inner = torch.searchsorted(indptr, targets, right=False).clamp(max=n_nodes)
    bounds = torch.cat([torch.zeros(1, dtype=torch.int64, device=dst.device), inner,
                        torch.full((1,), n_nodes, dtype=torch.int64, device=dst.device)])
    return torch.cummax(bounds, 0).values


class _DenseHalo(torch.autograd.Function):
    """all-gather of equal-sized padded shards; backward = reduce-scatter (sum)."""

    @staticmethod
    def forward(ctx, shard, group):
        ctx.group = group
        world = dist.get_world_size(group)
        out = shard.new_empty((world * shard.shape[0],) + tuple(shard.shape[1:]))
        dist.all_gather_into_tensor(out, shard.contiguous(), group=group)
        return out

    @staticmethod
    def backward(ctx, grad):
        world = dist.get_world_size(ctx.group)
        out = grad.new_empty((grad.shape[0] // world,) + tuple(grad.shape[1:]))
        dist.reduce_scatter_tensor(out, grad.contiguous(), op=dist.ReduceOp.SUM, group=ctx.group)
        return out, None


class _DenseHaloAsync(torch.autograd.Function):
    """`_DenseHalo` with the collectives started asynchronously so that the caller can put work between the start
    and the first use: forward leaves the work handle in ``state.fwd[key]``; backward uses the reduce-scatter that
    ``state.bwd[key]`` holds if the gradient hook already started one (``PartitionedGraph.gat``)."""

    @staticmethod
    def forward(ctx, shard, group, state, key):
        ctx.group, ctx.state, ctx.key = group, state, key
        world = dist.get_world_size(group)
        out = shard.new_empty((world * shard.shape[0],) + tuple(shard.shape[1:]))
        state.fwd[key] = dist.all_gather_into_tensor(out, shard.contiguous(), group=group, async_op=True)
        return out

    @staticmethod
    def backward(ctx, grad):
        pre = ctx.state.bwd.pop(ctx.key, None)
        if pre is not None:
            work, out = pre
            work.wait()
            return out, None, None, None
        world = dist.get_world_size(ctx.group)
        out = grad.new_empty((grad.shape[0] // world,) + tuple(grad.shape[1:]))
        dist.reduce_scatter_tensor(out, grad.contiguous(), op=dist.ReduceOp.SUM, group=ctx.group)
        return out, None, None, None


class _DenseHaloHeads(torch.autograd.Function):
    """`_DenseHaloAsync` for a (rows, H, D) table shipped one head range at a time: the forward starts one
    all-gather per range (``state.fwd_chunks``; the layer's ``pre_head`` hook waits for range i and copies it into
    place right before the kernel launch of range i, so range i+1 travels while range i is computed); the backward
    collects the per-range reduce-scatters the ``post_src_head`` hook started (``state.bwd_chunks``)."""

    @staticmethod
    def forward(ctx, shard, group, state, chunks):
        world = dist.get_world_size(group)
        ctx.group, ctx.state, ctx.chunks, ctx.shard_shape = group, state, chunks, tuple(shard.shape)
        state.out = shard.new_empty((world * shard.shape[0],) + tuple(shard.shape[1:]))
        state.fwd_chunks, state.bwd_chunks = [], []
        for hb, hc in chunks:
            piece = shard[:, hb:hb + hc].contiguous()
            buf = shard.new_empty((world * shard.shape[0], hc) + tuple(shard.shape[2:]))
            work = dist.all_gather_into_tensor(buf, piece, group=group, async_op=True)
            state.fwd_chunks.append((work, buf))
        return state.out

    @staticmethod
    def backward(ctx, grad):
        st, world = ctx.state, dist.get_world_size(ctx.group)
        res = grad.new_empty(ctx.shard_shape)
        if len(st.bwd_chunks) == len(ctx.chunks):
            for (hb, hc), (work, piece) in zip(ctx.chunks, st.bwd_chunks):
                work.wait()
                res[:, hb:hb + hc] = piece
        else:  # the hooks did not run (plain autograd use): one reduce-scatter of the whole gradient
            dist.reduce_scatter_tensor(res, grad.contiguous(), op=dist.ReduceOp.SUM, group=ctx.group)
        return res, None, None, None


class _HaloState:
    def __init__(self):
        self.fwd, self.bwd = {}, {}
        self.out, self.fwd_chunks, self.bwd_chunks = None, [], []


class _SparseHalo(torch.autograd.Function):
    """all-to-all of the referenced rows; backward sends the halo gradients home and adds them."""

    @staticmethod
    def forward(ctx, own, send_idx, send_counts, recv_counts, group):
        ctx.group, ctx.n_own = group, own.shape[0]
        ctx.send_counts, ctx.recv_counts = send_counts, recv_counts
        ctx.save_for_backward(send_idx)
        send = own.index_select(0, send_idx)
        recv = own.new_empty((sum(recv_counts),) + tuple(own.shape[1:]))
        dist.all_to_all_single(recv, send, output_split_sizes=recv_counts, input_split_sizes=send_counts, group=group)
        return torch.cat([own, recv], 0)

    @staticmethod
    def backward(ctx, grad):
        (send_idx,) = ctx.saved_tensors
        g_own = grad[: ctx.n_own].clone()
        g_halo = grad[ctx.n_own:].contiguous()
        back = grad.new_empty((sum(ctx.send_counts),) + tuple(grad.shape[1:]))
        dist.all_to_all_single(back, g_halo, output_split_sizes=ctx.send_counts, input_split_sizes=ctx.recv_counts,
                               group=ctx.group)
        g_own.index_add_(0, send_idx, back)  # several peers may reference one row: index_add_ accumulates
        return g_own, None, None, None, None


class P2PHalo:
    """Buffers of the peer-memory halo exchange of one layer shape (``botgat_halo_pull`` / ``botgat_halo_pull_reduce``,
    csrc/halo.cu).  Every rank holds the gathered source table ``[ft | el]`` (world * max_own rows of ``P`` = H*D + H
    floats padded to 128-byte rows) and its table of partial gradients in SYMMETRIC memory
    (``torch.distributed._symmetric_memory``: every rank maps every other rank's buffers; NVLink peer loads).  Rank r's
    own slice of ITS table is the authoritative copy of its rows: a producer (the projection GEMM, ``own_ft`` /
    ``own_el`` below) can write there directly and nothing is staged or repacked."""

    def __init__(self, pg, H, D):
        import ctypes as C

        import torch.distributed._symmetric_memory as symm_mem

        self.H, self.D, self.HD = H, D, H * D
        self.P = (self.HD + H + 31) // 32 * 32
        dev = pg.local.device
        group = pg.group if pg.group is not None else dist.group.WORLD
        rows = pg.max_own
        self.table = symm_mem.empty((pg.world * rows, self.P), dtype=torch.float32, device=dev)
        self.gtable = symm_mem.empty((pg.world * rows, self.P), dtype=torch.float32, device=dev)
        self.h_table = symm_mem.rendezvous(self.table, group)
        self.h_gtable = symm_mem.rendezvous(self.gtable, group)
        self.table.zero_()
        self.gtable.zero_()
        self.table_ptrs = (C.c_void_p * pg.world)(*[int(p) for p in self.h_table.buffer_ptrs])
        self.gtable_ptrs = (C.c_void_p * pg.world)(*[int(p) for p in self.h_gtable.buffer_ptrs])
        self.own = self.table[pg.rank * rows: pg.rank * rows + pg.n_own]
        # where a producer writes this rank's rows so that the layer does not copy them (strided views of the table)
        self.own_ft = self.own[:, :self.HD].unflatten(1, (H, D))
        self.own_el = self.own[:, self.HD:self.HD + H]
        # the exchange must find room BESIDE a gather kernel that fills the GPU: small blocks on a high-priority stream
        self.stream = torch.cuda.Stream(device=dev, priority=-1)
        self.blocks = int(os.environ.get("BOTGAT_HALO_BLOCKS", "592"))
        self.world, self.rank, self.rows = pg.world, pg.rank, rows
        self.fwd_pending = self.bwd_pending = False   # a forward / backward ran since the last barrier of the other kind
        torch.cuda.synchronize(dev)
        self.h_table.barrier(channel=0)

    def pull(self, col0, width):
        from . import _lib
        from .graph import _stream

        _lib.check(_lib.load().botgat_halo_pull(self.world, self.rank, self.table_ptrs, self.rows, self.P, col0, width, self.blocks,
                                                _stream()), "botgat_halo_pull")

    def pull_reduce(self, col0, width, out):
        from . import _lib
        from .graph import _stream

        _lib.check(_lib.load().botgat_halo_pull_reduce(self.world, self.rank, self.gtable_ptrs, self.rows, self.P, col0, width,
                                                       out.data_ptr(), out.stride(0), self.blocks, _stream()),
                   "botgat_halo_pull_reduce")


class _P2PGatFn(torch.autograd.Function):
    """The partitioned layer with the halo exchanged by this repo's own peer-memory kernels instead of NCCL collectives,
    pipelined per head range on a second (high-priority) stream:

      forward   [ft | el] of the owned rows sit in this rank's slice of its symmetric table -> inter-GPU barrier ->
                pull(head range k+1)  ||  gather kernel(head range k)          (edge staging runs beside the first pull)
      backward  src kernel(head range k+1) writes its partial grad_ft into the symmetric gradient table  ||
                barrier + pull_reduce(head range k) -> owned rows of grad_ft;  grad_el the same after the last range;
                the edge phase (grad_ee, grad_er) runs beside the tail of the exchange.
    """

    @staticmethod
    def forward(ctx, pg, hx, chunks, ft_own, el_own, er, ee, keep, attn_mul, src_scale, dst_scale, slope, attn_p, seed):
        from . import functional as Fn

        H, D, HD = hx.H, hx.D, hx.HD
        n_own = pg.n_own
        graph = pg.local
        main = torch.cuda.current_stream()
        # Before my rows are overwritten every peer must have finished pulling the previous version.  A peer's pulls
        # end before its forward kernels do, and the barrier at the start of the BACKWARD is passed only after every
        # rank's forward: in a training loop (forward, backward, forward, ...) that barrier already orders it.
        if hx.fwd_pending:
            hx.h_table.barrier(channel=0)
        hx.fwd_pending, hx.bwd_pending = True, False
        if ft_own.data_ptr() != hx.own_ft.data_ptr():
            hx.own[:, :HD].copy_(ft_own.reshape(n_own, HD))
        if el_own.data_ptr() != hx.own_el.data_ptr():
            hx.own_el.copy_(el_own.reshape(n_own, H))
        hx.h_table.barrier(channel=1)        # every rank's rows are written
        hx.stream.wait_stream(main)
        events = []
        with torch.cuda.stream(hx.stream):
            for i, (hb, hc) in enumerate(chunks):
                if i == 0:
                    hx.pull(HD, H)           # el of every source row
                hx.pull(hb * D, hc * D)
                ev = torch.cuda.Event()
                ev.record(hx.stream)
                events.append(ev)
        el_all = torch.empty((hx.table.shape[0], H), dtype=torch.float32, device=hx.table.device)

        def pre_kernel():
            # runs after the edge staging passes (they overlap the first pull): el arrives with head range 0
            main.wait_event(events[0])
            el_all.copy_(hx.table[:, HD:HD + H])

        def pre_head(i):
            if i > 0:
                main.wait_event(events[i])

        ee, ld_ee, keep, attn_mul, ld_am = Fn._check_edge_operands(graph, H, ee, keep, attn_mul)
        hooks = Fn.Hooks(pre_kernel=pre_kernel, head_chunks=chunks, pre_head=pre_head)
        out, row_max, row_sum, attn_p_used = Fn._forward_core(
            graph, hx.table, H, D, el_all, er, ee, ld_ee, keep, attn_mul, ld_am, src_scale, dst_scale, slope, attn_p, seed,
            hooks, True)
        ctx.pg, ctx.hx, ctx.chunks = pg, hx, chunks
        ctx.cfg = (H, D, Fn.edge_mode == "staged", float(slope), attn_p_used, int(seed))
        ctx.save_for_backward(el_all, er, ee, keep, attn_mul, src_scale, dst_scale, out, row_max, row_sum)
        return out

    @staticmethod
    def backward(ctx, gout):
        from . import functional as Fn

        pg, hx, chunks = ctx.pg, ctx.hx, ctx.chunks
        el_all, er, ee, keep, attn_mul, src_scale, dst_scale, out, row_max, row_sum = ctx.saved_tensors
        H, D, HD = hx.H, hx.D, hx.HD
        n_own = pg.n_own
        main = torch.cuda.current_stream()
        gout = gout.contiguous()
        gshard = torch.empty((hx.rows, hx.P), dtype=torch.float32, device=gout.device)
        gshard.record_stream(hx.stream)
        # Before my gradient table is overwritten every peer must have finished reading the previous one; the barrier of
        # a forward in between (passed only after every rank's previous backward, exchange included) already orders it.
        if hx.bwd_pending or not hx.fwd_pending:
            hx.h_gtable.barrier(channel=0)
        hx.bwd_pending, hx.fwd_pending = True, False

        def post_src_head(i, grad_ft, grad_el):
            hb, hc = chunks[i]
            last = i == len(chunks) - 1
            if last:
                hx.gtable[:, HD:HD + H].copy_(grad_el)      # complete only after the last head range
            ev = torch.cuda.Event()
            ev.record(main)
            with torch.cuda.stream(hx.stream):
                hx.stream.wait_event(ev)
                hx.h_gtable.barrier(channel=1 + i)          # every rank has written this column range
                hx.pull_reduce(hb * D, hc * D, gshard)
                if last:
                    hx.pull_reduce(HD, H, gshard)

        hooks = Fn.Hooks(head_chunks=chunks, post_src_head=post_src_head)
        hooks.force_chunked = True
        need_er = er is not None and ctx.needs_input_grad[5]
        need_ee = ee is not None and ctx.needs_input_grad[6]
        grad_el, grad_er, grad_ee = Fn._backward_core(
            pg.local, ctx.cfg, hooks, hx.table, el_all, er, ee, keep, attn_mul, src_scale, dst_scale, out, row_max, row_sum,
            gout, hx.gtable, need_er, need_ee)
        main.wait_stream(hx.stream)
        grad_ft_own = gshard[:n_own, :HD].unflatten(1, (H, D))
        grad_el_own = gshard[:n_own, HD:HD + H]
        return (None, None, None, grad_ft_own, grad_el_own, grad_er, grad_ee, None, None, None, None, None, None, None)


class PartitionedGraph:
    """This rank's share of a homogeneous graph.

    ``src``/``dst`` are the FULL graph's COO (every rank passes the same tensors); afterwards
    only the local edge set is kept.  Attributes:
      bounds        (P+1,) row ranges        lo, hi, n_own
      edge_gid      global edge id of every local edge (local edge order = global edge-id order)
      local         ``bot_b200.Graph`` block: n_dst = n_own destinations; sources are numbered
                    dense : owner*max_own + (gid - bounds[owner])     (n_src = P*max_own)
                    sparse: [owned rows | halo rows sorted by gid]    (n_src = n_own + n_halo)
      halo_gid      (sparse) global ids of the halo rows
    """

    def __init__(self, src, dst, n_nodes, world=None, rank=None, group=None, plan="auto", build_graph=True):
        self.group = group
        # per-head pipelining of the halo exchange in `gat` (see _gat_head_pipelined); opt-in until measured at N = 8
        self.pipeline_heads = os.environ.get("BOTGAT_PIPE_HEADS", "0") == "1"
        # halo exchange of the dense plan: "nccl" = all_gather_into_tensor / reduce_scatter_tensor of whole tables;
        # "p2p" = this repo's peer-memory kernels (csrc/halo.cu), pipelined per head range (needs NVLink peer access)
        # (measured on 8 B200s, profiles/r02_multi_gpu.md: p2p 2.98 vs nccl 3.19 ms/step at the proteins shape).  "auto" =
        # p2p on CUDA when the symmetric-memory rendezvous succeeds, else nccl.
        self.exchange = os.environ.get("BOTGAT_EXCHANGE", "auto")
        self.halo_chunks = int(os.environ.get("BOTGAT_HALO_CHUNKS", "0"))    # head ranges per exchange; 0 = auto (2)
        self._p2p, self._p2p_failed, self._p2p_error = {}, False, None
        self.world = dist.get_world_size(group) if world is None else world
        self.rank = dist.get_rank(group) if rank is None else rank
        self.n_nodes = n_nodes
        dev = src.device
        self.bounds = partition_bounds(dst, n_nodes, self.world)
        b = self.bounds.tolist()
        self.lo, self.hi = b[self.rank], b[self.rank + 1]
        self.n_own = self.hi - self.lo
        self.max_own = max(b[i + 1] - b[i] for i in range(self.world))

        mine = torch.nonzero((dst >= self.lo) & (dst < self.hi)).flatten()
        self.edge_gid = mine
        s, d = src.index_select(0, mine), dst.index_select(0, mine)
        ldst = d - self.lo
        owned = (s >= self.lo) & (s < self.hi)
        self.halo_gid = torch.unique(s[~owned])  # sorted
        if plan == "auto":
            # dense when this rank references most of the table anyway (uniformly random graphs)
            plan = "dense" if (self.halo_gid.numel() + self.n_own) * 2 >= n_nodes else "sparse"
            if dist.is_initialized() and self.world > 1:
                flag = torch.tensor([1 if plan == "dense" else 0], device=dev)
                dist.all_reduce(flag, op=dist.ReduceOp.MAX, group=group)  # ranks must agree
                plan = "dense" if int(flag.item()) else "sparse"
        self.plan = plan

        if plan == "dense":
            owner = torch.searchsorted(self.bounds, s, right=True) - 1
            lsrc = owner * self.max_own + (s - self.bounds.index_select(0, owner))
            n_src = self.world * self.max_own
            self.send_idx = self.send_counts = self.recv_counts = None
        else:
            lsrc = torch.where(owned, s - self.lo, self.n_own + torch.searchsorted(self.halo_gid, s))
            n_src = self.n_own + self.halo_gid.numel()
            self._plan_sparse(dev)
        self.lsrc, self.ldst, self.n_src_local = lsrc, ldst, n_src
        self.local = Graph(lsrc, ldst, n_src, self.n_own, is_block=True) if build_graph else None

    def _plan_sparse(self, dev):
        """Tell every owner which of its rows this rank needs (one all-to-all of id lists at setup)."""
        halo_owner = torch.searchsorted(self.bounds, self.halo_gid, right=True) - 1
        self.recv_counts = torch.bincount(halo_owner, minlength=self.world).tolist()
        if self.world == 1:
            self.send_counts, self.send_idx = [0], torch.zeros(0, dtype=torch.int64, device=dev)
            return
        rc = torch.tensor(self.recv_counts, dtype=torch.int64, device=dev)
        sc = torch.empty_like(rc)
        dist.all_to_all_single(sc, rc, group=self.group)
        self.send_counts = sc.tolist()
        want = torch.empty(sum(self.send_counts), dtype=torch.int64, device=dev)
        # halo_gid is sorted by gid, hence grouped by owner in rank order
        dist.all_to_all_single(want, self.halo_gid.contiguous(), output_split_sizes=self.send_counts,
                               input_split_sizes=self.recv_counts, group=self.group)
        self.send_idx = want - self.lo

    # ---- exchange ---------------------------------------------------------
    def _pad(self, t):
        if t.shape[0] == self.max_own:
            return t
        return torch.cat([t, t.new_zeros((self.max_own - t.shape[0],) + tuple(t.shape[1:]))], 0)

    def halo_gather(self, *owned_tables):
        """Local source tables (rows in ``local``'s source numbering) from row-sharded ones.

        Every argument is (n_own, ...).  One collective per table (the big feature table lands
        contiguous and aligned, ready for the gather kernels; the logit table is tiny).  Differentiable."""
        outs = []
        for t in owned_tables:
            if self.world == 1:
                outs.append(self._pad(t) if self.plan == "dense" else t)
            elif self.plan == "dense":
                outs.append(_DenseHalo.apply(self._pad(t), self.group))
            else:
                outs.append(_SparseHalo.apply(t, self.send_idx, self.send_counts, self.recv_counts, self.group))
        return outs[0] if len(outs) == 1 else tuple(outs)

    def gat(self, ft_own, el_own, er=None, ee=None, keep=None, attn_mul=None, src_scale=None, dst_scale=None,
            slope=0.2, attn_p=0.0, seed=0, edge_order="eid", halo_slot=0):
        """The partitioned layer in one call: halo exchange + ``gat_fused`` on the local block, with the collectives
        overlapped with the work that does not depend on them (dense plan):
          forward : all-gather of [ft], [el]  ||  edge staging            -> forward gather kernel
          backward: node + src pass -> reduce-scatter of grad_ft, grad_el  ||  edge phase (grad_ee, grad_er)
        ``src_scale`` is given for the LOCAL source numbering (``halo_gather`` a row-sharded one).  ``edge_order``:
        order of the per-edge operands' rows, "eid" = local edge order (``local_edges``), "canonical" = the local
        block's canonical order (``self.local.edge_perm()``), see ``functional.gat_fused``."""
        from .functional import Hooks, gat_fused, to_canonical

        if edge_order == "eid" and isinstance(self.local, Graph):
            ee, keep, attn_mul = (to_canonical(self.local, t) for t in (ee, keep, attn_mul))
        edge_order = "canonical"

        if self.world > 1 and self.plan == "dense" and self.exchange in ("p2p", "auto") and ft_own.is_cuda and ft_own.dim() == 3 \
                and isinstance(self.local, Graph) and self._p2p_usable(ft_own.shape[1], ft_own.shape[2], halo_slot):
            H, D = ft_own.shape[1], ft_own.shape[2]
            # the exchange buffers hold the gathered table until the layer's backward has run: layers whose forward /
            # backward overlap in time (a multi-layer model) each need their own ``halo_slot``
            hx = self.halo_buffers(H, D, halo_slot)
            n = max(1, min(H, self.halo_chunks if self.halo_chunks > 0 else 2))
            if self.local._info.n_slots_in or self.local._info.n_slots_out:
                n = 1     # split (heavy) rows need the full head range in one launch
            bounds = [round(i * H / n) for i in range(n + 1)]
            chunks = [(bounds[i], bounds[i + 1] - bounds[i]) for i in range(n) if bounds[i + 1] > bounds[i]]
            return _P2PGatFn.apply(self, hx, chunks, ft_own, el_own, er, ee, keep, attn_mul, src_scale, dst_scale, slope, attn_p,
                                   seed)
        if self.world == 1 or self.plan != "dense":
            ft_all, el_all = self.halo_gather(ft_own, el_own)
            return gat_fused(self.local, ft_all, el_all, er, ee, keep, attn_mul, src_scale, dst_scale, slope, attn_p, seed,
                             edge_order=edge_order)
        st = _HaloState()
        if self.pipeline_heads and ft_own.dim() == 3 and ft_own.shape[1] > 1:
            return self._gat_head_pipelined(st, ft_own, el_own, er, ee, keep, attn_mul, src_scale, dst_scale, slope, attn_p, seed)
        ft_all = _DenseHaloAsync.apply(self._pad(ft_own), self.group, st, "ft")
        el_all = _DenseHaloAsync.apply(self._pad(el_own), self.group, st, "el")

        def pre_kernel():
            st.fwd.pop("ft").wait()
            st.fwd.pop("el").wait()

        def post_src(grad_ft, grad_el):
            for key, g in (("ft", grad_ft), ("el", grad_el)):
                out = g.new_empty((g.shape[0] // self.world,) + tuple(g.shape[1:]))
                work = dist.reduce_scatter_tensor(out, g, op=dist.ReduceOp.SUM, group=self.group, async_op=True)
                st.bwd[key] = (work, out)

        out = gat_fused(self.local, ft_all, el_all, er, ee, keep, attn_mul, src_scale, dst_scale, slope, attn_p, seed,
                        hooks=Hooks(pre_kernel, post_src), edge_order=edge_order)
        return out

    def _gat_head_pipelined(self, st, ft_own, el_own, er, ee, keep, attn_mul, src_scale, dst_scale, slope, attn_p, seed):
        """`gat` with the feature exchange pipelined per head against per-head kernel launches (the kernels work
        head-major): all-gather of head h+1 || forward kernel of head h; backward src kernel of head h+1 ||
        reduce-scatter of head h's grad_ft.  Opt-in (``pipeline_heads`` / BOTGAT_PIPE_HEADS=1)."""
        from .functional import Hooks, gat_fused

        H = ft_own.shape[1]
        chunks = [(h, 1) for h in range(H)]
        ft_all = _DenseHaloHeads.apply(self._pad(ft_own), self.group, st, chunks)
        el_all = _DenseHaloAsync.apply(self._pad(el_own), self.group, st, "el")

        def pre_head(i):
            if i == 0:
                st.fwd.pop("el").wait()
            work, buf = st.fwd_chunks[i]
            work.wait()
            hb, hc = chunks[i]
            st.out[:, hb:hb + hc].copy_(buf)

        def post_src_head(i, grad_ft, grad_el):
            hb, hc = chunks[i]
            g = grad_ft[:, hb:hb + hc].contiguous()
            piece = g.new_empty((g.shape[0] // self.world,) + tuple(g.shape[1:]))
            work = dist.reduce_scatter_tensor(piece, g, op=dist.ReduceOp.SUM, group=self.group, async_op=True)
            st.bwd_chunks.append((work, piece))
            if i == len(chunks) - 1:
                out = grad_el.new_empty((grad_el.shape[0] // self.world,) + tuple(grad_el.shape[1:]))
                w = dist.reduce_scatter_tensor(out, grad_el, op=dist.ReduceOp.SUM, group=self.group, async_op=True)
                st.bwd["el"] = (w, out)

        return gat_fused(self.local, ft_all, el_all, er, ee, keep, attn_mul, src_scale, dst_scale, slope, attn_p, seed,
                         hooks=Hooks(head_chunks=chunks, pre_head=pre_head, post_src_head=post_src_head),
                         edge_order="canonical")

    def _p2p_usable(self, H, D, halo_slot):
        """Create (once) the peer-memory exchange buffers; with ``exchange = "auto"`` a failing symmetric-memory
        rendezvous (no peer access, an older torch) falls back to the NCCL collectives on EVERY rank."""
        if self.exchange == "p2p" or (H, D, halo_slot) in self._p2p:
            return True
        if self._p2p_failed:
            return False
        ok = 1
        try:
            self.halo_buffers(H, D, halo_slot)
        except Exception as ex:  # noqa: BLE001 - any failure means "use NCCL"
            ok = 0
            self._p2p_error = repr(ex)
        flag = torch.tensor([ok], device=self.local.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)     # the ranks must agree
        if int(flag.item()) == 0:
            self._p2p_failed = True
            self._p2p.pop((H, D, halo_slot), None)
            self.exchange = "nccl"
            return False
        self.exchange = "p2p"
        return True

    def halo_buffers(self, H, D, halo_slot=0):
        """The peer-memory exchange buffers of a (H, D) layer (``exchange = "p2p"``): write this rank's projected rows
        straight into ``.own_ft`` (n_own, H, D) / ``.own_el`` (n_own, H) and pass those views to ``gat`` — no copy."""
        hx = self._p2p.get((H, D, halo_slot))
        if hx is None:
            hx = self._p2p[(H, D, halo_slot)] = P2PHalo(self, H, D)
        return hx

    def owned_slice(self, full_table):
        """Rows of a replicated (N, ...) table this rank owns."""
        return full_table[self.lo:self.hi]

    def local_edges(self, edge_table):
        """Rows of a replicated (E, ...) edge table that belong to the local edges, local edge order."""
        return edge_table.index_select(0, self.edge_gid)


def partition_bounds_device(graph, n_parts):
    """The same bounds from the device in-CSR of an ingested graph (``botgat_partition_1d``)."""
    import ctypes as C

    from . import _lib
    from .graph import _stream

    out = (C.c_int64 * (n_parts + 1))()
    _lib.check(_lib.load().botgat_partition_1d(graph._ensure(), n_parts, out, _stream()), "botgat_partition_1d")
    return torch.tensor(list(out), dtype=torch.int64)


def partition_extract_device(graph, lo, hi):
    """Local edge set of destination rows [lo, hi) from the device structure (``botgat_partition_extract``):
    (global edge ids, global sources, local destinations), edge-id order."""
    import ctypes as C

    from . import _lib
    from .graph import _stream

    lib, h = _lib.load(), graph._ensure()
    n = C.c_int64()
    _lib.check(lib.botgat_partition_extract(h, lo, hi, None, None, None, C.byref(n), _stream()), "botgat_partition_extract")
    dev = graph.device
    eid = torch.empty(n.value, dtype=torch.int64, device=dev)
    src = torch.empty_like(eid)
    ldst = torch.empty_like(eid)
    if n.value:
        _lib.check(lib.botgat_partition_extract(h, lo, hi, _lib.ptr(eid), _lib.ptr(src), _lib.ptr(ldst), C.byref(n), _stream()),
                   "botgat_partition_extract")
    return eid, src, ldst
