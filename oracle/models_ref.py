"""Whole-model oracle: the forward bodies of the three GAT wrappers restated on top of ``oracle.modules_ref`` —
TEST INFRASTRUCTURE ONLY.

* ``gat_full_graph``  src/no-sampling/models.py:644-736      (``bot_b200.no_sampling.GAT``)
* ``proteins_gat``    src/ogbn-proteins/models.py:230-264    (``bot_b200.sampled.ProteinsGAT``)
* ``products_gat``    src/ogbn-products/models.py:168-265    (``bot_b200.sampled.ProductsGAT``)

Every function takes a model state_dict, the graph as COO in edge-id order (one :class:`Coo` per layer for sampled
blocks), features in edge-id order and the random draws of the step (:class:`Draws`), and runs in the dtype of the
node features (the tests use fp64).  It returns ``(y, stats)``: the model output and, in training mode, the
BatchNorm running statistics the step leaves behind (state_dict keys).  In eval mode with no draws the output is
pinned to the recorded reference models by tests/test_models_ref_cpu.py.
"""
from __future__ import annotations

from typing import NamedTuple

import torch
import torch.nn.functional as F

from . import modules_ref


class Coo(NamedTuple):
    """One layer's graph: (E,) int64 ``src`` / ``dst`` in edge-id order; ``is_block``: dst nodes are the first
    ``n_dst`` src nodes (a DGL message-flow block)."""
    src: torch.Tensor
    dst: torch.Tensor
    n_src: int
    n_dst: int
    is_block: bool = False


class Draws:
    """The random draws of one training step, as the model consumed them.

    ``keep``       per layer: (E,) bool edge-drop keep set in edge-id order, or None (no edge drop)
    ``attn_mul``   per layer: (E, H) attention-dropout multiplier (0 or 1/(1-p)) in edge-id order, or None
    ``input_drop`` multiplier (0 or 1/(1-p)) shaped like the input of the model's ``input_drop``, or None
    ``dropout``    one multiplier per call of the model's ``dropout``, in call order (one per layer that has it)
    """

    def __init__(self, keep=None, attn_mul=None, input_drop=None, dropout=()):
        self.keep, self.attn_mul, self.input_drop, self.dropout = keep, attn_mul, input_drop, list(dropout)


class _Step:
    """Hands the draws out in the order the model body asks for them; no draws = every dropout is the identity."""

    def __init__(self, draws, dtype):
        self.d, self.dtype, self._next = draws, dtype, 0

    def keep(self, i):
        return None if self.d is None or self.d.keep is None else self.d.keep[i]

    def attn_mul(self, i):
        if self.d is None or self.d.attn_mul is None or self.d.attn_mul[i] is None:
            return None
        return self.d.attn_mul[i].to(self.dtype)

    def input_drop(self, x):
        if self.d is None or self.d.input_drop is None:
            return x
        return x * self.d.input_drop.to(self.dtype)

    def dropout(self, x):
        if self.d is None or not self.d.dropout:
            return x
        m = self.d.dropout[self._next]
        self._next += 1
        return x * m.to(self.dtype)

    def done(self):
        if self.d is not None and self.d.dropout and self._next != len(self.d.dropout):
            raise ValueError(f"{len(self.d.dropout)} dropout masks given, the model body used {self._next}")


def _sub(sd, prefix):
    p = prefix + "."
    return {k[len(p):]: v for k, v in sd.items() if k.startswith(p)}


def _cast(sd, dtype):
    return {k: v.to(dtype) if v.is_floating_point() else v for k, v in sd.items()}


def _batch_norm(h, sd, prefix, training, stats, momentum, eps):
    """``nn.BatchNorm1d`` (affine, tracking running statistics): batch statistics and an updated running mean / unbiased
    variance in training mode, the running statistics in eval mode."""
    mean, var = sd[prefix + ".running_mean"].clone(), sd[prefix + ".running_var"].clone()
    y = F.batch_norm(h, mean, var, sd[prefix + ".weight"], sd[prefix + ".bias"], training, momentum, eps)
    if training:
        stats[prefix + ".running_mean"], stats[prefix + ".running_var"] = mean, var
        stats[prefix + ".num_batches_tracked"] = sd[prefix + ".num_batches_tracked"] + 1
    return y


def gat_full_graph(sd, graph: Coo, feat, *, n_layers, norm="none", residual=False, use_symmetric_norm=False,
                   activation=F.relu, training=False, draws=None, bn_momentum=0.1, bn_eps=1e-5):
    """src/no-sampling/models.py:644-736 (``GAT.forward``); ``norm`` "batch" or "none" (``ElementWiseLinear`` bias)."""
    dtype = feat.dtype
    sd = _cast(sd, dtype)
    d, stats = _Step(draws, dtype), {}
    h = d.input_drop(feat)
    h_last = None
    for i in range(n_layers):
        c = _sub(sd, f"convs.{i}")
        _, H, D = c["attn_l"].shape
        h = modules_ref.gatconv_v1(c, graph.src, graph.dst, graph.n_src, graph.n_dst, h, num_heads=H, out_feats=D,
                                   use_symmetric_norm=use_symmetric_norm, is_block=graph.is_block, keep=d.keep(i),
                                   attn_mul=d.attn_mul(i))
        if i < n_layers - 1:
            if residual and h_last is not None:                               # :720-731
                h = h + h_last
            h_last = h
            h = h.flatten(1)
            if norm == "batch":
                h = _batch_norm(h, sd, f"norms.{i}", training, stats, bn_momentum, bn_eps)
            else:
                h = h + sd[f"biases.{i}.bias"]
            h = d.dropout(activation(h))
    d.done()
    last = max(int(k.split(".")[1]) for k in sd if k.startswith("biases."))
    return h.mean(1) + sd[f"biases.{last}.bias"], stats


def _sampled_layers(sd, graphs, h, efeat, residual, activation, training, d, stats, bn_momentum, bn_eps):
    """The layer loop shared by the proteins and products models (src/ogbn-proteins/models.py:230-264)."""
    h_last = None
    for i, g in enumerate(graphs):
        c = _sub(sd, f"convs.{i}")
        H = c["attn_src_fc.weight"].shape[0]
        D = c["src_fc.weight"].shape[0] // H
        emb = None
        if efeat is not None and f"edge_encoder.{i}.weight" in sd:            # :245-247
            emb = F.relu(F.linear(efeat[i], sd[f"edge_encoder.{i}.weight"], sd[f"edge_encoder.{i}.bias"]))
        h = modules_ref.gatconv_v2(c, g.src, g.dst, g.n_src, g.n_dst, h, emb, n_heads=H, out_feats=D,
                                   is_block=g.is_block, keep=d.keep(i), attn_mul=d.attn_mul(i))
        h = h.flatten(1, -1)
        if h_last is not None and residual:                                   # :253-260
            h = h + h_last[: h.shape[0], :]
        h_last = h
        h = _batch_norm(h, sd, f"norms.{i}", training, stats, bn_momentum, bn_eps)
        h = d.dropout(activation(h))
    d.done()
    return F.linear(h, sd["pred_linear.weight"], sd["pred_linear.bias"])


def _graphs(graphs, n_layers):
    return list(graphs) if isinstance(graphs, (list, tuple)) and not isinstance(graphs, Coo) else [graphs] * n_layers


def proteins_gat(sd, graphs, feat, efeat=None, *, n_layers, activation=F.relu, training=False, draws=None,
                 bn_momentum=0.1, bn_eps=1e-5):
    """src/ogbn-proteins/models.py:230-264: node encoder + ReLU + input dropout, the per-layer edge encoder + ReLU
    feeding ``attn_edge_fc``, the unconditional residual, BatchNorm, ``pred_linear``.  ``graphs``: one :class:`Coo` (full
    graph) or one per layer (blocks, input layer first); ``efeat``: the raw edge features in edge-id order, one tensor
    (full graph) or one per layer, or None."""
    dtype = feat.dtype
    sd = _cast(sd, dtype)
    graphs = _graphs(graphs, n_layers)
    if efeat is not None and not isinstance(efeat, (list, tuple)):
        efeat = [efeat] * n_layers
    efeat = None if efeat is None else [e.to(dtype) for e in efeat]
    d, stats = _Step(draws, dtype), {}
    h = d.input_drop(F.relu(F.linear(feat, sd["node_encoder.weight"], sd["node_encoder.bias"])))
    return _sampled_layers(sd, graphs, h, efeat, True, activation, training, d, stats, bn_momentum, bn_eps), stats


def products_gat(sd, graphs, feat, *, n_layers, residual=False, activation=F.relu, training=False, draws=None,
                 bn_momentum=0.1, bn_eps=1e-5):
    """src/ogbn-products/models.py:168-265: input dropout on the raw features (the node encoder is never called), the
    residual gated by ``residual``, BatchNorm, ``pred_linear``; no edge features."""
    dtype = feat.dtype
    sd = _cast(sd, dtype)
    d, stats = _Step(draws, dtype), {}
    h = d.input_drop(feat)
    y = _sampled_layers(sd, _graphs(graphs, n_layers), h, None, residual, activation, training, d, stats, bn_momentum,
                        bn_eps)
    return y, stats
