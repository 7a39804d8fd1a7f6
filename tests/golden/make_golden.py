"""Generate the golden vectors under tests/golden/ by running the UNMODIFIED reference modules
(src/*/models.py of a reference checkout) on CPU on top of oracle/dgl_shim.py (DGL itself is not installable
offline; the shim restates only the DGL primitives, SURVEY.md Appendix B).

    BOT_REFERENCE=<reference checkout> python tests/golden/make_golden.py

Each case stores: the COO graph, the module's state_dict, the inputs, the output, the gradients of a fixed
scalar loss w.r.t. the inputs and parameters, and — for training-mode cases — the random edge-drop permutation
and attention-dropout multiplier the reference drew, so that a test can replay them.
"""
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import dgl_shim, graph_ref  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


class Recorder:
    """Capture what the reference draws: torch.randperm results and nn.Dropout multipliers."""

    def __init__(self):
        self.perms, self.drops = [], []

    def __enter__(self):
        self._randperm = torch.randperm
        self._dropout_fwd = torch.nn.Dropout.forward

        def randperm(*a, **k):
            p = self._randperm(*a, **k)
            self.perms.append(p.clone())
            return p

        rec = self

        def dropout_forward(mod, x):
            y = rec._dropout_fwd(mod, x)
            if mod.training and mod.p > 0 and getattr(mod, "_record", False):
                with torch.no_grad():
                    rec.drops.append(rec_mul(x, y, mod.p))
            return y

        torch.randperm = randperm
        torch.nn.Dropout.forward = dropout_forward
        return self

    def __exit__(self, *exc):
        torch.randperm = self._randperm
        torch.nn.Dropout.forward = self._dropout_fwd


def rec_mul(x, y, p):
    """multiplier y/x where x != 0; edge_softmax outputs are > 0 so this is exact enough to tell kept from dropped"""
    keep = (y != 0).float()
    return keep / (1.0 - p)


def make_graph(n, e, seed, self_loops):
    src, dst = graph_ref.synthetic_coo(n, e, seed)
    if self_loops:
        src, dst = graph_ref.add_self_loop(*graph_ref.remove_self_loop(src, dst), n)
    return src, dst


def run_case(name, ref_mod, kind, n, e, seed, self_loops, ctor, in_feats, train, edge_feats=0, block=None):
    torch.manual_seed(seed)
    src, dst = make_graph(n, e, seed, self_loops)
    n_dst = n
    if block is not None:  # bipartite block: dst nodes are the first `block` nodes
        n_dst = block
        keep = dst < block
        src, dst = src[keep], dst[keep]
    g = dgl_shim.ShimGraph(src, dst, n, n_dst, is_block=block is not None)
    conv = ref_mod.GATConv(**ctor)
    conv.train(train)
    conv.attn_drop._record = True
    x = torch.randn(n, in_feats, requires_grad=True)
    fe = torch.randn(len(src), edge_feats, requires_grad=True) if edge_feats else None
    if kind == "v2" and ctor.get("use_symmetric_norm"):
        deg = torch.bincount(torch.as_tensor(src), minlength=n).float().clamp(min=1)
        g.srcdata["deg"] = deg
        g.dstdata["deg"] = deg[:n_dst]
    with Recorder() as rec:
        y = conv(g, x) if kind == "v1" else conv(g, x, fe)
    w = torch.randn(y.shape, generator=torch.Generator().manual_seed(seed + 1))
    loss = (y * w).sum()
    loss.backward()
    case = {
        "kind": kind, "ctor": ctor, "train": train, "n": n, "n_dst": n_dst, "block": block is not None,
        "src": torch.as_tensor(src), "dst": torch.as_tensor(dst),
        "state_dict": {k: v.detach().clone() for k, v in conv.state_dict().items()},
        "x": x.detach().clone(), "fe": None if fe is None else fe.detach().clone(), "w": w,
        "y": y.detach().clone(), "gx": x.grad.clone(), "gfe": None if fe is None else fe.grad.clone(),
        "gparams": {k: p.grad.clone() for k, p in conv.named_parameters() if p.grad is not None},
        "perm": rec.perms[0] if rec.perms else None,
        "attn_mul": rec.drops[0] if rec.drops else None,
    }
    torch.save(case, os.path.join(OUT, name + ".pt"))
    print(name, tuple(y.shape), float(y.abs().max()), "perm" if rec.perms else "", "drop" if rec.drops else "")


def main():
    v1 = dgl_shim.import_reference("no-sampling")
    v2 = dgl_shim.import_reference("ogbn-proteins")
    # V1 (src/no-sampling/models.py:416-566)
    run_case("v1_eval_plain", v1, "v1", 60, 400, 0, True, dict(in_feats=12, out_feats=8, num_heads=3), 12, False)
    run_case("v1_eval_symm_attnr", v1, "v1", 60, 400, 1, True,
             dict(in_feats=12, out_feats=8, num_heads=3, use_symmetric_norm=True, non_interactive_attn=True), 12, False)
    run_case("v1_eval_nolinear_last", v1, "v1", 50, 300, 2, True,
             dict(in_feats=24, out_feats=7, num_heads=1, linear=False, use_symmetric_norm=True), 24, False)
    run_case("v1_train_edgedrop_attndrop", v1, "v1", 60, 500, 3, True,
             dict(in_feats=12, out_feats=8, num_heads=2, attn_drop=0.3, edge_drop=0.4, use_symmetric_norm=True), 12, True)
    run_case("v1_train_attndrop_only", v1, "v1", 40, 300, 4, True,
             dict(in_feats=10, out_feats=250 // 25, num_heads=3, attn_drop=0.1, non_interactive_attn=True), 10, True)
    # V2 (src/ogbn-proteins/models.py:19-168)
    run_case("v2_eval_edgefeat", v2, "v2", 60, 500, 5, False,
             dict(node_feats=16, edge_feats=6, out_feats=8, n_heads=3), 16, False, edge_feats=6)
    run_case("v2_eval_noedge_nodst", v2, "v2", 60, 500, 6, False,
             dict(node_feats=16, edge_feats=0, out_feats=12, n_heads=2, use_attn_dst=False), 16, False)
    run_case("v2_train_edgedrop", v2, "v2", 60, 600, 7, False,
             dict(node_feats=16, edge_feats=6, out_feats=8, n_heads=3, edge_drop=0.1), 16, True, edge_feats=6)
    run_case("v2_train_edgedrop_attndrop", v2, "v2", 50, 500, 8, False,
             dict(node_feats=8, edge_feats=4, out_feats=4, n_heads=6, edge_drop=0.25, attn_drop=0.2), 8, True, edge_feats=4)
    run_case("v2_eval_symm", v2, "v2", 50, 400, 9, False,
             dict(node_feats=8, edge_feats=4, out_feats=4, n_heads=2, use_symmetric_norm=True), 8, False, edge_feats=4)
    run_case("v2_eval_block", v2, "v2", 80, 900, 10, False,
             dict(node_feats=8, edge_feats=4, out_feats=4, n_heads=2), 8, False, edge_feats=4, block=25)
    run_case("v1_eval_block", v1, "v1", 80, 900, 11, False,
             dict(in_feats=8, out_feats=4, num_heads=2, allow_zero_in_degree=True, non_interactive_attn=True), 8, False,
             block=25)


def run_model_case(name, build, feed, n, e, seed, self_loops=False):
    """Whole-model golden vector (eval mode, so no random draws): state_dict, inputs, logits."""
    torch.manual_seed(seed)
    src, dst = make_graph(n, e, seed, self_loops)
    g = dgl_shim.ShimGraph(src, dst, n)
    model = build()
    model.eval()
    inputs = feed(g, len(src), n)
    with torch.no_grad():
        y = model(*inputs["call"](g))
    torch.save({"src": torch.as_tensor(src), "dst": torch.as_tensor(dst), "n": n,
                "state_dict": {k: v.detach().clone() for k, v in model.state_dict().items()},
                "tensors": inputs["tensors"], "y": y.detach().clone()}, os.path.join(OUT, name + ".pt"))
    print(name, tuple(y.shape), float(y.abs().max()))


def model_cases():
    v1 = dgl_shim.import_reference("no-sampling")
    prot = dgl_shim.import_reference("ogbn-proteins")
    prod = dgl_shim.import_reference("ogbn-products")

    def feed_v1(g, E, n):
        x = torch.randn(n, 20)
        return {"tensors": {"feat": x}, "call": lambda g: (g, x)}

    run_model_case("model_v1_gat_bn", lambda: v1.GAT(20, 0, 5, 8, 3, 2, F.relu, norm="batch", dropout=0.5, attn_drop=0.1,
                                                       use_symmetric_norm=True, linear=True, residual=True), feed_v1, 70, 500, 20, True)
    run_model_case("model_v1_gat_bias", lambda: v1.GAT(20, 0, 5, 8, 2, 3, F.relu, norm="none", non_interactive_attn=True),
                   feed_v1, 70, 500, 21, True)

    def feed_prot(g, E, n):
        x, ef = torch.randn(n, 8), torch.randn(E, 8)
        g.srcdata["feat"] = x
        g.edata["feat"] = ef
        return {"tensors": {"feat": x, "efeat": ef}, "call": lambda g: (g,)}

    run_model_case("model_proteins_gat", lambda: prot.GAT(8, 8, 11, 2, 3, 10, 16, F.relu, 0.25, 0.1, 0.0, 0.1), feed_prot, 60, 600, 22)

    def feed_prod(g, E, n):
        x = torch.randn(n, 9)
        g.srcdata["feat"] = x
        return {"tensors": {"feat": x}, "call": lambda g: (g,)}

    run_model_case("model_products_gat", lambda: prod.GAT(9, 0, 7, 2, 2, 6, 0, F.relu, 0.5, 0.1, 0.0, 0.1,
                                                          allow_zero_in_degree=True, residual=True), feed_prod, 60, 600, 23)


def gcn_cases():
    """GraphConv / GCN (SURVEY 8f rank 3): layer outputs + input gradients, model logits."""
    v1 = dgl_shim.import_reference("no-sampling")
    for name, ctor, fin, seed in (("gcn_both_wfirst", dict(in_feats=24, out_feats=8, norm="both"), 24, 30),
                                  ("gcn_right_aggfirst", dict(in_feats=8, out_feats=20, norm="right"), 8, 31),
                                  ("gcn_none_nobias", dict(in_feats=12, out_feats=12, norm="none", bias=False), 12, 32)):
        torch.manual_seed(seed)
        src, dst = make_graph(60, 500, seed, True)
        g = dgl_shim.ShimGraph(src, dst, 60)
        conv = v1.GraphConv(**ctor)
        x = torch.randn(60, fin, requires_grad=True)
        y = conv(g, x)
        w = torch.randn(y.shape, generator=torch.Generator().manual_seed(seed + 1))
        (y * w).sum().backward()
        torch.save({"ctor": ctor, "src": torch.as_tensor(src), "dst": torch.as_tensor(dst), "n": 60,
                    "state_dict": {k: v.detach().clone() for k, v in conv.state_dict().items()},
                    "x": x.detach().clone(), "w": w, "y": y.detach().clone(), "gx": x.grad.clone(),
                    "gparams": {k: p.grad.clone() for k, p in conv.named_parameters() if p.grad is not None}},
                   os.path.join(OUT, name + ".pt"))
        print(name, tuple(y.shape), float(y.abs().max()))

    def feed(g, E, n):
        x = torch.randn(n, 20)
        return {"tensors": {"feat": x}, "call": lambda g: (g, x)}

    run_model_case("model_v1_gcn", lambda: v1.GCN(20, 5, 16, 3, F.relu, norm="batch", norm_adj="symm", dropout=0.5,
                                                   residual=True, use_linear=True), feed, 70, 500, 33, True)


if __name__ == "__main__":
    main()
    model_cases()
    gcn_cases()
