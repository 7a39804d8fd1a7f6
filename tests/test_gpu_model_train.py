"""Whole-model TRAINING steps of the GAT wrappers against the fp64 restatement of oracle/models_ref.py — `-m gpu`.

Each test runs three consecutive training steps (Adam between them) of ``no_sampling.GAT``, ``sampled.ProteinsGAT`` or
``sampled.ProductsGAT`` and replays every step in fp64 on the CPU from the state_dict the step started from, with the
random draws the engine made.  Compared: the loss, the model output, every parameter gradient and the BatchNorm running
statistics the step leaves behind.  This reaches what the eval-mode model tests cannot: the production edge-drop keep
mask (a ``KeptEdges`` in canonical edge order), the in-kernel Philox attention dropout with a fresh seed per layer and
step, the fused edge encoder's gradients, the folded projections, the residual (sliced on blocks) under training-mode
BatchNorm, and the state carried from one step to the next (kept-edge subsets, ``HostFeed`` ring slots, the
``EdgeFrame`` canonical cache).

Recording the draws.  The engine's own draw function (``draw_edge_keep``) and layer entry points (``GATConvSampledFn``,
``gat_fused``) are wrapped: the wrappers record what was drawn (the keep mask, ``attn_p``, the seed) and call through
unchanged.  For the oracle the canonical keep mask goes to edge-id order through ``graph.canonical_edge_ids()``, and the
attention multiplier is the numpy Philox restatement keyed on the canonical edge number.  The node-feature dropouts
(torch's ``nn.Dropout``, not under test) are replaced by a module that draws its mask from a CPU generator and keeps it.

Tolerances: the loss, the output and the running statistics within ``FWD_TOL``, every gradient within ``GRAD_TOL``,
norm-relative per tensor."""
import time

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle import models_ref
from util import FWD_TOL, GRAD_TOL, philox_attn_mul, rel_err

pytestmark = pytest.mark.gpu
STEPS = 3
# an analytically zero gradient is judged against the gradient of its layer's weight (see _check_step)
ZERO_GRAD_TOL = 1e-5


def _power_law_graph(n, e, seed, in_alpha=0.8, out_alpha=0.0):
    """COO with destinations ~ rank^-in_alpha (and sources ~ rank^-out_alpha over another node order), self-loops
    removed and one added per node, edge ids shuffled so that the canonical order is a real permutation."""
    rng = np.random.default_rng(seed)

    def draw(alpha):
        if alpha <= 0:
            return rng.integers(0, n, size=e)
        w = np.arange(1, n + 1, dtype=np.float64) ** -alpha
        rank = np.minimum(np.searchsorted(np.cumsum(w / w.sum()), rng.random(e)), n - 1)
        return rng.permutation(n)[rank]

    dst, src = draw(in_alpha), draw(out_alpha)
    off = src != dst
    loop = np.arange(n)
    src, dst = np.concatenate([src[off], loop]), np.concatenate([dst[off], loop])
    p = rng.permutation(src.size)
    return torch.from_numpy(src[p].astype(np.int64)), torch.from_numpy(dst[p].astype(np.int64))


class RecordedDropout(nn.Module):
    """``nn.Dropout`` whose keep mask comes from a CPU generator and is kept for the oracle."""

    def __init__(self, p, seed):
        super().__init__()
        self.p, self.gen, self.masks = p, torch.Generator().manual_seed(seed), []

    def forward(self, x):
        if not self.training or self.p == 0:
            return x
        keep = torch.rand(x.shape, generator=self.gen) >= self.p
        self.masks.append(keep)
        return x * keep.to(x.device, x.dtype) * (1.0 / (1.0 - self.p))

    def take(self):
        """The multipliers drawn since the last call, in fp64."""
        out, self.masks = [m.double() / (1.0 - self.p) for m in self.masks], []
        return out


class Recorder:
    """Wraps the engine's edge-drop draw and the layer entry points the modules call.  Records the draws, changes
    nothing: the returned keep set (a ``KeptEdges`` on CUDA) and every argument go through as they were."""

    def __init__(self, monkeypatch):
        from bot_b200 import functional, no_sampling, sampled

        self.keeps, self.calls, self.edge_mlp = [], [], 0
        real_draw, real_fn, real_gf = no_sampling.draw_edge_keep, functional.GATConvSampledFn, functional.gat_fused
        real_mlp = functional.EdgeMLPLogits
        rec = self

        def draw_edge_keep(n_edges, edge_drop, device):
            keep, eids = real_draw(n_edges, edge_drop, device)
            rec.keeps.append((keep, eids))
            return keep, eids

        class SampledFn:
            @staticmethod
            def apply(*args):
                rec.calls.append({"attn_p": args[13], "seed": args[14]})
                return real_fn.apply(*args)

        class EdgeMLP:
            @staticmethod
            def apply(*args):
                rec.edge_mlp += 1
                return real_mlp.apply(*args)

        def gat_fused(*args, **kw):
            rec.calls.append({"attn_p": args[10], "seed": args[11]})
            return real_gf(*args, **kw)

        for mod in (no_sampling, sampled):
            monkeypatch.setattr(mod, "draw_edge_keep", draw_edge_keep)
            monkeypatch.setattr(mod, "gat_fused", gat_fused)
        monkeypatch.setattr(sampled, "GATConvSampledFn", SampledFn)
        monkeypatch.setattr(functional, "GATConvSampledFn", SampledFn)   # no_sampling imports it at call time
        monkeypatch.setattr(functional, "EdgeMLPLogits", EdgeMLP)

    def take(self):
        out = (self.keeps, self.calls, self.edge_mlp)
        self.keeps, self.calls, self.edge_mlp = [], [], 0
        return out


def _install_dropouts(model, seed):
    model.input_drop = RecordedDropout(model.input_drop.p, seed)
    model.dropout = RecordedDropout(model.dropout.p, seed + 1)


def _snapshot(model):
    return {k: v.detach().clone() for k, v in model.state_dict().items()}


def _train(model, forward, loss_fn, rec, steps=STEPS):
    """``steps`` training steps with an Adam step between them.  ``forward(step)`` returns ``(y, ctx)``; ``ctx`` carries
    what the oracle needs (engine graphs, CPU inputs, labels).  Returns one record per step."""
    opt = torch.optim.Adam(model.parameters(), lr=1e-2)
    out = []
    for step in range(steps):
        before = _snapshot(model)
        opt.zero_grad(set_to_none=True)
        y, ctx = forward(step)
        loss = loss_fn(y, ctx["labels"])
        loss.backward()
        keeps, calls, edge_mlp = rec.take()
        out.append(dict(before=before, after=_snapshot(model), loss=loss.detach().clone(), y=y.detach().clone(),
                        grads={n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None},
                        keeps=keeps, calls=calls, edge_mlp=edge_mlp, input_drop=model.input_drop.take(),
                        dropout=model.dropout.take(), ctx=ctx))
        opt.step()
    torch.cuda.synchronize()
    return out


def _draws(r, heads, edge_drop):
    """The step's draws in edge-id order, for the oracle."""
    from bot_b200.no_sampling import KeptEdges

    graphs = r["ctx"]["graphs"]
    keep = None
    if edge_drop > 0:
        assert len(r["keeps"]) == len(graphs)
        keep = []
        for (k, eids), g in zip(r["keeps"], graphs):
            E = g.number_of_edges()
            assert isinstance(eids, KeptEdges), "on CUDA the keep set is the selection draw's canonical mask"
            assert k.dtype == torch.uint8 and k.shape == (E,) and int(k.sum()) == E - int(E * edge_drop)
            cid = g.canonical_edge_ids()
            keep.append((k if cid is None else k[cid]).bool().cpu())
    else:
        assert not r["keeps"]
    assert len(r["calls"]) == len(graphs)
    attn = []
    for c, g, H in zip(r["calls"], graphs, heads):
        if c["attn_p"] > 0:   # the in-kernel stream is keyed on the canonical edge number
            cid = g.canonical_edge_ids()
            ids = np.arange(g.number_of_edges()) if cid is None else cid.cpu().numpy()
            attn.append(philox_attn_mul(c["seed"], 0, H, c["attn_p"], eids=ids).double())
        else:
            attn.append(None)
    inp = r["input_drop"]
    assert len(inp) <= 1
    return models_ref.Draws(keep=keep, attn_mul=attn, input_drop=inp[0] if inp else None, dropout=r["dropout"])


def _check_step(name, step, r, param_names, oracle_fn, loss_fn, heads, edge_drop, zero_grads=()):
    """One recorded engine step against the fp64 oracle run from the state_dict the step started from.  Returns
    {quantity: (error, bound)}."""
    sd = {k: v.cpu().double() if v.is_floating_point() else v.cpu() for k, v in r["before"].items()}
    for k in param_names:
        sd[k].requires_grad_(True)
    y, stats = oracle_fn(sd, _draws(r, heads, edge_drop), r["ctx"])
    loss = loss_fn(y, r["ctx"]["labels_cpu"])
    loss.backward()
    ref_loss = float(loss.detach())
    errs = {"loss": (abs(float(r["loss"]) - ref_loss) / abs(ref_loss), FWD_TOL),
            "out": (rel_err(r["y"], y), FWD_TOL)}
    for k in param_names:
        ref, got = sd[k].grad, r["grads"].get(k)
        assert (got is None) == (ref is None), f"{name} step {step}: gradient of {k} is {got is None} on the engine"
        if ref is None:
            continue
        if k in zero_grads:
            # the bias of dst_fc feeds a training-mode BatchNorm (directly and through every later residual), which
            # removes any per-column shift: its gradient is zero up to rounding and cannot be judged relative to itself
            w = zero_grads[k]
            scale = float(r["grads"][w].abs().max())
            assert float(ref.abs().max()) <= 1e-12 * float(sd[w].grad.abs().max())
            errs["|grad " + k + "|"] = (float(got.abs().max()) / scale, ZERO_GRAD_TOL)
        else:
            errs["grad " + k] = (rel_err(got, ref), GRAD_TOL)
    has_bn = any(k.endswith("running_mean") for k in sd)
    assert bool(stats) == has_bn, "training mode updates the running statistics of every BatchNorm, and nothing else"
    for k, v in stats.items():
        if k.endswith("num_batches_tracked"):
            assert int(r["after"][k]) == int(v), k
        else:
            errs[k] = (rel_err(r["after"][k], v), FWD_TOL)
    print(f"\n[{name} step {step}] " + " ".join(f"{k}={e:.1e}" for k, (e, _) in errs.items()))
    return errs


def _check_run(name, steps, model, oracle_fn, loss_fn, heads, edge_drop, zero_grads=()):
    """Every step of ``steps`` against the oracle; the draws must differ between layers and between steps."""
    names = [n for n, _ in model.named_parameters()]
    worst = {}
    for i, r in enumerate(steps):
        for k, (e, bound) in _check_step(name, i, r, names, oracle_fn, loss_fn, heads, edge_drop, zero_grads).items():
            assert e <= bound, f"{name} step {i}: {k} error {e:.3e} > {bound}"
            if k not in worst or e / bound > worst[k][0] / worst[k][1]:
                worst[k] = (e, bound)
    k, (e, bound) = max(worst.items(), key=lambda kv: kv[1][0] / kv[1][1])
    print(f"\n[{name}] worst: {k} {e:.2e} (bound {bound:.0e}, {bound / max(e, 1e-300):.0f}x margin)")
    keeps = [k for r in steps for k, _ in r["keeps"]]
    for a in range(len(keeps)):
        for b in range(a):
            if keeps[a].shape == keeps[b].shape:
                assert not torch.equal(keeps[a], keeps[b]), "edge-drop keep masks repeat between layers or steps"
    seeds = [c["seed"] for r in steps for c in r["calls"] if c["attn_p"] > 0]
    assert len(set(seeds)) == len(seeds), "attention-dropout seeds repeat between layers or steps"
    return worst


def _grads_identical(a, b):
    assert torch.equal(a["loss"], b["loss"]) and torch.equal(a["y"], b["y"])
    assert a["grads"].keys() == b["grads"].keys()
    for k in a["grads"]:
        assert torch.equal(a["grads"][k], b["grads"][k]), k


def _bce(y, labels):
    return F.binary_cross_entropy_with_logits(y, labels)


def _ce(y, labels):
    return F.cross_entropy(y, labels)


# ---- proteins, full graph ------------------------------------------------------------------------------------------

PROTEINS = dict(node_feats=8, edge_feats=8, n_classes=16, n_layers=3, n_heads=6, n_hidden=16, edge_emb=16, dropout=0.25,
                input_drop=0.1, attn_drop=0.0, edge_drop=0.1)


def _proteins_model(cuda, **over):
    from bot_b200.sampled import ProteinsGAT

    c = dict(PROTEINS, **over)
    torch.manual_seed(0)
    model = ProteinsGAT(c["node_feats"], c["edge_feats"], c["n_classes"], c["n_layers"], c["n_heads"], c["n_hidden"],
                        c["edge_emb"], F.relu, c["dropout"], c["input_drop"], c["attn_drop"], c["edge_drop"]).to(cuda)
    _install_dropouts(model, seed=5)
    return model.train(), c


def _dst_bias_pairs(n_layers):
    return {f"convs.{i}.dst_fc.bias": f"convs.{i}.dst_fc.weight" for i in range(n_layers)}


@pytest.mark.parametrize("knobs", ["default", "seg64", "rowwise"])
def test_proteins_full_graph_training(cuda, monkeypatch, knobs):
    """The bench's proteins step scaled down: 3 layers, 6 heads, fused edge encoder, edge drop, node dropouts, BCE.
    The features are fed as the benchmark feeds them (``HostFeed`` + ``edata.put_canonical``) and, from the same RNG
    state, through ``edata["feat"]`` in edge-id order: the two must be bit-identical.  ``seg64`` splits heavy rows of
    both CSRs into segments, ``rowwise`` forces the all-heads-per-row kernels."""
    import bot_b200

    t0 = time.time()
    env = {"default": {}, "seg64": {"BOTGAT_SEG": "64"}, "rowwise": {"BOTGAT_ROWWISE": "1"}}[knobs]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    n = 3000
    src, dst = _power_law_graph(n, 40000, seed=1, in_alpha=0.8, out_alpha=0.6)
    E = src.numel()
    gen = torch.Generator().manual_seed(2)
    x = torch.randn(n, PROTEINS["node_feats"], generator=gen)
    efeat = torch.rand(E, PROTEINS["edge_feats"], generator=gen)
    labels = (torch.rand(n, PROTEINS["n_classes"], generator=gen) > 0.5).float()
    g = bot_b200.Graph(src.to(cuda), dst.to(cuda), n)
    perm = g.edge_perm()
    assert perm is not None, "the test needs a graph whose canonical order is a real permutation"
    if knobs == "seg64":
        assert g._info.n_seg_in > 0 and g._info.n_seg_out > 0
    ctx = {"graphs": [g] * PROTEINS["n_layers"], "labels": labels.to(cuda), "labels_cpu": labels.double()}
    rec = Recorder(monkeypatch)
    runs = {}
    for feed in ("host", "eid"):
        model, c = _proteins_model(cuda)
        if feed == "host":
            hf = bot_b200.HostFeed(cuda, depth=2)
            host = [x.pin_memory(), efeat[perm.cpu()].contiguous().pin_memory()]
            hf.submit(*host)

            def forward(step):
                if step + 1 < STEPS:
                    hf.submit(*host)
                xd, fe = hf.take()
                g.srcdata["feat"] = xd.wait()
                g.edata.put_canonical("feat", fe.wait())      # static features stored canonically on the host
                return model(g), ctx
        else:
            xd, ed = x.to(cuda), efeat.to(cuda)

            def forward(step):
                g.srcdata["feat"] = xd
                g.edata["feat"] = ed                          # edge-id order (DGL's edata)
                return model(g), ctx
        torch.manual_seed(10)
        runs[feed] = _train(model, forward, _bce, rec)
    for a, b in zip(runs["host"], runs["eid"]):
        _grads_identical(a, b)
    assert all(r["edge_mlp"] == PROTEINS["n_layers"] for r in runs["host"]), "the fused edge-MLP path must run"

    coo = models_ref.Coo(src, dst, n, n)

    def oracle(sd, draws, ctx):
        return models_ref.proteins_gat(sd, coo, x.double(), efeat.double(), n_layers=c["n_layers"], training=True,
                                       draws=draws)

    _check_run(f"proteins-full-{knobs}", runs["host"], model, oracle, _bce, [c["n_heads"]] * c["n_layers"],
               c["edge_drop"], _dst_bias_pairs(c["n_layers"]))
    print(f"\n[proteins-full-{knobs}] {time.time() - t0:.1f} s")


# ---- proteins, sampled blocks --------------------------------------------------------------------------------------

def test_proteins_sampled_blocks_training(cuda, monkeypatch):
    """The proteins model on ``MultiLayerNeighborSampler`` blocks (a new batch and new blocks every step), edge drop and
    in-kernel attention dropout on: the residual ``h_last[: n_dst]`` of a block, block edge features ``parent[EID]``."""
    import bot_b200
    from bot_b200 import sampling

    t0 = time.time()
    n = 4000
    src, dst = _power_law_graph(n, 50000, seed=3, in_alpha=0.8)
    gen = torch.Generator().manual_seed(4)
    x = torch.randn(n, PROTEINS["node_feats"], generator=gen)
    efeat = torch.rand(src.numel(), PROTEINS["edge_feats"], generator=gen)
    labels = (torch.rand(n, PROTEINS["n_classes"], generator=gen) > 0.5).float()
    g = bot_b200.Graph(src.to(cuda), dst.to(cuda), n)
    g.ndata["feat"], g.edata["feat"] = x.to(cuda), efeat.to(cuda)
    rec = Recorder(monkeypatch)
    model, c = _proteins_model(cuda, attn_drop=0.1)
    sampler = sampling.MultiLayerNeighborSampler([12, 10, 8])
    order = torch.randperm(n, generator=gen)

    def forward(step):
        seeds = order[step * 600:(step + 1) * 600]
        blocks = sampler.sample_blocks(g, seeds.to(cuda), seed=100 + step)
        assert all(b.number_of_src_nodes() > b.number_of_dst_nodes() for b in blocks)
        return model(blocks), {"graphs": blocks, "labels": labels[seeds].to(cuda), "labels_cpu": labels[seeds].double(),
                               "seeds": seeds}

    torch.manual_seed(11)
    steps = _train(model, forward, _bce, rec)
    assert all(r["edge_mlp"] == c["n_layers"] for r in steps)

    def oracle(sd, draws, ctx):
        blocks = ctx["graphs"]
        coo = [models_ref.Coo(b.edges()[0].cpu(), b.edges()[1].cpu(), b.number_of_src_nodes(), b.number_of_dst_nodes(),
                              True) for b in blocks]
        fe = [efeat[b.edata[sampling.EID].cpu()].double() for b in blocks]
        feat = x[blocks[0].srcdata[sampling.NID].cpu()].double()
        assert torch.equal(blocks[-1].dstdata[sampling.NID].cpu(), ctx["seeds"])
        return models_ref.proteins_gat(sd, coo, feat, fe, n_layers=c["n_layers"], training=True, draws=draws)

    _check_run("proteins-blocks", steps, model, oracle, _bce, [c["n_heads"]] * c["n_layers"], c["edge_drop"],
               _dst_bias_pairs(c["n_layers"]))
    print(f"\n[proteins-blocks] {time.time() - t0:.1f} s")


# ---- products, full graph ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("residual", [True, False], ids=["residual", "no_residual"])
def test_products_training(cuda, monkeypatch, residual):
    """The products model (no edge features, no node encoder in the data path), edge drop, node dropouts,
    cross-entropy, with and without its residual."""
    import bot_b200
    from bot_b200.sampled import ProductsGAT

    t0 = time.time()
    n, feats, classes, layers, heads, hidden = 3000, 12, 10, 3, 4, 8
    src, dst = _power_law_graph(n, 40000, seed=6, in_alpha=0.9)
    gen = torch.Generator().manual_seed(7)
    x = torch.randn(n, feats, generator=gen)
    labels = torch.randint(0, classes, (n,), generator=gen)
    g = bot_b200.Graph(src.to(cuda), dst.to(cuda), n)
    assert g.edge_perm() is not None
    g.ndata["feat"] = x.to(cuda)
    ctx = {"graphs": [g] * layers, "labels": labels.to(cuda), "labels_cpu": labels}
    rec = Recorder(monkeypatch)
    torch.manual_seed(0)
    model = ProductsGAT(feats, 0, classes, layers, heads, hidden, 0, F.relu, 0.5, 0.1, 0.0, 0.1, residual=residual).to(cuda)
    _install_dropouts(model, seed=8)
    model.train()
    torch.manual_seed(12)
    steps = _train(model, lambda step: (model(g), ctx), _ce, rec)
    assert all(r["grads"].get("node_encoder.weight") is None for r in steps)

    coo = models_ref.Coo(src, dst, n, n)

    def oracle(sd, draws, ctx):
        return models_ref.products_gat(sd, coo, x.double(), n_layers=layers, residual=residual, training=True, draws=draws)

    name = f"products-{'residual' if residual else 'no_residual'}"
    _check_run(name, steps, model, oracle, _ce, [heads] * layers, 0.1, _dst_bias_pairs(layers))
    print(f"\n[{name}] {time.time() - t0:.1f} s")


# ---- no_sampling.GAT (arxiv / reddit settings) ---------------------------------------------------------------------

@pytest.mark.parametrize("variant", ["batch_norm", "bias"])
def test_full_graph_gat_training(cuda, monkeypatch, variant):
    """``no_sampling.GAT``: ``batch_norm`` is the arxiv setting (BatchNorm, symmetric norm, ``linear`` and residual:
    the folded projections), ``bias`` takes the ``ElementWiseLinear`` path with ``non_interactive_attn`` and no
    ``res_fc`` (the unfolded layer).  Both with in-kernel attention dropout, edge drop, node dropouts, a one-head last
    layer and cross-entropy."""
    import bot_b200
    from bot_b200.no_sampling import GAT

    t0 = time.time()
    n, feats, classes, layers, heads, hidden = 3000, 16, 8, 3, 3, 12
    kw = dict(norm="batch", use_symmetric_norm=True, linear=True, residual=True) if variant == "batch_norm" else \
        dict(norm="none", non_interactive_attn=True)
    src, dst = _power_law_graph(n, 40000, seed=9, in_alpha=0.8, out_alpha=0.5)
    gen = torch.Generator().manual_seed(10)
    x = torch.randn(n, feats, generator=gen)
    labels = torch.randint(0, classes, (n,), generator=gen)
    g = bot_b200.Graph(src.to(cuda), dst.to(cuda), n)
    assert g.edge_perm() is not None
    xd = x.to(cuda)
    ctx = {"graphs": [g] * layers, "labels": labels.to(cuda), "labels_cpu": labels}
    rec = Recorder(monkeypatch)
    torch.manual_seed(0)
    model = GAT(feats, 0, classes, hidden, layers, heads, F.relu, dropout=0.5, input_drop=0.25, attn_drop=0.1,
                edge_drop=0.1, **kw).to(cuda)
    _install_dropouts(model, seed=13)
    model.train()
    torch.manual_seed(14)
    steps = _train(model, lambda step: (model(g, xd), ctx), _ce, rec)

    coo = models_ref.Coo(src, dst, n, n)

    def oracle(sd, draws, ctx):
        return models_ref.gat_full_graph(sd, coo, x.double(), n_layers=layers, norm=kw["norm"],
                                         residual=kw.get("residual", False),
                                         use_symmetric_norm=kw.get("use_symmetric_norm", False), training=True,
                                         draws=draws)

    _check_run(f"gat-{variant}", steps, model, oracle, _ce, [heads] * (layers - 1) + [1], 0.1)
    print(f"\n[gat-{variant}] {time.time() - t0:.1f} s")

