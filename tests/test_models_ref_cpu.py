"""The whole-model oracle (oracle/models_ref.py) against the recorded reference models (CPU).

In eval mode with no draws, the fp64 restatement of each GAT wrapper must give the ``y`` the unmodified reference model
recorded in tests/golden/model_*gat*.pt, to the 5e-5 the engine is held to in
test_gpu_golden.test_whole_model_matches_reference.  This ties the oracle of test_gpu_model_train.py to reference data."""
import glob
import os

import pytest
import torch

from oracle import models_ref
from util import rel_err

GOLDEN_GAT_MODELS = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "model_*gat*.pt")))

# the constructor arguments of test_gpu_golden._build_model, as the oracle's keywords
CTOR = {
    # GAT(20, 0, 5, 8, 3, 2, F.relu, norm="batch", dropout=0.5, attn_drop=0.1, use_symmetric_norm=True, linear=True,
    #     residual=True)
    "model_v1_gat_bn": ("full", dict(n_layers=3, norm="batch", residual=True, use_symmetric_norm=True)),
    # GAT(20, 0, 5, 8, 2, 3, F.relu, norm="none", non_interactive_attn=True)
    "model_v1_gat_bias": ("full", dict(n_layers=2, norm="none", residual=False, use_symmetric_norm=False)),
    # ProteinsGAT(8, 8, 11, 2, 3, 10, 16, F.relu, 0.25, 0.1, 0.0, 0.1)
    "model_proteins_gat": ("proteins", dict(n_layers=2)),
    # ProductsGAT(9, 0, 7, 2, 2, 6, 0, F.relu, 0.5, 0.1, 0.0, 0.1, allow_zero_in_degree=True, residual=True)
    "model_products_gat": ("products", dict(n_layers=2, residual=True)),
}


def oracle_model_forward(case, name, dtype=torch.float64):
    kind, kw = CTOR[name]
    sd = case["state_dict"]
    t = {k: v.to(dtype) for k, v in case["tensors"].items()}
    g = models_ref.Coo(case["src"], case["dst"], case["n"], case["n"])
    if kind == "full":
        return models_ref.gat_full_graph(sd, g, t["feat"], **kw)
    if kind == "proteins":
        return models_ref.proteins_gat(sd, g, t["feat"], t.get("efeat"), **kw)
    return models_ref.products_gat(sd, g, t["feat"], **kw)


def test_every_golden_gat_model_has_a_constructor():
    names = [os.path.basename(p)[:-3] for p in GOLDEN_GAT_MODELS]
    assert sorted(names) == sorted(CTOR)


@pytest.mark.parametrize("path", GOLDEN_GAT_MODELS, ids=[os.path.basename(p)[:-3] for p in GOLDEN_GAT_MODELS])
def test_model_oracle_matches_reference(path):
    case = torch.load(path, weights_only=False)
    name = os.path.basename(path)[:-3]
    y, stats = oracle_model_forward(case, name)
    assert stats == {}   # eval mode: the running statistics are read, not updated
    assert y.dtype == torch.float64 and y.shape == case["y"].shape
    err = rel_err(y, case["y"])
    print(f"\n[{name}] fp64 oracle vs reference: {err:.2e}")
    assert err <= 5e-5


def test_model_oracle_train_mode_batch_norm():
    """Training mode: batch statistics, and running statistics updated like nn.BatchNorm1d's (unbiased variance)."""
    path = os.path.join(os.path.dirname(__file__), "golden", "model_products_gat.pt")
    case = torch.load(path, weights_only=False)
    sd = case["state_dict"]
    g = models_ref.Coo(case["src"], case["dst"], case["n"], case["n"])
    x = case["tensors"]["feat"].double()
    y_eval, _ = models_ref.products_gat(sd, g, x, n_layers=2, residual=True)
    y, stats = models_ref.products_gat(sd, g, x, n_layers=2, residual=True, training=True)
    assert set(stats) == {f"norms.{i}.{k}" for i in range(2) for k in ("running_mean", "running_var", "num_batches_tracked")}
    assert not torch.allclose(y, y_eval)
    # layer 0 by hand: the pre-norm activations of the first layer, then nn.BatchNorm1d's own update
    from oracle import modules_ref

    c = {k[len("convs.0."):]: v.double() for k, v in sd.items() if k.startswith("convs.0.")}
    h0 = modules_ref.gatconv_v2(c, g.src, g.dst, g.n_src, g.n_dst, x, n_heads=2, out_feats=6).flatten(1)
    bn = torch.nn.BatchNorm1d(12).double().train()
    bn.load_state_dict({k[len("norms.0."):]: v for k, v in sd.items() if k.startswith("norms.0.")})
    bn(h0)
    assert torch.allclose(stats["norms.0.running_mean"], bn.running_mean, rtol=1e-12, atol=1e-14)
    assert torch.allclose(stats["norms.0.running_var"], bn.running_var, rtol=1e-12, atol=1e-14)
    assert int(stats["norms.0.num_batches_tracked"]) == int(sd["norms.0.num_batches_tracked"]) + 1
    # the state_dict the oracle was given is left as it was
    assert torch.equal(sd["norms.0.running_mean"], case["state_dict"]["norms.0.running_mean"])


def test_model_oracle_applies_draws():
    """A keep set, an attention multiplier and node-dropout masks reach the places the model body uses them."""
    path = os.path.join(os.path.dirname(__file__), "golden", "model_v1_gat_bias.pt")
    case = torch.load(path, weights_only=False)
    sd = case["state_dict"]
    g = models_ref.Coo(case["src"], case["dst"], case["n"], case["n"])
    x = case["tensors"]["feat"].double()
    kw = dict(n_layers=2, norm="none", residual=False)
    base, _ = models_ref.gat_full_graph(sd, g, x, **kw)
    E = g.src.numel()
    ones = [torch.ones(E, dtype=torch.bool)] * 2
    unit = models_ref.Draws(keep=ones, attn_mul=[torch.ones(E, 3), torch.ones(E, 1)], input_drop=torch.ones_like(x),
                            dropout=[torch.ones(case["n"], 24)])
    same, _ = models_ref.gat_full_graph(sd, g, x, draws=unit, **kw)
    assert torch.allclose(same, base, rtol=1e-12, atol=1e-12)
    gen = torch.Generator().manual_seed(0)
    for draws in (models_ref.Draws(keep=[torch.rand(E, generator=gen) > 0.3, None]),
                  models_ref.Draws(attn_mul=[None, (torch.rand(E, 1, generator=gen) > 0.3) / 0.7]),
                  models_ref.Draws(input_drop=(torch.rand(x.shape, generator=gen) > 0.3) / 0.7),
                  models_ref.Draws(dropout=[(torch.rand(case["n"], 24, generator=gen) > 0.3) / 0.7])):
        y, _ = models_ref.gat_full_graph(sd, g, x, draws=draws, **kw)
        assert rel_err(y, base) > 1e-3
    with pytest.raises(ValueError, match="dropout masks"):
        models_ref.gat_full_graph(sd, g, x, draws=models_ref.Draws(dropout=[torch.ones(case["n"], 24)] * 2), **kw)
