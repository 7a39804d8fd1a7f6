"""Parity of the CUDA path (through the C ABI) against the oracle — `-m gpu`."""
import zlib

import numpy as np
import pytest
import torch

from oracle import graph_ref
from util import check_case, engine_run, make_case, oracle_run, rel_err, FWD_TOL

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("canonical", [False, True])
@pytest.mark.parametrize("n,e,seed", [(1, 0, 0), (7, 3, 1), (100, 1000, 2), (2708, 13264, 3), (5000, 200000, 4)])
def test_structure_bit_exact(cuda, n, e, seed, canonical):
    """DGL's order (stable by edge id inside a row) and the default canonical order (neighbour lists sorted by id);
    row pointers, degrees and the edge-id maps are exact in both."""
    import bot_b200

    src, dst = graph_ref.synthetic_coo(n, e, seed, power_law=0.8 if seed == 4 else 0.0)
    ref = graph_ref.build_formats(src, dst, n, n, canonical=canonical)
    g = bot_b200.Graph(torch.from_numpy(src).to(cuda), torch.from_numpy(dst).to(cuda), n, canonical=canonical)
    if canonical and e > 1:
        assert np.array_equal(g.canonical_edge_ids().cpu().numpy(), graph_ref.canonical_edge_ids(src, dst))
        assert g._info.in_eid_identity == 1
    for name, arr in ref.items():
        got = g.structure(name).cpu().numpy()
        assert got.dtype == np.int64 and got.shape == arr.shape, name
        assert np.array_equal(got, arr), name
    assert g.has_zero_in_degree == bool((ref["in_deg"] == 0).any())


def test_block_structure(cuda):
    import bot_b200

    rng = np.random.default_rng(0)
    n_src, n_dst, e = 300, 40, 2000
    src = rng.integers(0, n_src, e)
    dst = rng.integers(0, n_dst, e)
    for canonical in (False, True):
        ref = graph_ref.build_formats(src, dst, n_src, n_dst, canonical=canonical)
        g = bot_b200.create_block((src, dst), n_src, n_dst, device=cuda, canonical=canonical)
        for name, arr in ref.items():
            assert np.array_equal(g.structure(name).cpu().numpy(), arr), name


def test_preprocess_bit_exact(cuda):
    """to_bidirected -> remove_self_loop -> add_self_loop (run.py:133-148)."""
    import bot_b200

    n, e = 500, 4000
    src, dst = graph_ref.synthetic_coo(n, e, 7)
    g = bot_b200.graph((src, dst), num_nodes=n, device=cuda)
    g2 = bot_b200.to_bidirected(g)
    rs, rd = graph_ref.to_bidirected(src, dst, n)
    assert np.array_equal(g2.edges()[0].cpu().numpy(), rs) and np.array_equal(g2.edges()[1].cpu().numpy(), rd)
    g3 = g2.remove_self_loop().add_self_loop()
    rs, rd = graph_ref.add_self_loop(*graph_ref.remove_self_loop(rs, rd), n)
    assert np.array_equal(g3.edges()[0].cpu().numpy(), rs) and np.array_equal(g3.edges()[1].cpu().numpy(), rd)
    assert g3.number_of_edges() == rs.shape[0]
    assert not g3.has_zero_in_degree


CASES = {
    # name: (n_src, n_dst, E, H, D, kwargs)
    "src_only_H3_D8": (200, 200, 3000, 3, 8, dict(er=False)),
    "er_H2_D16": (300, 300, 4000, 2, 16, dict()),
    "proteins_like_H6_D80_er_ee": (400, 400, 30000, 6, 80, dict(ee=True)),
    "proteins_like_edge_drop": (400, 400, 30000, 6, 80, dict(ee=True, keep_p=0.1)),
    "products_like_H4_D120": (500, 500, 20000, 4, 120, dict(keep_p=0.1)),
    "arxiv_like_H3_D250_symm": (600, 600, 9000, 3, 250, dict(er=False, symm=True, self_loops=True, attn_p=0.1)),
    "reddit_like_H4_D64_symm": (300, 300, 60000, 4, 64, dict(er=False, symm=True, attn_p=0.1)),
    "last_layer_H1_D40": (500, 500, 8000, 1, 40, dict(er=False, symm=True)),
    "last_layer_H1_D41_scalar": (500, 500, 8000, 1, 41, dict(er=False, symm=True)),
    "cora_like_H8_D8": (2708, 2708, 10556, 8, 8, dict(er=True, keep_p=0.5, self_loops=True)),
    "cora_last_H1_D7": (2708, 2708, 10556, 1, 7, dict(er=False, keep_p=0.5, self_loops=True, symm=True)),
    "block_Nd_lt_Ns": (900, 120, 5000, 4, 32, dict(ee=True)),
    "power_law_skew": (2000, 2000, 100000, 2, 64, dict(power_law=1.0, ee=True)),
    "zero_in_degree_rows": (300, 300, 200, 2, 24, dict(ee=True, keep_p=0.3)),
    "wide_D512": (100, 100, 2000, 1, 512, dict()),
    "odd_D250_H1": (150, 150, 3000, 1, 250, dict(ee=True, attn_p=0.2, keep_p=0.2)),
}


@pytest.mark.parametrize("name", list(CASES))
def test_fwd_bwd_parity(cuda, name):
    n_src, n_dst, e, H, D, kw = CASES[name]
    c = make_case(n_src, n_dst, e, H, D, seed=zlib.crc32(name.encode()) % 1000, **kw)
    errs = check_case(c, cuda)
    print(name, {k: f"{v:.2e}" for k, v in errs.items()})


def test_empty_graph(cuda):
    c = make_case(10, 10, 0, 2, 8, ee=True)
    out, g, _ = engine_run(c, cuda)
    assert out.shape == (10, 2, 8) and float(out.abs().max()) == 0.0
    assert float(g["ft"].abs().max()) == 0.0 and float(g["el"].abs().max()) == 0.0
    assert g["ee"].shape == (0, 2)


def test_all_edges_dropped_rows(cuda):
    """Rows whose every in-edge is dropped must produce 0 (reference: softmax over the kept edge subgraph)."""
    c = make_case(50, 50, 400, 2, 16, ee=True)
    keep = torch.ones(400, dtype=torch.bool)
    keep[c["dst"] < 10] = False
    c["keep"] = keep
    errs = check_case(c, cuda)
    out, _, _ = engine_run(c, cuda)
    assert float(out[:10].abs().max()) == 0.0
    assert torch.isfinite(out).all()


def test_column_parts_forward(cuda, monkeypatch):
    """Forcing a tiny L2 slab budget splits heads into column parts; results must not change."""
    c = make_case(3000, 3000, 20000, 2, 128, ee=True, seed=5)
    ref, _ = oracle_run(c)
    monkeypatch.setenv("BOTGAT_SLAB_MB", "1")
    monkeypatch.setenv("BOTGAT_ROWWISE", "0")   # the budget also steers the family choice; this test is about column parts
    out, _, _ = engine_run(c, cuda)
    assert rel_err(out, ref) <= FWD_TOL


def _gather_kernels(fn):
    """Normalised names of the gather kernels ``fn()`` launches (torch.profiler, CUDA activity)."""
    from torch.profiler import ProfilerActivity, profile

    from test_gpu_kernel_coverage import normalise

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {n for n in (normalise(e.name) for e in prof.events()) if n}


def test_forced_group_sizes(cuda, monkeypatch):
    """BOTGAT_G forces the lanes per neighbour of the head-major kernels; each shape is one the forced G covers (one
    vector slot per lane at G = D/4 and below), and the trace shows that G ran in both passes."""
    monkeypatch.setenv("BOTGAT_LOWDEG", "0")
    monkeypatch.setenv("BOTGAT_ROWWISE", "0")
    monkeypatch.setenv("BOTGAT_BWD_TMA", "0")
    for G, H, D in ((1, 2, 4), (2, 2, 8), (4, 2, 12), (8, 2, 16), (16, 2, 64), (32, 2, 64)):
        c = make_case(300, 300, 20000, H, D, ee=True, seed=6)
        monkeypatch.setenv("BOTGAT_G", str(G))
        names = _gather_kernels(lambda: check_case(c, cuda))
        gsh = G.bit_length() - 1
        assert {n.split("<")[0] for n in names} == {"botgat::gat_fwd_kernel", "botgat::gat_bwd_src_kernel"}, (G, names)
        assert all(n.split("<")[1].split(",")[1] == str(gsh) for n in names), (G, names)


@pytest.mark.parametrize("D", [301, 514])
def test_wide_heads_train(cuda, D):
    """Heads wider than the backward covers at their vector width (odd D > 256, D = 2 mod 4 > 512) are zero-padded to a
    multiple of 4 and train; the output and gradients keep the caller's width."""
    c = make_case(150, 150, 2000, 1, D, ee=True, keep_p=0.1, seed=D)
    check_case(c, cuda)


def test_too_wide_heads_are_rejected(cuda):
    """D > 1024 with gradients is rejected before any launch, naming the limit; with no input requiring grad it runs."""
    import bot_b200
    from bot_b200.functional import gat_fused

    c = make_case(50, 50, 300, 1, 1100, seed=3)
    g = bot_b200.Graph(c["src"].to(cuda), c["dst"].to(cuda), 50)
    ft = c["ft"].to(cuda).requires_grad_(True)
    with pytest.raises(ValueError, match="1024"):
        gat_fused(g, ft, c["el"].to(cuda), c["er"].to(cuda))
    out = gat_fused(g, ft.detach(), c["el"].to(cuda), c["er"].to(cuda))
    ref, _ = oracle_run(c)
    assert rel_err(out, ref) <= FWD_TOL


def test_deterministic(cuda):
    c = make_case(2000, 2000, 100000, 4, 64, ee=True, power_law=0.8, seed=9)
    o1, g1, _ = engine_run(c, cuda)
    o2, g2, _ = engine_run(c, cuda)
    assert torch.equal(o1, o2)
    for k in g1:
        assert torch.equal(g1[k], g2[k]), k


def test_softmax_rows_sum_to_one(cuda):
    """With ft = 1 the output is the row sum of attention = 1 on every row with an in-edge."""
    c = make_case(500, 500, 5000, 3, 16, ee=True, seed=11)
    c["ft"] = torch.ones_like(c["ft"])
    out, _, g = engine_run(c, cuda)
    has = (g.in_degrees() > 0).cpu()
    assert torch.allclose(out.cpu()[has], torch.ones_like(out.cpu()[has]), atol=2e-6)
    assert float(out.cpu()[~has].abs().max() if (~has).any() else 0.0) == 0.0


def test_padded_edge_records(cuda):
    """ee given as (E, 8) with H = 6 (32-byte records): same result, gradient padded with zeros."""
    import bot_b200
    from bot_b200.functional import gat_fused

    c = make_case(400, 400, 30000, 6, 80, ee=True, keep_p=0.1, seed=21)
    ref_out, ref_g = oracle_run(c)
    g = bot_b200.Graph(c["src"].to(cuda), c["dst"].to(cuda), 400)
    ee_pad = torch.zeros(30000, 8, device=cuda)
    ee_pad[:, :6] = c["ee"].to(cuda)
    ee_pad[:, 6:] = 123.0  # padding content must be ignored
    ee_pad.requires_grad_(True)
    ft = c["ft"].to(cuda).requires_grad_(True)
    el = c["el"].to(cuda).requires_grad_(True)
    er = c["er"].to(cuda).requires_grad_(True)
    out = gat_fused(g, ft, el, er, ee_pad, c["keep"].to(cuda))
    out.backward(c["gout"].to(cuda))
    assert rel_err(out, ref_out) <= FWD_TOL
    assert ee_pad.grad.shape == (30000, 8)
    assert float(ee_pad.grad[:, 6:].abs().max()) == 0.0
    assert rel_err(ee_pad.grad[:, :6], ref_g["ee"]) <= 1e-4
    assert rel_err(er.grad, ref_g["er"]) <= 1e-4 and rel_err(ft.grad, ref_g["ft"]) <= 1e-4


@pytest.mark.parametrize("rowwise", ["0", "1"])
@pytest.mark.parametrize("mode", ["staged", "direct"])
def test_edge_modes_agree(cuda, monkeypatch, mode, rowwise):
    """Staged and direct edge operands, with and without the all-heads-per-row kernels.  Those take no operand by edge
    id, so rowwise = 1 with the direct mode runs the head-major src pass; the plan of the src pass decides the record
    layout before the node phase, which therefore runs exactly once per backward."""
    from torch.profiler import ProfilerActivity, profile

    from bot_b200 import functional

    monkeypatch.setenv("BOTGAT_ROWWISE", rowwise)
    c = make_case(500, 500, 20000, 4, 32, ee=True, keep_p=0.2, attn_p=0.1, seed=22)
    old = functional.edge_mode
    functional.edge_mode = mode
    try:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            check_case(c, cuda)  # one forward and one backward
            torch.cuda.synchronize()
    finally:
        functional.edge_mode = old
    assert sum("gat_bwd_node_kernel" in e.name for e in prof.events()) == 1


@pytest.mark.parametrize("lowdeg", ["0", "1000000"])
@pytest.mark.parametrize("name", ["proteins_like_edge_drop", "arxiv_like_H3_D250_symm", "cora_like_H8_D8", "last_layer_H1_D41_scalar",
                                  "block_Nd_lt_Ns", "power_law_skew", "zero_in_degree_rows", "products_like_H4_D120"])
def test_both_kernel_families(cuda, monkeypatch, name, lowdeg):
    """Warp-per-row (BOTGAT_LOWDEG=0) and group-per-row (forced) kernels on the same cases."""
    monkeypatch.setenv("BOTGAT_LOWDEG", lowdeg)
    n_src, n_dst, e, H, D, kw = CASES[name]
    c = make_case(n_src, n_dst, e, H, D, seed=zlib.crc32(name.encode()) % 1000 + 1, **kw)
    check_case(c, cuda)


@pytest.mark.parametrize("lowdeg", ["0", "1000000"])
@pytest.mark.parametrize("seg", ["32", "64", "100"])
def test_row_splitting(cuda, monkeypatch, seg, lowdeg):
    """Heavy rows split into segments (segment length forced small), in the warp-per-row kernels (LDG and TMA src pass)
    and in the group-per-row family: same results, still deterministic."""
    monkeypatch.setenv("BOTGAT_SEG", seg)
    monkeypatch.setenv("BOTGAT_LOWDEG", lowdeg)
    c = make_case(600, 600, 60000, 3, 40, ee=True, keep_p=0.1, power_law=1.2, symm=True, seed=31)
    errs = check_case(c, cuda)
    o1, g1, g = engine_run(c, cuda)
    o2, g2, _ = engine_run(c, cuda)
    assert g._info.n_slots_in > 0 and g._info.n_slots_out >= 0
    assert torch.equal(o1, o2) and all(torch.equal(g1[k], g2[k]) for k in g1)


@pytest.mark.parametrize("lowdeg", ["0", "1000000"])
def test_row_splitting_all_dropped_segment(cuda, monkeypatch, lowdeg):
    """A whole segment of a split row dropped by edge-drop (max = -inf in that slot)."""
    monkeypatch.setenv("BOTGAT_SEG", "32")
    monkeypatch.setenv("BOTGAT_LOWDEG", lowdeg)
    c = make_case(100, 100, 3000, 2, 16, ee=True, power_law=1.5, seed=32)
    # drop the first 40 in-edges (edge-id order = CSR order inside a row) of the heaviest row
    keep = torch.ones(3000, dtype=torch.bool)
    idx = torch.nonzero(c["dst"] == 0).flatten()
    keep[idx[:40]] = False
    c["keep"] = keep
    check_case(c, cuda)


@pytest.mark.parametrize("E,C,H", [(0, 16, 6), (1000, 16, 6), (5000, 8, 4), (777, 5, 3), (3000, 64, 4), (2000, 16, 8), (100, 12, 1),
                                   (700001, 16, 6), (40003, 48, 6), (5001, 32, 8), (9000, 20, 5)])
def test_edge_logit_projection(cuda, E, C, H):
    """Streaming attn_edge_fc kernels (botgat_edge_proj_*) against torch's Linear, forward and backward."""
    from bot_b200.functional import edge_logits, pad_heads

    g = torch.Generator().manual_seed(E + C + H)
    x = torch.randn(E, C, generator=g).to(cuda).requires_grad_(True)
    w = torch.randn(H, C, generator=g).to(cuda).requires_grad_(True)
    y = edge_logits(x, w)
    assert y.shape == (E, pad_heads(H))
    ref = torch.nn.functional.linear(x.detach().double(), w.detach().double())
    assert rel_err(y[:, :H], ref) <= 1e-6
    if pad_heads(H) > H and E:
        assert float(y[:, H:].abs().max()) == 0.0
    gy = torch.randn(E, pad_heads(H), generator=g).to(cuda)
    y.backward(gy)
    gx_ref = gy[:, :H].double() @ w.detach().double()
    gw_ref = gy[:, :H].double().t() @ x.detach().double()
    assert rel_err(x.grad, gx_ref) <= 1e-6
    assert rel_err(w.grad, gw_ref) <= 1e-5
    # deterministic reduction
    x2 = x.detach().clone().requires_grad_(True)
    w2 = w.detach().clone().requires_grad_(True)
    edge_logits(x2, w2).backward(gy)
    assert torch.equal(w2.grad, w.grad) and torch.equal(x2.grad, x.grad)


def test_deferred_edge_features(cuda):
    """feat_edge produced on another stream (bot_b200.Deferred) gives the same result as a plain tensor."""
    import bot_b200
    from bot_b200.ogbn_proteins import GATConv

    torch.manual_seed(0)
    n, e = 300, 8000
    src = torch.randint(0, n, (e,), device=cuda)
    dst = torch.randint(0, n, (e,), device=cuda)
    g = bot_b200.Graph(src, dst, n)
    conv = GATConv(32, 16, 8, n_heads=6).to(cuda).eval()
    x = torch.randn(n, 32, device=cuda)
    fe_host = torch.randn(e, 16).pin_memory()
    y0 = conv(g, x, fe_host.to(cuda))
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        fe = fe_host.to(cuda, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(st)
    y1 = conv(g, x, bot_b200.Deferred(fe, ev))
    torch.cuda.synchronize()
    assert torch.equal(y0, y1)


@pytest.mark.parametrize("E,C,M,H", [(0, 8, 16, 6), (1000, 8, 16, 6), (5003, 8, 16, 8), (777, 5, 13, 3), (4000, 4, 16, 1),
                                     (3000, 3, 7, 2), (600011, 8, 16, 6)])
def test_edge_mlp_logits(cuda, E, C, M, H):
    """Fused edge encoder + ReLU + attn_edge_fc (botgat_edge_mlp_*) against the oracle restatement in fp64."""
    from bot_b200.functional import EdgeMLPLogits, pad_heads
    from oracle.modules_ref import edge_mlp_logits

    g = torch.Generator().manual_seed(E + C + M + H)
    x = torch.randn(E, C, generator=g)
    w1, b1, w2 = torch.randn(M, C, generator=g), torch.randn(M, generator=g), torch.randn(H, M, generator=g)
    gy = torch.randn(E, pad_heads(H), generator=g)
    ref_in = [t.double().requires_grad_(True) for t in (w1, b1, w2)]
    ref = edge_mlp_logits(x.double(), *ref_in)
    ref.backward(gy[:, :H].double())
    dev = [t.to(cuda).requires_grad_(True) for t in (w1, b1, w2)]
    y = EdgeMLPLogits.apply(x.to(cuda), *dev)
    assert y.shape == (E, pad_heads(H))
    y.backward(gy.to(cuda))
    if E:
        assert rel_err(y[:, :H], ref) <= 1e-6
        if pad_heads(H) > H:
            assert float(y[:, H:].abs().max()) == 0.0
        for got, want in zip(dev, ref_in):
            assert rel_err(got.grad, want.grad) <= 1e-5
    else:
        assert all(float(t.grad.abs().max()) == 0.0 for t in dev)
    dev2 = [t.detach().clone().requires_grad_(True) for t in dev]   # deterministic reduction
    EdgeMLPLogits.apply(x.to(cuda), *dev2).backward(gy.to(cuda))
    assert all(torch.equal(a.grad, b.grad) for a, b in zip(dev, dev2))


def test_edge_embedding_fused_equals_materialised(cuda):
    """GATConv given a lazy EdgeEmbedding (fused kernel) == given relu(encoder(efeat)) (the reference's data flow)."""
    import bot_b200
    from bot_b200.ogbn_proteins import GATConv

    torch.manual_seed(0)
    n, e = 300, 8000
    g = bot_b200.Graph(torch.randint(0, n, (e,), device=cuda), torch.randint(0, n, (e,), device=cuda), n)
    conv = GATConv(32, 16, 8, n_heads=6).to(cuda).eval()
    enc = torch.nn.Linear(8, 16).to(cuda)
    x = torch.randn(n, 32, device=cuda)
    efeat = torch.randn(e, 8, device=cuda)
    y0 = conv(g, x, torch.relu(enc(efeat)))
    y0.square().sum().backward()
    g0 = [p.grad.clone() for p in list(enc.parameters()) + [conv.attn_edge_fc.weight]]
    enc.zero_grad(), conv.zero_grad()
    y1 = conv(g, x, bot_b200.EdgeEmbedding(efeat, enc))
    y1.square().sum().backward()
    g1 = [p.grad for p in list(enc.parameters()) + [conv.attn_edge_fc.weight]]
    assert rel_err(y1, y0) <= FWD_TOL
    for a, b in zip(g1, g0):
        assert rel_err(a, b) <= 1e-4
    # unsupported width (edge_emb 32): falls back to the materialised embedding
    conv2 = GATConv(32, 32, 8, n_heads=6).to(cuda).eval()
    enc2 = torch.nn.Linear(8, 32).to(cuda)
    assert rel_err(conv2(g, x, bot_b200.EdgeEmbedding(efeat, enc2)), conv2(g, x, torch.relu(enc2(efeat)))) <= FWD_TOL


@pytest.mark.parametrize("E,n_drop,seed", [(1, 0, 1), (1, 1, 2), (2, 1, 3), (1001, 370, 4), (100000, 10000, 5),
                                           (3000001, 300000, 6), (50000, 49999, 7), (50000, 1, (1 << 61) + 12345),
                                           (9000001, 900000, 8)])
def test_edge_drop_draw_exact(cuda, E, n_drop, seed):
    """botgat_edge_drop_draw: exactly n_drop zeros, bit-identical to 'drop the n_drop smallest Philox keys'."""
    from bot_b200.functional import edge_drop_keep
    from util import philox_edge_drop_keep

    keep = edge_drop_keep(E, n_drop, seed, cuda)
    assert keep.dtype == torch.uint8 and keep.shape == (E,)
    assert int(keep.sum()) == E - n_drop
    assert torch.equal(keep.cpu(), philox_edge_drop_keep(seed, E, n_drop))
    assert torch.equal(keep, edge_drop_keep(E, n_drop, seed, cuda))


def test_edge_drop_draw_is_uniform(cuda):
    """Every edge is dropped with probability n_drop / E (the reference's randperm prefix): 400 draws on 2000 edges."""
    from bot_b200.functional import edge_drop_keep

    E, n_drop, draws = 2000, 600, 400
    freq = torch.zeros(E, device=cuda)
    for s in range(draws):
        freq += (edge_drop_keep(E, n_drop, 1000 + s, cuda) == 0).float()
    p = n_drop / E
    sd = (p * (1 - p) / draws) ** 0.5
    assert abs(float(freq.mean()) / draws - p) < 1e-9 + 1e-6           # exact count in every draw
    assert float((freq / draws - p).abs().max()) < 5.5 * sd            # no position favoured
    z = (freq / draws - p) / sd
    assert abs(float(z.std()) - 1.0) < 0.1


def test_module_edge_drop_uses_selection(cuda):
    """GATConv in training mode: the drawn mask has exactly int(E * p) zeros and follows torch's seed."""
    from bot_b200 import no_sampling

    torch.manual_seed(3)
    k1, ids1 = no_sampling.draw_edge_keep(10000, 0.37, cuda)
    torch.manual_seed(3)
    k2, _ = no_sampling.draw_edge_keep(10000, 0.37, cuda)
    k3, _ = no_sampling.draw_edge_keep(10000, 0.37, cuda)
    assert int(k1.sum()) == 10000 - 3700 and torch.equal(k1, k2) and not torch.equal(k1, k3)
    assert ids1.numel() == 6300 and torch.equal(ids1.ids(), torch.nonzero(k1).flatten())


@pytest.mark.parametrize("kind", ["lowdeg", "dense", "heavy_rows", "block", "symm_no_attn_dst"])
def test_folded_projections_match_unfolded(cuda, monkeypatch, kind):
    """sampled.GATConv with the four node-side Linears folded into two GEMMs (kernels reading ft / writing grad_ft
    inside the wide buffers, row stride != H*D) == the reference's op-by-op sequence, forward and every gradient."""
    import bot_b200
    from bot_b200 import sampled

    torch.manual_seed(1)
    n_src, n_dst, e, block = 400, 400, 3000, False
    kw = dict(n_heads=3, edge_drop=0.0)
    if kind == "dense":
        e = 60000
    elif kind == "heavy_rows":
        e = 60000
        monkeypatch.setenv("BOTGAT_SEG", "64")
    elif kind == "block":
        n_dst, block = 90, True
    elif kind == "symm_no_attn_dst":
        kw.update(use_symmetric_norm=True, use_attn_dst=False)
    src = torch.randint(0, n_src, (e,), device=cuda)
    dst = torch.randint(0, n_dst, (e,), device=cuda)
    if kind == "heavy_rows":
        dst[: e // 2] = 7
    g = bot_b200.Graph(src, dst, n_src, n_dst, is_block=block)
    if kw.get("use_symmetric_norm"):
        deg = g.out_degrees().float().clamp(min=1)
        g.srcdata["deg"], g.dstdata["deg"] = deg, deg[:n_dst]
    conv = sampled.GATConv(24, 16, 20, **kw).to(cuda).eval()
    x = torch.randn(n_src, 24, device=cuda)
    fe = torch.randn(e, 16, device=cuda)
    gy = torch.randn(n_dst, 3, 20, device=cuda)
    res = {}
    for fold in (False, True):
        monkeypatch.setattr(sampled, "fold_projections", fold)
        xi, fi = x.clone().requires_grad_(True), fe.clone().requires_grad_(True)
        conv.zero_grad()
        y = conv(g, xi, fi)
        y.backward(gy)
        res[fold] = [y.detach(), xi.grad, fi.grad] + [p.grad.clone() for p in conv.parameters()]
    assert rel_err(res[True][0], res[False][0]) <= FWD_TOL
    for a, b in zip(res[True][1:], res[False][1:]):
        assert a.shape == b.shape and rel_err(a, b) <= 1e-4


def test_host_feed_pipeline(cuda):
    """bot_b200.HostFeed: steps prefetched one ahead through two device buffer sets give the values and
    gradients of the same steps fed serially."""
    import bot_b200
    from bot_b200.ogbn_proteins import GATConv

    torch.manual_seed(0)
    n, e, steps = 300, 8000, 5
    src = torch.randint(0, n, (e,), device=cuda)
    dst = torch.randint(0, n, (e,), device=cuda)
    g = bot_b200.Graph(src, dst, n)
    conv = GATConv(32, 16, 8, n_heads=6).to(cuda).eval()
    xs = [torch.randn(n, 32).pin_memory() for _ in range(steps)]
    fes = [torch.randn(e, 16).pin_memory() for _ in range(steps)]

    def run(x, fe):
        y = conv(g, x, fe)
        y.square().sum().backward()
        return y.detach().clone()

    want = []
    for x, fe in zip(xs, fes):
        xd, fd = x.to(cuda).requires_grad_(True), fe.to(cuda).requires_grad_(True)
        want.append((run(xd, fd), xd.grad.clone(), fd.grad.clone()))

    feed = bot_b200.HostFeed(cuda, depth=2)
    feed.submit(xs[0], fes[0])
    with pytest.raises(RuntimeError):
        feed.submit(xs[0], fes[0]), feed.submit(xs[0], fes[0])
    feed = bot_b200.HostFeed(cuda, depth=2)
    feed.submit(xs[0], fes[0])
    for i in range(steps):
        if i + 1 < steps:
            feed.submit(xs[i + 1], fes[i + 1])
        x, fe = feed.take(requires_grad=(0, 1))
        y = run(x, fe)
        gx, gfe = x.tensor.grad, fe.tensor.grad
        assert torch.equal(y, want[i][0]) and torch.equal(gx, want[i][1]) and torch.equal(gfe, want[i][2])
    with pytest.raises(RuntimeError):
        feed.take()


@pytest.mark.parametrize("H", [1, 3, 6])
def test_fused_philox_attention_dropout(cuda, H):
    """In-kernel attention dropout (Philox keyed on seed, edge id, head): forward and both backward passes agree with
    the oracle run on the multiplier the same generator yields on the host."""
    from util import philox_attn_mul

    p, seed = 0.3, 0x1234_5678_9ABC_DEF1
    c = make_case(300, 300, 9000, H, 16, ee=True, keep_p=0.1, seed=40 + H)
    # the stream is keyed on the graph's canonical edge number
    c["attn_mul"] = philox_attn_mul(seed, 9000, H, p, eids=graph_ref.canonical_edge_ids(c["src"].numpy(), c["dst"].numpy()))
    frac = float((c["attn_mul"] == 0).float().mean())
    assert abs(frac - p) < 0.03
    ref_out, ref_g = oracle_run(c)
    c_gpu = dict(c, attn_mul=None)
    out, g, _ = engine_run(c_gpu, cuda, attn_p=p, seed=seed)
    assert rel_err(out, ref_out) <= FWD_TOL
    for k in ("ft", "el", "er", "ee"):
        assert rel_err(g[k], ref_g[k]) <= 1e-4, k


@pytest.mark.parametrize("parts", [1, 2, 4, 8])
def test_partition_abi_bit_exact(cuda, parts):
    """botgat_partition_1d / botgat_partition_extract against the partition oracle (bit-exact)."""
    import bot_b200
    from bot_b200.partition import partition_bounds, partition_bounds_device, partition_extract_device

    n, e = 700, 9000
    src, dst = graph_ref.synthetic_coo(n, e, 12, power_law=0.7)
    f = graph_ref.build_formats(src, dst, n, n)
    ref_b = graph_ref.partition_bounds(f["in_indptr"], parts)
    # ABI-level check in the library's own edge numbering: build from the COO as given
    g = bot_b200.Graph(torch.from_numpy(src).to(cuda), torch.from_numpy(dst).to(cuda), n, canonical=False)
    assert np.array_equal(partition_bounds_device(g, parts).numpy(), ref_b)
    assert np.array_equal(partition_bounds(torch.from_numpy(dst).to(cuda), n, parts).cpu().numpy(), ref_b)
    for r in range(parts):
        loc = graph_ref.partition_local(src, dst, n, ref_b, r)
        eid, s, ld = partition_extract_device(g, int(ref_b[r]), int(ref_b[r + 1]))
        assert np.array_equal(eid.cpu().numpy(), loc["edge_gid"])
        assert np.array_equal(s.cpu().numpy(), src[loc["edge_gid"]])
        assert np.array_equal(ld.cpu().numpy(), loc["ldst"])


def test_rows_gather_scatter_abi(cuda):
    import ctypes as C

    from bot_b200 import _lib
    from bot_b200.graph import _stream

    lib = _lib.load()
    t = torch.randn(50, 12, device=cuda)
    rows = torch.tensor([3, 7, 49, 0], device=cuda)
    out = torch.empty(4, 10, device=cuda)
    _lib.check(lib.botgat_rows_gather(_lib.ptr(t), 12, 10, _lib.ptr(rows), 4, _lib.ptr(out), _stream()), "rows_gather")
    assert torch.equal(out, t[rows, :10])
    before = t.clone()
    _lib.check(lib.botgat_rows_scatter_add(_lib.ptr(t), 12, 10, _lib.ptr(rows), 4, _lib.ptr(out), _stream()), "rows_scatter_add")
    exp = before.clone()
    exp[rows, :10] += out
    assert torch.equal(t, exp)


def test_partitioned_layer_on_gpu(cuda):
    """PartitionedGraph.gat on the GPU (NCCL group of one rank): the hook path that starts the collectives around
    the kernels gives the single-call result and gradients of the right shapes."""
    import socket

    import torch.distributed as dist

    import bot_b200
    from bot_b200.functional import gat_fused
    from bot_b200.partition import PartitionedGraph

    if dist.is_initialized():
        pytest.skip("a process group is already initialised")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=0, world_size=1,
                            device_id=torch.device(cuda))
    try:
        c = make_case(300, 300, 9000, 3, 32, ee=True, keep_p=0.2, seed=31)
        src, dst = c["src"].to(cuda), c["dst"].to(cuda)
        pg = PartitionedGraph(src, dst, 300)
        g = bot_b200.Graph(src, dst, 300)
        args = [c[k].to(cuda) for k in ("ft", "el", "er", "ee")]
        keep, gout = c["keep"].to(cuda), c["gout"].to(cuda)
        a = [t.clone().requires_grad_(True) for t in args]
        b = [t.clone().requires_grad_(True) for t in args]
        out_a = pg.gat(a[0], a[1], a[2], pg.local_edges(a[3]), pg.local_edges(keep))
        out_b = gat_fused(g, b[0], b[1], b[2], b[3], keep)
        out_a.backward(gout)
        out_b.backward(gout)
        assert rel_err(out_a, out_b) <= FWD_TOL
        for x, y in zip(a, b):
            assert x.grad.shape == y.grad.shape and rel_err(x.grad, y.grad) <= 1e-4
    finally:
        dist.destroy_process_group()


def test_full_size_properties(cuda):
    """BASELINE.json's north-star size (proteins shape: N = 132,534, E = 39,561,252, H = 6, D = 80, edge logits,
    edge_drop 0.1) is beyond the oracle; size-independent properties instead:
      1. ft = 1  ->  every row with a kept in-edge sums its attention to 1
      2. the layer is linear in ft for fixed logits
      3. adjoint identity <gout, out(ft)> == <grad_ft, ft>  (backward gather against forward gather)
      4. dropped edges receive exactly zero grad_ee; reruns are bit-identical"""
    import bot_b200
    from bot_b200.functional import edge_drop_keep, gat_fused

    N, E, H, D = 132534, 39561252, 6, 80
    g = torch.Generator(device=cuda).manual_seed(0)
    src = torch.randint(0, N, (E,), device=cuda, generator=g)
    dst = torch.randint(0, N, (E,), device=cuda, generator=g)
    graph = bot_b200.Graph(src, dst, N)
    el = torch.randn(N, H, device=cuda, generator=g).requires_grad_(True)
    er = torch.randn(N, H, device=cuda, generator=g).requires_grad_(True)
    ee = torch.randn(E, 8, device=cuda, generator=g).requires_grad_(True)
    keep = edge_drop_keep(E, int(E * 0.1), 7, cuda)
    assert int(keep.sum()) == E - int(E * 0.1)

    def layer(ft):
        return gat_fused(graph, ft, el, er, ee, keep)

    # 1. rows sum to one
    kept_in = torch.zeros(N, device=cuda).index_add_(0, dst, keep.float())
    ones = layer(torch.ones(N, H, D, device=cuda)).detach()
    has = kept_in > 0
    assert float((ones[has] - 1.0).abs().max()) <= 2e-5
    assert float(ones[~has].abs().max() if (~has).any() else 0.0) == 0.0
    del ones
    # 2. linearity
    f1 = torch.randn(N, H, D, device=cuda, generator=g)
    f2 = torch.randn(N, H, D, device=cuda, generator=g)
    o1, o2 = layer(f1).detach(), layer(f2).detach()
    o12 = layer(0.5 * f1 - 2.0 * f2).detach()
    assert rel_err(o12, 0.5 * o1 - 2.0 * o2) <= FWD_TOL
    del o2, o12, f2
    # 3. adjoint identity, 4. dropped edges, determinism
    ft = f1.requires_grad_(True)
    gout = torch.randn(N, H, D, device=cuda, generator=g)
    out = layer(ft)
    out.backward(gout)
    lhs = float((gout.double() * out.detach().double()).sum())
    rhs = float((ft.grad.double() * ft.detach().double()).sum())
    assert abs(lhs - rhs) <= 1e-5 * max(abs(lhs), abs(rhs), 1.0)
    assert float(ee.grad[keep == 0].abs().max()) == 0.0 and float(ee.grad[:, H:].abs().max()) == 0.0
    assert torch.isfinite(ee.grad).all() and torch.isfinite(el.grad).all() and torch.isfinite(er.grad).all()
    first = (out.detach().clone(), ft.grad.clone(), el.grad.clone(), er.grad.clone(), ee.grad.clone())
    for t in (ft, el, er, ee):
        t.grad = None
    out2 = layer(ft)
    out2.backward(gout)
    again = (out2.detach(), ft.grad, el.grad, er.grad, ee.grad)
    assert all(torch.equal(a, b) for a, b in zip(first, again))


@pytest.mark.parametrize("name", ["proteins_like_edge_drop", "arxiv_like_H3_D250_symm", "cora_like_H8_D8"])
def test_head_range_launches(cuda, name):
    """Forward and backward src phase launched one head range at a time (botgat_*_args.h_begin / h_count, the hook
    protocol of the head-pipelined halo exchange) give bit-identical results to the single launch."""
    import bot_b200
    from bot_b200.functional import Hooks, gat_fused

    n_src, n_dst, e, H, D, kw = CASES[name]
    c = make_case(n_src, n_dst, e, H, D, seed=3, **kw)
    g = bot_b200.Graph(c["src"].to(cuda), c["dst"].to(cuda), n_src, n_dst)
    names = ["ft", "el"] + (["er"] if c.get("er") is not None else []) + (["ee"] if c.get("ee") is not None else [])
    keep = c["keep"].to(cuda) if c.get("keep") is not None else None
    cs = c["src_scale"].to(cuda) if c.get("src_scale") is not None else None
    ds = c["dst_scale"].to(cuda) if c.get("dst_scale") is not None else None
    seen = []
    chunks = [(0, 1), (1, H - 1)] if H > 2 else [(h, 1) for h in range(H)]
    hooks = Hooks(head_chunks=chunks, pre_head=lambda i: seen.append(("f", i)),
                  post_src_head=lambda i, gft, gel: seen.append(("b", i, tuple(gft.shape))))
    res = []
    for hk in (None, hooks):
        t = {k: c[k].to(cuda).clone().requires_grad_(True) for k in names}
        am = c["attn_mul"].to(cuda) if c.get("attn_mul") is not None else None
        out = gat_fused(g, t["ft"], t["el"], t.get("er"), t.get("ee"), keep, am, cs, ds, 0.2, 0.0, 0, hooks=hk)
        out.backward(c["gout"].to(cuda))
        res.append([out.detach()] + [t[k].grad for k in names])
    assert all(torch.equal(a, b) for a, b in zip(*res))
    assert seen == [("f", i) for i in range(len(chunks))] + [("b", i, (n_src, H, D)) for i in range(len(chunks))]


def test_out_of_range_node_id_is_a_clean_error(cuda):
    """An id outside [0, n) must come back as an error BEFORE it is used as an index (no out-of-bounds histogram
    write, no sticky device fault): the device keeps working afterwards."""
    import bot_b200
    from bot_b200 import sampling

    src = torch.tensor([0, 1, 2, 50_000_000, 3], device=cuda)
    dst = torch.tensor([1, 2, 3, 0, -7], device=cuda)
    with pytest.raises(RuntimeError, match="out of range"):
        bot_b200.Graph(src, dst, 10).create_formats_()
    torch.cuda.synchronize()                                        # would raise on a sticky illegal-address fault
    c = make_case(50, 50, 400, 2, 8, seed=3)
    check_case(c, cuda)
    g = bot_b200.Graph(c["src"].to(cuda), c["dst"].to(cuda), 50)
    with pytest.raises(RuntimeError, match="out of range"):
        sampling.sample_neighbors(g, torch.tensor([1, 2, 10**9], device=cuda), 4, 0)
    with pytest.raises(RuntimeError, match="out of range"):
        sampling.to_block(g, torch.tensor([1, 99], device=cuda), torch.tensor([1, 2], device=cuda),
                          torch.tensor([0, 1], device=cuda), torch.tensor([0, 1], device=cuda))
    torch.cuda.synchronize()
    check_case(c, cuda)


def test_block_without_destination_rows_has_zero_gradients(cuda):
    """A rank whose row range is empty still owns halo sources: its gradients must be written (zeros), they are
    reduce-scattered into the other ranks' gradients (bot_b200/partition.py)."""
    import bot_b200
    from bot_b200.functional import gat_fused

    g = bot_b200.create_block((torch.empty(0, dtype=torch.int64), torch.empty(0, dtype=torch.int64)), 40, 0, device=cuda)
    ft = torch.randn(40, 2, 8, device=cuda, requires_grad=True)
    el = torch.randn(40, 2, device=cuda, requires_grad=True)
    er = torch.randn(0, 2, device=cuda, requires_grad=True)
    out = gat_fused(g, ft, el, er)
    assert out.shape == (0, 2, 8)
    # poison the caching allocator so that an unwritten gradient buffer would not read as zeros
    junk = torch.full((40, 2, 8), float("nan"), device=cuda)
    del junk
    out.backward(torch.empty(0, 2, 8, device=cuda))
    assert float(ft.grad.abs().max()) == 0.0 and float(el.grad.abs().max()) == 0.0


@pytest.mark.parametrize("lowdeg", ["0", "1000000"])
def test_zero_negative_slope(cuda, monkeypatch, lowdeg):
    """negative_slope = 0 (a valid GATConv argument): the -inf logit of a dropped edge / a lane past the row end must
    not become NaN through -inf * 0."""
    monkeypatch.setenv("BOTGAT_LOWDEG", lowdeg)
    c = make_case(300, 300, 5000, 3, 24, ee=True, keep_p=0.3, seed=21)
    ref_out, ref_g = oracle_run(c, slope=0.0)
    out, g, _ = engine_run(c, cuda, slope=0.0)
    assert torch.isfinite(out).all()
    assert rel_err(out, ref_out) <= FWD_TOL
    for k in ("ft", "el", "er", "ee"):
        assert rel_err(g[k], ref_g[k]) <= 1e-4, k


@pytest.mark.parametrize("tiles", [None, "3,2", "1,4"])
def test_canonical_edge_operands(cuda, monkeypatch, tiles):
    """Operands given in the graph's canonical order (no permutation pass) give bit-identical results to the same
    operands given in edge-id order; the cache-blocked out-CSR traversal (forced here on a small graph) changes the
    order edges are visited in, never a value."""
    import bot_b200
    from bot_b200.functional import gat_fused

    if tiles:
        monkeypatch.setenv("BOTGAT_TILES", tiles)
    c = make_case(500, 500, 40000, 6, 16, ee=True, keep_p=0.2, attn_p=0.3, seed=77)
    ref_out, ref_g = oracle_run(c)
    g = bot_b200.Graph(c["src"].to(cuda), c["dst"].to(cuda), 500)
    perm = g.edge_perm()
    assert perm is not None and g._info.in_eid_identity == 1
    if tiles:
        assert (g._info.tiles_src, g._info.tiles_dst) == tuple(int(x) for x in tiles.split(","))

    def run(order):
        ft, el, er = (c[k].to(cuda).clone().requires_grad_(True) for k in ("ft", "el", "er"))
        ee, keep, mul = c["ee"].to(cuda), c["keep"].to(cuda), c["attn_mul"].to(cuda)
        if order == "canonical":
            ee, keep, mul = ee[perm], keep[perm], mul[perm]
        ee = ee.clone().requires_grad_(True)
        out = gat_fused(g, ft, el, er, ee, keep, mul, edge_order=order)
        out.backward(c["gout"].to(cuda))
        return out.detach(), ft.grad, el.grad, er.grad, ee.grad

    a, b = run("eid"), run("canonical")
    assert rel_err(a[0], ref_out) <= FWD_TOL
    for x, k in zip(a[1:], ("ft", "el", "er", "ee")):
        assert rel_err(x, ref_g[k]) <= 1e-4, k
    for x, y in zip(a[:4], b[:4]):
        assert torch.equal(x, y)
    assert torch.equal(a[4][perm], b[4])


def test_edge_frame_canonical_view(cuda):
    """graph.edata speaks edge ids; .canonical(key) is the same rows in canonical order, permuted once per assignment."""
    import bot_b200

    src, dst = graph_ref.synthetic_coo(50, 400, 5)
    g = bot_b200.Graph(torch.from_numpy(src).to(cuda), torch.from_numpy(dst).to(cuda), 50)
    x = torch.randn(400, 3, device=cuda)
    g.edata["feat"] = x
    c1 = g.edata.canonical("feat")
    assert g.edata["feat"] is x and torch.equal(c1, x[g.edge_perm()]) and g.edata.canonical("feat") is c1
    with g.local_scope():
        g.edata["feat"] = x * 2
        assert torch.equal(g.edata.canonical("feat"), (x * 2)[g.edge_perm()])
    assert torch.equal(g.edata.canonical("feat"), x[g.edge_perm()])
    # a COO already sorted by (dst, src) needs no permutation at all
    order = np.lexsort((src, dst))
    g2 = bot_b200.Graph(torch.from_numpy(src[order]).to(cuda), torch.from_numpy(dst[order]).to(cuda), 50)
    assert g2.edge_perm() is None and g2.canonical_edge_ids() is None


@pytest.mark.parametrize("kind", ["symm_attn_r", "plain", "block", "train_drops"])
def test_v1_folded_logits_match_unfolded(cuda, kind):
    """no_sampling.GATConv with el / er folded into the fc / res_fc GEMMs (SURVEY 8f rank 2, models.py:517-521) against
    the op-by-op sequence: outputs and every parameter gradient."""
    import bot_b200
    from bot_b200.no_sampling import GATConv

    torch.manual_seed(3)
    n_src, n_dst = (300, 80) if kind == "block" else (300, 300)
    src = torch.randint(0, n_src, (6000,), device=cuda)
    dst = torch.randint(0, n_dst, (6000,), device=cuda)
    if kind != "block":
        src, dst = torch.cat([src, torch.arange(300, device=cuda)]), torch.cat([dst, torch.arange(300, device=cuda)])
    g = bot_b200.Graph(src, dst, n_src, n_dst, is_block=kind == "block")
    conv = GATConv(40, 16, num_heads=3, use_symmetric_norm=kind == "symm_attn_r", non_interactive_attn=kind != "plain",
                   edge_drop=0.3 if kind == "train_drops" else 0.0, attn_drop=0.2 if kind == "train_drops" else 0.0).to(cuda)
    conv.train(kind == "train_drops")
    x = torch.randn(n_src, 40, device=cuda)
    res = []
    for fold in (True, False):
        conv.fold_logits = fold
        conv.zero_grad()
        xi = x.clone().requires_grad_(True)
        torch.manual_seed(11)          # the same draws in both passes
        y = conv(g, xi)
        y.square().sum().backward()
        res.append((y.detach(), xi.grad, {k: p.grad.clone() for k, p in conv.named_parameters()}))
    (y1, gx1, gp1), (y2, gx2, gp2) = res
    assert rel_err(y1, y2) <= FWD_TOL * 2 and rel_err(gx1, gx2) <= 1e-4
    for k in gp1:
        assert rel_err(gp1[k], gp2[k]) <= 1e-4, k


@pytest.mark.parametrize("tma", ["0", "1"])
@pytest.mark.parametrize("H,D,kw", [
    (6, 80, dict(ee=True, keep_p=0.1)),              # proteins: G = 4, five slots, no idle lanes
    (4, 64, dict(er=False, symm=True, attn_p=0.1)),  # Reddit
    (4, 120, dict(keep_p=0.1)),                      # products: G = 8, ragged last slot
    (2, 16, dict()), (3, 32, dict(ee=True)), (2, 48, dict()), (1, 96, dict(symm=True)), (2, 128, dict(ee=True)),
    (3, 40, dict(er=False)), (1, 160, dict(ee=True, keep_p=0.3)),
    (2, 72, dict(ee=True)),                          # a width the TMA kernel is not instantiated for: LDG either way
    (12, 32, dict(ee=True)), (12, 120, dict(keep_p=0.2)),   # H > 8: edge records wider than one 32-byte sector
    (5, 40, dict(ee=True, keep_p=0.1)), (8, 16, dict(er=False, attn_p=0.2)), (1, 128, dict(er=False, symm=True)),
    (3, 160, dict(attn_p=0.1)),
])
def test_src_pass_tma_and_ldg(cuda, monkeypatch, tma, H, D, kw):
    """The warp-per-row backward src pass in both data-movement variants (BOTGAT_BWD_TMA unset or 1: the TMA gather4
    ring; 0: LDG into registers) on every head width the TMA kernel is instantiated for, and D = 72, which it is not (LDG
    either way): rows of 0, 1, < 32, exactly 32/64 and several hundred out-edges.  The trace shows which one ran."""
    monkeypatch.setenv("BOTGAT_LOWDEG", "0")
    monkeypatch.setenv("BOTGAT_BWD_TMA", tma)
    n = 260
    c = make_case(n, n, 12000, H, D, seed=7 * D + H, power_law=0.0, **kw)
    # re-draw the sources so that out-degrees are ragged: a few hot rows, rows of exactly 32 and 64, empty rows
    rng = np.random.default_rng(D)
    deg = np.concatenate([[0, 1, 31, 32, 33, 64, 65, 96, 700, 1500], rng.integers(0, 90, size=n - 10)])
    src = np.repeat(np.arange(n), deg)[:12000]
    src = np.concatenate([src, rng.integers(0, n, size=12000 - src.shape[0])])
    c["src"] = torch.from_numpy(rng.permutation(src).astype(np.int64))
    if c["src_scale"] is not None:
        f = graph_ref.build_formats(c["src"].numpy(), c["dst"].numpy(), n, n)
        c["src_scale"] = torch.from_numpy(graph_ref.deg_scale(f["out_deg"], -0.5))
    names = _gather_kernels(lambda: check_case(c, cuda))
    src = {n.split("<")[0] for n in names if "bwd" in n}
    want = "botgat::gat_bwd_src_tma_kernel" if tma == "1" and D != 72 else "botgat::gat_bwd_src_kernel"
    assert src == {want}, (tma, D, names)


@pytest.mark.parametrize("tma", ["1", "2"])
@pytest.mark.parametrize("H", [2, 6])
def test_src_pass_tma_philox(cuda, monkeypatch, H, tma):
    """In-kernel attention dropout through the TMA src pass (warp-per-row forced; 2 = the persistent form)."""
    from util import philox_attn_mul

    monkeypatch.setenv("BOTGAT_LOWDEG", "0")
    monkeypatch.setenv("BOTGAT_BWD_TMA", tma)
    p, seed = 0.25, 0x0BAD_5EED_1234_5678
    c = make_case(200, 200, 20000, H, 80, ee=True, keep_p=0.1, seed=90 + H)
    c["attn_mul"] = philox_attn_mul(seed, 20000, H, p, eids=graph_ref.canonical_edge_ids(c["src"].numpy(), c["dst"].numpy()))
    ref_out, ref_g = oracle_run(c)
    out, g, _ = engine_run(dict(c, attn_mul=None), cuda, attn_p=p, seed=seed)
    assert rel_err(out, ref_out) <= FWD_TOL
    for k in ("ft", "el", "er", "ee"):
        assert rel_err(g[k], ref_g[k]) <= 1e-4, k


@pytest.mark.parametrize("family", ["warp", "group", "split", "rowwise"])
@pytest.mark.parametrize("model_kind", ["proteins", "products_res", "products_nores", "v1_bn", "v1_bias", "v1_bn_linear"])
def test_fused_layer_tail_inference(cuda, monkeypatch, family, model_kind):
    """Inference with the layer tail (residual adds, eval-mode BatchNorm / bias, ReLU) fused into the forward kernel's
    epilogue — in the warp-per-row kernel, the group-per-row kernel and the split-row combine — against the same model run
    op by op (gradients enabled selects the unfused path)."""
    import torch.nn.functional as F

    import bot_b200
    from bot_b200 import functional
    from bot_b200.no_sampling import GAT as V1GAT
    from bot_b200.ogbn_products import GAT as ProductsGAT
    from bot_b200.ogbn_proteins import GAT as ProteinsGAT

    monkeypatch.setenv("BOTGAT_LOWDEG", "1000000" if family == "group" else "0")
    monkeypatch.setenv("BOTGAT_ROWWISE", "1" if family == "rowwise" else "0")
    if family == "split":
        monkeypatch.setenv("BOTGAT_SEG", "32")
    torch.manual_seed(5)
    n, e = 500, 30000
    c = make_case(n, n, e, 1, 8, power_law=0.8 if family == "split" else 0.0, self_loops=True, seed=77)
    g = bot_b200.Graph(c["src"].to(cuda), c["dst"].to(cuda), n)
    E = g.number_of_edges()
    if model_kind == "proteins":
        model = ProteinsGAT(8, 8, 5, 3, 3, 16, 16, F.relu, 0.1, 0.1, 0.0, 0.1)
        g.srcdata["feat"] = torch.randn(n, 8, device=cuda)
        g.edata["feat"] = torch.rand(E, 8, device=cuda)
        call = lambda m: m(g)
    elif model_kind.startswith("products"):
        model = ProductsGAT(12, 0, 5, 3, 2, 20, 0, F.relu, 0.1, 0.1, 0.0, 0.1, residual=model_kind == "products_res")
        g.srcdata["feat"] = torch.randn(n, 12, device=cuda)
        call = lambda m: m(g)
    else:
        model = V1GAT(12, 0, 5, 16, 3, 2, F.relu, norm="none" if model_kind == "v1_bias" else "batch", dropout=0.1,
                      use_symmetric_norm=True, residual=True, linear=model_kind == "v1_bn_linear",
                      non_interactive_attn=model_kind == "v1_bn_linear")
        x = torch.randn(n, 12, device=cuda)
        call = lambda m: m(g, x)
    model = model.to(cuda)
    for m in model.modules():   # non-trivial running statistics / biases
        if isinstance(m, torch.nn.BatchNorm1d):
            m.running_mean.normal_(); m.running_var.uniform_(0.5, 2.0); m.weight.data.normal_(1.0, 0.2); m.bias.data.normal_()
    for name, p_ in model.named_parameters():
        if "biases" in name:
            p_.data.normal_()
    model.eval()
    from bot_b200 import sampled
    calls = []
    real = functional.gat_conv_inference

    def counted(*a, **k):
        calls.append(1)
        return real(*a, **k)

    real2 = functional.gat_fused_inference

    def counted2(*a, **k):
        calls.append(1)
        return real2(*a, **k)

    monkeypatch.setattr(functional, "gat_conv_inference", counted)
    monkeypatch.setattr(functional, "gat_fused_inference", counted2)
    monkeypatch.setattr(sampled, "gat_conv_inference", counted)
    with torch.no_grad():
        y_fused = call(model)
    n_fused = len(calls)
    y_plain = call(model).detach()    # gradients enabled: the op-by-op path
    assert n_fused >= 2 and len(calls) == n_fused, "the fused tail must run in inference and only there"
    assert y_fused.shape == y_plain.shape
    assert rel_err(y_fused, y_plain) <= 2e-6


# ---------------------------------------------------------------------------
# all-heads-per-row kernels (gat_rowwise.cu): selected automatically only for tables far beyond the L2, forced here
# ---------------------------------------------------------------------------
ROWWISE_CASES = dict(CASES)
ROWWISE_CASES.update({
    "rw_H2_D48": (300, 300, 9000, 2, 48, dict(ee=True)),                      # 16 lanes per head, one slot
    "rw_H1_D512": (100, 100, 3000, 1, 512, dict(keep_p=0.2)),                 # 32 lanes per head, four slots
    "rw_H3_D32_symm": (400, 400, 12000, 3, 32, dict(er=False, symm=True, attn_p=0.2)),   # an idle head group
    "rw_H5_D20": (200, 200, 8000, 5, 20, dict(ee=True, keep_p=0.1)),          # 4 lanes per head, three idle groups
    "rw_H8_D128": (150, 150, 5000, 8, 128, dict(ee=True)),                    # 4 lanes per head, eight slots
    "rw_H4_D256": (120, 120, 4000, 4, 256, dict()),                           # 8 lanes per head, eight slots
    "rw_long_rows": (64, 64, 40000, 4, 120, dict(ee=True, keep_p=0.1)),       # ~20 chunks per row: the online rescale
})


@pytest.mark.parametrize("bulk", ["1", "0"])
@pytest.mark.parametrize("name", list(ROWWISE_CASES))
def test_rowwise_kernels(cuda, monkeypatch, name, bulk):
    """One warp per row for all heads (forward and backward src pass; the latter with its rows staged by bulk copies
    into a shared-memory ring, or through the register ring) against the fp64 oracle on every parity case; shapes the
    family does not cover (vector width < 4) take the head-major kernels.  The trace shows which family ran."""
    monkeypatch.setenv("BOTGAT_ROWWISE", "1")
    monkeypatch.setenv("BOTGAT_RW_BULK", bulk)
    n_src, n_dst, e, H, D, kw = ROWWISE_CASES[name]
    c = make_case(n_src, n_dst, e, H, D, seed=zlib.crc32(name.encode()) % 1000 + 2, **kw)
    names = _gather_kernels(lambda: check_case(c, cuda))
    families = {n.split("<")[0] for n in names}
    if D % 4 == 0 and H <= 8 and D // 4 <= 8 * (32 // (1 << (H - 1).bit_length())):
        assert families == {"botgat::gat_fwd_rowwise_kernel",
                            "botgat::gat_bwd_src_rowbulk_kernel" if bulk == "1" else "botgat::gat_bwd_src_rowwise_kernel"}, names
    else:
        assert not any("rowwise" in f or "rowbulk" in f for f in families), names
    o1, g1, _ = engine_run(c, cuda)
    o2, g2, _ = engine_run(c, cuda)
    assert torch.equal(o1, o2) and all(g1[k] is None or torch.equal(g1[k], g2[k]) for k in g1)


def test_rowwise_is_selected(cuda, monkeypatch):
    """The family really runs when forced (launch names differ only in the profiler, so compare against the head-major
    result: close, but not bit-identical — the summation order differs) and is not selected for small tables."""
    c = make_case(500, 500, 20000, 4, 120, keep_p=0.1, seed=5)
    monkeypatch.setenv("BOTGAT_ROWWISE", "0")
    o0, g0, _ = engine_run(c, cuda)
    monkeypatch.delenv("BOTGAT_ROWWISE")
    oa, ga, _ = engine_run(c, cuda)          # auto: a 240 KB slab is L2-resident -> head-major
    assert torch.equal(o0, oa) and torch.equal(g0["ft"], ga["ft"])
    monkeypatch.setenv("BOTGAT_ROWWISE", "1")
    o1, g1, _ = engine_run(c, cuda)
    assert rel_err(o1, o0) <= 1e-6 and rel_err(g1["ft"], g0["ft"]) <= 1e-6
    assert not torch.equal(g1["ft"], g0["ft"])
    monkeypatch.setenv("BOTGAT_ROWWISE_MB", "0")   # auto with a zero threshold: selected by table size
    monkeypatch.delenv("BOTGAT_ROWWISE")
    o2, g2, _ = engine_run(c, cuda)
    assert torch.equal(o2, o1) and torch.equal(g2["ft"], g1["ft"])


@pytest.mark.parametrize("bulk", ["1", "0"])
@pytest.mark.parametrize("seg", ["32", "100"])
def test_rowwise_row_splitting(cuda, monkeypatch, seg, bulk):
    """Heavy rows split into segments through the all-heads-per-row kernels (same scratch slots and combine kernels)."""
    monkeypatch.setenv("BOTGAT_SEG", seg)
    monkeypatch.setenv("BOTGAT_ROWWISE", "1")
    monkeypatch.setenv("BOTGAT_RW_BULK", bulk)
    c = make_case(600, 600, 60000, 3, 40, ee=True, keep_p=0.1, power_law=1.2, symm=True, seed=31)
    check_case(c, cuda)
    o1, g1, g = engine_run(c, cuda)
    o2, g2, _ = engine_run(c, cuda)
    assert g._info.n_slots_in > 0
    assert torch.equal(o1, o2) and all(torch.equal(g1[k], g2[k]) for k in g1)


@pytest.mark.parametrize("bulk", ["1", "0"])
@pytest.mark.parametrize("H", [1, 4, 6])
def test_rowwise_philox(cuda, monkeypatch, H, bulk):
    """In-kernel attention dropout through the all-heads-per-row kernels."""
    from util import philox_attn_mul

    monkeypatch.setenv("BOTGAT_ROWWISE", "1")
    monkeypatch.setenv("BOTGAT_RW_BULK", bulk)
    p, seed = 0.25, 0x0BAD_5EED_1234_5678
    c = make_case(200, 200, 20000, H, 80, ee=True, keep_p=0.1, seed=190 + H)
    c["attn_mul"] = philox_attn_mul(seed, 20000, H, p, eids=graph_ref.canonical_edge_ids(c["src"].numpy(), c["dst"].numpy()))
    ref_out, ref_g = oracle_run(c)
    out, g, _ = engine_run(dict(c, attn_mul=None), cuda, attn_p=p, seed=seed)
    assert rel_err(out, ref_out) <= FWD_TOL
    for k in ("ft", "el", "er", "ee"):
        assert rel_err(g[k], ref_g[k]) <= 1e-4, k


@pytest.mark.parametrize("name", ["proteins_like_edge_drop", "products_like_H4_D120", "reddit_like_H4_D64_symm",
                                  "H12_in_halves"])
def test_rowwise_head_range_launches(cuda, monkeypatch, name):
    """Head-range launches (the head-pipelined halo exchange's protocol) through the all-heads-per-row kernels: a range
    of heads is a narrower row; results are bit-identical to the single launch when the lane geometry is the same and
    within rounding otherwise (fewer heads per launch -> more lanes per head -> another summation order).
    H12_in_halves: one launch of 12 heads is not covered by the all-heads-per-row kernels, so the node phase writes the
    per-destination records head-major, and the two 6-head src passes run the row-wise kernel on them."""
    import bot_b200
    from torch.profiler import ProfilerActivity, profile

    from bot_b200.functional import Hooks, gat_fused
    from util import GRAD_TOL

    monkeypatch.setenv("BOTGAT_ROWWISE", "1")
    if name == "H12_in_halves":
        n_src, n_dst, e, H, D, kw = 500, 500, 20000, 12, 32, dict(ee=True, keep_p=0.1)
        chunks = [(0, 6), (6, 6)]
    else:
        n_src, n_dst, e, H, D, kw = CASES[name]
        chunks = [(0, 1), (1, H - 1)]
    c = make_case(n_src, n_dst, e, H, D, seed=3, **kw)
    g = bot_b200.Graph(c["src"].to(cuda), c["dst"].to(cuda), n_src, n_dst)
    names = ["ft", "el"] + (["er"] if c.get("er") is not None else []) + (["ee"] if c.get("ee") is not None else [])
    keep = c["keep"].to(cuda) if c.get("keep") is not None else None
    cs = c["src_scale"].to(cuda) if c.get("src_scale") is not None else None
    ds = c["dst_scale"].to(cuda) if c.get("dst_scale") is not None else None
    hooks = Hooks(head_chunks=chunks, pre_head=lambda i: None, post_src_head=lambda i, gft, gel: None)
    res = []
    for hk in (None, hooks):
        t = {k: c[k].to(cuda).clone().requires_grad_(True) for k in names}
        am = c["attn_mul"].to(cuda) if c.get("attn_mul") is not None else None
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            out = gat_fused(g, t["ft"], t["el"], t.get("er"), t.get("ee"), keep, am, cs, ds, 0.2, 0.0, 0, hooks=hk)
            out.backward(c["gout"].to(cuda))
            torch.cuda.synchronize()
        res.append([out.detach()] + [t[k].grad for k in names])
    for a, b in zip(*res):
        assert rel_err(b, a) <= 2e-6
    # the last (chunked) run's src passes: all heads per row, one launch per chunk
    assert sum("gat_bwd_src_row" in e.name for e in prof.events()) == len(chunks)
    if name == "H12_in_halves":
        ref_out, ref_g = oracle_run(c)
        assert rel_err(res[1][0], ref_out) <= FWD_TOL
        for k, got in zip(names, res[1][1:]):
            assert rel_err(got, ref_g[k]) <= GRAD_TOL, k
