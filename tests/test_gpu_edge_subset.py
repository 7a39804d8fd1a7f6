"""The per-step kept adjacency (``botgat_edge_subset``): with an edge-drop ``keep`` mask the staging pass writes a CSR of the
kept edges in both orders and the gather kernels walk it instead of the graph's, so a dropped edge costs them nothing.
Checked here: the subset itself against a torch restatement, bit-identity with the same step on the kept subgraph in
every kernel family, the fp64 oracle on the cases the compaction changes, and that a call without ``keep`` launches
nothing new."""
import zlib

import numpy as np
import pytest
import torch

from oracle import graph_ref
from util import FWD_TOL, check_case, engine_run, make_case, oracle_run, rel_err

pytestmark = pytest.mark.gpu


def _segments(indptr, L):
    """Row segments of a CSR whose longest row exceeds L (csrc/segments.cu), else None."""
    deg = indptr[1:] - indptr[:-1]
    if deg.numel() == 0 or int(deg.max()) <= L:
        return None
    beg, end = [], []
    for r in range(deg.numel()):
        b, e = int(indptr[r]), int(indptr[r + 1])
        for s in range(max(1, -(-(e - b) // L))):
            beg.append(b + s * L)
            end.append(min(e, b + (s + 1) * L))
    return torch.tensor(beg), torch.tensor(end)


@pytest.mark.parametrize("seg", [None, "64"])
@pytest.mark.parametrize("canonical", [True, False])
@pytest.mark.parametrize("order", ["in", "out"])
def test_subset_matches_restatement(cuda, monkeypatch, order, canonical, seg):
    import bot_b200
    from bot_b200 import _lib, functional

    if seg:
        monkeypatch.setenv("BOTGAT_SEG", seg)
    n, E, H = 700, 40000, 3
    src, dst = graph_ref.synthetic_coo(n, E, 5, power_law=1.0)
    if canonical:   # given sorted by (dst, src): the library's edge numbering is the edge id
        o = np.lexsort((src, dst))
        src, dst = src[o], dst[o]
    g = bot_b200.Graph(torch.from_numpy(src).to(cuda), torch.from_numpy(dst).to(cuda), n, canonical=canonical)
    g._ensure()
    assert g._info.in_eid_identity == int(canonical)
    gen = torch.Generator().manual_seed(1)
    keep = (torch.rand(E, generator=gen) >= 0.3).to(torch.uint8)
    keep[: E // 50] = 0
    ee = torch.randn(E, 4, generator=gen)
    ords = _lib.ORDER_IN if order == "in" else _lib.ORDER_OUT
    eb, Hb, am, kept = functional.edge_stage(g, ords, H, ee.to(cuda), keep.to(cuda), kept=True, kept_eid=True)
    torch.cuda.synchronize()
    assert Hb == H and am is None and kept is not None

    indptr = g.structure(f"{order}_indptr").cpu()
    indices = g.structure(f"{order}_indices").cpu()
    eid = g.structure(f"{order}_eid").cpu()
    flag = keep[eid].long()
    X = torch.cat([torch.zeros(1, dtype=torch.long), flag.cumsum(0)])
    Ek = int(X[-1])
    W = E // 32 + 1
    bits = torch.zeros(W * 32, dtype=torch.long)
    bits[:E] = flag
    words = (bits.view(W, 32) << torch.arange(32)).sum(1)
    assert torch.equal(kept.kept.cpu().long() & 0xFFFFFFFF, words)
    assert torch.equal(kept.base.cpu().long(), X[torch.arange(W) * 32])
    assert torch.equal(kept.indptr.cpu().long(), X[indptr])
    sel = flag.bool()
    assert torch.equal(kept.indices[:Ek].cpu().long(), indices[sel])
    assert torch.equal(kept.eid[:Ek].cpu().long(), eid[sel])
    assert torch.equal(eb[:, :Ek].cpu(), ee[eid[sel], :H].t())
    segs = _segments(indptr, int(seg or 2048))
    n_seg = g._info.n_seg_in if order == "in" else g._info.n_seg_out
    if segs is None:
        assert n_seg == 0 and kept.seg_beg is None
    else:
        assert n_seg == segs[0].numel()
        assert torch.equal(kept.seg_beg.cpu().long(), X[segs[0]]) and torch.equal(kept.seg_end.cpu().long(), X[segs[1]])


# kernel families forced through the planner's knobs: (forward, src pass)
FAMILIES = {
    "warp_tma": dict(BOTGAT_LOWDEG="0", BOTGAT_ROWWISE="0"),
    "warp_ldg": dict(BOTGAT_LOWDEG="0", BOTGAT_ROWWISE="0", BOTGAT_BWD_TMA="0"),
    "lowdeg": dict(BOTGAT_LOWDEG="1000000", BOTGAT_ROWWISE="0"),
    "rowwise_bulk": dict(BOTGAT_ROWWISE="1"),
    "rowwise_ring": dict(BOTGAT_ROWWISE="1", BOTGAT_RW_BULK="0"),
}
SUBGRAPH_CASES = {
    "proteins_like_edge_drop": (400, 400, 30000, 6, 80, dict(ee=True, keep_p=0.1)),
    "products_like_H4_D120": (500, 500, 20000, 4, 120, dict(keep_p=0.1)),
}


@pytest.mark.parametrize("family", list(FAMILIES))
@pytest.mark.parametrize("name", list(SUBGRAPH_CASES))
def test_bit_identical_to_kept_subgraph(cuda, monkeypatch, name, family):
    """A step on (graph, keep) is the same computation as a step on the graph of the kept edges: the output, grad_ft and
    grad_el are bit-identical, and grad_ee is the subgraph's at kept edges and exactly 0 at dropped ones.  grad_er is
    reduced from the full grad_ee (dropped records are zeros in other lanes), so it agrees to fp32 rounding."""
    for k, v in FAMILIES[family].items():
        monkeypatch.setenv(k, v)
    n_src, n_dst, e, H, D, kw = SUBGRAPH_CASES[name]
    c = make_case(n_src, n_dst, e, H, D, seed=zlib.crc32(name.encode()) % 1000, **kw)
    keep = c["keep"]
    # without edge logits the keep mask is what makes the staged logit term (zeros) exist; an all-kept mask gives the
    # subgraph the same operands and so the same kernel instantiation
    sub_keep = None if c["ee"] is not None else torch.ones(int(keep.sum()), dtype=torch.bool)
    sub = dict(c, src=c["src"][keep], dst=c["dst"][keep], keep=sub_keep, ee=None if c["ee"] is None else c["ee"][keep])
    out, g, _ = engine_run(c, cuda)
    out_s, g_s, _ = engine_run(sub, cuda)
    assert torch.equal(out, out_s)
    for k in ("ft", "el"):
        assert torch.equal(g[k], g_s[k]), k
    assert rel_err(g["er"], g_s["er"]) <= 1e-6
    if c["ee"] is not None:
        kd = keep.to(cuda)
        assert torch.equal(g["ee"][kd], g_s["ee"])
        assert int(torch.count_nonzero(g["ee"][~kd])) == 0


def test_dropped_out_rows_and_attn_mul(cuda):
    """Sources whose every out-edge is dropped (empty rows of the kept out-CSR) and destinations whose every in-edge is,
    with an explicit attention-dropout multiplier compacted beside the logits: against the fp64 oracle."""
    c = make_case(300, 300, 12000, 4, 32, ee=True, keep_p=0.1, attn_p=0.2, seed=77)
    c["keep"] = c["keep"] & (c["src"] >= 20) & (c["dst"] >= 10)
    check_case(c, cuda)
    out, g, _ = engine_run(c, cuda)
    assert float(g["ft"][:20].abs().max()) == 0.0 and float(g["el"][:20].abs().max()) == 0.0
    assert float(out[:10].abs().max()) == 0.0


def test_power_law_split_rows(cuda, monkeypatch):
    """Heavy rows split into segments on both sides, keep plus in-kernel attention dropout against the oracle."""
    from util import philox_attn_mul

    monkeypatch.setenv("BOTGAT_SEG", "64")
    p, seed = 0.2, 99
    c = make_case(800, 800, 50000, 3, 40, ee=True, keep_p=0.15, power_law=1.2, seed=78)
    ids = graph_ref.canonical_edge_ids(c["src"].numpy(), c["dst"].numpy())
    ref_c = dict(c, attn_mul=philox_attn_mul(seed, 50000, 3, p, eids=ids))
    ref_out, ref_g = oracle_run(ref_c)
    out, g, gr = engine_run(c, cuda, attn_p=p, seed=seed)
    assert gr._info.n_seg_in > 0 and gr._info.n_seg_out > 0
    assert rel_err(out, ref_out) <= FWD_TOL
    for k in ("ft", "el", "er", "ee"):
        assert rel_err(g[k], ref_g[k]) <= 1e-4, k


def test_no_keep_launches_nothing_new(cuda):
    """Without keep the staging path is the one without a subset: no scan, no bound translation."""
    import bot_b200
    from bot_b200.functional import gat_fused
    from torch.profiler import ProfilerActivity, profile

    c = make_case(400, 400, 30000, 6, 80, ee=True, keep_p=0.1, seed=3)
    g = bot_b200.Graph(c["src"].to(cuda), c["dst"].to(cuda), 400)
    g._ensure()   # the graph build (its own CUB scans) happens outside the traced steps
    ft, el, er, ee = (c[k].to(cuda).requires_grad_(True) for k in ("ft", "el", "er", "ee"))
    gout, keep = c["gout"].to(cuda), c["keep"].to(cuda)
    torch.cuda.synchronize()

    def names(k):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            gat_fused(g, ft, el, er, ee, k).backward(gout)
            torch.cuda.synchronize()
        return {e.name for e in prof.events()}

    without, with_keep = names(None), names(keep)
    assert not any("k_subset_bounds" in n or "DeviceScan" in n for n in without)
    assert any("k_subset_bounds" in n for n in with_keep) and any("DeviceScan" in n for n in with_keep)
