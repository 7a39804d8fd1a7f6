"""Host-side mirror of the reference interface (CPU): constructors, parameter names/shapes/initialisation,
#Params known-answer values (SURVEY.md section 4), helper arithmetic."""
import os

import pytest
import torch
import torch.nn.functional as F


def golden(name):
    """A case recorded from the unmodified reference modules by tests/golden/make_golden.py."""
    return torch.load(os.path.join(os.path.dirname(__file__), "golden", name + ".pt"), weights_only=True)


def n_params(m):
    return sum(p.numel() for p in m.parameters() if p.requires_grad)


def test_param_counts_known_answers():
    from bot_b200.no_sampling import GAT
    from bot_b200.ogbn_products import GAT as ProductsGAT
    from bot_b200.ogbn_proteins import GAT as ProteinsGAT

    # run.py:1009 (cmd :1002): arxiv GAT --use-labels, 3 layers, 3 heads, hidden 250, BN, linear
    arxiv = GAT(128 + 40, 0, 40, 250, 3, 3, F.relu, norm="batch", dropout=0.75, input_drop=0.1, attn_drop=0.1,
                edge_drop=0, use_symmetric_norm=True, linear=True)
    assert n_params(arxiv) == 1441580
    # proteins gat.py:377 / :385
    assert n_params(ProteinsGAT(8, 8, 112, 6, 6, 80, 16, F.relu, 0.25, 0.1, 0.0, 0.1)) == 2475232
    assert n_params(ProteinsGAT(8 + 112, 8, 112, 6, 6, 80, 16, F.relu, 0.25, 0.1, 0.0, 0.1)) == 2484192
    # products gat.py:441
    assert n_params(ProductsGAT(100, 0, 47, 3, 4, 120, 0, F.relu, 0.5, 0.1, 0.0, 0.1, allow_zero_in_degree=True)) == 1065127
    # run.py:902 / :974 were logged when every layer had attn_r (today's --non-interactive-attn)
    cora = GAT(1433, 0, 7, 8, 2, 8, F.relu, norm="none", dropout=0.6, attn_drop=0.6, edge_drop=0.5, non_interactive_attn=True)
    assert n_params(cora) == 92373
    reddit = GAT(602, 0, 41, 64, 3, 4, F.relu, norm="batch", non_interactive_attn=True, linear=True)
    assert n_params(reddit) == 462459


# reference-recorded GATConv layer cases under tests/golden/ -> the torch.manual_seed make_golden.py set right before
# it built the reference module (make_golden.py main: run_case seeds)
V1_CASES = {"v1_eval_plain": 0, "v1_eval_symm_attnr": 1, "v1_eval_nolinear_last": 2, "v1_train_edgedrop_attndrop": 3,
            "v1_train_attndrop_only": 4, "v1_eval_block": 11}
V2_CASES = {"v2_eval_edgefeat": 5, "v2_eval_noedge_nodst": 6, "v2_train_edgedrop": 7, "v2_train_edgedrop_attndrop": 8,
            "v2_eval_symm": 9, "v2_eval_block": 10}


@pytest.mark.parametrize("case", V1_CASES)
def test_v1_state_dict_and_init_match_reference(case):
    from bot_b200.no_sampling import GATConv

    rec = golden(case)
    sd_t = rec["state_dict"]   # the reference's GATConv(**ctor), built under the same seed
    torch.manual_seed(V1_CASES[case])
    ours = GATConv(**rec["ctor"])
    sd_o = ours.state_dict()
    assert list(sd_t) == list(sd_o)
    for k in sd_t:
        assert torch.equal(sd_t[k], sd_o[k]), k  # same names, shapes AND values under the same seed
    ours.load_state_dict(sd_t, strict=True)


@pytest.mark.parametrize("case", V2_CASES)
def test_v2_state_dict_and_init_match_reference(case):
    """Recorded from src/ogbn-proteins/models.py; bot_b200.ogbn_proteins and bot_b200.ogbn_products share this GATConv,
    and the products reference's layers are checked inside its whole model (test_model_state_dicts_interchange)."""
    from bot_b200.sampled import GATConv

    rec = golden(case)
    sd_t = rec["state_dict"]
    torch.manual_seed(V2_CASES[case])
    ours = GATConv(**rec["ctor"])
    sd_o = ours.state_dict()
    assert sorted(sd_t) == sorted(sd_o)
    for k in sd_t:
        assert torch.equal(sd_t[k], sd_o[k]), k


def test_model_state_dicts_interchange():
    """The reference-recorded whole models (make_golden.py model_cases: seed, constructor arguments): same parameter
    and buffer names, same initial values under the same seed, and their state_dicts load strictly into ours."""
    from bot_b200.no_sampling import GAT
    from bot_b200.ogbn_products import GAT as ProductsGAT
    from bot_b200.ogbn_proteins import GAT as ProteinsGAT

    for name, seed, build in (
            ("model_v1_gat_bn", 20, lambda: GAT(20, 0, 5, 8, 3, 2, F.relu, norm="batch", dropout=0.5, attn_drop=0.1,
                                                use_symmetric_norm=True, linear=True, residual=True)),
            ("model_v1_gat_bias", 21, lambda: GAT(20, 0, 5, 8, 2, 3, F.relu, norm="none", non_interactive_attn=True)),
            ("model_proteins_gat", 22, lambda: ProteinsGAT(8, 8, 11, 2, 3, 10, 16, F.relu, 0.25, 0.1, 0.0, 0.1)),
            ("model_products_gat", 23, lambda: ProductsGAT(9, 0, 7, 2, 2, 6, 0, F.relu, 0.5, 0.1, 0.0, 0.1,
                                                           allow_zero_in_degree=True, residual=True))):
        t = golden(name)["state_dict"]
        torch.manual_seed(seed)
        o = build()
        assert sorted(t) == sorted(o.state_dict()), name
        for k, v in t.items():
            assert torch.equal(v, o.state_dict()[k]), (name, k)
        o.load_state_dict(t, strict=True)


def test_v2_residual_false_is_rejected_like_the_reference():
    """The reference's GATConv(residual=False) fails in its constructor (nn.Parameter(int) at
    src/ogbn-proteins/models.py:49); ours rejects it explicitly."""
    from bot_b200.sampled import GATConv

    with pytest.raises(TypeError):
        GATConv(4, 0, 4, residual=False)


def test_edge_keep_follows_reference_draw():
    from bot_b200.no_sampling import draw_edge_keep

    torch.manual_seed(5)
    perm = torch.randperm(100)
    torch.manual_seed(5)
    keep, eids = draw_edge_keep(100, 0.37, torch.device("cpu"))
    bound = int(100 * 0.37)
    assert torch.equal(eids, perm[bound:]) and int(keep.sum()) == 100 - bound
    assert not keep[perm[:bound]].any()


def test_pad_heads():
    from bot_b200.functional import pad_heads

    assert [pad_heads(h) for h in (1, 2, 3, 4, 5, 6, 8, 9, 12)] == [1, 2, 4, 4, 8, 8, 8, 12, 12]


def test_lazy_frame_gathers_parent_rows():
    from bot_b200.sampling import NID, _LazyFrame

    parent = {"feat": torch.arange(20.0).view(10, 2), "deg": torch.arange(10)}
    ids = torch.tensor([7, 2, 2, 9])
    f = _LazyFrame(parent, ids)
    assert torch.equal(f[NID], ids) and "feat" in f and "nope" not in f
    assert torch.equal(f["feat"], parent["feat"][ids]) and torch.equal(f["deg"], ids)
    f["feat"] = f["feat"] + 1          # the reference's add_labels overwrites srcdata["feat"] (gat.py:88-100)
    assert torch.equal(f["feat"], parent["feat"][ids] + 1)
    assert set(f.keys()) == {NID, "feat", "deg"}
    with pytest.raises(KeyError):
        f["nope"]


def test_sampling_restatement_properties():
    """The numpy restatement the GPU sampler is checked against: exact counts, no repeats, real in-edges,
    and a uniform draw (direct and complement paths)."""
    import numpy as np

    from oracle import graph_ref
    from util import sample_neighbors_ref, to_block_ref

    src, dst = graph_ref.synthetic_coo(120, 3000, 1, power_law=0.9)
    ref = graph_ref.build_formats(src, dst, 120, 120)
    seeds = np.arange(0, 120, 3)
    for fanout in (3, 20, -1):
        s, d, e, off = sample_neighbors_ref(ref["in_indptr"], ref["in_indices"], ref["in_eid"], seeds, fanout, 99)
        deg = ref["in_deg"][seeds]
        assert np.array_equal(np.diff(off), deg if fanout <= 0 else np.minimum(deg, fanout))
        assert np.unique(e).size == e.size
        assert np.array_equal(src[e], s) and np.array_equal(dst[e], seeds[d])
        nodes, local = to_block_ref(120, seeds, s)
        assert np.array_equal(nodes[: seeds.size], seeds) and np.unique(nodes).size == nodes.size
        assert np.array_equal(nodes[local], s)
    indptr, idx = np.array([0, 30]), np.arange(30)
    for k in (6, 24):
        freq = np.zeros(30)
        for sd in range(600):
            _, _, e, _ = sample_neighbors_ref(indptr, idx, idx, np.array([0]), k, sd)
            assert e.size == k
            freq[e] += 1
        p = k / 30
        z = (freq / 600 - p) / (p * (1 - p) / 600) ** 0.5
        assert np.abs(z).max() < 4.5


def test_edge_drop_restatement_counts():
    from util import philox_edge_drop_keep

    for E, n_drop in ((1, 0), (7, 3), (1000, 370), (1001, 1000)):
        keep = philox_edge_drop_keep(5, E, n_drop)
        assert int(keep.sum()) == E - n_drop
    a, b = philox_edge_drop_keep(1, 5000, 500), philox_edge_drop_keep(2, 5000, 500)
    assert not torch.equal(a, b)


def test_bench_algorithmic_bytes_match_survey():
    """SURVEY.md section 8d: 1,983 B/edge forward and 3,996 B/edge backward at the proteins shape (the figure
    `roofline.achieved` is computed from), 78.4 + 158.1 GB per layer."""
    import bench

    E, N, H, D = 39561252, 132534, 6, 80
    bf, bb = bench.algorithmic_bytes(E, N, N, H, D)
    assert round(bf / E) == 1983 and round(bb / E) == 3996
    assert abs(bf / 1e9 - 78.4) < 0.1 and abs(bb / 1e9 - 158.1) < 0.1
    # products shape (no edge features): 2,018 + 4,148 B/edge
    bf, bb = bench.algorithmic_bytes(61859140, 2449029, 2449029, 4, 120, er=True, ee=False)
    assert abs(bf / 61859140 - 2018) < 1.5 and abs(bb / 61859140 - 4148) < 2.5


class _RefBatchSampler:
    """Restatement of the reference's BatchSampler (src/ogbn-proteins/utils.py:22-32): infinite, ``None`` ends an epoch."""

    def __init__(self, n, batch_size):
        self.n, self.batch_size = n, batch_size

    def __iter__(self):
        while True:
            for b in torch.randperm(self.n).split(self.batch_size):
                yield b
            yield None


class _RefDataLoaderWrapper:
    """Restatement of DataLoaderWrapper (utils.py:8-19): ONE iter() reused every epoch, any exception ends the epoch."""

    def __init__(self, dataloader):
        self.iter = iter(dataloader)

    def __iter__(self):
        return self

    def __next__(self):
        try:
            return next(self.iter)
        except Exception:
            raise StopIteration() from None


def test_node_dataloader_with_the_reference_batch_sampler_over_epochs():
    """`NodeDataLoader(..., batch_sampler=BatchSampler(n, bs))` wrapped in `DataLoaderWrapper`
    (src/ogbn-proteins/gat.py:179-189) must yield every node once per epoch, for several epochs, with and
    without the wrapper; `len()` = batches per epoch."""
    from bot_b200 import sampling

    class FakeBlock:
        def __init__(self, seeds):
            self.srcdata = {sampling.NID: seeds}

    class FakeSampler:
        def sample_blocks(self, g, seeds):
            return [FakeBlock(seeds)]

    class FakeGraph:
        device = torch.device("cpu")

    nids = torch.arange(100, 137)
    loader = sampling.NodeDataLoader(FakeGraph(), nids, FakeSampler(), batch_sampler=_RefBatchSampler(37, 10), num_workers=10)
    assert len(loader) == 4
    wrapped = _RefDataLoaderWrapper(loader)
    for _ in range(3):
        got = [out for _, out, _ in wrapped]
        assert len(got) == 4 and torch.equal(torch.cat(got).sort().values, nids)
    loader = sampling.NodeDataLoader(FakeGraph(), nids, FakeSampler(), batch_sampler=_RefBatchSampler(37, 10))
    for _ in range(3):   # plain `for ... in loader` also sees one epoch per loop
        got = [out for _, out, _ in loader]
        assert len(got) == 4 and torch.equal(torch.cat(got).sort().values, nids)
    # finite batch samplers restart every epoch
    loader = sampling.NodeDataLoader(FakeGraph(), nids, FakeSampler(), batch_sampler=[[0, 1], [2]])
    for _ in range(2):
        assert [o.tolist() for _, o, _ in loader] == [[100, 101], [102]]


def test_bench_numa_pinning_is_harmless_without_nvml():
    """`bench.pin_to_gpu_numa`: a no-op for one rank, and on a machine without NVML (this container) it reports the
    failure and leaves the process affinity as it was."""
    import os

    import bench

    before = os.sched_getaffinity(0)
    assert bench.pin_to_gpu_numa(0, 1) is None
    got = bench.pin_to_gpu_numa(0, 2)
    assert got is None or isinstance(got, dict)
    if isinstance(got, dict) and ("error" in got or got.get("cpus") == 0):
        assert os.sched_getaffinity(0) == before
    os.sched_setaffinity(0, before)
