"""Shared helpers for the parity tests (oracle = checker only)."""
import numpy as np
import torch

from oracle import gat_ref, graph_ref

FWD_TOL = 1e-5   # north_star: fp32 layer outputs within 1e-5 relative
GRAD_TOL = 1e-4  # north_star: gradients within 1e-4 relative


def rel_err(x, ref):
    """max|x-ref| / max|ref| (norm-relative; elementwise relative error is ill-defined near 0)."""
    x = x.detach().double().cpu()
    ref = ref.detach().double().cpu()
    assert x.shape == ref.shape, (x.shape, ref.shape)
    if ref.numel() == 0:
        return 0.0
    denom = ref.abs().max().item()
    return (x - ref).abs().max().item() / (denom if denom > 0 else 1.0)


def make_case(n_src, n_dst, n_edges, H, D, *, er=True, ee=False, keep_p=0.0, attn_p=0.0, symm=False,
              seed=0, power_law=0.0, self_loops=False):
    """Random inputs of the sparse section, on CPU, fp32.  Returns a dict."""
    g = torch.Generator().manual_seed(seed)
    rng = np.random.default_rng(seed)
    src = rng.integers(0, n_src, size=n_edges, dtype=np.int64)
    if power_law > 0:
        w = np.arange(1, n_dst + 1, dtype=np.float64) ** (-power_law)
        cdf = np.cumsum(w / w.sum())
        dst = np.minimum(np.searchsorted(cdf, rng.random(n_edges)), n_dst - 1).astype(np.int64)
    else:
        dst = rng.integers(0, n_dst, size=n_edges, dtype=np.int64)
    if self_loops:
        assert n_src == n_dst
        src, dst = graph_ref.add_self_loop(*graph_ref.remove_self_loop(src, dst), n_src)
    E = src.shape[0]
    c = {
        "src": torch.from_numpy(src), "dst": torch.from_numpy(dst), "n_src": n_src, "n_dst": n_dst, "H": H, "D": D,
        "ft": torch.randn(n_src, H, D, generator=g),
        "el": torch.randn(n_src, H, generator=g),
        "er": torch.randn(n_dst, H, generator=g) if er else None,
        "ee": torch.randn(E, H, generator=g) if ee else None,
        "keep": None, "attn_mul": None, "src_scale": None, "dst_scale": None,
        "gout": torch.randn(n_dst, H, D, generator=g),
    }
    if keep_p > 0:
        perm = torch.randperm(E, generator=g)
        keep = torch.ones(E, dtype=torch.bool)
        keep[perm[: int(E * keep_p)]] = False
        c["keep"] = keep
    if attn_p > 0:
        m = (torch.rand(E, H, generator=g) >= attn_p).float() / (1.0 - attn_p)
        c["attn_mul"] = m
    if symm:
        f = graph_ref.build_formats(src, dst, n_src, n_dst)
        c["src_scale"] = torch.from_numpy(graph_ref.deg_scale(f["out_deg"], -0.5))
        c["dst_scale"] = torch.from_numpy(graph_ref.deg_scale(f["in_deg"], 0.5))
    return c


def oracle_run(c, dtype=torch.float64, slope=0.2):
    """Forward + gradients from the oracle (autograd).  Returns (out, grads dict)."""
    def cvt(t, grad):
        if t is None:
            return None
        t = t.to(dtype).clone()
        return t.requires_grad_(grad)

    ft, el = cvt(c["ft"], True), cvt(c["el"], True)
    er, ee = cvt(c["er"], True), cvt(c["ee"], True)
    out = gat_ref.gat_sparse(c["src"], c["dst"], c["n_dst"], ft, el, er, ee, c["keep"],
                             cvt(c["attn_mul"], False), slope, cvt(c["src_scale"], False), cvt(c["dst_scale"], False))
    out.backward(c["gout"].to(dtype))
    grads = {"ft": ft.grad, "el": el.grad, "er": None if er is None else er.grad, "ee": None if ee is None else ee.grad}
    return out.detach(), grads


def engine_run(c, device, slope=0.2, attn_p=0.0, seed=0):
    """Same through bot_b200 (CUDA).  Returns (out, grads dict)."""
    import bot_b200
    from bot_b200.functional import gat_fused

    def dev(t, grad):
        if t is None:
            return None
        t = t.to(device).clone()
        return t.requires_grad_(grad)

    g = bot_b200.Graph(c["src"].to(device), c["dst"].to(device), c["n_src"], c["n_dst"],
                       is_block=c["n_src"] != c["n_dst"])
    ft, el = dev(c["ft"], True), dev(c["el"], True)
    er, ee = dev(c["er"], True), dev(c["ee"], True)
    out = gat_fused(g, ft, el, er, ee, dev(c["keep"], False), dev(c["attn_mul"], False), dev(c["src_scale"], False),
                    dev(c["dst_scale"], False), slope, attn_p, seed)
    out.backward(c["gout"].to(device))
    torch.cuda.synchronize()
    grads = {"ft": ft.grad, "el": el.grad, "er": None if er is None else er.grad, "ee": None if ee is None else ee.grad}
    return out.detach(), grads, g


def check_case(c, device, **kw):
    """Forward and gradients against the fp64 oracle, norm-relative and row-normalised (``gat_rows.row_rel_err``, each
    row by its own magnitude floored at 1e-3 (forward) / 1e-2 (gradients) of the global one, as test_gpu_fullsize)."""
    from oracle.gat_rows import row_rel_err

    ref_out, ref_g = oracle_run(c)
    out, g, _ = engine_run(c, device, **kw)
    errs = {"out": rel_err(out, ref_out)}
    assert errs["out"] <= FWD_TOL, f"forward rel err {errs['out']:.3e} > {FWD_TOL}"
    r = row_rel_err(out, ref_out, 1e-3)
    assert r <= FWD_TOL, f"forward row-normalised err {r:.3e} > {FWD_TOL}"
    for k in ("ft", "el", "er", "ee"):
        if ref_g[k] is None:
            assert g[k] is None
            continue
        errs[k] = rel_err(g[k], ref_g[k])
        assert errs[k] <= GRAD_TOL, f"grad_{k} rel err {errs[k]:.3e} > {GRAD_TOL}"
        r = row_rel_err(g[k], ref_g[k], 1e-2)
        assert r <= GRAD_TOL, f"grad_{k} row-normalised err {r:.3e} > {GRAD_TOL}"
    return errs


def philox_attn_mul(seed, n_edges, n_heads, p, eids=None):
    """numpy restatement of `philox_dropout_mul` (bot_b200/csrc/common.cuh): Philox4x32-10 keyed on the 64-bit
    seed, counter (edge id, head >> 2, 0x9E3779B9, 0xBB67AE85), component head & 3; keep iff u >= p.
    ``eids``: evaluate only these edge ids (rows of the result follow it) instead of 0..n_edges-1."""
    import numpy as np

    M0, M1, W0, W1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), np.uint32(0x9E3779B9), np.uint32(0xBB67AE85)
    eid = np.arange(n_edges, dtype=np.uint32) if eids is None else np.asarray(eids).astype(np.uint32)
    n_edges = eid.shape[0]
    out = np.zeros((n_edges, n_heads), dtype=np.float32)
    for h in range(n_heads):
        c0 = eid.copy()
        c1 = np.full(n_edges, h >> 2, dtype=np.uint32)
        c2 = np.full(n_edges, 0x9E3779B9, dtype=np.uint32)
        c3 = np.full(n_edges, 0xBB67AE85, dtype=np.uint32)
        k0, k1 = np.uint32(seed & 0xFFFFFFFF), np.uint32((seed >> 32) & 0xFFFFFFFF)
        for _ in range(10):
            p0 = M0 * c0.astype(np.uint64)
            p1 = M1 * c2.astype(np.uint64)
            hi0, lo0 = (p0 >> np.uint64(32)).astype(np.uint32), p0.astype(np.uint32)
            hi1, lo1 = (p1 >> np.uint64(32)).astype(np.uint32), p1.astype(np.uint32)
            c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
            k0, k1 = np.uint32((int(k0) + int(W0)) & 0xFFFFFFFF), np.uint32((int(k1) + int(W1)) & 0xFFFFFFFF)
        x = (c0, c1, c2, c3)[h & 3]
        u = (x >> np.uint32(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)
        out[:, h] = np.where(u >= np.float32(p), np.float32(1.0 / (1.0 - p)), np.float32(0.0))
    return torch.from_numpy(out)


def philox_edge_drop_keep(seed, n_edges, n_drop):
    """numpy restatement of `botgat_edge_drop_draw` (bot_b200/csrc/edge_drop.cu): 64-bit Philox4x32-10 keys, counter
    (pair, 0x80000000 | pair >> 32, 0x9E3779B9, 0xBB67AE85) for the edges (2*pair, 2*pair+1) = words (0,1) / (2,3);
    the n_drop smallest keys are dropped."""
    import numpy as np

    M0, M1, W0, W1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), 0x9E3779B9, 0xBB67AE85
    n_pairs = (n_edges + 1) // 2
    pair = np.arange(n_pairs, dtype=np.uint64)
    c0 = pair.astype(np.uint32)
    c1 = (np.uint32(0x80000000) | (pair >> np.uint64(32)).astype(np.uint32))
    c2 = np.full(n_pairs, W0, dtype=np.uint32)
    c3 = np.full(n_pairs, W1, dtype=np.uint32)
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    for _ in range(10):
        p0 = M0 * c0.astype(np.uint64)
        p1 = M1 * c2.astype(np.uint64)
        hi0, lo0 = (p0 >> np.uint64(32)).astype(np.uint32), p0.astype(np.uint32)
        hi1, lo1 = (p1 >> np.uint64(32)).astype(np.uint32), p1.astype(np.uint32)
        c0, c1, c2, c3 = hi1 ^ c1 ^ np.uint32(k0), lo1, hi0 ^ c3 ^ np.uint32(k1), lo0
        k0, k1 = (k0 + W0) & 0xFFFFFFFF, (k1 + W1) & 0xFFFFFFFF
    keys = np.empty(2 * n_pairs, dtype=np.uint64)
    keys[0::2] = (c0.astype(np.uint64) << np.uint64(32)) | c1.astype(np.uint64)
    keys[1::2] = (c2.astype(np.uint64) << np.uint64(32)) | c3.astype(np.uint64)
    keys = keys[:n_edges]
    keep = np.ones(n_edges, dtype=np.uint8)
    keep[np.argsort(keys, kind="stable")[:n_drop]] = 0
    return torch.from_numpy(keep)


def _philox4x32(seed, c0, c1, c2, c3):
    """numpy Philox4x32-10 over arrays of counter words (uint32); returns the four output words."""
    import numpy as np

    M0, M1, W0, W1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), 0x9E3779B9, 0xBB67AE85
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint32) for c in (c0, c1, c2, c3))
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    for _ in range(10):
        p0 = M0 * c0.astype(np.uint64)
        p1 = M1 * c2.astype(np.uint64)
        hi0, lo0 = (p0 >> np.uint64(32)).astype(np.uint32), p0.astype(np.uint32)
        hi1, lo1 = (p1 >> np.uint64(32)).astype(np.uint32), p1.astype(np.uint32)
        c0, c1, c2, c3 = hi1 ^ c1 ^ np.uint32(k0), lo1, hi0 ^ c3 ^ np.uint32(k1), lo0
        k0, k1 = (k0 + W0) & 0xFFFFFFFF, (k1 + W1) & 0xFFFFFFFF
    return c0, c1, c2, c3


def sample_neighbors_ref(indptr, indices, eids, seeds, fanout, seed):
    """numpy restatement of `botgat_sample_neighbors` (bot_b200/csrc/sampling.cu): per seed v with in-degree d > fanout
    the candidate stream c_n = mulhi64(philox64(seed; n>>1, 0x40000000, v, 0x5BD1E995)[n&1], d), n = 0, 1, ...,
    accepted when new until m = fanout picks (or, when fanout > d // 2, m = d - fanout EXCLUDED positions, the rest
    emitted in row order).  Returns (src, dst_pos, eid, offsets)."""
    import numpy as np

    src, dst, eid, offsets = [], [], [], [0]
    for i, v in enumerate(np.asarray(seeds)):
        beg, d = int(indptr[v]), int(indptr[v + 1] - indptr[v])
        if fanout <= 0 or d <= fanout:
            pos = list(range(d))
        else:
            complement = fanout > d // 2
            m = d - fanout if complement else fanout
            picks, n0 = [], 0
            while len(picks) < m:
                n = np.arange(n0, n0 + 32, dtype=np.uint64)
                w = _philox4x32(seed, (n >> np.uint64(1)).astype(np.uint32), np.full(32, 0x40000000, np.uint32),
                                np.full(32, v, np.uint32), np.full(32, 0x5BD1E995, np.uint32))
                for j in range(32):
                    hi, lo = (w[2][j], w[3][j]) if (n0 + j) & 1 else (w[0][j], w[1][j])
                    c = (((int(hi) << 32) | int(lo)) * d) >> 64
                    if c not in picks and len(picks) < m:
                        picks.append(c)
                n0 += 32
            pos = [j for j in range(d) if j not in set(picks)] if complement else picks
        src += [int(indices[beg + j]) for j in pos]
        eid += [int(eids[beg + j]) for j in pos]
        dst += [i] * len(pos)
        offsets.append(len(src))
    return (np.asarray(src, dtype=np.int64), np.asarray(dst, dtype=np.int64), np.asarray(eid, dtype=np.int64),
            np.asarray(offsets, dtype=np.int64))


def to_block_ref(n_parent, seeds, src):
    """numpy restatement of `botgat_block_compact`: src nodes = seeds, then the other sampled sources ascending."""
    import numpy as np

    seeds = np.asarray(seeds, dtype=np.int64)
    extra = np.setdiff1d(np.unique(src), seeds)
    nodes = np.concatenate([seeds, extra])
    where = np.full(n_parent, -1, dtype=np.int64)
    where[nodes] = np.arange(nodes.size)
    return nodes, where[np.asarray(src, dtype=np.int64)]
