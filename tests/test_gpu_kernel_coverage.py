"""Every instantiated gather kernel against the fp64 oracle, with the launch trace confirming which one ran.

The layer's hot path is a set of template kernels; host code picks one instantiation per launch from the shape, the
pointer alignment, the graph's degrees and a few knobs (``plan_forward`` / ``plan_src`` in csrc/plan.cu, with
``choose_tiling``, ``rowwise_wanted`` / ``rowwise_geometry`` and the low-degree threshold).  An off-by-one in the lane /
slot arithmetic of one instantiation only shows when that instantiation runs, and a case that quietly falls back to
another family still passes.  So each case below

* sets shape, alignment and knobs, and predicts the forward and backward src-pass instantiation with a restatement of
  the selection functions (``expected_kernels``; a drift between it and the C++ code fails the trace assertion);
* runs a training step and a fused-tail inference step under ``torch.profiler`` and asserts that exactly the predicted
  gather kernels were launched;
* compares the output and every gradient with ``oracle/gat_ref.py`` in fp64, norm-relative and row-normalised, and
  checks that a rerun is bit-identical.

The last test checks that the cases together ran every gather instantiation in the built library.
"""
from __future__ import annotations

import os
import re
import shutil
import subprocess
import time
import types

import numpy as np
import pytest
import torch

from oracle import gat_rows
from util import FWD_TOL, GRAD_TOL, oracle_run, philox_attn_mul, rel_err

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "bot_b200", "libbotgat.so")
KNOBS = ("BOTGAT_ROWWISE", "BOTGAT_ROWWISE_FWD", "BOTGAT_ROWWISE_BWD", "BOTGAT_ROWWISE_MB", "BOTGAT_LOWDEG",
         "BOTGAT_LOWDEG_BWD", "BOTGAT_BWD_TMA", "BOTGAT_RW_BULK", "BOTGAT_G", "BOTGAT_VW", "BOTGAT_NOALIGN",
         "BOTGAT_SLAB_MB", "BOTGAT_SEG", "BOTGAT_FUSE_TAIL")


# ---------------------------------------------------------------------------
# restatement of the kernel selection (csrc/plan.cu; the instantiation lists are in common.cuh and params.cuh)
# ---------------------------------------------------------------------------
def _combos():
    """BG_COMBOS (common.cuh): the head-major (VW, GSH, VPL) geometries."""
    small, full, big = (1, 2), tuple(range(1, 9)), (5, 6, 7, 8)
    rows = [(4, 0, small), (4, 1, small), (4, 2, small), (4, 3, full), (4, 4, big), (4, 5, big),
            (2, 0, small), (2, 1, small), (2, 2, small), (2, 3, small), (2, 4, full), (2, 5, big),
            (1, 0, small), (1, 1, small), (1, 2, small), (1, 3, small), (1, 4, small), (1, 5, full)]
    return {(vw, g, v) for vw, g, vpls in rows for v in vpls}


COMBOS = _combos()
TMA_COMBOS = {(4, 2), (8, 2), (12, 2), (16, 2), (20, 2), (24, 2), (32, 2), (10, 3), (30, 3), (40, 3)}  # BG_TMA_COMBOS (params.cuh)
BULK_RING = 8        # kBulkRing (params.cuh)


def _env_int(env, name, dflt):
    s = env.get(name, "")
    return int(s) if s else dflt


def _pow2ceil(x):
    p = 1
    while p < x:
        p <<= 1
    return p


def choose_tiling(H, D, ld_g, pg, ld_o, po, parts_req, n_rows, env):
    """plan.cu choose_tiling: returns (vw, gshift, vpl, col_parts).  ``pg`` / ``po``: pointer addresses (or their
    residues modulo 128)."""
    def ok(vw):
        return D % vw == 0 and ld_g % vw == 0 and ld_o % vw == 0 and pg % (vw * 4) == 0 and po % (vw * 4) == 0

    vw = 4 if ok(4) else (2 if ok(2) else 1)
    fvw = _env_int(env, "BOTGAT_VW", 0)
    if fvw in (1, 2) and fvw < vw:
        vw = fvw
    gline = 32 // vw
    can_align = (ld_g * 4) % 128 == 0 and pg % 128 == 0 and _env_int(env, "BOTGAT_NOALIGN", 0) == 0
    if parts_req == 1 and can_align and D > (256 - gline) * vw:
        can_align = False
    cap = (256 - (gline if can_align else 0)) * vw
    parts = parts_req
    if parts <= 0:
        budget = _env_int(env, "BOTGAT_SLAB_MB", 64) << 20
        parts = max(1, -(-n_rows * D * 4 // budget))
        parts = min(parts, max(1, D // (16 * vw)))

    def part_cols(n):
        return -(-(-(-D // n)) // vw) * vw

    while part_cols(parts) > cap:
        parts += 1
    pc = part_cols(parts)
    col_parts = -(-D // pc)
    nv = -(-pc // vw)
    G = min(gline, _pow2ceil(nv))
    fg = _env_int(env, "BOTGAT_G", 0)
    if 1 <= fg <= 32 and fg & (fg - 1) == 0:
        G = fg
    while True:
        gsh = G.bit_length() - 1
        omask = min(G, gline) - 1 if can_align else 0
        omax = max([((h * D + cp * pc) // vw) & omask for h in range(H) for cp in range(col_parts)]) if omask else 0
        need = -(-(nv + omax) // G)
        vpl = next((c for c in range(need, 9) if (vw, gsh, c) in COMBOS), -1)
        if vpl > 0 or G >= 32:
            break
        G <<= 1
    return vw, gsh, vpl, col_parts


def use_lowdeg(n_edges, n_rows, backward, env):
    """plan.cu low_degree with the threshold of Knobs::read."""
    s = env.get("BOTGAT_LOWDEG_BWD" if backward else "BOTGAT_LOWDEG", "") or env.get("BOTGAT_LOWDEG", "")
    thr = int(s) if s else (96 if backward else 20)
    return n_rows > 0 and n_edges < thr * n_rows


def rowwise_geometry(heads, D):
    """plan.cu rowwise_geometry: (log2 lanes per head, slots per lane) or None."""
    if heads < 1 or heads > 8 or D % 4:
        return None
    g = 32 // _pow2ceil(heads)
    need = -(-(D // 4) // g)
    return None if need > 8 else (g.bit_length() - 1, need)


def rowwise_wanted(D, n_rows_table, n_edges, n_csr_rows, backward, env):
    """plan.cu rowwise_wanted."""
    s = env.get("BOTGAT_ROWWISE_BWD" if backward else "BOTGAT_ROWWISE_FWD", "") or env.get("BOTGAT_ROWWISE", "")
    if s:
        return s[0] != "0"
    always = _env_int(env, "BOTGAT_ROWWISE_MB", 256 if backward else 96) << 20
    resident = min(_env_int(env, "BOTGAT_SLAB_MB", 64) << 20, always)
    max_parts = D // 64 if (not backward and D // 64 > 0) else 1
    part_bytes = n_rows_table * D * 4 // max_parts
    if part_bytes <= resident:
        return False
    low = n_edges < 96 * n_csr_rows and (not backward or n_edges >= 8 * n_csr_rows)
    return low or part_bytes > always


def _b(x):
    return "true" if x else "false"


def expected_kernels(c, env, edge_mode):
    """(forward training kernel, forward inference kernel, backward src-pass kernel) for case ``c`` (see ``make_inputs``),
    as botgat::name<args> strings: the family order of plan.cu plan_forward (row-wise, low-degree, warp) and plan_src
    (row-wise with bulk or register ring, TMA unless low-degree, low-degree, warp)."""
    H, D, n_src, n_dst, E = c["H"], c["D"], c["n_src"], c["n_dst"], c["E"]
    direct = edge_mode == "direct"
    has_edge_ops = c["ee"] or c["keep"] or c["attn_mul"]
    # forward: the gathered table is ft (storage offset c["off"] floats); out / residuals / y / scale / shift are fresh
    ft_ptr = 4 * c["off"]
    vw, gsh, vpl, parts = choose_tiling(H, D, H * D, ft_ptr, H * D, 0, 0, n_src, env)
    fwd = []
    for ep in (False, True):
        rw = rowwise_geometry(H, D)
        if vw == 4 and not (direct and has_edge_ops) and rowwise_wanted(D, n_src, E, n_dst, False, env) and rw:
            fwd.append(f"botgat::gat_fwd_rowwise_kernel<{rw[0]}, {rw[1]}, {_b(ep)}>")
        elif use_lowdeg(E, n_dst, False, env):
            fwd.append(f"botgat::gat_fwd_lowdeg_kernel<{vw}, {gsh}, {vpl}, {_b(ep)}>")
        else:
            fwd.append(f"botgat::gat_fwd_kernel<{vw}, {gsh}, {vpl}, {_b(ep)}>")
    # backward src pass: the gathered table is g' (fresh, ld H*D); ft and grad_ft only constrain the vector width
    vw, gsh, vpl, parts = choose_tiling(H, D, H * D, 0, H * D, ft_ptr, 1, n_dst, env)
    assert parts == 1
    need_gz = c["er"] or c["ee"]
    gz_e = direct and need_gz
    by_eid = direct and has_edge_ops
    rw = rowwise_geometry(H, D)
    lowdeg = use_lowdeg(E, n_src, True, env)
    if vw == 4 and not by_eid and not gz_e and rowwise_wanted(D, n_dst, E, n_src, True, env) and rw:
        bulk = env.get("BOTGAT_RW_BULK", "")[:1] != "0" and BULK_RING * (-(-H * D * 4 // 128) * 128) <= 96 * 1024
        src = f"botgat::gat_bwd_src_{'rowbulk' if bulk else 'rowwise'}_kernel<{rw[0]}, {rw[1]}>"
    elif (not lowdeg and env.get("BOTGAT_BWD_TMA", "")[:1] != "0" and vw == 4 and D % 8 == 0
          and (D // 4, 2 if (D // 4) % 4 == 0 and D // 4 <= 32 else 3) in TMA_COMBOS):
        dv = D // 4
        eb = not direct and (c["ee"] or c["keep"])
        am = not direct and c["attn_mul"]
        mode = 0 if (by_eid or gz_e) else (1 if (eb and need_gz and not am and not c["attn_p"]) else 2)
        src = f"botgat::gat_bwd_src_tma_kernel<{dv}, {2 if dv % 4 == 0 and dv <= 32 else 3}, {mode}>"
    elif lowdeg:
        src = f"botgat::gat_bwd_src_lowdeg_kernel<{vw}, {gsh}, {vpl}>"
    else:
        src = f"botgat::gat_bwd_src_kernel<{vw}, {gsh}, {vpl}>"
    return fwd[0], fwd[1], src


def normalise(name):
    """'void botgat::gat_fwd_kernel<4, 3, 3, false>(botgat::FwdParams)' -> 'botgat::gat_fwd_kernel<4,3,3,0>'; None for
    anything that is not a gather kernel."""
    m = re.search(r"(botgat::gat_(?:fwd|bwd)_\w*kernel)<([^>]*)>", name)
    if not m:
        return None
    args = [{"true": "1", "false": "0"}.get(a.strip(), a.strip()) for a in m.group(2).split(",")]
    return f"{m.group(1)}<{','.join(args)}>"


def binary_instantiations():
    """Gather-kernel instantiations compiled into the built library (cuobjdump from the toolkit of the Makefile's NVCC)."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cuobjdump = os.path.join(os.path.dirname(nvcc), "cuobjdump")
    if not os.path.exists(cuobjdump):
        cuobjdump = shutil.which("cuobjdump")
    assert cuobjdump, "cuobjdump not found next to nvcc"
    syms = subprocess.run([cuobjdump, "-symbols", LIB], check=True, capture_output=True, text=True).stdout
    mangled = sorted({w for w in syms.split() if w.startswith("_ZN6botgat") and "gat_" in w})
    demangled = subprocess.run(["c++filt"], input="\n".join(mangled), check=True, capture_output=True, text=True).stdout
    return {n for n in map(normalise, demangled.splitlines()) if n}


# ---------------------------------------------------------------------------
# inputs, runs and checks
# ---------------------------------------------------------------------------
def _degrees(rng, n, G, total=None):
    special = sorted({0, 1, max(G - 1, 0), G, G + 1, 31, 32, 33, 64, 65, 300})
    deg = np.concatenate([special, rng.integers(0, 13, size=n - len(special))]).astype(np.int64)
    return deg, len(special)


def make_inputs(c):
    """COO (sorted by (dst, src), so the canonical edge order is the edge-id order) whose in- and out-degrees both take
    the chunk and slot boundaries 0, 1, G-1, G, G+1, 31, 32, 33, 64, 65 and 300, plus the operands of case ``c``."""
    rng = np.random.default_rng(c["seed"])
    gen = torch.Generator().manual_seed(c["seed"])
    n_src, n_dst, H, D = c["n_src"], c["n_dst"], c["H"], c["D"]
    ind, ns_d = _degrees(rng, n_dst, c["Gdeg"])
    outd, ns_s = _degrees(rng, n_src, c["Gdeg"])
    diff = int(ind.sum() - outd.sum())   # balance the totals on the rows without a boundary degree
    np.add.at(outd if diff > 0 else ind, rng.integers(ns_s if diff > 0 else ns_d, n_src if diff > 0 else n_dst, abs(diff)), 1)
    dst = np.repeat(np.arange(n_dst), ind)
    src = rng.permutation(np.repeat(np.arange(n_src), outd))
    order = np.lexsort((src, dst))
    src, dst = src[order], dst[order]
    E = src.shape[0]
    d = {"src": torch.from_numpy(src), "dst": torch.from_numpy(dst), "n_src": n_src, "n_dst": n_dst, "E": E}
    d["ft"] = torch.randn(n_src, H, D, generator=gen)
    d["el"] = torch.randn(n_src, H, generator=gen)
    d["er"] = torch.randn(n_dst, H, generator=gen) if c["er"] else None
    d["ee"] = torch.randn(E, H, generator=gen) if c["ee"] else None
    d["keep"] = d["attn_mul"] = d["src_scale"] = d["dst_scale"] = None
    if c["keep"]:
        keep = torch.rand(E, generator=gen) >= 0.1
        keep[torch.from_numpy(dst == int(np.nonzero(ind == 33)[0][0]))] = False   # a row whose every in-edge is dropped
        d["keep"] = keep
    if c["attn_mul"]:
        d["attn_mul"] = (torch.rand(E, H, generator=gen) >= 0.15).float() / 0.85
    if c["attn_p"]:
        d["attn_mul"] = philox_attn_mul(c["attn_seed"], E, H, c["attn_p"])   # what the in-kernel dropout draws
    if c["symm"]:
        d["src_scale"] = torch.from_numpy(np.maximum(outd, 1) ** -0.5).float()
        d["dst_scale"] = torch.from_numpy(np.maximum(ind, 1) ** 0.5).float()
    d["gout"] = torch.randn(n_dst, H, D, generator=gen)
    d["res"] = torch.randn(n_dst, H * D, generator=gen)
    d["h_last"] = torch.randn(n_dst, H * D, generator=gen)
    d["scale"] = torch.rand(H * D, generator=gen) + 0.5
    d["shift"] = torch.randn(H * D, generator=gen)
    return d


def _dev(t, dev, grad=False):
    return None if t is None else t.to(dev).clone().requires_grad_(grad)


def run_train(c, d, dev, graph):
    """One forward + backward through ``gat_fused``; ft is a contiguous view at storage offset c["off"] floats."""
    from bot_b200.functional import gat_fused

    n = d["ft"].numel()
    buf = torch.empty(n + c["off"], device=dev)
    ft = buf[c["off"]:].view(d["ft"].shape)
    ft.copy_(d["ft"])
    ft.requires_grad_(True)
    assert ft.data_ptr() % 128 == 4 * c["off"]
    el, er, ee = _dev(d["el"], dev, True), _dev(d["er"], dev, True), _dev(d["ee"], dev, True)
    am = None if c["attn_p"] else _dev(d["attn_mul"], dev)
    out = gat_fused(graph, ft, el, er, ee, _dev(d["keep"], dev), am, _dev(d["src_scale"], dev), _dev(d["dst_scale"], dev),
                    0.2, c["attn_p"], c["attn_seed"])
    out.backward(d["gout"].to(dev))
    return {"out": out.detach(), "ft": ft.grad, "el": el.grad, "er": None if er is None else er.grad,
            "ee": None if ee is None else ee.grad}


def run_infer(c, d, dev, graph):
    """The same forward with the layer tail (residual, h_last, scale / shift, ReLU) fused into the kernel epilogue."""
    from bot_b200.functional import LayerTail, gat_fused_inference

    n = d["ft"].numel()
    buf = torch.empty(n + c["off"], device=dev)
    ft = buf[c["off"]:].view(d["ft"].shape)
    ft.copy_(d["ft"])
    norm = types.SimpleNamespace(weight=d["scale"].to(dev), bias=d["shift"].to(dev))
    tail = LayerTail(h_last=d["h_last"].to(dev), norm=norm, relu=True)
    return gat_fused_inference(graph, ft, _dev(d["el"], dev), _dev(d["er"], dev), _dev(d["ee"], dev), _dev(d["keep"], dev),
                               _dev(d["attn_mul"], dev), _dev(d["src_scale"], dev), _dev(d["dst_scale"], dev), 0.2, tail,
                               res=d["res"].to(dev))


def _check(name, got, want, tol, floor):
    assert got.shape == want.shape, (name, got.shape, want.shape)
    assert torch.isfinite(got).all(), f"{name}: non-finite values"
    e, r = rel_err(got, want), gat_rows.row_rel_err(got, want, floor)
    assert e <= tol, f"{name}: rel err {e:.3e} > {tol}"
    assert r <= tol, f"{name}: row-normalised err {r:.3e} > {tol} (floor {floor})"
    return e, r


# ---------------------------------------------------------------------------
# case table
# ---------------------------------------------------------------------------
# operand sets, used in rotation: (er, ee, keep, attn_mul, attn_p, symm)
OPERANDS = [
    dict(er=True, ee=True, keep=True, attn_mul=False, attn_p=0.0, symm=False),    # proteins: edge logits + edge drop
    dict(er=False, ee=False, keep=False, attn_mul=True, attn_p=0.0, symm=True),   # arxiv: symmetric norm, dropout mask
    dict(er=True, ee=False, keep=True, attn_mul=False, attn_p=0.1, symm=False),   # in-kernel Philox attention dropout
    dict(er=True, ee=False, keep=False, attn_mul=False, attn_p=0.0, symm=False),  # plain
]

# Head-major geometries (VW, GSH, VPL) -> (H, D, ft storage offset in floats, BOTGAT_VW, BOTGAT_NOALIGN, BOTGAT_G).
# Every one of the 60 is reached by both the warp-per-row and the group-per-row family.
HEAD_MAJOR = {
    (1, 0, 1): (2, 1, 2, 0, 0, 0), (1, 0, 2): (2, 2, 1, 0, 0, 1), (1, 1, 1): (2, 2, 1, 0, 0, 0),
    (1, 1, 2): (2, 3, 2, 0, 0, 1), (1, 2, 1): (3, 4, 0, 1, 0, 0), (1, 2, 2): (2, 8, 1, 0, 0, 1),
    (1, 3, 1): (2, 8, 1, 0, 0, 0), (1, 3, 2): (2, 9, 2, 0, 0, 1), (1, 4, 1): (12, 9, 0, 0, 0, 0),
    (1, 4, 2): (2, 17, 2, 0, 0, 1), (1, 5, 1): (2, 8, 1, 0, 0, 32), (1, 5, 2): (2, 33, 2, 0, 0, 0),
    (1, 5, 3): (3, 68, 0, 1, 1, 0), (1, 5, 4): (2, 97, 2, 0, 0, 0), (1, 5, 5): (2, 129, 2, 0, 0, 0),
    (1, 5, 6): (1, 161, 0, 0, 0, 0), (1, 5, 7): (2, 193, 2, 0, 0, 0), (1, 5, 8): (1, 225, 0, 0, 0, 0),
    (2, 0, 1): (2, 2, 2, 0, 0, 0), (2, 0, 2): (2, 4, 2, 0, 0, 1), (2, 1, 1): (2, 4, 2, 0, 0, 0),
    (2, 1, 2): (2, 8, 2, 0, 0, 1), (2, 2, 1): (12, 6, 0, 0, 0, 0), (2, 2, 2): (2, 10, 2, 0, 0, 1),
    (2, 3, 1): (2, 12, 0, 2, 1, 0), (2, 3, 2): (2, 18, 2, 0, 0, 1), (2, 4, 1): (2, 8, 2, 0, 0, 16),
    (2, 4, 2): (2, 34, 2, 0, 0, 0), (2, 4, 3): (2, 66, 2, 0, 0, 0), (2, 4, 4): (3, 100, 0, 2, 0, 0),
    (2, 4, 5): (2, 130, 2, 0, 0, 0), (2, 4, 6): (2, 162, 2, 0, 0, 0), (2, 4, 7): (2, 194, 2, 0, 0, 0),
    (2, 4, 8): (1, 226, 0, 0, 0, 0), (2, 5, 5): (2, 8, 2, 0, 0, 32), (2, 5, 6): (1, 322, 2, 0, 0, 0),
    (2, 5, 7): (1, 386, 2, 0, 0, 0), (2, 5, 8): (1, 450, 2, 0, 0, 0),
    (4, 0, 1): (2, 4, 0, 0, 0, 0), (4, 0, 2): (2, 8, 0, 0, 0, 1), (4, 1, 1): (2, 8, 0, 0, 0, 0),
    (4, 1, 2): (2, 12, 0, 0, 0, 1), (4, 2, 1): (12, 12, 0, 0, 0, 0), (4, 2, 2): (2, 20, 0, 0, 0, 1),
    (4, 3, 1): (2, 8, 0, 0, 0, 8), (4, 3, 2): (12, 36, 0, 0, 0, 0), (4, 3, 3): (6, 80, 0, 0, 0, 0),
    (4, 3, 4): (2, 100, 0, 0, 0, 0), (4, 3, 5): (2, 132, 0, 0, 0, 0), (4, 3, 6): (2, 164, 0, 0, 0, 0),
    (4, 3, 7): (2, 196, 0, 0, 0, 0), (4, 3, 8): (2, 228, 0, 0, 0, 0), (4, 4, 5): (2, 8, 0, 0, 0, 16),
    (4, 4, 6): (1, 324, 0, 0, 0, 0), (4, 4, 7): (1, 388, 0, 0, 0, 0), (4, 4, 8): (1, 452, 0, 0, 0, 0),
    (4, 5, 5): (2, 8, 0, 0, 0, 32), (4, 5, 6): (1, 644, 0, 0, 0, 0), (4, 5, 7): (1, 772, 0, 0, 0, 0),
    (4, 5, 8): (1, 900, 0, 0, 0, 0),
}

# all-heads-per-row geometries (GSH, VPL): 32 / 2**GSH lanes per head -> (H, D)
ROWWISE = {}
for _gsh, _heads in ((5, (1,)), (4, (2,)), (3, (3, 4)), (2, (5, 6, 7, 8))):
    for _vpl in range(1, 9):
        _H = _heads[_vpl % len(_heads)]
        _cols = 4 << _gsh                       # columns one slot of a head's lanes covers
        ROWWISE[(_gsh, _vpl)] = (_H, _cols * _vpl - (4 if _vpl % 2 else 0))   # odd slot counts: a ragged last slot

TMA_WIDTHS = (16, 32, 48, 64, 80, 96, 128, 40, 120, 160)


def _case(i, family, H, D, off=0, vw=0, noalign=0, G=0, env=None, ops=None, block=None, edge_mode="staged"):
    ops = dict(OPERANDS[i % len(OPERANDS)] if ops is None else ops)
    block = (i % 3 == 0) if block is None else block
    e = {"BOTGAT_VW": str(vw) if vw else "", "BOTGAT_NOALIGN": "1" if noalign else "", "BOTGAT_G": str(G) if G else ""}
    e.update(env or {})
    gdeg = G or 8
    return dict(family=family, H=H, D=D, off=off, env={k: v for k, v in e.items() if v}, edge_mode=edge_mode,
                n_src=400 if block else 320, n_dst=150 if block else 320, Gdeg=gdeg, seed=1000 + i, attn_seed=77 + i, **ops)


def build_cases():
    cases = {}
    for i, (geo, (H, D, off, vw, noal, G)) in enumerate(sorted(HEAD_MAJOR.items())):
        mode = "direct" if i % 5 == 4 else "staged"
        base = dict(H=H, D=D, off=off, vw=vw, noalign=noal, G=G, edge_mode=mode)
        cases[f"warp_{geo[0]}_{geo[1]}_{geo[2]}"] = _case(i, "warp", env={"BOTGAT_LOWDEG": "0", "BOTGAT_BWD_TMA": "0",
                                                                          "BOTGAT_ROWWISE": "0"}, **base)
        cases[f"group_{geo[0]}_{geo[1]}_{geo[2]}"] = _case(i, "group", env={"BOTGAT_LOWDEG": "1000000",
                                                                                "BOTGAT_ROWWISE": "0"}, **base)
    for i, (geo, (H, D)) in enumerate(sorted(ROWWISE.items())):
        for bulk in ("1", "0"):
            cases[f"rowwise_{geo[0]}_{geo[1]}_bulk{bulk}"] = _case(i + int(bulk), "rowwise", H, D, off=4 * (i % 2),
                                                                  env={"BOTGAT_ROWWISE": "1", "BOTGAT_RW_BULK": bulk})
    for i, D in enumerate(TMA_WIDTHS):
        H = (1, 2, 3, 6)[i % 4]
        for mode, ops, em in ((0, OPERANDS[0], "direct"), (1, OPERANDS[0], "staged"), (2, OPERANDS[2 - i % 2], "staged")):
            cases[f"tma_D{D}_mode{mode}"] = _case(3 * i + mode, "tma", H, D, ops=ops, edge_mode=em,
                                                 env={"BOTGAT_LOWDEG": "0", "BOTGAT_ROWWISE": "0"})
    # a forward split into column parts (a tiny L2 budget per slab); the backward covers the head in one part
    cases["colparts_H1_D512"] = dict(_case(7, "warp", 1, 512, block=False, env={
        "BOTGAT_LOWDEG": "0", "BOTGAT_ROWWISE": "0", "BOTGAT_BWD_TMA": "0", "BOTGAT_SLAB_MB": "1"}), n_src=600, n_dst=600)
    return cases


CASES = build_cases()
_state = {"ran": set(), "passed": set(), "t0": None}


# ---------------------------------------------------------------------------
# fixtures and tests
# ---------------------------------------------------------------------------
@pytest.fixture
def trace():
    """trace(fn) runs fn() under torch.profiler (CUDA activity) and returns the normalised names of the gather kernels
    it launched."""
    from torch.profiler import ProfilerActivity, profile

    def run(fn):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            res = fn()
            torch.cuda.synchronize()
        names = {n for n in (normalise(e.name) for e in prof.events()) if n}
        return names, res

    return run


@pytest.fixture
def knobs(monkeypatch):
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)
    return monkeypatch


def test_trace_sees_library_launches(cuda, trace, knobs):
    """The profiler sees the library's launches (made through ctypes): a proteins-like layer runs gat_fwd_kernel<4,3,3>."""
    import bot_b200
    from util import make_case

    from bot_b200.functional import gat_fused

    c = make_case(400, 400, 30000, 6, 80, ee=True, keep_p=0.1, seed=0)
    g = bot_b200.Graph(c["src"].to(cuda), c["dst"].to(cuda), 400)
    names, _ = trace(lambda: gat_fused(g, c["ft"].to(cuda), c["el"].to(cuda), c["er"].to(cuda), c["ee"].to(cuda),
                                       c["keep"].to(cuda)))
    assert normalise("botgat::gat_fwd_kernel<4, 3, 3, false>") in names, sorted(names)


_oracle_cache = {}


def _oracle(c, d):
    key = (c["seed"], c["H"], c["D"], c["n_src"], c["n_dst"])   # the warp / group pair of a geometry shares its inputs
    if key not in _oracle_cache:
        _oracle_cache.clear()
        ref_out, ref_g = oracle_run(d)
        ref_h = ref_out.reshape(c["n_dst"], -1) + d["res"].double() + d["h_last"].double()
        ref_y = torch.relu(ref_h * d["scale"].double() + d["shift"].double())
        _oracle_cache[key] = (ref_out, ref_g, ref_h, ref_y)
    return _oracle_cache[key]


@pytest.mark.parametrize("name", list(CASES))
def test_instantiation(cuda, trace, knobs, name):
    """One case: the predicted forward / src-pass instantiations run (and only they), and match the fp64 oracle."""
    import bot_b200
    from bot_b200 import functional

    if _state["t0"] is None:
        _state["t0"] = time.time()
    _state["ran"].add(name)
    c = dict(CASES[name])
    for k, v in c["env"].items():
        knobs.setenv(k, v)
    knobs.setattr(functional, "edge_mode", c["edge_mode"])
    d = make_inputs(c)
    c["E"] = d["E"]
    f_train, f_infer, src = (normalise(k) for k in expected_kernels(c, c["env"], c["edge_mode"]))
    g = bot_b200.Graph(d["src"].to(cuda), d["dst"].to(cuda), c["n_src"], c["n_dst"], is_block=c["n_src"] != c["n_dst"])
    assert g.edge_perm() is None   # the COO is in canonical order: per-edge operands need no permutation

    names, got = trace(lambda: run_train(c, d, cuda, g))
    assert names == {f_train, src}, f"training launched {sorted(names)}, expected {sorted({f_train, src})}"
    names_i, (h, y) = trace(lambda: run_infer(c, d, cuda, g))
    assert names_i == {f_infer}, f"inference launched {sorted(names_i)}, expected {f_infer}"

    ref_out, ref_g, ref_h, ref_y = _oracle(c, d)
    _check(f"out of {f_train}", got["out"], ref_out, FWD_TOL, 1e-3)
    for k in ("ft", "el", "er", "ee"):
        if ref_g[k] is None:
            assert got[k] is None, k
        else:
            _check(f"grad_{k} of {f_train} + {src}", got[k], ref_g[k], GRAD_TOL, 1e-2)
    _check(f"h (fused tail) of {f_infer}", h, ref_h, FWD_TOL, 1e-3)
    _check(f"y (fused tail) of {f_infer}", y, ref_y, FWD_TOL, 1e-3)

    again = run_train(c, d, cuda, g)
    torch.cuda.synchronize()
    for k, v in got.items():
        assert v is None or torch.equal(v, again[k]), f"{k}: a rerun is not bit-identical"
    _state["passed"].add(name)
    _state.setdefault("kernels", set()).update({f_train, f_infer, src})


def test_coverage_of_every_instantiation():
    """Last in the file: the passing cases together ran every gather instantiation of the built library."""
    if len(_state["ran"]) < len(CASES):
        pytest.skip("only part of the case table ran (-k / deselection)")
    have = binary_instantiations()
    ran = _state.get("kernels", set())
    missing = sorted(have - ran)
    extra = sorted(ran - have)
    took = time.time() - _state["t0"]
    print(f"\n{len(have & ran)}/{len(have)} gather instantiations ran and matched the fp64 oracle "
          f"({len(_state['passed'])}/{len(CASES)} cases, {took:.0f} s)")
    assert not extra, f"traced kernels the binary does not list: {extra}"
    assert not missing, f"{len(missing)} instantiations never ran in a passing case:\n" + "\n".join(missing)
