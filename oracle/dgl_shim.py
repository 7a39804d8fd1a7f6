"""Minimal stand-in for the DGL 0.5 API surface the reference touches — TEST
INFRASTRUCTURE ONLY.

DGL 0.5.* (README.md:9 of the reference) is not installable offline, so the
reference's ``models.py`` files cannot be imported as they are.  ``install()``
registers a fake ``dgl`` package in ``sys.modules`` whose graph object implements —
in plain differentiable torch ops on CPU — exactly the calls the reference's
``GATConv``/``GAT`` make (SURVEY.md section 2b K1-K13, Appendix B).  With it,
``tests/golden/make_golden.py`` imports the UNMODIFIED reference modules from a
reference checkout and records their outputs, so the reference's own orchestration
(aliasing before scaling, +0.5 exponent, in-place adds, randperm edge-drop ...)
is what the golden vectors pin; only the DGL primitives are restated here.
"""
from __future__ import annotations

import contextlib
import sys
import types

import torch

from . import gat_ref

ALL = "__ALL__"


class DGLError(Exception):
    pass


# ---- dgl.function descriptors -------------------------------------------------
class _Msg:
    def __init__(self, kind, a, b, out):
        self.kind, self.a, self.b, self.out = kind, a, b, out


class _Red:
    def __init__(self, kind, msg, out):
        self.kind, self.msg, self.out = kind, msg, out


def u_add_v(lhs, rhs, out):
    return _Msg("u_add_v", lhs, rhs, out)


def u_mul_e(lhs, rhs, out):
    return _Msg("u_mul_e", lhs, rhs, out)


def copy_u(u, out):
    return _Msg("copy_u", u, None, out)


def copy_src(src, out):
    return _Msg("copy_u", src, None, out)


def copy_e(e, out):
    return _Msg("copy_e", e, None, out)


def fsum(msg, out):
    return _Red("sum", msg, out)


class ShimGraph:
    """The DGLGraph subset of SURVEY.md section 8b ('graph argument protocol')."""

    def __init__(self, src, dst, n_src, n_dst=None, is_block=False):
        self._src = torch.as_tensor(src, dtype=torch.int64)
        self._dst = torch.as_tensor(dst, dtype=torch.int64)
        self._n_src = int(n_src)
        self._n_dst = int(n_src if n_dst is None else n_dst)
        self.is_block = bool(is_block)
        self.edata = {}
        if self.is_block or self._n_src != self._n_dst:
            self.srcdata, self.dstdata = {}, {}
            self.ndata = self.srcdata
        else:
            self.ndata = {}
            self.srcdata = self.dstdata = self.ndata

    device = torch.device("cpu")

    @contextlib.contextmanager
    def local_scope(self):
        saved = [dict(d) for d in (self.srcdata, self.dstdata, self.edata)]
        try:
            yield
        finally:
            for d, s in zip((self.srcdata, self.dstdata, self.edata), saved):
                d.clear()
                d.update(s)

    def edges(self, order="eid"):
        return self._src, self._dst

    def number_of_edges(self):
        return self._src.numel()

    def number_of_nodes(self):
        return self._n_src

    def number_of_src_nodes(self):
        return self._n_src

    def number_of_dst_nodes(self):
        return self._n_dst

    def in_degrees(self):
        return torch.bincount(self._dst, minlength=self._n_dst)

    def out_degrees(self):
        return torch.bincount(self._src, minlength=self._n_src)

    def to(self, device):
        return self

    def cpu(self):
        return self

    def create_formats_(self):
        return None

    def apply_edges(self, m):
        if m.kind == "u_add_v":
            self.edata[m.out] = self.srcdata[m.a].index_select(0, self._src) + \
                self.dstdata[m.b].index_select(0, self._dst)
        elif m.kind == "copy_u":
            self.edata[m.out] = self.srcdata[m.a].index_select(0, self._src)
        else:
            raise DGLError(m.kind)

    def update_all(self, m, r):
        if r.kind != "sum":
            raise DGLError(r.kind)
        if m.kind == "u_mul_e":
            msg = self.srcdata[m.a].index_select(0, self._src) * self.edata[m.b]
        elif m.kind == "copy_u":
            msg = self.srcdata[m.a].index_select(0, self._src)
        elif m.kind == "copy_e":
            msg = self.edata[m.a]
        else:
            raise DGLError(m.kind)
        out = torch.zeros((self._n_dst,) + tuple(msg.shape[1:]), dtype=msg.dtype)
        self.dstdata[r.out] = out.index_add(0, self._dst, msg)


def edge_softmax(graph, e, eids=ALL, norm_by="dst"):
    """DGL 0.5 ``dgl.ops.edge_softmax``; with ``eids`` the softmax runs over the
    edge-induced subgraph and returns ``len(eids)`` rows in ``eids`` order."""
    assert norm_by == "dst"
    dst = graph._dst if isinstance(eids, str) else graph._dst.index_select(0, eids)
    return gat_ref.edge_softmax(dst, e, graph._n_dst)


def expand_as_pair(in_feats, g=None):
    if isinstance(in_feats, tuple):
        return in_feats
    return in_feats, in_feats


def install():
    """Register the fake ``dgl`` package.  Idempotent."""
    if "dgl" in sys.modules and getattr(sys.modules["dgl"], "__botgat_shim__", False):
        return sys.modules["dgl"]

    def mod(name):
        m = types.ModuleType(name)
        sys.modules[name] = m
        return m

    dgl = mod("dgl")
    dgl.__botgat_shim__ = True
    fn = mod("dgl.function")
    fn.u_add_v, fn.u_mul_e, fn.copy_u, fn.copy_src, fn.copy_e, fn.sum = \
        u_add_v, u_mul_e, copy_u, copy_src, copy_e, fsum
    dgl.function = fn
    nn_ = mod("dgl.nn")
    nnpt = mod("dgl.nn.pytorch")
    nnutils = mod("dgl.nn.pytorch.utils")
    nnutils.Identity = torch.nn.Identity
    nn_.pytorch = nnpt
    nnpt.utils = nnutils
    dgl.nn = nn_
    ffi = mod("dgl._ffi")
    ffibase = mod("dgl._ffi.base")
    ffibase.DGLError = DGLError
    ffi.base = ffibase
    dgl._ffi = ffi
    base = mod("dgl.base")
    base.ALL, base.DGLError = ALL, DGLError
    dgl.base = base
    ops = mod("dgl.ops")
    ops.edge_softmax = edge_softmax
    dgl.ops = ops
    utils = mod("dgl.utils")
    utils.expand_as_pair = expand_as_pair
    dgl.utils = utils
    dgl.DGLError = DGLError
    return dgl


def import_reference(which):
    """Import an unmodified reference ``models.py`` ('no-sampling', 'ogbn-proteins',
    'ogbn-products') of the reference checkout named by ``BOT_REFERENCE`` under a unique module name."""
    import importlib.util
    import os

    root = os.environ.get("BOT_REFERENCE")
    if not root:
        raise RuntimeError("set BOT_REFERENCE to a checkout of the reference (AiRyunn/BoT)")
    install()
    path = os.path.join(root, "src", which, "models.py")
    spec = importlib.util.spec_from_file_location(f"_bot_ref_{which.replace('-', '_')}", path)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    torch.set_printoptions(profile="default")  # reference sets precision=20 at import
    return m
