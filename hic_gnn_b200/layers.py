"""Graph-conv layers of the hot path, same names / parameters / state_dict keys as the
reference (``layers.SAGEConv``: layers.py:12-83; PyG 1.7.2 ``GATConv`` as constructed at
models.py:619,1013), with the message passing done by the CSR kernels of conv.cu.

The dense projections (``lin_l``/``lin_r``) stay ``torch.nn.Linear`` (cuBLAS): they are plain
library GEMMs and not part of the rewritten subsystems (SURVEY.md section 8a-5).
"""
from __future__ import annotations

import math
import os

import torch
from torch import nn

from . import _native as N
from .graph import CSRGraph, _addr, as_graph
from . import ops as _ops
from .ops import _cuda, _stream


class _SageAggregate(torch.autograd.Function):
    """``matmul(D^-1 A, x)`` (layers.py:75-79); backward through the transposed weights."""

    @staticmethod
    def forward(ctx, x, graph: CSRGraph):
        _cuda(x)
        x = x.contiguous()
        r32, c32 = graph.i32()
        w, _ = graph.sage_weights()
        out = torch.empty_like(x)
        N.check(N.lib().hicgat_spmm_csr_f32(r32.data_ptr(), _addr(c32), _addr(w), x.data_ptr(), graph.n, x.shape[1], out.data_ptr(), _stream()), "hicgat_spmm_csr_f32")
        ctx.graph = graph
        return out

    @staticmethod
    def backward(ctx, g):
        graph = ctx.graph
        g = g.contiguous()
        r32, c32 = graph.i32()
        _, wt = graph.sage_weights()
        dx = torch.empty_like(g)
        N.check(N.lib().hicgat_spmm_csr_f32(r32.data_ptr(), _addr(c32), _addr(wt), g.data_ptr(), graph.n, g.shape[1], dx.data_ptr(), _stream()), "hicgat_spmm_csr_f32")
        return dx, None


def _sage_aggregate_rows(x, graph: CSRGraph):
    """Rows ``[g0, g1)`` of ``D^-1 A x`` for a row-block view of the graph (``x`` holds all rows).  No backward: ``x`` is the
    model input, which needs no gradient."""
    _cuda(x)
    if x.requires_grad:
        raise NotImplementedError("SAGEConv on a row block: the aggregation has no backward (its input x must not require grad)")
    x = x.contiguous().float()
    g0, g1 = graph.rows
    r32, c32 = graph.i32()
    w, _ = graph.sage_weights()
    out = torch.empty(g1 - g0, x.shape[1], dtype=torch.float32, device=x.device)
    N.check(N.lib().hicgat_spmm_csr_rows_f32(r32.data_ptr(), _addr(c32), _addr(w), x.data_ptr(), graph.n, g0, g1, x.shape[1], _addr(out), _stream()),
            "hicgat_spmm_csr_rows_f32")
    return out


class SAGEConv(nn.Module):
    """``lin_l(D^-1 A x) + lin_r(trunc(x))`` -- layers.py:57-73, including the reference's
    ``x.long()`` truncation of the root features (layers.py:64; ``trunc_root=False`` disables
    the quirk).  ``reset_parameters`` is never called in the reference (layers.py:34), so the
    Linears keep ``nn.Linear``'s default init."""

    def __init__(self, in_channels: int, out_channels: int, normalize: bool = False, root_weight: bool = True, bias: bool = True, trunc_root: bool = True):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.normalize, self.root_weight, self.trunc_root = normalize, root_weight, trunc_root
        self.lin_l = _ops.Linear(in_channels, out_channels, bias=bias)
        if root_weight:
            self.lin_r = _ops.Linear(in_channels, out_channels, bias=False)

    def forward(self, x, edge_index, edge_attr=None, size=None):
        graph = as_graph(edge_index, edge_attr, x.shape[0])
        if graph.block is not None:  # row block: the block's rows of the aggregation and of the root term
            g0, g1 = graph.block
            out = _sage_aggregate_rows(x, graph)
            x = x[g0:g1]
        else:
            out = _SageAggregate.apply(x.float(), graph)
        out = self.lin_l(out)
        if self.root_weight:
            x_r = torch.trunc(x).float() if self.trunc_root else x.float()
            out = out + self.lin_r(x_r)
        if self.normalize:
            out = torch.nn.functional.normalize(out, p=2.0, dim=-1)
        return out

    def __repr__(self):
        return f"{self.__class__.__name__}({self.in_channels}, {self.out_channels})"


# CSR GAT backward: "fused" (one 2 KB-per-edge gather pass) or "split" (two passes); env HICGAT_GAT_BWD overrides
GAT_BACKWARD = os.environ.get("HICGAT_GAT_BWD", "fused")

# (heads, channels per head) the GAT kernels are compiled for, on both message-passing paths (conv.cu HICGAT_DISPATCH_HQ)
GAT_SHAPES = ((1, 128), (1, 256), (1, 512), (2, 128), (2, 256), (2, 512), (4, 128), (4, 256))


def gat_shape_supported(heads: int, channels: int) -> bool:
    return (heads, channels) in GAT_SHAPES


class _GatWorkspace:
    _cache: dict = {}

    @classmethod
    def get(cls, device, n, nnz, heads, channels):
        key = (device.index, n, nnz, heads, channels)
        ws = cls._cache.get(key)
        if ws is None:
            need = N.lib().hicgat_gat_bwd_workspace_bytes(n, nnz, heads, channels)
            if need == 0:
                raise RuntimeError(f"GATConv kernels do not support heads={heads}, channels={channels}")
            ws = torch.zeros(need, dtype=torch.uint8, device=device)
            cls._cache[key] = ws
        return ws


class _GatAttend(torch.autograd.Function):
    """Per-edge LeakyReLU logits -> segmented softmax -> gather-SpMM (+ bias), and its
    backward in the same CSR order.  Saves O(N*H*C + nnz*H), never an [nnz,H,C] tensor."""

    @staticmethod
    def forward(ctx, xl, att_l, att_r, bias, graph: CSRGraph, heads: int, channels: int, slope: float):
        _cuda(xl)
        xl = xl.contiguous()
        att_l_f, att_r_f, bias_f = att_l.contiguous().view(-1), att_r.contiguous().view(-1), bias.contiguous()
        r32, c32, _ = graph.with_self_loops()
        n, nnz = graph.n, c32.numel()
        dev = xl.device
        a_src = torch.empty(n, heads, dtype=torch.float32, device=dev)
        a_dst = torch.empty(n, heads, dtype=torch.float32, device=dev)
        alpha = torch.empty(nnz, heads, dtype=torch.float32, device=dev)
        out = torch.empty(n, heads * channels, dtype=torch.float32, device=dev)
        N.check(
            N.lib().hicgat_gat_fwd(r32.data_ptr(), c32.data_ptr(), n, heads, channels, xl.data_ptr(), att_l_f.data_ptr(), att_r_f.data_ptr(), bias_f.data_ptr(), slope,
                                   a_src.data_ptr(), a_dst.data_ptr(), alpha.data_ptr(), out.data_ptr(), _stream()),
            "hicgat_gat_fwd",
        )
        ctx.save_for_backward(xl, att_l_f, att_r_f, bias_f, a_src, a_dst, alpha, out)
        ctx.graph, ctx.hc, ctx.slope, ctx.att_shape = graph, (heads, channels), slope, att_l.shape
        return out

    @staticmethod
    def backward(ctx, g):
        xl, att_l_f, att_r_f, bias_f, a_src, a_dst, alpha, out = ctx.saved_tensors
        graph, (heads, channels) = ctx.graph, ctx.hc
        g = g.contiguous()
        r32, c32, perm = graph.with_self_loops()
        n, nnz = graph.n, c32.numel()
        dxl = torch.empty_like(xl)
        datt_l, datt_r, dbias = torch.empty_like(att_l_f), torch.empty_like(att_r_f), torch.empty(heads * channels, dtype=torch.float32, device=xl.device)
        ws = _GatWorkspace.get(xl.device, n, nnz, heads, channels)
        if GAT_BACKWARD == "fused":  # one gather pass (default); "split" = the two-pass kernels, kept for A/B and as a cross-check
            N.check(
                N.lib().hicgat_gat_bwd_fused(r32.data_ptr(), c32.data_ptr(), perm.data_ptr(), n, nnz, heads, channels, xl.data_ptr(), att_l_f.data_ptr(), att_r_f.data_ptr(),
                                             bias_f.data_ptr(), ctx.slope, a_src.data_ptr(), a_dst.data_ptr(), alpha.data_ptr(), out.data_ptr(), g.data_ptr(), dxl.data_ptr(),
                                             datt_l.data_ptr(), datt_r.data_ptr(), dbias.data_ptr(), ws.data_ptr(), ws.numel(), _stream()),
                "hicgat_gat_bwd_fused",
            )
        else:
            N.check(
                N.lib().hicgat_gat_bwd(r32.data_ptr(), c32.data_ptr(), perm.data_ptr(), n, nnz, heads, channels, xl.data_ptr(), att_l_f.data_ptr(), att_r_f.data_ptr(), ctx.slope,
                                       a_src.data_ptr(), a_dst.data_ptr(), alpha.data_ptr(), g.data_ptr(), dxl.data_ptr(), datt_l.data_ptr(), datt_r.data_ptr(), dbias.data_ptr(),
                                       ws.data_ptr(), ws.numel(), _stream()),
                "hicgat_gat_bwd",
            )
        return dxl, datt_l.view(ctx.att_shape), datt_r.view(ctx.att_shape), dbias, None, None, None, None


class _GatAttendRows(torch.autograd.Function):
    """:class:`_GatAttend` on the target rows ``[g0, g1)`` of a row-block view: ``xl`` is the projection of ALL rows, the output
    the block's rows.  The backward returns PARTIAL gradients (``dxl`` on every row, the att / bias gradients) that, summed over a
    partition of the rows, are the full-graph gradients."""

    @staticmethod
    def forward(ctx, xl, att_l, att_r, bias, graph: CSRGraph, heads: int, channels: int, slope: float):
        _cuda(xl)
        xl = xl.contiguous()
        att_l_f, att_r_f, bias_f = att_l.contiguous().view(-1), att_r.contiguous().view(-1), bias.contiguous()
        r32, c32, _ = graph.with_self_loops()
        (g0, g1), (e0, e1) = graph.rows, graph.block_entries()
        n, dev = graph.n, xl.device
        a_src = torch.empty(n, heads, dtype=torch.float32, device=dev)
        a_dst = torch.empty(n, heads, dtype=torch.float32, device=dev)
        alpha = torch.empty(e1 - e0, heads, dtype=torch.float32, device=dev)
        out = torch.empty(g1 - g0, heads * channels, dtype=torch.float32, device=dev)
        N.check(
            N.lib().hicgat_gat_fwd_rows(r32.data_ptr(), c32.data_ptr(), n, g0, g1, e0, heads, channels, xl.data_ptr(), att_l_f.data_ptr(), att_r_f.data_ptr(),
                                        bias_f.data_ptr(), slope, a_src.data_ptr(), a_dst.data_ptr(), _addr(alpha), _addr(out), _stream()),
            "hicgat_gat_fwd_rows",
        )
        ctx.save_for_backward(xl, att_l_f, att_r_f, bias_f, a_src, a_dst, alpha, out)
        ctx.graph, ctx.hc, ctx.slope, ctx.att_shape = graph, (heads, channels), slope, att_l.shape
        return out

    @staticmethod
    def backward(ctx, g):
        xl, att_l_f, att_r_f, bias_f, a_src, a_dst, alpha, out = ctx.saved_tensors
        graph, (heads, channels) = ctx.graph, ctx.hc
        g = g.contiguous()
        r32, c32, perm = graph.with_self_loops()
        (g0, g1), (e0, _) = graph.rows, graph.block_entries()
        n, nnz = graph.n, c32.numel()
        dxl = torch.empty_like(xl)
        datt_l, datt_r, dbias = torch.empty_like(att_l_f), torch.empty_like(att_r_f), torch.empty(heads * channels, dtype=torch.float32, device=xl.device)
        ws = _GatWorkspace.get(xl.device, n, nnz, heads, channels)
        N.check(
            N.lib().hicgat_gat_bwd_fused_rows(r32.data_ptr(), c32.data_ptr(), perm.data_ptr(), n, nnz, g0, g1, e0, heads, channels, xl.data_ptr(), att_l_f.data_ptr(),
                                              att_r_f.data_ptr(), bias_f.data_ptr(), ctx.slope, a_src.data_ptr(), a_dst.data_ptr(), _addr(alpha), _addr(out), _addr(g),
                                              dxl.data_ptr(), datt_l.data_ptr(), datt_r.data_ptr(), dbias.data_ptr(), ws.data_ptr(), ws.numel(), _stream()),
            "hicgat_gat_bwd_fused_rows",
        )
        return dxl, datt_l.view(ctx.att_shape), datt_r.view(ctx.att_shape), dbias, None, None, None, None


class _GatAttendDense(torch.autograd.Function):
    """Dense-tile path of :class:`_GatAttend` for near-dense graphs (csrc/gat_dense.cu): the same
    attention, evaluated as register-tiled fp32 GEMMs whose attention tiles are regenerated from
    the logit halves, the row statistics and a bit mask of the pattern.  Saves O(N*H*C)."""

    @staticmethod
    def forward(ctx, xl, att_l, att_r, bias, graph: CSRGraph, heads: int, channels: int, slope: float):
        _cuda(xl)
        xl = xl.contiguous()
        att_l_f, att_r_f, bias_f = att_l.contiguous().view(-1), att_r.contiguous().view(-1), bias.contiguous()
        r32, c32, _ = graph.with_self_loops()
        mask = graph.dense_mask()
        n, dev, lib = graph.n, xl.device, N.lib()
        a_src = torch.empty(n, heads, dtype=torch.float32, device=dev)
        a_dst = torch.empty(n, heads, dtype=torch.float32, device=dev)
        out = torch.empty(n, heads * channels, dtype=torch.float32, device=dev)
        need = lib.hicgat_gat_dense_workspace_bytes(n, heads, channels)
        if need == 0:
            raise RuntimeError(f"dense GAT kernels do not support heads={heads}, channels={channels}")
        ws = torch.empty(need, dtype=torch.uint8, device=dev)  # holds the row statistics until backward
        s = _stream()
        N.check(lib.hicgat_gat_logits(n, heads, channels, xl.data_ptr(), att_l_f.data_ptr(), att_r_f.data_ptr(), a_src.data_ptr(), a_dst.data_ptr(), s), "hicgat_gat_logits")
        N.check(lib.hicgat_gat_dense_fwd(r32.data_ptr(), c32.data_ptr(), mask.data_ptr(), n, heads, channels, xl.data_ptr(), a_src.data_ptr(), a_dst.data_ptr(),
                                         bias_f.data_ptr(), slope, out.data_ptr(), ws.data_ptr(), ws.numel(), s), "hicgat_gat_dense_fwd")
        ctx.save_for_backward(xl, att_l_f, att_r_f, bias_f, a_src, a_dst, out, ws)
        ctx.graph, ctx.hc, ctx.slope, ctx.att_shape = graph, (heads, channels), slope, att_l.shape
        return out

    @staticmethod
    def backward(ctx, g):
        xl, att_l_f, att_r_f, bias_f, a_src, a_dst, out, ws = ctx.saved_tensors
        graph, (heads, channels) = ctx.graph, ctx.hc
        g = g.contiguous()
        n, dev, lib = graph.n, xl.device, N.lib()
        mask = graph.dense_mask()
        dxl = torch.empty_like(xl)
        d_src = torch.empty(n, heads, dtype=torch.float32, device=dev)
        d_dst = torch.empty(n, heads, dtype=torch.float32, device=dev)
        datt_l, datt_r = torch.empty_like(att_l_f), torch.empty_like(att_r_f)
        dbias = torch.empty(heads * channels, dtype=torch.float32, device=dev)
        s = _stream()
        N.check(lib.hicgat_gat_dense_bwd(mask.data_ptr(), n, heads, channels, xl.data_ptr(), a_src.data_ptr(), a_dst.data_ptr(), att_l_f.data_ptr(), att_r_f.data_ptr(),
                                         bias_f.data_ptr(), ctx.slope, out.data_ptr(), g.data_ptr(), dxl.data_ptr(), d_src.data_ptr(), d_dst.data_ptr(),
                                         ws.data_ptr(), ws.numel(), s), "hicgat_gat_dense_bwd")
        pws = torch.empty(lib.hicgat_gat_param_grads_workspace_bytes(n, heads, channels), dtype=torch.uint8, device=dev)
        N.check(lib.hicgat_gat_param_grads(n, heads, channels, xl.data_ptr(), g.data_ptr(), d_src.data_ptr(), d_dst.data_ptr(), datt_l.data_ptr(), datt_r.data_ptr(),
                                           dbias.data_ptr(), pws.data_ptr(), pws.numel(), s), "hicgat_gat_param_grads")
        return dxl, datt_l.view(ctx.att_shape), datt_r.view(ctx.att_shape), dbias, None, None, None, None


def _glorot_(t: torch.Tensor) -> None:
    s = math.sqrt(6.0 / (t.size(-2) + t.size(-1)))
    with torch.no_grad():
        t.uniform_(-s, s)


class GATConv(nn.Module):
    """torch-geometric 1.7.2 ``GATConv(in, C, heads=H, concat=True)`` on a SparseTensor input:
    one shared bias-free projection (``lin_r is lin_l``), self loops via ``set_diag``, edge
    values ignored, slope 0.2, softmax ``exp(e-max)/(sum+1e-16)``, no attention dropout.
    Parameter names and init (glorot / zeros, same RNG order) follow 1.7.2 so reference
    ``state_dict``s load unchanged."""

    def __init__(self, in_channels: int, out_channels: int, heads: int = 1, concat: bool = True, negative_slope: float = 0.2, dropout: float = 0.0, add_self_loops: bool = True, bias: bool = True):
        super().__init__()
        if not concat or dropout != 0.0 or not add_self_loops or not bias:
            raise NotImplementedError("only the configuration the reference uses: concat=True, dropout=0, add_self_loops=True, bias=True")
        if not gat_shape_supported(heads, out_channels):
            raise NotImplementedError(f"GATConv kernels support (heads, out_channels) in {', '.join(map(str, GAT_SHAPES))}; "
                                      f"got ({heads}, {out_channels})")
        self.in_channels, self.out_channels, self.heads, self.negative_slope = in_channels, out_channels, heads, negative_slope
        # message-passing path: "auto" = dense tiles when >= dense_threshold of all pairs are edges
        # (and the kernels support the shape), else the CSR warp-per-row kernels; "csr" / "dense" force one
        self.path, self.dense_threshold, self.dense_max_n = "auto", 0.35, 32768
        self.lin_l = _ops.Linear(in_channels, heads * out_channels, bias=False)
        self.lin_r = self.lin_l
        self.att_l = nn.Parameter(torch.empty(1, heads, out_channels))
        self.att_r = nn.Parameter(torch.empty(1, heads, out_channels))
        self.bias = nn.Parameter(torch.empty(heads * out_channels))
        self.reset_parameters()

    def reset_parameters(self):
        _glorot_(self.lin_l.weight)
        _glorot_(self.lin_r.weight)
        _glorot_(self.att_l)
        _glorot_(self.att_r)
        with torch.no_grad():
            self.bias.zero_()

    # torch-geometric >= 2.0 renamed the parameters (lin_src / lin_dst / att_src / att_dst, later a single `lin`);
    # checkpoints written there load into the 1.7.2 names the reference uses (SURVEY.md Appendix A.3)
    _PYG2_KEYS = {"lin_src.weight": "lin_l.weight", "lin_dst.weight": "lin_r.weight", "lin.weight": "lin_l.weight", "att_src": "att_l", "att_dst": "att_r"}

    def _load_from_state_dict(self, state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys, error_msgs):
        for new, old in self._PYG2_KEYS.items():
            if prefix + new in state_dict:
                state_dict.setdefault(prefix + old, state_dict.pop(prefix + new))
        l, r = prefix + "lin_l.weight", prefix + "lin_r.weight"   # one shared projection under two names (lin_r is lin_l)
        if l in state_dict and r not in state_dict:
            state_dict[r] = state_dict[l]
        elif r in state_dict and l not in state_dict:
            state_dict[l] = state_dict[r]
        super()._load_from_state_dict(state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys, error_msgs)

    def forward(self, x, edge_index, edge_weight=None, size=None):
        graph = as_graph(edge_index, edge_weight, x.shape[0])
        xl = self.lin_l(x)
        if graph.block is not None:  # row block: CSR kernels with the one-pass backward only
            if self.path == "dense":
                raise ValueError("GATConv: the dense-tile path has no row-block form; use path='csr' or 'auto' with a row-block graph")
            if GAT_BACKWARD != "fused":
                raise ValueError(f"GATConv: the {GAT_BACKWARD!r} backward has no row-block form; a row-block graph needs the fused backward")
            return _GatAttendRows.apply(xl, self.att_l, self.att_r, self.bias, graph, self.heads, self.out_channels, self.negative_slope)
        dense_ok = gat_shape_supported(self.heads, self.out_channels) and graph.n <= self.dense_max_n
        use_dense = self.path == "dense" or (self.path == "auto" and dense_ok and graph.n >= 256 and graph.density() >= self.dense_threshold)
        if use_dense and not dense_ok:
            raise RuntimeError(f"dense GAT path: needs at most dense_max_n = {self.dense_max_n} loci and (heads, channels) in {GAT_SHAPES}")
        fn = _GatAttendDense if use_dense else _GatAttend
        return fn.apply(xl, self.att_l, self.att_r, self.bias, graph, self.heads, self.out_channels, self.negative_slope)

    def __repr__(self):
        return f"{self.__class__.__name__}({self.in_channels}, {self.out_channels}, heads={self.heads})"
