"""Device-side graph handle: what ``data.edge_index`` is in the reference (a symmetric
``torch_sparse.SparseTensor``, utils.py:70-71), plus the derived index arrays the conv
kernels use (built once instead of on every forward, cf. layers.py:41-54 and PyG's set_diag).
"""
from __future__ import annotations

import torch

from . import _native as N
from .ops import _addr, _cuda, _stream


class _Storage:
    """``SparseTensor.storage`` look-alike (``rowptr()/col()/value()/row()``)."""

    def __init__(self, g):
        self._g = g

    def rowptr(self):
        return self._g.rowptr

    def col(self):
        return self._g.col

    def value(self):
        return self._g.value

    def row(self):
        counts = self._g.rowptr[1:] - self._g.rowptr[:-1]
        return torch.repeat_interleave(torch.arange(self._g.n, device=self._g.col.device), counts)


class CSRGraph:
    """Symmetric CSR graph on the GPU.

    ``rowptr`` int64[n+1], ``col`` int64[nnz], ``value`` f32[nnz] are the reference-visible
    arrays (bit-exact with ``load_input``); everything else is derived lazily and cached.
    """

    def __init__(self, rowptr: torch.Tensor, col: torch.Tensor, value: torch.Tensor, n: int):
        _cuda(rowptr, col, value)
        self.rowptr, self.col, self.value, self.n = rowptr.contiguous(), col.contiguous(), value.contiguous(), int(n)
        self.nnz = int(col.numel())
        self.storage = _Storage(self)
        self._cache: dict = {}
        self.block: tuple[int, int] | None = None  # (g0, g1) of a row-block view, see row_block

    # -- SparseTensor-like surface ------------------------------------------------
    def sizes(self):
        return [self.n, self.n]

    def sparse_sizes(self):
        return (self.n, self.n)

    @property
    def device(self):
        return self.col.device

    @classmethod
    def from_edge_index(cls, edge_index: torch.Tensor, edge_weight: torch.Tensor | None, n: int):
        """``forward(x, edge_index, edge_weight)`` with a ``[2,E]`` LongTensor: sort row-major
        (what SparseTensor's constructor does).  The pattern must be symmetric and duplicate-free (what
        ``load_input`` produces); that is checked when the conv layers derive their index arrays."""
        _cuda(edge_index)
        row, col = edge_index[0].long(), edge_index[1].long()
        if edge_weight is None:
            edge_weight = torch.ones(row.numel(), dtype=torch.float32, device=row.device)
        order = torch.argsort(row * n + col, stable=True)
        row, col, val = row[order], col[order], edge_weight.float()[order]
        rowptr = torch.zeros(n + 1, dtype=torch.int64, device=row.device)
        rowptr[1:] = torch.cumsum(torch.bincount(row, minlength=n), 0)
        return cls(rowptr, col, val, n)

    def row_block(self, g0: int, g1: int) -> "CSRGraph":
        """View of target rows ``[g0, g1)`` for a GNN whose rows are sharded across GPUs: the conv layers given it take the
        full input ``x [n, F]`` and return the block's ``g1 - g0`` rows (CSR kernels only).  It shares this graph's arrays and
        its cache of derived index arrays, so blocks of one graph build them once."""
        g0, g1 = int(g0), int(g1)
        if not 0 <= g0 <= g1 <= self.n:
            raise ValueError(f"CSRGraph.row_block: need 0 <= g0 <= g1 <= n = {self.n}, got [{g0}, {g1})")
        view = object.__new__(CSRGraph)
        view.__dict__.update(self.__dict__)
        view.storage = _Storage(view)
        view.block = (g0, g1)
        return view

    @property
    def rows(self) -> tuple[int, int]:
        """(g0, g1): the target rows the conv layers produce, ``(0, n)`` unless this is a row-block view."""
        return self.block if self.block is not None else (0, self.n)

    def block_entries(self) -> tuple[int, int]:
        """(e0, e1): the block's entries ``[rowptr[g0] + g0, rowptr[g1] + g1)`` in the self-loop pattern (read once, cached)."""
        g0, g1 = self.rows
        return self._get(("block_entries", g0, g1), lambda: tuple(int(v) + g for v, g in zip(self.rowptr[[g0, g1]].tolist(), (g0, g1))))

    # -- derived arrays -----------------------------------------------------------
    def _get(self, key, builder):
        if key not in self._cache:
            self._cache[key] = builder()
        return self._cache[key]

    def i32(self):
        """(rowptr32, col32) of the stored pattern."""

        def build():
            r32 = torch.empty(self.n + 1, dtype=torch.int32, device=self.device)
            c32 = torch.empty(max(self.nnz, 1), dtype=torch.int32, device=self.device)
            N.check(N.lib().hicgat_csr_pack_i32(self.rowptr.data_ptr(), self.col.data_ptr(), self.n, self.nnz, r32.data_ptr(), c32.data_ptr(), _stream()), "hicgat_csr_pack_i32")
            return r32, c32[: self.nnz]

        return self._get("i32", build)

    def with_self_loops(self):
        """(rowptr32, col32, perm32) of set_diag(pattern); perm = transposed-entry index."""

        def build():
            r32, c32 = self.i32()
            if self.nnz and bool((self.storage.row() == self.col).any()):
                raise RuntimeError("CSRGraph.with_self_loops: the stored pattern already has diagonal entries")
            orow = torch.empty(self.n + 1, dtype=torch.int32, device=self.device)
            ocol = torch.empty(self.nnz + self.n, dtype=torch.int32, device=self.device)
            N.check(N.lib().hicgat_csr_add_self_loops_i32(r32.data_ptr(), _addr(c32), self.n, orow.data_ptr(), ocol.data_ptr(), _stream()), "hicgat_csr_add_self_loops_i32")
            perm = torch.empty(self.nnz + self.n, dtype=torch.int32, device=self.device)
            N.check(N.lib().hicgat_csr_transpose_perm(orow.data_ptr(), ocol.data_ptr(), self.n, perm.data_ptr(), _stream()), "hicgat_csr_transpose_perm")
            _check_transpose_perm(perm, "CSRGraph.with_self_loops")
            return orow, ocol, perm

        return self._get("self_loops", build)

    def density(self) -> float:
        """Fraction of all ordered pairs (incl. self loops) that are edges of the GAT pattern."""
        return (self.nnz + self.n) / float(self.n * self.n)

    def dense_mask(self):
        """Bit mask u32[n, ceil(n/32)] of the self-loop pattern for the dense-tile GAT path."""

        def build():
            r32, c32, _ = self.with_self_loops()
            words = (self.n + 31) // 32
            mask = torch.empty(self.n, words, dtype=torch.int32, device=self.device)
            N.check(N.lib().hicgat_gat_dense_build_mask(r32.data_ptr(), c32.data_ptr(), self.n, mask.data_ptr(), _stream()), "hicgat_gat_dense_build_mask")
            return mask

        return self._get("dense_mask", build)

    def sage_weights(self):
        """(norm_val, norm_val_t): D^-1 A values (layers.py:41-54) and their transposed-entry
        gather, both f32[nnz] in CSR order; built once."""

        def build():
            r32, c32 = self.i32()
            colsum = torch.empty(self.n, dtype=torch.float32, device=self.device)
            norm = torch.empty(max(self.nnz, 1), dtype=torch.float32, device=self.device)
            N.check(N.lib().hicgat_sage_norm_values(r32.data_ptr(), _addr(c32), _addr(self.value), self.n, colsum.data_ptr(), norm.data_ptr(), _stream()), "hicgat_sage_norm_values")
            perm = torch.empty(max(self.nnz, 1), dtype=torch.int32, device=self.device)
            N.check(N.lib().hicgat_csr_transpose_perm(r32.data_ptr(), _addr(c32), self.n, perm.data_ptr(), _stream()), "hicgat_csr_transpose_perm")
            norm = norm[: self.nnz]
            _check_transpose_perm(perm[: self.nnz], "CSRGraph.sage_weights")
            return norm, norm[perm[: self.nnz].long()].contiguous()

        return self._get("sage", build)


def _check_transpose_perm(perm: torch.Tensor, what: str) -> None:
    """The backward kernels index ``alpha[perm]`` / ``dz[perm]``: every stored entry (i, j) needs its
    transposed entry (j, i) exactly once.  ``hicgat_csr_transpose_perm`` writes -1 where (j, i) is missing;
    duplicates break the involution.  One host read at graph-build time (the build already syncs)."""
    if perm.numel() == 0:
        return
    p = perm.long()
    if bool((p < 0).any()):
        raise RuntimeError(f"{what}: the edge pattern is not symmetric (an entry (i, j) has no (j, i)); "
                           "the conv backward kernels need a symmetric pattern, as utils.load_input builds it")
    if not bool((p[p] == torch.arange(p.numel(), device=p.device)).all()):
        raise RuntimeError(f"{what}: the edge pattern holds duplicate entries; coalesce the edge list first")


def as_graph(edge_index, edge_weight=None, n: int | None = None) -> CSRGraph:
    """Accept what the reference's models accept as ``edge_index``: a CSR handle (ours, or
    anything SparseTensor-like with ``.storage.rowptr()/col()/value()``), or a ``[2,E]``
    LongTensor with optional ``edge_weight``."""
    if isinstance(edge_index, CSRGraph):
        return edge_index
    if hasattr(edge_index, "storage") and hasattr(edge_index.storage, "rowptr"):
        st = edge_index.storage
        sizes = edge_index.sizes()
        return CSRGraph(st.rowptr().cuda(), st.col().cuda(), st.value().cuda().float(), sizes[0])
    if torch.is_tensor(edge_index) and edge_index.dim() == 2 and edge_index.shape[0] == 2:
        if n is None:
            raise RuntimeError("as_graph: need n for a [2,E] edge_index")
        return CSRGraph.from_edge_index(edge_index, edge_weight, n)
    raise TypeError(f"unsupported edge_index type {type(edge_index)}")
