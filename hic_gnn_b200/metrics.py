"""Evaluation metrics of the reference on the GPU (SURVEY.md section 8 row f-3, "next").

``dscc`` is the reference's headline accuracy number: the Spearman correlation between the
strict-upper-triangle wish distances and the reconstructed pairwise distances
(``scipy.stats.spearmanr``, HiC-GNN_main.py:135-139, HiC_GAT_generalize_directly.py:242) with
AVERAGE ranks for ties -- every zero-contact pair has wish distance exactly 1.0, so ties are the
rule, not the exception.  The distances come from the library's pair-distance kernel; the rank
transform is sort-based torch glue (evaluation runs once per model, not per step).
:class:`DsccMeter` is the per-step form (the reference also evaluates ``spearmanr`` every iteration,
HiC_GAT_generalize_directly.py:242): histogram mid-ranks entirely on the device, graph-capturable.
"""
from __future__ import annotations

import torch

from . import ops


def average_ranks(v: torch.Tensor) -> torch.Tensor:
    """``scipy.stats.rankdata(v, method="average")`` as f64, on the device of ``v``."""
    sv, order = torch.sort(v)
    _, inverse, counts = torch.unique_consecutive(sv, return_inverse=True, return_counts=True)
    last = torch.cumsum(counts, 0).to(torch.float64)          # 1-based rank of the last member of each tie group
    avg = last - (counts.to(torch.float64) - 1.0) / 2.0
    ranks = torch.empty(v.numel(), dtype=torch.float64, device=v.device)
    ranks[order] = avg[inverse]
    return ranks


def _pearson(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    a = a - a.mean()
    b = b - b.mean()
    return (a * b).sum() / torch.sqrt((a * a).sum() * (b * b).sum())


def upper_pairs(coords: torch.Tensor, truth: torch.Tensor):
    """(dist_truth, dist_out) over i<j like the reference's ``triu_indices`` gathers
    (HiC_GAT_generalize_directly.py:210-214); ``truth`` is the dense N x N wish matrix (any float
    dtype) or a full-matrix :class:`ops.WishTarget`."""
    if isinstance(truth, ops.WishTarget):
        if truth.r0 != 0 or truth.r1 != truth.n:
            raise RuntimeError("dscc needs the full target (gather the row blocks first)")
        truth = truth.dense()
    n = truth.shape[0]
    idx = torch.triu_indices(n, n, 1, device=truth.device)
    d = ops.pairdist(coords.detach().float())
    return truth[idx[0], idx[1]], d[idx[0], idx[1]]


NBINS = 1 << 22      # histogram resolution of the streamed dSCC: rank error <= half a bin population, ~1e-7 relative
STREAM_FROM = 4096    # loci from which dscc() switches to the streamed evaluation (the exact one sorts P = N(N-1)/2 pairs)


def _midranks(hist: torch.Tensor) -> torch.Tensor:
    """Average rank (1-based, f64) of the members of every histogram bin, the bin being one tie group."""
    h = hist.to(torch.float64)
    below = torch.cumsum(h, 0) - h
    return below + (h + 1.0) / 2.0


def _spearman_from_tables(hist_d, hist_t, cross, npairs: float) -> float:
    hd, ht = hist_d.to(torch.float64), hist_t.to(torch.float64)
    rd, rt = _midranks(hist_d), _midranks(hist_t)
    mean = (npairs + 1.0) / 2.0                      # average ranks always sum to P(P+1)/2
    var_d = float((hd * (rd - mean) ** 2).sum())
    var_t = float((ht * (rt - mean) ** 2).sum())
    cov = float(cross) - npairs * mean * mean        # sum (rd - mean)(rt - mean) = sum rd rt - P mean^2
    return cov / (var_d * var_t) ** 0.5


def _implicit_target_ranks(tv: torch.Tensor, fill: float, npairs: float):
    """Average ranks of an implicit target's i<j values: ``tv`` (f64) holds the stored pairs, the other ``npairs - len(tv)`` pairs are
    ``fill``.  Returns (rank of every stored value, rank of the fill group, var_t = sum (rank - mean)^2 over all pairs), the last two as
    0-d device tensors."""
    n_stored = tv.numel()
    vals, inv, counts = torch.unique(torch.cat((tv, torch.tensor([float(fill)], dtype=torch.float64, device=tv.device))), return_inverse=True, return_counts=True)
    counts = counts.to(torch.float64)
    fill_slot = inv[-1]
    counts[fill_slot] += npairs - n_stored - 1.0   # the appended marker itself is not a pair
    below = torch.cumsum(counts, 0) - counts
    rank_vals = below + (counts + 1.0) / 2.0
    mean = (npairs + 1.0) / 2.0
    return rank_vals[inv[:-1]], rank_vals[fill_slot], (counts * (rank_vals - mean) ** 2).sum()


def dscc_streamed(coords: torch.Tensor, target, nbins: int = NBINS, reduce=None) -> float:
    """dSCC without the N x N distance matrix, the ``triu_indices`` gathers or a sort (``hicgat_rank_*``): two streaming passes over
    the target (dense :class:`ops.WishTarget`, any row block) or one compute-only pass plus O(nnz) work (implicit
    :class:`ops.SparseWishTarget`).  ``reduce(tensor)`` all-reduces in place when the target is row-sharded.  Ranks are histogram
    mid-ranks: within ~1e-7 of scipy's average ranks at the default resolution."""
    from . import _native as N

    c = coords.detach().float().contiguous()
    ops._cuda(c)
    n = c.shape[0]
    npairs = n * (n - 1) / 2.0
    dev = c.device
    span = (c.max(dim=0).values - c.min(dim=0).values).double()
    dmax = float(torch.sqrt((span * span).sum())) * (1.0 + 1e-6) + 1e-30   # bounding-box diagonal >= every pair distance
    d_scale = nbins / dmax
    hist_d = torch.zeros(nbins, dtype=torch.int64, device=dev)
    lib, st = N.lib(), ops._stream()
    if isinstance(target, ops.SparseWishTarget):
        r0, r1 = target.r0, target.r1
        N.check(lib.hicgat_dist_histogram(c.data_ptr(), n, r0, r1, d_scale, nbins, hist_d.data_ptr(), st), "hicgat_dist_histogram")
        if reduce is not None:
            reduce(hist_d)
        rank_d = _midranks(hist_d)
        # stored pairs i < j of this rank's rows: their wish value and the bin of their reconstructed distance
        bins = torch.empty(max(target.col.numel(), 1), dtype=torch.int32, device=dev)
        N.check(lib.hicgat_edge_dist_bins(c.data_ptr(), target.rowptr.data_ptr(), target.col.data_ptr(), n, r0, r1, d_scale, nbins, bins.data_ptr(), st),
                "hicgat_edge_dist_bins")
        k0, k1 = int(target.rowptr[r0]), int(target.rowptr[r1])
        b = bins[k0:k1]
        up = b >= 0
        tv, bd = target.tval[k0:k1][up].double(), b[up].long()
        # rank of t: the stored values (all ranks' values are needed: gather them when sharded) and the fill group
        if reduce is not None:
            raise NotImplementedError("row-sharded dSCC of an implicit target: gather the stored values first (use the dense streamed form per rank)")
        rt, r_fill, var_t = _implicit_target_ranks(tv, target.fill, npairs)
        r_fill, var_t = float(r_fill), float(var_t)
        mean = (npairs + 1.0) / 2.0
        hd = hist_d.to(torch.float64)
        sum_rd_all = float((hd * rank_d).sum())
        rd = rank_d[bd]
        cross = float((rt * rd).sum()) + r_fill * (sum_rd_all - float(rd.sum()))
        var_d = float((hd * (rank_d - mean) ** 2).sum())
        return (cross - npairs * mean * mean) / (var_d * var_t) ** 0.5
    if not isinstance(target, ops.WishTarget):
        raise TypeError("dscc_streamed expects a WishTarget or a SparseWishTarget")
    tmax = float(target.data.max()) if target.data.numel() else 1.0
    if reduce is not None:
        tm = torch.tensor([tmax], dtype=torch.float64, device=dev)
        tmax = float(reduce(tm, "max"))
    t_scale = nbins / (max(tmax, 1e-30) * (1.0 + 1e-6))
    hist_t = torch.zeros(nbins, dtype=torch.int64, device=dev)
    args = (c.data_ptr(), target.data.data_ptr(), target.pitch, n, target.r0, target.r1, d_scale, t_scale, nbins)
    N.check(lib.hicgat_rank_histograms(*args, hist_d.data_ptr(), hist_t.data_ptr(), st), "hicgat_rank_histograms")
    if reduce is not None:
        reduce(hist_d)
        reduce(hist_t)
    rank_d, rank_t = _midranks(hist_d), _midranks(hist_t)
    cross = torch.zeros(1, dtype=torch.float64, device=dev)
    N.check(lib.hicgat_rank_cross_sum(*args, rank_d.data_ptr(), rank_t.data_ptr(), cross.data_ptr(), st), "hicgat_rank_cross_sum")
    if reduce is not None:
        reduce(cross)
    return _spearman_from_tables(hist_d, hist_t, cross, npairs)


class DsccMeter:
    """dSCC of a full target at every training step (``spearmanr`` per iteration, HiC_GAT_generalize_directly.py:242), on the device.

    ``DsccMeter(target)`` takes a dense :class:`ops.WishTarget` or an implicit :class:`ops.SparseWishTarget` of all ``n`` rows and does
    the target-side work once: the rank table of the target (``hicgat_dscc_target_ranks``), or the ranks of the stored values and of
    the fill group.  It allocates every buffer here.  ``meter(coords)`` then returns the dSCC as a 0-d f64 CUDA tensor with no host
    read and no allocation (``hicgat_dscc_dense`` / ``hicgat_dscc_implicit``), so it can be captured in a CUDA graph.  The same tensor
    is returned and overwritten by every call.  Histogram mid-ranks with ``nbins`` bins, the bins of :func:`dscc_streamed`: the two
    agree to summation order.  NaN for constant distances or targets, as scipy gives."""

    def __init__(self, target, nbins: int = NBINS):
        from . import _native as N

        if not isinstance(target, (ops.WishTarget, ops.SparseWishTarget)):
            raise TypeError("DsccMeter expects a WishTarget or a SparseWishTarget")
        if target.r0 != 0 or target.r1 != target.n:
            raise ValueError("DsccMeter needs the full target (rows [0, n)); a row block would need the histograms all-reduced every step")
        nbins = int(nbins)
        if nbins <= 0:
            raise ValueError(f"nbins must be positive, got {nbins}")
        self.target, self.n, self.nbins = target, target.n, nbins
        lib, n = N.lib(), target.n
        dev = target.data.device if isinstance(target, ops.WishTarget) else target.tval.device
        ws_bytes = lib.hicgat_dscc_workspace_bytes(n, nbins)
        if ws_bytes == 0:
            raise ValueError(f"DsccMeter: unsupported size n={n}, nbins={nbins}")
        self._ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        self.rho = torch.full((), float("nan"), dtype=torch.float64, device=dev)
        npairs = n * (n - 1) / 2.0
        if isinstance(target, ops.WishTarget):
            tmax = float(target.data.max()) if target.data.numel() else 1.0
            self._t_scale = nbins / (max(tmax, 1e-30) * (1.0 + 1e-6))          # the rule of dscc_streamed
            self._rank_t = torch.empty(nbins, dtype=torch.float64, device=dev)
            self._var_t = torch.empty((), dtype=torch.float64, device=dev)
            N.check(lib.hicgat_dscc_target_ranks(target.data.data_ptr(), target.pitch, n, self._t_scale, nbins, self._rank_t.data_ptr(),
                                                 self._var_t.data_ptr(), self._ws.data_ptr(), ws_bytes, ops._stream()), "hicgat_dscc_target_ranks")
        else:
            row = torch.repeat_interleave(torch.arange(n, device=dev), target.rowptr[1:].long() - target.rowptr[:-1].long())
            up = target.col.long() > row
            rt, r_fill, var_t = _implicit_target_ranks(target.tval[up].double(), target.fill, npairs)
            self._rank_t = torch.zeros(max(target.col.numel(), 1), dtype=torch.float64, device=dev)
            self._rank_t[: target.col.numel()][up] = rt
            self._rank_fill, self._var_t = r_fill.reshape(()).clone(), var_t.reshape(()).clone()
        self._ws_bytes = ws_bytes

    def __call__(self, coords: torch.Tensor) -> torch.Tensor:
        from . import _native as N

        ops._cuda(coords)
        if coords.dtype != torch.float32 or coords.dim() != 2 or tuple(coords.shape) != (self.n, 3) or not coords.is_contiguous():
            raise RuntimeError(f"coords must be contiguous float32 [n,3] with n={self.n}, got {coords.dtype} {tuple(coords.shape)}")
        lib, t = N.lib(), self.target
        if isinstance(t, ops.WishTarget):
            rc = lib.hicgat_dscc_dense(coords.data_ptr(), t.data.data_ptr(), t.pitch, self.n, self._t_scale, self.nbins, self._rank_t.data_ptr(),
                                       self._var_t.data_ptr(), self.rho.data_ptr(), self._ws.data_ptr(), self._ws_bytes, ops._stream())
            N.check(rc, "hicgat_dscc_dense")
        else:
            rc = lib.hicgat_dscc_implicit(coords.data_ptr(), t.rowptr.data_ptr(), t.col.data_ptr(), self._rank_t.data_ptr(), self.n,
                                          self._rank_fill.data_ptr(), self._var_t.data_ptr(), self.nbins, self.rho.data_ptr(), self._ws.data_ptr(),
                                          self._ws_bytes, ops._stream())
            N.check(rc, "hicgat_dscc_implicit")
        return self.rho


def dscc(coords: torch.Tensor, truth) -> float:
    """Distance Spearman correlation coefficient of a reconstructed structure (CUDA tensors).  Maps of up to ``STREAM_FROM``
    loci with a full dense target: exact average ranks (sort-based, like scipy); larger maps, row blocks and implicit targets:
    the streamed histogram evaluation (:func:`dscc_streamed`)."""
    if isinstance(truth, ops.SparseWishTarget) or (isinstance(truth, ops.WishTarget) and (truth.n > STREAM_FROM or truth.r0 != 0 or truth.r1 != truth.n)):
        return dscc_streamed(coords, truth)
    t, d = upper_pairs(coords, truth)
    return float(_pearson(average_ranks(t.double()), average_ranks(d.double())))


def pearson(coords: torch.Tensor, truth) -> float:
    """``scipy.stats.pearsonr`` of the same two vectors (HiC_GAT_generalize_directly.py:220)."""
    t, d = upper_pairs(coords, truth)
    return float(_pearson(t.double(), d.double()))
