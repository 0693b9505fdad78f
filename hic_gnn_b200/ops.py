"""Torch-facing wrappers of the C ABI (device memory, streams and autograd only).

Every function requires CUDA tensors and enqueues on torch's current stream; none has a CPU
path.  Reference call sites are cited on each wrapper.
"""
from __future__ import annotations

import os

import torch

from . import _native as N

_MODES = {
    "mse": N.PAIR_GRAD_MSE,
    # per-step training mode of the MSE + Pearson loop: only the coordinate-dependent statistics
    # are accumulated; sum t / sum t^2 are constants of the target (WishTarget.t_moments)
    "mse_moments": N.PAIR_GRAD_MSE | N.PAIR_MOMENTS_D,
    "mse_moments_full": N.PAIR_GRAD_MSE | N.PAIR_MOMENTS,
    "contrastive": N.PAIR_GRAD_L1 | N.PAIR_MOMENTS,
    "moments": N.PAIR_MOMENTS,
    "value": 0,
}


def _cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("hic_gnn_b200 ops need CUDA tensors (there is no CPU fallback)")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _ptr(t):
    return None if t is None else t.data_ptr()


_PLACEHOLDER: dict = {}


def _addr(t: torch.Tensor) -> int:
    """``t.data_ptr()``, or for an empty ``t`` (whose ``data_ptr()`` is 0) the address of a small placeholder on its device: the
    C ABI refuses null arrays, and a pattern without edges (a map with no off-diagonal contact, a single locus) has empty ``col``
    and value arrays, which the kernels -- bounded by ``rowptr`` -- never read."""
    if t.numel():
        return t.data_ptr()
    buf = _PLACEHOLDER.get(t.device)
    if buf is None:
        buf = _PLACEHOLDER[t.device] = torch.zeros(4, dtype=torch.int32, device=t.device)
    return buf.data_ptr()


# ------------------------------------------------------------------------------ target
class WishTarget:
    """f32 wish-distance row block ``rows [r0, r1) x n`` with a 16-byte-aligned pitch.

    The layout the fused loss kernel streams (``truth.float()`` of HiC-GNN_main.py:127,
    stored once instead of re-cast every iteration)."""

    def __init__(self, data: torch.Tensor, n: int, r0: int, r1: int, symmetric: bool | None = None):
        _cuda(data)
        assert data.dtype == torch.float32 and data.dim() == 2 and data.stride(1) == 1
        assert data.shape[0] == r1 - r0 and data.stride(0) % 4 == 0 and data.stride(0) >= n
        self.data, self.n, self.r0, self.r1 = data, n, r0, r1
        # True: t_ij == t_ji verified (or promised by the builder) -> column-side gradient is complete;
        # False: verified asymmetric -> the row-side term is added by a second pass (MSE modes);
        # None: a row block built without sight of the full matrix: the caller's contract, as documented in hicgat.h
        self.symmetric = symmetric

    @property
    def pitch(self) -> int:
        return self.data.stride(0)

    @staticmethod
    def pitch_for(n: int) -> int:
        return (n + 3) // 4 * 4

    @classmethod
    def empty(cls, n: int, r0: int = 0, r1: int | None = None, device="cuda", symmetric: bool | None = None):
        r1 = n if r1 is None else r1
        buf = torch.zeros(max(r1 - r0, 1), cls.pitch_for(n), dtype=torch.float32, device=device)
        return cls(buf[: r1 - r0], n, r0, r1, symmetric)

    @classmethod
    def from_dense(cls, truth: torch.Tensor, r0: int = 0, r1: int | None = None, symmetric: bool | None = None):
        """Copy rows [r0,r1) of an N x N (f32/f64) CUDA matrix into the padded layout.  ``truth`` is the FULL
        matrix, so its symmetry (of rows [r0,r1) against columns [r0,r1)) is checked here, once, unless the
        caller states it (the reference does not symmetrise ``y``: utils.py:29-35)."""
        _cuda(truth)
        n = truth.shape[0]
        r1 = n if r1 is None else r1
        out = cls.empty(n, r0, r1, truth.device)
        out.data[:, :n].copy_(truth[r0:r1])
        if symmetric is None:
            # judged on the f32 values the kernel will stream (an f64 matrix whose asymmetry vanishes in the cast is symmetric for the kernel)
            ref = truth if truth.dtype == torch.float32 else (out.data if (r0 == 0 and r1 == n) else truth.float())
            symmetric = asymmetry(ref, r0, r1) == 0.0
        out.symmetric = bool(symmetric)
        return out

    def dense(self) -> torch.Tensor:
        return self.data[:, : self.n]

    def t_moments(self) -> torch.Tensor:
        """f64[8] holding this row block's ``sum_{i<j} t`` and ``sum_{i<j} t^2`` in slots 4 and 5
        (zeros elsewhere): the target-only Pearson moments, computed once by a full-moment launch
        and added to the per-step ``HICGAT_PAIR_MOMENTS_D`` result."""
        if getattr(self, "_tmom", None) is None:
            zeros = torch.zeros(self.n, 3, dtype=torch.float32, device=self.data.device)
            m, _ = pairloss_raw(zeros, self, N.PAIR_MOMENTS, 0.0, 0.0)
            out = torch.zeros_like(m)
            out[4:6] = m[4:6]
            self._tmom = out
        return self._tmom


class SparseWishTarget:
    """Implicit wish-distance target of a sparse map (SURVEY.md section 8 row f-4): the symmetric,
    diagonal-free CSR pattern of ``load_input`` with the wish distance of every stored pair;
    all other off-diagonal pairs are ``fill`` (1.0 after ``cont2dist``: zero contacts map to
    max/max, utils.py:78-80) and the diagonal is 0.  Rows ``[r0, r1)`` are this rank's share."""

    def __init__(self, n: int, rowptr32: torch.Tensor, col32: torch.Tensor, tval: torch.Tensor, fill: float = 1.0, r0: int = 0, r1: int | None = None):
        _cuda(rowptr32, col32, tval)
        assert rowptr32.dtype == torch.int32 and col32.dtype == torch.int32 and tval.dtype == torch.float32
        assert rowptr32.numel() == n + 1 and col32.numel() == tval.numel()
        self.n, self.rowptr, self.col, self.tval, self.fill = n, rowptr32.contiguous(), col32.contiguous(), tval.contiguous(), float(fill)
        self.r0, self.r1 = r0, n if r1 is None else r1

    @classmethod
    def from_graph(cls, graph, adj: torch.Tensor | None, factor: float, r0: int = 0, r1: int | None = None):
        """Wish distances at the stored pairs: ``(1/a)^factor / max`` like ``cont2dist`` (utils.py:75-80).
        With the dense f64 contact matrix ``adj`` the values are gathered from it (bit-identical to the dense
        target at those pairs); without it they come from the graph's f32 edge values."""
        r32, c32 = graph.i32()
        row = graph.storage.row()
        a = adj[row, graph.col].double() if adj is not None else graph.value.double()
        dist = (1.0 / a) ** factor
        tval = (dist / dist.max()).float()
        return cls(graph.n, r32, c32, tval, 1.0, r0, r1)

    @classmethod
    def from_values(cls, graph, value64: torch.Tensor, factor: float, r0: int = 0, r1: int | None = None):
        """Same from the f64 contact value of every stored entry (``utils.load_input_sparse``: there is no dense matrix to gather
        from): ``(1/a)^factor / max`` in f64, cast to f32 -- the values ``cont2dist`` gives the stored pairs (utils.py:75-80)."""
        r32, c32 = graph.i32()
        dist = (1.0 / value64.double()) ** factor
        tval = (dist / dist.max()).float()
        return cls(graph.n, r32, c32, tval, 1.0, r0, r1)

    def rows(self, r0: int, r1: int):
        return SparseWishTarget(self.n, self.rowptr, self.col, self.tval, self.fill, r0, r1)

    def t_moments(self) -> torch.Tensor:
        if getattr(self, "_tmom", None) is None:
            zeros = torch.zeros(self.n, 3, dtype=torch.float32, device=self.tval.device)
            m, _ = pairloss_raw(zeros, self, N.PAIR_MOMENTS, 0.0, 0.0)
            out = torch.zeros_like(m)
            out[4:6] = m[4:6]
            self._tmom = out
        return self._tmom


def asymmetry(mat: torch.Tensor, r0: int = 0, r1: int | None = None) -> float:
    """``max |M_ij - M_ji|`` over rows [r0,r1) of a full row-major f32/f64 CUDA matrix (``hicgat_asymmetry_*``);
    one host read -- a build-time check, never per step."""
    _cuda(mat)
    if mat.dim() != 2 or mat.stride(1) != 1 or mat.shape[0] > mat.shape[1] or mat.dtype not in (torch.float32, torch.float64):
        raise RuntimeError("asymmetry expects a row-major float32/float64 CUDA matrix with at least as many columns as rows")
    n = mat.shape[0]
    r1 = n if r1 is None else r1
    out = torch.empty(1, dtype=torch.float64, device=mat.device)
    fn = N.lib().hicgat_asymmetry_f32 if mat.dtype == torch.float32 else N.lib().hicgat_asymmetry_f64
    N.check(fn(mat.data_ptr(), mat.stride(0), n, r0, r1, out.data_ptr(), _stream()), "hicgat_asymmetry")
    return float(out)


# ------------------------------------------------------------------------------ pair loss
class _PairWorkspace:
    """Per (device, n, row block) scratch for the cross-CTA reductions, re-sized when the kernel
    tuning changes (``_native.set_pairloss_tuning`` bumps the epoch)."""

    _cache: dict = {}

    @classmethod
    def get(cls, device, n, r0, r1, sparse: bool = False, sym: bool = False):
        key = (device.index, n, r0, r1, N.tuning_epoch(), sparse, sym)
        ws = cls._cache.get(key)
        if ws is None:
            if sparse:
                need = N.lib().hicgat_pairloss_sparse_workspace_bytes(n, r0, r1)
            else:
                need = N.lib().hicgat_pairloss_workspace_bytes_mode(n, r0, r1, N.PAIR_SYMMETRIC if sym else 0)
            # zero-filled once and used for nothing else: calls pass HICGAT_PAIR_WS_CLEAN
            ws = torch.zeros(need, dtype=torch.uint8, device=device)
            cls._cache[key] = ws
        return ws


_USE_UPPER = os.environ.get("HICGAT_NO_UPPER", "0") != "1"  # A/B switch: stream the full row block even for symmetric targets


def uses_upper_triangle(target) -> bool:
    """True when the loss kernels stream only the upper triangle of ``target`` (``HICGAT_PAIR_SYMMETRIC``): the target's
    symmetry has been verified or stated when it was built.  Row blocks of a sharded run are then balanced by
    upper-triangle area (``sharding.row_block(..., balance="upper")``)."""
    if isinstance(target, SparseWishTarget):
        return _USE_UPPER  # the CSR pattern of load_input is symmetric by construction, the background constant
    return _USE_UPPER and target.symmetric is True


def pairloss_raw(coords: torch.Tensor, target: WishTarget, mode: int, c_mse: float, c_l1: float, moments=None, grad=None):
    """One launch of ``hicgat_pairloss_fwd_bwd`` (dense f32 target) or ``hicgat_pairloss_sparse_fwd_bwd``
    (implicit target): returns ``(moments f64[8], grad f32[n,3])``."""
    if isinstance(target, SparseWishTarget):
        _cuda(coords)
        if coords.dtype != torch.float32 or coords.shape != (target.n, 3):
            raise RuntimeError(f"coords must be float32 [n,3] with n={target.n}, got {coords.dtype} {tuple(coords.shape)}")
        coords = coords.contiguous()
        n = target.n
        if moments is None:
            moments = torch.empty(N.PAIR_NMOM, dtype=torch.float64, device=coords.device)
        if grad is None and (mode & 3):
            grad = torch.empty(n, 3, dtype=torch.float32, device=coords.device)
        ws = _PairWorkspace.get(coords.device, n, target.r0, target.r1, sparse=True, sym=_USE_UPPER)  # the layout depends on the mode
        rc = N.lib().hicgat_pairloss_sparse_fwd_bwd(
            coords.data_ptr(), target.rowptr.data_ptr(), _addr(target.col), _addr(target.tval), target.fill, n, target.r0, target.r1,
            mode | N.PAIR_WS_CLEAN | (N.PAIR_SYMMETRIC if _USE_UPPER else 0), c_mse, c_l1, moments.data_ptr(), _ptr(grad), ws.data_ptr(), ws.numel(), _stream(),
        )
        N.check(rc, "hicgat_pairloss_sparse_fwd_bwd")
        return moments, grad
    _cuda(coords, target.data)
    if coords.dtype != torch.float32 or coords.shape != (target.n, 3):
        raise RuntimeError(f"coords must be float32 [n,3] with n={target.n}, got {coords.dtype} {tuple(coords.shape)}")
    coords = coords.contiguous()
    n = target.n
    if moments is None:
        moments = torch.empty(N.PAIR_NMOM, dtype=torch.float64, device=coords.device)
    if grad is None and (mode & 3):
        grad = torch.empty(n, 3, dtype=torch.float32, device=coords.device)
    sym = uses_upper_triangle(target)
    ws = _PairWorkspace.get(coords.device, n, target.r0, target.r1, sym=sym)
    asym = target.symmetric is False and (mode & 3)
    if asym and (mode & N.PAIR_GRAD_L1):
        raise NotImplementedError("the contrastive (L1, i<j) gradient needs a symmetric target: t_ij != t_ji found when the target was built "
                                  "(symmetrise it, e.g. (T + T.T)/2 or triu(T) + triu(T, 1).T, whichever the experiment means)")
    rc = N.lib().hicgat_pairloss_fwd_bwd(
        coords.data_ptr(), target.data.data_ptr(), target.pitch, n, target.r0, target.r1, mode | N.PAIR_WS_CLEAN | (N.PAIR_SYMMETRIC if sym else 0),
        0.5 * c_mse if asym else c_mse, c_l1, moments.data_ptr(), _ptr(grad), ws.data_ptr(), ws.numel(), _stream(),
    )
    N.check(rc, "hicgat_pairloss_fwd_bwd")
    if asym:  # autograd of MSELoss(cdist(x), T) for T != T^T: column-side and row-side terms, (2/N^2) each
        rc = N.lib().hicgat_pairloss_rowside_add(coords.data_ptr(), target.data.data_ptr(), target.pitch, n, target.r0, target.r1, 0.5 * c_mse,
                                                 grad.data_ptr(), _stream())
        N.check(rc, "hicgat_pairloss_rowside_add")
    return moments, grad


def pearson_grad_raw(coords: torch.Tensor, target, moments: torch.Tensor, with_mse: bool, grad=None) -> torch.Tensor:
    """Second pass of the differentiable Pearson modes (``hicgat_pairloss_pearson_grad`` / ``_sparse_pearson_grad``): this row
    block's contribution to the gradient of ``1 - r`` (``with_mse=False``) or of ``MSE + alpha (1 - r)`` with alpha held
    constant (``with_mse=True``), from the GLOBAL f64 moments ``moments`` (pass 1 + the target constants), read on the device."""
    _cuda(coords, moments)
    n = target.n
    if coords.dtype != torch.float32 or coords.shape != (n, 3):
        raise RuntimeError(f"coords must be float32 [n,3] with n={n}, got {coords.dtype} {tuple(coords.shape)}")
    if moments.dtype != torch.float64 or moments.numel() != N.PAIR_NMOM or not moments.is_contiguous():
        raise RuntimeError("moments must be a contiguous float64 CUDA tensor of HICGAT_PAIR_NMOM elements")
    coords = coords.contiguous()
    if grad is None:
        grad = torch.empty(n, 3, dtype=torch.float32, device=coords.device)
    mode = N.PAIR_WS_CLEAN | (N.PAIR_GRAD_MSE if with_mse else 0)
    c_mse = 4.0 / (float(n) * float(n))
    if isinstance(target, SparseWishTarget):
        ws = _PairWorkspace.get(coords.device, n, target.r0, target.r1, sparse=True, sym=_USE_UPPER)
        rc = N.lib().hicgat_pairloss_sparse_pearson_grad(
            coords.data_ptr(), target.rowptr.data_ptr(), _addr(target.col), _addr(target.tval), target.fill, n, target.r0, target.r1,
            mode | (N.PAIR_SYMMETRIC if _USE_UPPER else 0), moments.data_ptr(), c_mse, int(with_mse), grad.data_ptr(), ws.data_ptr(), ws.numel(), _stream(),
        )
        N.check(rc, "hicgat_pairloss_sparse_pearson_grad")
        return grad
    _cuda(target.data)
    if target.symmetric is False:
        raise NotImplementedError("the differentiable Pearson gradient needs a symmetric target: t_ij != t_ji found when the target was built "
                                  "(symmetrise it, e.g. (T + T.T)/2 or triu(T) + triu(T, 1).T, whichever the experiment means)")
    sym = uses_upper_triangle(target)
    ws = _PairWorkspace.get(coords.device, n, target.r0, target.r1, sym=sym)
    rc = N.lib().hicgat_pairloss_pearson_grad(
        coords.data_ptr(), target.data.data_ptr(), target.pitch, n, target.r0, target.r1, mode | (N.PAIR_SYMMETRIC if sym else 0),
        moments.data_ptr(), c_mse, int(with_mse), grad.data_ptr(), ws.data_ptr(), ws.numel(), _stream(),
    )
    N.check(rc, "hicgat_pairloss_pearson_grad")
    return grad


def pearson_from_moments(m: torch.Tensor, npairs: float) -> torch.Tensor:
    """Pearson r of (d, t) over i<j from raw f64 moments (scipy.stats.pearsonr's value,
    HiC_GAT_generalize_directly.py:220)."""
    sd, sdd, st, stt, sdt = m[2], m[3], m[4], m[5], m[6]
    cov = sdt - sd * st / npairs
    vd = sdd - sd * sd / npairs
    vt = stt - st * st / npairs
    return (cov / torch.sqrt(vd * vt)).clamp(-1.0, 1.0)


# differentiable Pearson modes of pairwise_loss: pass 1 (moments) -> global moments -> pass 2 (gradient)
_PEARSON_MODES = ("pearson", "mse_pearson_grad")


def pearson_loss_from_moments(m: torch.Tensor, n: int, with_mse: bool) -> torch.Tensor:
    """f64 value of ``1 - r`` (``with_mse=False``) or of ``MSE + alpha (1 - r)``, ``alpha = min(1, 0.1 + 1/(MSE + 1e-6))`` with
    the f32 MSE (``with_mse=True``: the value of the ``mse_pearson`` training loss, HiC_GAT_generalize_directly.py:219-225).
    r is NaN when ``v_d v_t <= 0`` or is not finite (n <= 2, coincident loci, a constant target), as scipy gives."""
    npairs = n * (n - 1) / 2.0
    vd = m[3] - m[2] * m[2] / npairs
    vt = m[5] - m[4] * m[4] / npairs
    prod = vd * vt
    r = torch.where((prod > 0) & torch.isfinite(prod), pearson_from_moments(m, npairs), torch.full_like(prod, float("nan")))
    if not with_mse:
        return 1.0 - r
    mse = (m[0] / (float(n) * float(n))).to(torch.float32).double()
    alpha = torch.clamp(0.1 + 1.0 / (mse + 1e-6), max=1.0)
    return mse + alpha * (1.0 - r)


class _PairLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, coords, target, mode_name, reducer):
        n = target.n
        npairs = n * (n - 1) / 2.0
        if mode_name in _PEARSON_MODES:
            with_mse = mode_name == "mse_pearson_grad"
            if reducer is not None:
                moments, grad = reducer(coords.detach())
            else:
                moments, _ = pairloss_raw(coords.detach(), target, N.PAIR_MOMENTS_D, 0.0, 0.0)
                moments = moments + target.t_moments()
                grad = pearson_grad_raw(coords.detach(), target, moments, with_mse)
            ctx.save_for_backward(grad)
            ctx.mark_non_differentiable(moments)
            return pearson_loss_from_moments(moments, n, with_mse), moments
        mode = _MODES[mode_name]
        c_mse, c_l1 = 4.0 / (float(n) * float(n)), 0.1 / max(npairs, 1.0)
        if reducer is not None:  # row-sharded: local block + one packed all-reduce (sharding.py)
            moments, grad = reducer(coords.detach())
        else:
            moments, grad = pairloss_raw(coords.detach(), target, mode, c_mse, c_l1)
            if mode & N.PAIR_MOMENTS_D and not mode & N.PAIR_MOMENTS:
                moments = moments + target.t_moments()
        ctx.save_for_backward(grad)
        ctx.mark_non_differentiable(moments)
        if mode_name == "contrastive":
            loss = 0.1 * moments[1] / npairs  # f64, like the reference (:131-134)
        else:
            loss = (moments[0] / (float(n) * float(n))).to(torch.float32)  # MSELoss over N x N
        return loss, moments

    @staticmethod
    def backward(ctx, g_loss, _g_moments):
        (grad,) = ctx.saved_tensors
        return grad * g_loss.to(grad.dtype), None, None, None


def pairwise_loss(coords: torch.Tensor, target: WishTarget, mode: str = "mse", reducer=None):
    """Fused replacement of ``cdist`` + loss + backward.  Returns ``(loss, moments)``.

    mode ``"mse"``          MSELoss(cdist(coords), truth)            HiC-GNN_main.py:126-127
         ``"mse_moments"``  same + Pearson/L1 moments in one pass    HiC_GAT_generalize_directly.py:206-225
         ``"contrastive"``  0.1*mean_{i<j}|t-d| (f64)                train_and_test_same_res_GAT_node2vec.py:131-134
         ``"pearson"``      1 - r over i<j (f64), with its gradient
         ``"mse_pearson_grad"``  MSE + alpha (1 - r) (f64, the value of the mse_pearson training loss), alpha held constant
                            and the gradient of BOTH terms (the reference's r is a float without one)
    The two Pearson modes run two passes (moments, then the gradient from the global moments) and need a symmetric target.
    """
    if mode not in ("mse", "mse_moments", "mse_moments_full", "contrastive") + _PEARSON_MODES:
        raise ValueError(mode)
    return _PairLossFn.apply(coords, target, mode, reducer)


def sharded_reducer(target: WishTarget, mode: str, group=None, transport: str = "auto"):
    """``reducer`` for :func:`pairwise_loss` when ``target`` is this rank's row block.
    ``transport``: see :func:`sharding.make_sharded_pair_loss` (the two-pass modes ``pearson`` / ``mse_pearson_grad`` take
    ``"p2p"``, ``"nccl"`` or ``"auto"``)."""
    import torch.distributed as dist

    from . import sharding

    n = target.n
    npairs = n * (n - 1) / 2.0
    device = target.tval.device if isinstance(target, SparseWishTarget) else target.data.device
    if mode in _PEARSON_MODES:
        if transport == "p2p_oneshot":
            raise NotImplementedError(f"mode {mode!r}: the one-shot p2p exchange is not extended to the two-pass modes (use 'p2p' or 'nccl')")
        with_mse = mode == "mse_pearson_grad"

        def moments_fn(coords, out):
            pairloss_raw(coords, target, N.PAIR_MOMENTS_D, 0.0, 0.0, moments=out)

        def grad_fn(coords, moments, grad=None):
            return pearson_grad_raw(coords, target, moments.contiguous(), with_mse, grad=grad)

        const = sharding.allreduce_packed(target.t_moments().clone(), group)
        multi = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
        if transport == "p2p" or (transport == "auto" and multi and device.type == "cuda"):
            try:
                return sharding.P2PTwoPassShardedPairLoss(n, moments_fn, grad_fn, device, group, moment_const=const)
            except Exception as e:  # no symmetric memory on this system: the NCCL exchange is equivalent
                if transport == "p2p":
                    raise
                import warnings

                warnings.warn(f"symmetric-memory exchange unavailable ({e!r}); using two NCCL all-reduces")
        return sharding.TwoPassShardedPairLoss(n, moments_fn, grad_fn, device, group, moment_const=const)
    m = _MODES[mode]
    c_mse, c_l1 = 4.0 / (float(n) * float(n)), 0.1 / max(npairs, 1.0)
    fn = sharding.cuda_local_fn(target, m, c_mse, c_l1)
    split_fn = sharding.cuda_local_split_fn(target, m, c_mse, c_l1)
    const = None
    if m & N.PAIR_MOMENTS_D and not m & N.PAIR_MOMENTS:
        const = sharding.allreduce_packed(target.t_moments().clone(), group)  # global sum t, sum t^2: once
    return sharding.make_sharded_pair_loss(n, fn, device, group, moment_const=const, transport=transport, local_split_fn=split_fn)


def pair_moments(coords: torch.Tensor, target: WishTarget) -> torch.Tensor:
    """Moments only (no gradient): evaluation-time Pearson / MSE / dRMSD inputs."""
    m, _ = pairloss_raw(coords.detach(), target, _MODES["moments"], 0.0, 0.0)
    return m


class _PairDistFn(torch.autograd.Function):
    """Materialised ``torch.cdist(x, x, p=2)`` (models.py:39) for API parity of forward()."""

    @staticmethod
    def forward(ctx, coords):
        _cuda(coords)
        c = coords.detach().contiguous().float()
        n = c.shape[0]
        out = torch.empty(n, n, dtype=torch.float32, device=c.device)
        N.check(N.lib().hicgat_pairdist_fwd(c.data_ptr(), n, out.data_ptr(), n, _stream()), "hicgat_pairdist_fwd")
        ctx.save_for_backward(c)
        return out

    @staticmethod
    def backward(ctx, g):
        (c,) = ctx.saved_tensors
        n = c.shape[0]
        g = g.contiguous().float()
        gc = torch.empty_like(c)
        N.check(N.lib().hicgat_pairdist_bwd(c.data_ptr(), n, g.data_ptr(), n, gc.data_ptr(), _stream()), "hicgat_pairdist_bwd")
        return gc


def pairdist(coords: torch.Tensor) -> torch.Tensor:
    return _PairDistFn.apply(coords)


# ------------------------------------------------------------------------------ builders
def cont2dist(adj: torch.Tensor, factor: float, want_f64: bool = True, want_f32: bool = False, r0: int = 0, r1: int | None = None, max_reduce=None,
              symmetric: bool | None = None):
    """``utils.cont2dist`` (utils.py:75-80) on the GPU.  ``adj``: f64 CUDA rows [r0,r1) x n.

    Returns ``(f64 matrix or None, WishTarget or None)``.  ``max_reduce`` (sharded builds) is
    called on the device scalar between the two passes (an all-reduce(max)).  ``symmetric``: what the caller
    knows about the contact matrix (the wish distance is elementwise, so it inherits the symmetry); a full
    matrix (r0 = 0, r1 = n) is checked here when nothing is stated."""
    _cuda(adj)
    if adj.dtype != torch.float64 or adj.dim() != 2 or adj.stride(1) != 1:
        raise RuntimeError("cont2dist expects a row-major float64 CUDA matrix")
    n = adj.shape[1]
    r1 = n if r1 is None else r1
    if adj.shape[0] != r1 - r0:
        raise RuntimeError("adj must hold exactly rows [r0, r1)")
    lib = N.lib()
    mx = torch.empty(1, dtype=torch.float64, device=adj.device)
    ws = torch.empty(lib.hicgat_cont2dist_workspace_bytes(n, r0, r1), dtype=torch.uint8, device=adj.device)
    N.check(lib.hicgat_cont2dist_max_f64(adj.data_ptr(), adj.stride(0), n, r0, r1, float(factor), mx.data_ptr(), ws.data_ptr(), ws.numel(), _stream()), "hicgat_cont2dist_max_f64")
    if max_reduce is not None:
        max_reduce(mx)
    if symmetric is None and want_f32 and r0 == 0 and r1 == n:
        symmetric = asymmetry(adj) == 0.0
    o64 = torch.empty(r1 - r0, n, dtype=torch.float64, device=adj.device) if want_f64 else None
    tgt = WishTarget.empty(n, r0, r1, adj.device, symmetric) if want_f32 else None
    N.check(
        lib.hicgat_cont2dist_apply_f64(
            adj.data_ptr(), adj.stride(0), n, r0, r1, float(factor), mx.data_ptr(),
            _ptr(o64), n, _ptr(tgt.data) if tgt is not None else None, tgt.pitch if tgt is not None else 0, _stream(),
        ),
        "hicgat_cont2dist_apply_f64",
    )
    return o64, tgt


def csr_from_dense(adj: torch.Tensor, with_self_loops: bool = False):
    """Graph half of ``utils.load_input`` (utils.py:33-71) on the GPU: returns
    ``(rowptr int64[n+1], col int64[nnz], value f32[nnz])``, bit-exact with the reference."""
    _cuda(adj)
    if adj.dtype != torch.float64 or adj.dim() != 2 or adj.shape[0] != adj.shape[1] or adj.stride(1) != 1:
        raise RuntimeError("csr_from_dense expects a square row-major float64 CUDA matrix")
    n = adj.shape[0]
    lib = N.lib()
    counts = torch.empty(n, dtype=torch.int64, device=adj.device)
    rowptr = torch.empty(n + 1, dtype=torch.int64, device=adj.device)
    s = _stream()
    N.check(lib.hicgat_csr_count_f64(adj.data_ptr(), adj.stride(0), n, int(with_self_loops), counts.data_ptr(), s), "hicgat_csr_count_f64")
    N.check(lib.hicgat_csr_scan_i64(counts.data_ptr(), n, rowptr.data_ptr(), s), "hicgat_csr_scan_i64")
    nnz = int(rowptr[-1].item())  # one host sync, at build time only
    col = torch.empty(nnz, dtype=torch.int64, device=adj.device)
    val = torch.empty(nnz, dtype=torch.float32, device=adj.device)
    if nnz == 0:
        return rowptr, col, val
    N.check(lib.hicgat_csr_fill_f64(adj.data_ptr(), adj.stride(0), n, int(with_self_loops), rowptr.data_ptr(), col.data_ptr(), val.data_ptr(), s), "hicgat_csr_fill_f64")
    return rowptr, col, val


# ------------------------------------------------------------------------------ MLP-head glue
class _LnReluAddFn(torch.autograd.Function):
    """``relu(layer_norm(x)) [+ residual]`` in one kernel each way (``hicgat_ln_relu_add_fwd/bwd``)."""

    @staticmethod
    def forward(ctx, x, residual, weight, bias, eps):
        _cuda(x, residual, weight, bias)
        if x.dtype != torch.float32 or x.dim() != 2:
            raise RuntimeError("ln_relu_add expects a float32 [n, c] tensor")
        x = x.contiguous()
        res = residual.contiguous() if residual is not None else None
        if res is not None and res.shape != x.shape:
            raise RuntimeError("ln_relu_add: residual must have the shape of x")
        n, c = x.shape
        w, b = weight.detach().contiguous(), bias.detach().contiguous()
        y = torch.empty_like(x)
        mean = torch.empty(n, dtype=torch.float32, device=x.device)
        rstd = torch.empty(n, dtype=torch.float32, device=x.device)
        N.check(N.lib().hicgat_ln_relu_add_fwd(x.data_ptr(), _ptr(res), w.data_ptr(), b.data_ptr(), float(eps), n, c, y.data_ptr(), mean.data_ptr(),
                                               rstd.data_ptr(), _stream()), "hicgat_ln_relu_add_fwd")
        ctx.save_for_backward(x, mean, rstd, w, b)
        ctx.has_res = residual is not None
        return y

    @staticmethod
    def backward(ctx, gy):
        x, mean, rstd, w, b = ctx.saved_tensors
        gy = gy.contiguous()
        n, c = x.shape
        dx = torch.empty_like(x)
        dgamma = torch.empty_like(w)
        dbeta = torch.empty_like(b)
        ws = torch.empty(N.lib().hicgat_ln_relu_add_bwd_workspace_bytes(n, c), dtype=torch.uint8, device=x.device)
        N.check(N.lib().hicgat_ln_relu_add_bwd(gy.data_ptr(), x.data_ptr(), mean.data_ptr(), rstd.data_ptr(), w.data_ptr(), b.data_ptr(), n, c, dx.data_ptr(),
                                               dgamma.data_ptr(), dbeta.data_ptr(), ws.data_ptr(), ws.numel(), _stream()), "hicgat_ln_relu_add_bwd")
        return dx, (gy if ctx.has_res else None), dgamma, dbeta, None


def ln_relu_add(x: torch.Tensor, norm: torch.nn.LayerNorm, residual: torch.Tensor | None = None) -> torch.Tensor:
    """``F.relu(norm(x)) + residual`` of the GAT net's MLP head (models.py:670-690) as one fused kernel per
    direction; ``norm`` stays an ``nn.LayerNorm`` module (same parameters / ``state_dict`` keys)."""
    if tuple(norm.normalized_shape) != (x.shape[-1],) or norm.weight is None or norm.bias is None:
        raise RuntimeError("ln_relu_add: LayerNorm over the last dimension with affine parameters expected")
    return _LnReluAddFn.apply(x, residual, norm.weight, norm.bias, norm.eps)


# ------------------------------------------------------------------------------ Linear layers on the tcgen05 tensor cores (3xTF32)
TF32X3_MIN_ROWS = int(os.environ.get("HICGAT_TF32X3_MIN_ROWS", "4096"))  # below this the cuBLAS fp32 GEMM is launch-bound anyway
_split_cache: dict = {}


def split_tf32(x: torch.Tensor, pattern: int, transpose: bool = False, cache: bool = False) -> torch.Tensor:
    """``hicgat_split_tf32``: ``[s0 | s1 | s2]`` along the reduction dimension, ``s_p`` = hi or lo TF32 part by bit p of ``pattern``
    (0b100 for the left operand, 0b010 for the right one).  ``cache``: memoise for a constant tensor (the input features)."""
    _cuda(x)
    if x.dtype != torch.float32 or x.dim() != 2 or x.stride(1) != 1:
        raise RuntimeError("split_tf32 expects a row-major float32 CUDA matrix")
    key = (x.data_ptr(), x._version, tuple(x.shape), x.stride(0), pattern, transpose)
    hit = _split_cache.get(key)
    if hit is not None and hit[0] is x:  # the entry holds a reference to its source, so the address cannot have been recycled
        return hit[1]
    rows, cols = x.shape
    red = rows if transpose else cols
    kpad = (red + 31) // 32 * 32
    out = torch.empty(cols if transpose else rows, 3 * kpad, dtype=torch.float32, device=x.device)
    N.check(N.lib().hicgat_split_tf32(x.data_ptr(), rows, cols, x.stride(0), out.data_ptr(), pattern, int(transpose), _stream()), "hicgat_split_tf32")
    # memo: constant tensors (`cache`: the input features, split once per run) and, briefly, the latest activations (two Linear
    # layers that read the same tensor -- densea / align_densea -- share one split)
    if not cache:
        for k in [k for k, v in _split_cache.items() if not v[2]]:
            if len(_split_cache) > 6:
                del _split_cache[k]
    elif len(_split_cache) > 12:
        _split_cache.clear()
    _split_cache[key] = (x, out, cache)
    return out


def gemm_tf32_tn(a_s: torch.Tensor, b_s: torch.Tensor, bias: torch.Tensor | None = None) -> torch.Tensor:
    """``hicgat_gemm_tf32_tn``: ``a_s [m, k'] . b_s [n, k']^T (+ bias)`` on tcgen05 (operands from :func:`split_tf32`)."""
    m, k = a_s.shape
    n = b_s.shape[0]
    assert b_s.shape[1] == k
    d = torch.empty(m, n, dtype=torch.float32, device=a_s.device)
    lib = N.lib()
    wsb = lib.hicgat_gemm_tf32_workspace_bytes(m, n, k, 3)
    ws = torch.empty(max(wsb, 16), dtype=torch.uint8, device=a_s.device)
    N.check(lib.hicgat_gemm_tf32_tn(a_s.data_ptr(), a_s.stride(0), b_s.data_ptr(), b_s.stride(0), m, n, k, 3, _ptr(bias), d.data_ptr(), d.stride(0),
                                    ws.data_ptr(), ws.numel(), _stream()), "hicgat_gemm_tf32_tn")
    return d


class _Linear3xTF32(torch.autograd.Function):
    """``F.linear`` with all three GEMMs (y = x W^T + b, dx = dy W, dW = dy^T x) on the tensor cores at fp32 accuracy."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        x = x.contiguous()
        w = weight.detach().contiguous()
        y = gemm_tf32_tn(split_tf32(x.detach(), 0b100, cache=not x.requires_grad), split_tf32(w, 0b010), None if bias is None else bias.detach().contiguous())
        ctx.save_for_backward(x, w)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, gy):
        x, w = ctx.saved_tensors
        gy = gy.contiguous()
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:  # dx[m, k] = dy[m, n] . (W^T)[k, n]^T : reduction over the output features
            gx = gemm_tf32_tn(split_tf32(gy, 0b100), split_tf32(w, 0b010, transpose=True))
        if ctx.needs_input_grad[1]:  # dW[n, k] = (dy^T)[n, m] . (x^T)[k, m]^T : reduction over the rows
            gw = gemm_tf32_tn(split_tf32(gy, 0b100, transpose=True), split_tf32(x, 0b010, transpose=True, cache=not x.requires_grad))
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = gy.sum(dim=0)
        return gx, gw, gb


def linear(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor | None = None) -> torch.Tensor:
    """``torch.nn.functional.linear`` of the MLP heads / the GATConv projection.  Maps of at least ``TF32X3_MIN_ROWS`` loci run the
    three GEMMs on the tcgen05 tensor cores (3xTF32 split: fp32-level accuracy); smaller ones stay on the cuBLAS fp32 GEMM."""
    # measured at 49 850 rows (profiles/r2_gemm.json): 512x512 and 512x256 layers run 1.5-2x faster than the cuBLAS fp32 GEMM incl. the
    # split kernels, 256x128 and smaller are a wash or slower (the splits dominate): those stay on cuBLAS
    if x.is_cuda and x.dim() == 2 and x.dtype == torch.float32 and x.shape[0] >= TF32X3_MIN_ROWS and weight.numel() >= 100000 and TF32X3_MIN_ROWS > 0:
        return _Linear3xTF32.apply(x, weight, bias)
    return torch.nn.functional.linear(x, weight, bias)


class Linear(torch.nn.Linear):
    """``torch.nn.Linear`` (same parameters, init and ``state_dict`` keys) whose forward goes through :func:`linear`."""

    def forward(self, x):
        return linear(x, self.weight, self.bias)


# ------------------------------------------------------------------------------ host-buffer entry
class HostPairLoss:
    """Pairwise loss for a target that lives in (pinned) HOST memory: the row blocks are
    streamed host->device through two staging buffers while the fused kernel consumes the
    previous block (copy stream / compute stream, events), partial moments and gradients are
    summed on the device and read back once.  This is the end-to-end path ``bench.py`` times
    (``e2e``): PCIe-bound by construction; a training loop keeps the target resident instead.

    The gradient is the column-side sum of the fused kernel, complete only for a symmetric target (``t_ij == t_ji``), in both
    modes: an asymmetric host target is not supported.  ``symmetric=True`` only selects the upper-triangle upload (columns from
    each block's diagonal 128-column strip on); the columns left of it are never uploaded and never enter the result.
    """

    def __init__(self, n: int, r0: int = 0, r1: int | None = None, block_rows: int = 2048, device="cuda", reduce=None, symmetric: bool = False):
        self.n, self.r0, self.r1 = n, r0, n if r1 is None else r1
        self.reduce = reduce  # row-sharded runs: all-reduce of the packed device buffer before the read-back
        # symmetric=True: the caller has verified t_ij == t_ji (ops.asymmetry on the host matrix's device copy, or a target built
        # from a symmetric map): only the columns at or right of each row block's diagonal are uploaded and streamed
        self.symmetric = bool(symmetric) and _USE_UPPER
        self.block_rows = block_rows
        self.device = torch.device(device)
        self.pitch = WishTarget.pitch_for(n)
        self.stage = [torch.empty(block_rows, self.pitch, dtype=torch.float32, device=device) for _ in range(2)]
        self.copy_stream = torch.cuda.Stream(device=device)
        self.ready = [torch.cuda.Event() for _ in range(2)]
        self.free = [torch.cuda.Event() for _ in range(2)]
        self.coords_dev = torch.empty(n, 3, dtype=torch.float32, device=device)
        self.packed = torch.zeros(N.PAIR_NMOM + 3 * n, dtype=torch.float64, device=device)
        self.acc = torch.zeros_like(self.packed)
        self.out_host = torch.empty(N.PAIR_NMOM + 3 * n, dtype=torch.float64, pin_memory=True)
        self.h2d_bytes = 0
        self.d2h_bytes = 0

    def __call__(self, coords_host: torch.Tensor, target_host: torch.Tensor, mode: int, c_mse: float, c_l1: float):
        """``coords_host`` f32 [n,3] (pinned), ``target_host`` f32 [r1-r0, pitch] (pinned)."""
        assert not coords_host.is_cuda and not target_host.is_cuda
        assert target_host.shape == (self.r1 - self.r0, self.pitch) and target_host.dtype == torch.float32
        main = torch.cuda.current_stream()
        # the first two blocks of a call write the staging buffers without waiting on a `free` event: order them after
        # whatever the caller queued on its stream (work that still reads or writes that memory)
        self.copy_stream.wait_stream(main)
        self.coords_dev.copy_(coords_host, non_blocking=True)
        self.acc.zero_()
        self.h2d_bytes = coords_host.numel() * 4
        lib = N.lib()
        nblk = (self.r1 - self.r0 + self.block_rows - 1) // self.block_rows
        for b in range(nblk):
            s = b & 1
            lo = b * self.block_rows
            hi = min(lo + self.block_rows, self.r1 - self.r0)
            c0 = ((self.r0 + lo) // 128) * 128 if self.symmetric else 0  # first column strip that holds a pair with row <= column
            with torch.cuda.stream(self.copy_stream):
                if b >= 2:
                    self.copy_stream.wait_event(self.free[s])
                if c0 == 0:
                    self.stage[s][: hi - lo].copy_(target_host[lo:hi], non_blocking=True)
                else:
                    N.check(lib.hicgat_memcpy2d_h2d_async(self.stage[s].data_ptr() + 4 * c0, 4 * self.pitch, target_host.data_ptr() + 4 * (lo * self.pitch + c0),
                                                          4 * self.pitch, 4 * (self.pitch - c0), hi - lo, self.copy_stream.cuda_stream), "hicgat_memcpy2d_h2d_async")
                self.ready[s].record(self.copy_stream)
            self.h2d_bytes += (hi - lo) * (self.pitch - c0) * 4
            main.wait_event(self.ready[s])
            ws = _PairWorkspace.get(self.device, self.n, self.r0 + lo, self.r0 + hi, sym=self.symmetric)
            rc = lib.hicgat_pairloss_fwd_bwd_packed(
                self.coords_dev.data_ptr(), self.stage[s].data_ptr(), self.pitch, self.n, self.r0 + lo, self.r0 + hi,
                mode | N.PAIR_WS_CLEAN | (N.PAIR_SYMMETRIC if self.symmetric else 0), c_mse, c_l1, self.packed.data_ptr(), ws.data_ptr(), ws.numel(), main.cuda_stream,
            )
            N.check(rc, "hicgat_pairloss_fwd_bwd_packed")
            self.acc.add_(self.packed)
            self.free[s].record(main)
        if self.reduce is not None:
            self.reduce(self.acc)
        self.out_host.copy_(self.acc, non_blocking=True)
        self.d2h_bytes = self.out_host.numel() * 8
        main.synchronize()
        return self.out_host[: N.PAIR_NMOM], self.out_host[N.PAIR_NMOM:].view(self.n, 3)
