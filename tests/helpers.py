"""Shared helpers for the GPU parity tests (oracle = checker, CUDA path = thing under test)."""
import numpy as np
import torch


def rel_err(got: torch.Tensor, want: torch.Tensor) -> float:
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    return float((got - want).abs().max() / want.abs().max().clamp(min=1e-30))


def random_coords(n: int, seed: int = 0, scale: float = 0.3) -> torch.Tensor:
    g = torch.Generator().manual_seed(seed)
    return scale * torch.randn(n, 3, generator=g)


def wish_from_map(adj: torch.Tensor, factor: float = 1.0) -> torch.Tensor:
    from oracle.wish import cont2dist

    return cont2dist(adj.clone().double(), factor)


def small_map(n: int, density: float, seed: int = 0) -> torch.Tensor:
    from hic_gnn_b200 import synth

    return synth.synthetic_map(n, density, seed=seed)


def pair_block_reference(coords: torch.Tensor, rows: torch.Tensor, r0: int, upper: bool, mode: int, c_mse: float = 0.0, c_l1: float = 0.0,
                         chunk: int = 2048, with_slack: bool = False):
    """f64 reference of ONE row block ``[r0, r0 + len(rows))`` of the fused pair loss, on the device of ``rows``: what the kernel
    returns for that block as ``(moments f64[8], grad f64[n,3])``.

    ``upper=False`` (full rows): moment 0 = sum of e^2 over the whole rows, gradient = the column-side sum
    ``g_j = sum_i w_ij (x_j - x_i)``.  ``upper=True`` (``HICGAT_PAIR_SYMMETRIC``): only pairs with column >= row count, moment 0 =
    ``t_ii^2 + 2 sum_{j>i} e^2`` and the gradient adds the row-side sum ``g_i -= sum_{j>i} w_ij (x_j - x_i)``; entries left of the
    diagonal are never looked at (they may be NaN).  Moments 1..7 are the i<j sums (``sum |e|, d, d^2, t, t^2, d t, e^2``), zero
    where ``mode`` does not produce them (light set: no 1, 4, 5).  ``w = c_mse e / d`` (GRAD_MSE) plus ``c_l1 sign(e) / d`` (GRAD_L1).

    ``with_slack=True`` also returns, per gradient element, how far the kernel may lawfully be from the reference: the L1 weight
    jumps at e = 0, and where |e| is within the f32 error of the kernel's distance (2e-6 d) either sign is right, so every such pair
    may move the element by up to 2 c_l1 |x_j - x_i| / d (see :func:`grad_within`)."""
    mom_full, mom_d = 4, 8
    if (mode & mom_d) and (mode & 2):
        mode |= mom_full
    dev = rows.device
    c = coords.double().to(dev)
    n = c.shape[0]
    m = torch.zeros(8, dtype=torch.float64, device=dev)
    grad = torch.zeros(n, 3, dtype=torch.float64, device=dev)
    slack = torch.zeros(n, 3, dtype=torch.float64, device=dev)
    jj = torch.arange(n, device=dev).unsqueeze(0)
    for k0 in range(0, rows.shape[0], chunk):
        k1 = min(k0 + chunk, rows.shape[0])
        t = rows[k0:k1].double()
        ci = c[r0 + k0:r0 + k1]
        d = torch.cdist(ci, c, compute_mode="donot_use_mm_for_euclid_dist")
        ii = torch.arange(r0 + k0, r0 + k1, device=dev).unsqueeze(1)
        up = ii < jj
        e = torch.where(ii <= jj, d - t, torch.zeros_like(d)) if upper else d - t
        eu = torch.where(up, e, torch.zeros_like(e))
        zero = torch.zeros_like(d)
        m[0] += (2 * (eu * eu).sum() + (e[ii == jj] ** 2).sum()) if upper else (e * e).sum()
        m[1] += eu.abs().sum()
        m[2] += torch.where(up, d, zero).sum()
        m[3] += torch.where(up, d * d, zero).sum()
        m[4] += torch.where(up, t, zero).sum()
        m[5] += torch.where(up, t * t, zero).sum()
        m[6] += torch.where(up, d * t, zero).sum()
        m[7] += (eu * eu).sum()
        live = (up if upper else torch.ones_like(up)) & (d > 0)
        w = torch.zeros_like(d)
        if mode & 1:
            w = w + c_mse * torch.where(live, e / d.clamp(min=1e-300), zero)
        if mode & 2:
            w = w + c_l1 * torch.where(live, torch.sign(e) / d.clamp(min=1e-300), zero)
        amb = 2 * c_l1 * torch.where(live & (e.abs() <= 2e-6 * d), 1.0 / d.clamp(min=1e-300), zero) if mode & 2 else zero
        if mode & 3:
            for q in range(3):
                diff = c[:, q].unsqueeze(0) - ci[:, q].unsqueeze(1)  # x_j - x_i
                grad[:, q] += (w * diff).sum(0)
                slack[:, q] += (amb * diff.abs()).sum(0)
                if upper:
                    grad[r0 + k0:r0 + k1, q] -= (w * diff).sum(1)
                    slack[r0 + k0:r0 + k1, q] += (amb * diff.abs()).sum(1)
    if not mode & mom_full:
        m[1] = m[4] = m[5] = 0.0
        if not mode & mom_d:
            m[2] = m[3] = m[6] = m[7] = 0.0
    return (m, grad, slack) if with_slack else (m, grad)


def grad_within(got: torch.Tensor, want: torch.Tensor, slack: torch.Tensor, tol: float) -> bool:
    """Every element of ``got`` within ``tol * max|want|`` of ``want``, plus its sign-ambiguity ``slack``
    (:func:`pair_block_reference`; zero without an L1 term, where this is ``rel_err(got, want) < tol``)."""
    got, want, slack = (x.detach().double().cpu() for x in (got, want, slack))
    return bool(((got - want).abs() <= tol * float(want.abs().max()) + slack).all())





def poison_lower(rows: torch.Tensor, r0: int, seed: int) -> torch.Tensor:
    """Rows [r0, r0 + len(rows)) of an upper-triangle target with what HICGAT_PAIR_SYMMETRIC allows left of the diagonal: NaN in every
    column left of the row's diagonal 128-column strip, finite garbage (|x| <= 1e3) below the diagonal inside that strip."""
    g = torch.Generator(device=rows.device).manual_seed(seed)
    ii = torch.arange(r0, r0 + rows.shape[0], device=rows.device).unsqueeze(1)
    jj = torch.arange(rows.shape[1], device=rows.device).unsqueeze(0)
    garbage = 2e3 * torch.rand(rows.shape, generator=g, device=rows.device, dtype=rows.dtype) - 1e3
    out = torch.where(jj < ii, garbage, rows)
    return torch.where(jj < ii // 128 * 128, torch.full_like(out, float("nan")), out)
