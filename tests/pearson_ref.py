"""Reference (test infrastructure) for the differentiable Pearson modes: plain differentiable torch over the
upper-triangle pairs of ``oracle.loss.triu_pairs``, in the dtype of the inputs (f64 for the parity tests).

Degenerate moments (``v_d v_t <= 0`` or not finite) give a NaN value, as ``scipy.stats.pearsonr``, and a zero
Pearson gradient.
"""
from __future__ import annotations

import math

import numpy as np
import torch
from torch.optim import Adam

from oracle import loss as L


def _pearson_r(coords: torch.Tensor, truth: torch.Tensor):
    dist_truth, dist_out = L.triu_pairs(truth.to(coords.dtype), coords)
    dm = dist_out - dist_out.mean()
    tm = dist_truth - dist_truth.mean()
    vd, vt, c = (dm * dm).sum(), (tm * tm).sum(), (dm * tm).sum()
    prod = float((vd * vt).detach())
    if not (prod > 0.0 and math.isfinite(prod)):
        return torch.full((), float("nan"), dtype=coords.dtype) + 0.0 * dist_out.sum()  # NaN value, zero gradient
    return c / torch.sqrt(vd * vt)


def pearson_loss(coords: torch.Tensor, truth: torch.Tensor) -> torch.Tensor:
    """``1 - r`` over the pairs i<j, with its gradient."""
    return 1.0 - _pearson_r(coords, truth)


def mse_pearson_grad_loss(coords: torch.Tensor, truth: torch.Tensor):
    """``MSE + alpha (1 - r)`` of HiC_GAT_generalize_directly.py:219-225 with alpha = min(1, 0.1 + 1/(MSE + 1e-6)) held
    constant (a Python float, as there) and r differentiable.  MSE over the full N x N matrix in the inputs' dtype.
    Returns (total, mse, alpha)."""
    out = torch.cdist(coords, coords, p=2)
    mse = ((out - truth.to(coords.dtype)) ** 2).mean()
    alpha = min(1.0, 0.1 + 1.0 / (float(np.float32(mse.item())) + 1e-6))
    return mse + alpha * pearson_loss(coords, truth), mse, alpha


def closed_form_grad(x: np.ndarray, t: np.ndarray, with_mse: bool) -> np.ndarray:
    """numpy mirror of the closed form: g_i = sum_{j != i} [c_mse (d - t) + lambda A rho_ij] (x_i - x_j) / d_ij with
    rho = t - beta d - kappa (the quantities of hicgat.h's Pearson section), in f64."""
    n = x.shape[0]
    diff = x[:, None, :] - x[None, :, :]
    d = np.sqrt((diff**2).sum(-1))
    iu = np.triu_indices(n, 1)
    dp, tp = d[iu], t[iu]
    p = n * (n - 1) / 2.0
    sd, sdd, st, stt, sdt = dp.sum(), (dp * dp).sum(), tp.sum(), (tp * tp).sum(), (dp * tp).sum()
    vd, vt, c = sdd - sd * sd / p, stt - st * st / p, sdt - sd * st / p
    prod = vd * vt
    lam_a = beta = kappa = 0.0
    if prod > 0 and np.isfinite(prod):
        beta = c / vd
        kappa = st / p - beta * sd / p
        lam_a = -1.0 / np.sqrt(prod)
    mse = ((d - t) ** 2).mean()
    if with_mse:
        lam_a *= min(1.0, 0.1 + 1.0 / (float(np.float32(mse)) + 1e-6))
    w = lam_a * (t - beta * d - kappa)
    if with_mse:
        w = w + 4.0 / (n * n) * (d - t)
    np.fill_diagonal(w, 0.0)
    inv = np.divide(1.0, d, out=np.zeros_like(d), where=d > 0)
    return ((w * inv)[:, :, None] * diff).sum(1)


def train(model, x, edge_index, truth, lr: float = 1e-3, max_steps: int = 10, thresh: float = 1e-8):
    """``oracle.loop.train``'s loop with the ``mse_pearson_grad`` body: one forward to coordinates, the differentiable
    total, backward, Adam.  Returns ``(loss_history, grads)`` with every parameter gradient of every step."""
    optimizer = Adam(model.parameters(), lr=lr)
    old, diff = 1.0, 1.0
    hist, grads = [], []
    while diff > thresh and len(hist) < max_steps:
        model.train()
        optimizer.zero_grad()
        coords = model.get_model(x, edge_index)
        total, _, _ = mse_pearson_grad_loss(coords, truth)
        value = float(total.detach())
        diff = abs(old - value)
        total.backward()
        grads.append({k: p.grad.detach().clone() for k, p in model.named_parameters() if p.grad is not None})
        optimizer.step()
        old = value
        hist.append(value)
    return hist, grads
