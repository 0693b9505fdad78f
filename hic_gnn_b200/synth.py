"""Seeded synthetic Hi-C contact maps for the benchmark / parity configurations
(SURVEY.md section 8d): counts follow the Hi-C distance decay ``c(s) = c0 * s^-1.08``, the map is
symmetric with a zero diagonal, the +-1 off-diagonals are forced non-zero (no isolated loci),
then balanced (Sinkhorn / KR fixed point, f64) to unit row sums and ``round(., 6)`` like
``r_utils.R:90``.

Everything is a pure function of ``(i, j, seed)`` through an integer hash, so a row block can
be generated on its own (row-sharded builds) and is symmetric by construction.
Pure torch; runs on CPU or GPU (input generation, not part of the hot path).
"""
from __future__ import annotations

import math

import torch

CHR1_LOCI = {"100kb": 2493, "25kb": 9970, "5kb": 49850}  # chr1 = 249 Mb


def _hash_uniform(i: torch.Tensor, j: torch.Tensor, seed: int) -> torch.Tensor:
    """U[0,1) from (min(i,j), max(i,j), seed): 32-bit mix in int64 arithmetic."""
    lo, hi = torch.minimum(i, j), torch.maximum(i, j)
    h = (lo * 0x9E3779B1 + hi * 0x85EBCA77 + seed * 0xC2B2AE3D) & 0xFFFFFFFF
    h = (h ^ (h >> 15)) * 0x2C1B3C6D & 0xFFFFFFFF
    h = (h ^ (h >> 12)) * 0x297A2D39 & 0xFFFFFFFF
    h = h ^ (h >> 15)
    return h.to(torch.float64) / 4294967296.0


def solve_c0(n: int, density: float) -> float:
    """c0 such that the mean over pairs of P(count>0) = 1-exp(-c0 s^-1.08) equals ``density``."""
    s = torch.arange(1, n, dtype=torch.float64)
    wts = (n - s) / (n * (n - 1) / 2.0)
    decay = s.pow(-1.08)
    lo, hi = 1e-6, 1e12
    for _ in range(200):
        mid = math.sqrt(lo * hi)
        d = float((wts * (1 - torch.exp(-mid * decay))).sum())
        lo, hi = (mid, hi) if d < density else (lo, mid)
    return math.sqrt(lo * hi)


def raw_block(n: int, r0: int, r1: int, c0: float, seed: int, device="cpu") -> torch.Tensor:
    """Rows [r0,r1) of the raw (unnormalised) synthetic count matrix, f64."""
    i = torch.arange(r0, r1, device=device, dtype=torch.int64).unsqueeze(1)
    j = torch.arange(0, n, device=device, dtype=torch.int64).unsqueeze(0)
    s = (i - j).abs().to(torch.float64)
    mean = c0 * s.clamp(min=1.0).pow(-1.08)
    present = _hash_uniform(i, j, seed) < (1.0 - torch.exp(-mean))
    present |= s == 1.0
    value = torch.ceil(mean * (0.5 + _hash_uniform(i, j, seed + 7919))).clamp(min=1.0)
    out = torch.where(present, value, torch.zeros_like(value))
    out[s == 0.0] = 0.0
    return out


def balance(a: torch.Tensor, iters: int = 300, tol: float = 1e-10) -> torch.Tensor:
    """Symmetric matrix balancing to unit row sums (the fixed point KR converges to)."""
    x = torch.ones(a.shape[0], dtype=torch.float64, device=a.device)
    for _ in range(iters):
        r = x * (a @ x)
        if float((r - 1).abs().max()) < tol:
            break
        x = x / torch.sqrt(r)
    return torch.round((x.unsqueeze(1) * a) * x.unsqueeze(0), decimals=6)


def synthetic_map(n: int, density: float, seed: int | None = None, device="cpu") -> torch.Tensor:
    """Dense balanced N x N f64 contact matrix (configs C3/C4; N up to ~10-20k)."""
    seed = 1234 + n if seed is None else seed
    raw = raw_block(n, 0, n, solve_c0(n, density), seed, device)
    return balance(raw)


def synthetic_features(n: int, dim: int = 512, seed: int | None = None, device="cpu") -> torch.Tensor:
    """``0.25 * randn(N, 512)`` f32 seeded random node features: a cheap stand-in for the LINE embeddings (not carried by
    this package) and for node2vec embeddings where their cost is not wanted; :mod:`hic_gnn_b200.node2vec` computes the
    real node2vec embeddings of a graph."""
    g = torch.Generator().manual_seed((1234 + n if seed is None else seed) + 1)
    return (0.25 * torch.randn(n, dim, generator=g)).to(device)


def synthetic_map_chunked(n: int, density: float, seed: int | None = None, device="cuda", chunk_rows: int = 2048,
                          iters: int = 300, tol: float = 1e-10) -> torch.Tensor:
    """Same matrix as :func:`synthetic_map`, built in row chunks and balanced in place so that
    the 50k-locus map (20 GB of f64) needs one resident N x N buffer plus chunk-sized
    temporaries.  Bench input generation (outside every timed region)."""
    seed = 1234 + n if seed is None else seed
    c0 = solve_c0(n, density)
    a = torch.empty(n, n, dtype=torch.float64, device=device)
    for r0 in range(0, n, chunk_rows):
        r1 = min(r0 + chunk_rows, n)
        a[r0:r1] = raw_block(n, r0, r1, c0, seed, device)
    x = torch.ones(n, dtype=torch.float64, device=device)
    for it in range(iters):
        r = x * torch.mv(a, x)
        if it % 10 == 9 and float((r - 1).abs().max()) < tol:
            break
        x = x / torch.sqrt(r)
    for r0 in range(0, n, chunk_rows):
        r1 = min(r0 + chunk_rows, n)
        blk = a[r0:r1]
        blk.mul_(x[r0:r1].unsqueeze(1)).mul_(x.unsqueeze(0))
        torch.round(blk, decimals=6, out=blk)
    return a
