"""Differentiable Pearson modes, host side (no GPU): the f64 reference against scipy and the closed form, the invariants
of the gradient, the degenerate-moment rule, the two-exchange sharded reducer on gloo with CPU stand-ins for the two
kernel passes, and argument validation of the new C entry points."""
import ctypes
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
from scipy.stats import pearsonr

import pearson_ref as R
from hic_gnn_b200 import _native as N
from hic_gnn_b200 import sharding
from hic_gnn_b200.ops import pearson_loss_from_moments


def _problem(n, seed=0, noise=0.3):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, 3, generator=g, dtype=torch.float64)
    t = torch.cdist(x, x) + noise * torch.rand(n, n, generator=g, dtype=torch.float64)
    t = (t + t.t()) / 2
    t.fill_diagonal_(0)
    coords = 0.5 * torch.randn(n, 3, generator=g, dtype=torch.float64)
    return coords, t


def _autograd(fn, coords, truth):
    c = coords.clone().requires_grad_(True)
    out = fn(c, truth)
    val = out[0] if isinstance(out, tuple) else out
    (g,) = torch.autograd.grad(val, c)
    return val.detach(), g


@pytest.mark.parametrize("n", [3, 17, 120])
def test_value_matches_scipy(n):
    coords, truth = _problem(n, seed=n)
    val = R.pearson_loss(coords, truth)
    iu = np.triu_indices(n, 1)
    d = torch.cdist(coords, coords).numpy()
    r = pearsonr(truth.numpy()[iu], d[iu])[0]
    assert abs(float(val) - (1.0 - r)) < 1e-12
    total, mse, alpha = R.mse_pearson_grad_loss(coords, truth)
    assert abs(float(total) - (float(mse) + alpha * (1.0 - r))) < 1e-12


@pytest.mark.parametrize("with_mse", [False, True])
@pytest.mark.parametrize("n", [3, 40, 150])
def test_autograd_matches_closed_form(n, with_mse):
    coords, truth = _problem(n, seed=n + 7)
    fn = R.mse_pearson_grad_loss if with_mse else R.pearson_loss
    _, g = _autograd(fn, coords, truth)
    want = R.closed_form_grad(coords.numpy(), truth.numpy(), with_mse)
    assert np.abs(g.numpy() - want).max() <= 1e-10 * np.abs(want).max()


@pytest.mark.parametrize("n", [5, 90])
def test_gradient_invariants(n):
    coords, truth = _problem(n, seed=3 * n)
    for fn in (R.pearson_loss, R.mse_pearson_grad_loss):
        _, g = _autograd(fn, coords, truth)
        assert float(g.sum(0).abs().max()) < 1e-12 * float(g.abs().max()) * n  # translation invariance
    _, g = _autograd(R.pearson_loss, coords, truth)
    # r is invariant under scaling every distance: <g, x> = d(1 - r)/ds at s = 1 = 0
    assert abs(float((g * coords).sum())) < 1e-12 * float(g.abs().max() * coords.abs().max()) * n


def test_degenerate_moments_nan_value_zero_pearson_gradient():
    coords, truth = _problem(6, seed=1)
    cases = [
        (coords[:2], truth[:2, :2]),                 # n = 2: one pair, no variance
        (torch.zeros(6, 3, dtype=torch.float64), truth),  # every locus coincident
        (coords, torch.ones(6, 6, dtype=torch.float64) - torch.eye(6, dtype=torch.float64)),  # constant target
    ]
    for c, t in cases:
        val, g = _autograd(R.pearson_loss, c, t)
        assert torch.isnan(val)
        assert torch.equal(g, torch.zeros_like(g))
        total, g2 = _autograd(R.mse_pearson_grad_loss, c, t)
        assert torch.isnan(total)
        _, g_mse = _autograd(lambda x, y: ((torch.cdist(x, x) - y) ** 2).mean(), c, t)
        assert torch.allclose(g2, g_mse, rtol=0, atol=1e-15)
        assert np.allclose(R.closed_form_grad(c.numpy(), t.numpy(), False), 0.0)


def test_loss_from_moments_degenerate_and_regular():
    n = 30
    coords, truth = _problem(n, seed=11)
    iu = torch.triu_indices(n, n, 1)
    d = torch.cdist(coords, coords)
    dp, tp = d[iu[0], iu[1]], truth[iu[0], iu[1]]
    m = torch.tensor([float(((d - truth) ** 2).sum()), 0.0, float(dp.sum()), float((dp * dp).sum()), float(tp.sum()), float((tp * tp).sum()),
                      float((dp * tp).sum()), 0.0], dtype=torch.float64)
    assert abs(float(pearson_loss_from_moments(m, n, False)) - float(R.pearson_loss(coords, truth))) < 1e-12
    # the training loss takes its MSE term as MSELoss returns it (f32), the reference keeps it in f64
    want = float(R.mse_pearson_grad_loss(coords, truth)[0])
    assert abs(float(pearson_loss_from_moments(m, n, True)) - want) < 1e-7 * want
    flat = m.clone()
    flat[4], flat[5] = float(tp.numel()), float(tp.numel())  # a constant target of ones
    assert torch.isnan(pearson_loss_from_moments(flat, n, False))
    assert torch.isnan(pearson_loss_from_moments(flat, n, True))


# ------------------------------------------------------------------------------ sharded reducer on gloo
def _block_moments(c, t, r0, r1, out):
    """Pass-1 stand-in: HICGAT_PAIR_MOMENTS_D of rows [r0, r1) (slots 4, 5 come from the target constants)."""
    n = c.shape[0]
    d = torch.cdist(c[r0:r1], c)
    tb = t[r0:r1]
    up = torch.arange(r0, r1).unsqueeze(1) < torch.arange(n).unsqueeze(0)
    out.zero_()
    out[0] = ((d - tb) ** 2).sum()
    out[2], out[3], out[6], out[7] = d[up].sum(), (d[up] ** 2).sum(), (d[up] * tb[up]).sum(), ((d - tb)[up] ** 2).sum()


def _block_grad(c, t, r0, r1, m, with_mse):
    """Pass-2 stand-in: column-side sums of rows [r0, r1) with the coefficients of the GLOBAL moments m."""
    n = c.shape[0]
    p = n * (n - 1) / 2.0
    sd, sdd, st, stt, sdt = (float(m[k]) for k in (2, 3, 4, 5, 6))
    vd, vt, cov = sdd - sd * sd / p, stt - st * st / p, sdt - sd * st / p
    beta, kappa, lam_a = 0.0, 0.0, 0.0
    if vd * vt > 0:
        beta = cov / vd
        kappa = st / p - beta * sd / p
        lam_a = -1.0 / np.sqrt(vd * vt)
    if with_mse:
        lam_a *= min(1.0, 0.1 + 1.0 / (float(np.float32(float(m[0]) / n**2)) + 1e-6))
    d = torch.cdist(c[r0:r1], c)
    tb = t[r0:r1]
    w = lam_a * (tb - beta * d - kappa) + ((4.0 / n**2) * (d - tb) if with_mse else 0.0)
    w = torch.where(d > 0, w / d.clamp(min=1e-300), torch.zeros_like(d))
    diff = c.unsqueeze(0) - c[r0:r1].unsqueeze(1)  # x_j - x_i
    return (w.unsqueeze(-1) * diff).sum(0)


def _worker(rank, world, port, n, tmpdir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        coords, truth = _problem(n, seed=5)
        iu = torch.triu_indices(n, n, 1)
        tp = truth[iu[0], iu[1]]
        # target constants of THIS block, all-reduced once (WishTarget.t_moments of each rank's rows)
        r0, r1 = sharding.row_block(n, rank, world)
        mine = (iu[0] >= r0) & (iu[0] < r1)
        const = torch.zeros(8, dtype=torch.float64)
        const[4], const[5] = tp[mine].sum(), (tp[mine] ** 2).sum()
        const = sharding.allreduce_packed(const)
        for with_mse in (False, True):
            red = sharding.TwoPassShardedPairLoss(
                n, lambda c, out: _block_moments(c, truth, r0, r1, out), lambda c, m: _block_grad(c, truth, r0, r1, m, with_mse), "cpu",
                moment_const=const)
            moments, grad = red(coords)
            fn = R.mse_pearson_grad_loss if with_mse else R.pearson_loss
            val, g = _autograd(fn, coords, truth)
            tol = 1e-7 if with_mse else 1e-12  # the total's MSE term is the f32 value MSELoss returns
            assert abs(float(pearson_loss_from_moments(moments, n, with_mse)) - float(val)) < tol * max(1.0, abs(float(val)))
            assert float((grad.double() - g).abs().max() / g.abs().max()) < 1e-6  # f32 result of an f64 sum
        open(os.path.join(tmpdir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,n", [(2, 37), (3, 10)])
def test_two_exchange_reducer_gloo(tmp_path, world, n):
    port = 31500 + os.getpid() % 2000 + world
    mp.spawn(_worker, args=(world, port, n, str(tmp_path)), nprocs=world, join=True)
    assert all((tmp_path / f"ok{r}").exists() for r in range(world))


# ------------------------------------------------------------------------------ C ABI argument validation (no CUDA call is reached)
@pytest.fixture(scope="module")
def lib():
    from hic_gnn_b200 import build

    build.build()
    return N.lib()


def test_pearson_entry_points_reject_bad_arguments(lib):
    buf = (ctypes.c_double * 64)()
    p = ctypes.addressof(buf)
    dense = lambda mode, mom, grad: lib.hicgat_pairloss_pearson_grad(p, p, 8, 8, 0, 8, mode, mom, 0.0, 0, grad, p, 64, None)
    sparse = lambda mode, mom, grad: lib.hicgat_pairloss_sparse_pearson_grad(p, p, p, p, 1.0, 8, 0, 8, mode, mom, 0.0, 0, grad, p, 64, None)
    for call in (dense, sparse):
        assert call(0, None, p) == -1 and b"null" in lib.hicgat_last_error()
        assert call(0, p, None) == -1 and b"null" in lib.hicgat_last_error()
        for bad in (N.PAIR_GRAD_L1, N.PAIR_GRAD_MSE | N.PAIR_GRAD_L1, N.PAIR_MOMENTS, N.PAIR_MOMENTS_D, 64, 128, 1 << 31):
            assert call(bad, p, p) == -1, bad
            assert b"mode" in lib.hicgat_last_error()
    # the internal Pearson bit is not accepted by the one-pass entry points either
    assert lib.hicgat_pairloss_fwd_bwd(p, p, 8, 8, 0, 8, 64, 0.0, 0.0, p, p, p, 64, None) == -1
    assert b"unknown mode bits" in lib.hicgat_last_error()
