"""The routes into the fused pair loss other than the resident ``hicgat_pairloss_fwd_bwd`` call, and the read contract of the
upper-triangle mode (HICGAT_PAIR_SYMMETRIC):

* the lower-triangle contract: columns left of a row's diagonal 128-column strip never enter the result (NaN there changes
  nothing), entries below the diagonal inside the strip are cancelled exactly -- for every kernel variant;
* ``hicgat_pairloss_fwd_bwd_packed`` (the buffer a sharded run all-reduces) against the unpacked call, bit for bit;
* ``ops.sharded_reducer`` on one process (the NCCL transport's ``local_fn``), alone and as emulated ranks;
* ``ops.HostPairLoss`` (target in pinned host memory, streamed through two staging buffers) against a resident replay."""
import pytest
import torch

from helpers import grad_within, pair_block_reference, poison_lower, random_coords, rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-5
VARIANTS = (0, 1, 2, 3, 4)
MODES = ("value", "moments", "mse", "mse_moments", "mse_moments_full", "contrastive")


def _sym_matrix(n, seed):
    """Symmetric f32 target on the device with a non-zero diagonal (MSELoss over the full matrix counts t_ii^2)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    t = torch.rand(n, n, generator=g, device="cuda")
    t = torch.triu(t) + torch.triu(t, 1).t()
    t.diagonal().mul_(0.05)
    return t


def _coefs(n):
    return 4.0 / (float(n) * float(n)), 0.1 / max(n * (n - 1) / 2.0, 1.0)


def _block(full, r0, r1, symmetric, rows=None):
    import hic_gnn_b200 as hg

    n = full.shape[0]
    blk = hg.WishTarget.empty(n, r0, r1, symmetric=symmetric)
    if r1 > r0:
        blk.data[:, :n].copy_(full[r0:r1] if rows is None else rows)
    return blk


def _equal(a, b):
    """Bit-identical up to the sign of zero (a weight of 0 times a negative residual is -0)."""
    return a is None and b is None or torch.equal(a, b)


# ------------------------------------------------------------------------------ lower-triangle contract
@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("n,cuts", [(1, [0, 1]), (2, [0, 1, 1, 2]), (130, [0, 3, 3, 67, 130]), (1001, [0, 5, 133, 700, 1001]),
                                    (3001, [0, 250, 1003, 1003, 3001]), (19500, [100, 6045])])
def test_lower_triangle_never_enters_the_result(n, cuts, variant):
    """Every variant in upper-triangle mode: a block with NaN left of each row's diagonal strip and finite garbage below the diagonal
    inside it gives moments and gradient bit-identical to a clean copy of the same symmetric rows, in every mode and in the Pearson
    pass.  19 500 loci: more than 148 strips (staggered chunk tables), a block that starts inside a strip."""
    from hic_gnn_b200 import _native as N
    from hic_gnn_b200 import ops

    full = _sym_matrix(n, seed=n)
    coords = random_coords(n, seed=n + 1).cuda()
    c_mse, c_l1 = _coefs(n)
    glob = ops.pairloss_raw(coords, _block(full, 0, n, True), N.PAIR_MOMENTS, 0.0, 0.0)[0].clone()  # moments for the Pearson pass
    try:
        N.set_pairloss_tuning(0, variant)
        for r0, r1 in zip(cuts[:-1], cuts[1:]):
            clean = _block(full, r0, r1, True)
            bad = _block(full, r0, r1, True, rows=poison_lower(full[r0:r1], r0, seed=r0) if r1 > r0 else None)
            if r1 - r0 > 0 and r0 // 128 * 128 > 0:
                assert bool(bad.dense().isnan().any())
            for mode in MODES:
                m1, g1 = (None if x is None else x.clone() for x in ops.pairloss_raw(coords, clean, ops._MODES[mode], c_mse, c_l1))
                m2, g2 = ops.pairloss_raw(coords, bad, ops._MODES[mode], c_mse, c_l1)
                assert _equal(m1, m2) and _equal(g1, g2), (mode, r0, r1)
                assert bool(torch.isfinite(m2).all()), (mode, r0, r1)
            for with_mse in (False, True):
                g1 = ops.pearson_grad_raw(coords, clean, glob, with_mse).clone()
                g2 = ops.pearson_grad_raw(coords, bad, glob, with_mse)
                assert torch.equal(g1, g2), ("pearson", with_mse, r0, r1)
    finally:
        N.set_pairloss_tuning(0, 0)


# ------------------------------------------------------------------------------ packed entry point
def _packed(coords, blk, bits, c_mse, c_l1):
    from hic_gnn_b200 import _native as N

    n = blk.n
    lib = N.lib()
    ws = torch.zeros(lib.hicgat_pairloss_workspace_bytes_mode(n, blk.r0, blk.r1, bits), dtype=torch.uint8, device="cuda")
    out = torch.full((N.PAIR_NMOM + 3 * n,), float("nan"), dtype=torch.float64, device="cuda")
    N.check(lib.hicgat_pairloss_fwd_bwd_packed(coords.data_ptr(), blk.data.data_ptr(), blk.pitch, n, blk.r0, blk.r1, bits, c_mse, c_l1, out.data_ptr(),
                                               ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream), "hicgat_pairloss_fwd_bwd_packed")
    return out


def _unpacked(coords, blk, bits, c_mse, c_l1):
    from hic_gnn_b200 import _native as N

    n = blk.n
    lib = N.lib()
    ws = torch.zeros(lib.hicgat_pairloss_workspace_bytes_mode(n, blk.r0, blk.r1, bits), dtype=torch.uint8, device="cuda")
    m = torch.full((N.PAIR_NMOM,), float("nan"), dtype=torch.float64, device="cuda")
    g = torch.full((n, 3), float("nan"), dtype=torch.float32, device="cuda")
    N.check(lib.hicgat_pairloss_fwd_bwd(coords.data_ptr(), blk.data.data_ptr(), blk.pitch, n, blk.r0, blk.r1, bits, c_mse, c_l1, m.data_ptr(),
                                        g.data_ptr() if bits & 3 else None, ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream),
            "hicgat_pairloss_fwd_bwd")
    return m, g


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("n,cuts,combine", [(3001, [0, 5, 1000, 1003, 1003, 3001], (5, 3)), (3001, [0, 5, 1000, 1003, 1003, 3001], (1, 96)), (30000, [2000, 2100], None)])
@pytest.mark.parametrize("upper", [False, True])
def test_packed_matches_unpacked_bit_for_bit(n, cuts, combine, upper, variant):
    """``packed[:8] == moments`` and ``packed[8:] == grad.double()`` exactly, into a buffer pre-filled with NaN: every element is
    written.  Modes without a gradient and empty blocks give a zero gradient part.  The segmented row-side combine is on (5, 3 and
    the default at 30 000 loci on a short block) and off (1, 96)."""
    import hic_gnn_b200 as hg
    from hic_gnn_b200 import _native as N
    from hic_gnn_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(n)
    coords = random_coords(n, seed=n).cuda()
    c_mse, c_l1 = _coefs(n)
    try:
        N.set_pairloss_tuning(0, variant)
        if combine is not None:
            N.set_pairloss_combine(*combine)
        for r0, r1 in zip(cuts[:-1], cuts[1:]):
            blk = hg.WishTarget.empty(n, r0, r1, symmetric=True if upper else None)
            if r1 > r0:
                blk.data[:, :n].copy_(torch.rand(r1 - r0, n, generator=g, device="cuda"))
            for mode in MODES:
                bits = ops._MODES[mode] | (N.PAIR_SYMMETRIC if upper else 0)
                p = _packed(coords, blk, bits, c_mse, c_l1)
                m, gr = _unpacked(coords, blk, bits, c_mse, c_l1)
                assert torch.equal(p[:N.PAIR_NMOM], m), (mode, r0, r1)
                if bits & 3:
                    assert torch.equal(p[N.PAIR_NMOM:], gr.reshape(-1).double()), (mode, r0, r1)
                else:
                    assert float(p[N.PAIR_NMOM:].abs().sum()) == 0.0, (mode, r0, r1)  # zeros, not NaN
                if r1 == r0:
                    assert float(p.abs().sum()) == 0.0
    finally:
        N.set_pairloss_tuning(0, 0)
        N.set_pairloss_combine()


# ------------------------------------------------------------------------------ sharded reducer, one process
@pytest.mark.parametrize("n", [1500, 3001])
@pytest.mark.parametrize("mode", ["mse", "mse_moments", "contrastive"])
def test_sharded_reducer_single_process(n, mode):
    """Without torch.distributed, ``sharded_reducer`` is the packed kernel behind ``ShardedPairLoss``: on the full block it equals
    the plain call bit for bit; one reducer per block of a W-way upper-area split (W = 3, 8), summed, equals the full call and the
    f64 reference."""
    import hic_gnn_b200 as hg
    from hic_gnn_b200 import _native as N
    from hic_gnn_b200 import ops, sharding

    full = _sym_matrix(n, seed=n + 5)
    coords = random_coords(n, seed=n + 6).cuda()
    tgt = hg.WishTarget.from_dense(full)
    assert tgt.symmetric is True
    c = coords.clone().requires_grad_(True)
    loss, m = hg.pairwise_loss(c, tgt, mode)
    (g,) = torch.autograd.grad(loss, c)
    red = ops.sharded_reducer(tgt, mode)
    assert isinstance(red, sharding.ShardedPairLoss)
    c2 = coords.clone().requires_grad_(True)
    loss2, m2 = hg.pairwise_loss(c2, tgt, mode, reducer=red)
    (g2,) = torch.autograd.grad(loss2, c2)
    assert torch.equal(loss, loss2) and torch.equal(m, m2) and torch.equal(g, g2)
    bits = ops._MODES[mode]
    c_mse, c_l1 = _coefs(n)
    want_m, want_g, slack = pair_block_reference(coords, full, 0, True, bits | N.PAIR_MOMENTS, c_mse, c_l1, with_slack=True)
    if not bits & N.PAIR_MOMENTS:
        want_m[1] = 0.0
        if not bits & N.PAIR_MOMENTS_D:
            want_m[2:] = 0.0
    for world in (3, 8):
        m_sum = torch.zeros_like(m)
        g_sum = torch.zeros(n, 3, dtype=torch.float64, device="cuda")
        for r in range(world):
            r0, r1 = sharding.row_block(n, r, world, "upper")
            blk = hg.WishTarget(tgt.data[r0:r1], n, r0, r1, symmetric=True)
            rr = ops.sharded_reducer(blk, mode)
            mb, _ = rr(coords)
            m_sum += mb
            g_sum += rr.packed[N.PAIR_NMOM:].view(n, 3)
        assert rel_err(m_sum, m) < 1e-7, world
        assert rel_err(g_sum, g) < 1e-6, world
        assert rel_err(m_sum, want_m) < TOL and grad_within(g_sum, want_g, slack, TOL), world


def test_sharded_reducer_asymmetric_target_matches_autograd():
    """An asymmetric target goes through the split call (column-side kernel + row-side pass) and a pack: the reducer on the full
    block equals the plain call, and 3 row blocks summed match the oracle's autograd."""
    import hic_gnn_b200 as hg
    from hic_gnn_b200 import ops, sharding
    from oracle import loss as oloss

    n = 700
    g = torch.Generator().manual_seed(n)
    truth = torch.rand(n, n, generator=g, dtype=torch.float64)
    truth.fill_diagonal_(0)
    truth = truth.float().double()
    coords = random_coords(n, seed=3)
    cc = coords.clone().requires_grad_(True)
    (want_g,) = torch.autograd.grad(oloss.mse_loss(cc, truth), cc)
    tgt = hg.WishTarget.from_dense(truth.cuda())
    assert tgt.symmetric is False
    c = coords.cuda().requires_grad_(True)
    loss, m = hg.pairwise_loss(c, tgt, "mse")
    (gp,) = torch.autograd.grad(loss, c)
    red = ops.sharded_reducer(tgt, "mse")
    c2 = coords.cuda().requires_grad_(True)
    loss2, m2 = hg.pairwise_loss(c2, tgt, "mse", reducer=red)
    (g2,) = torch.autograd.grad(loss2, c2)
    assert torch.equal(loss, loss2) and torch.equal(m, m2) and torch.equal(gp, g2)
    g_sum = torch.zeros(n, 3, dtype=torch.float64, device="cuda")
    for r in range(3):
        r0, r1 = sharding.row_block(n, r, 3)
        blk = hg.WishTarget.from_dense(truth.cuda(), r0, r1)
        assert blk.symmetric is False
        rr = ops.sharded_reducer(blk, "mse")
        rr(coords.cuda())
        g_sum += rr.packed[8:].view(n, 3)
    assert rel_err(g_sum, want_g) < TOL


# ------------------------------------------------------------------------------ host-buffer path
@pytest.mark.parametrize("symmetric", [False, True])
@pytest.mark.parametrize("n", [2, 130, 3001, 19500])
def test_host_pair_loss_matches_resident_replay(n, symmetric):
    """``HostPairLoss`` with NaN in its staging buffers (and, upper-triangle mode, NaN in every host column left of each row's
    diagonal strip): bit-identical to one resident ``pairloss_raw`` per block of the same cuts, accumulated in f64 in block order,
    for every variant, block size and mode; within 1e-5 of the f64 reference (plus the sign ambiguity of the L1 gradient at e = 0,
    which a few of the 1.9e8 pairs at 19 500 loci reach); two calls bit-identical; ``reduce`` called once with the accumulated buffer;
    ``h2d_bytes`` = coordinates + the uploaded part of every block.  The NaN fill is queued on the current stream right before the
    first call: the staging uploads must be ordered after it."""
    import hic_gnn_b200 as hg
    from hic_gnn_b200 import _native as N
    from hic_gnn_b200 import ops

    if symmetric and not ops._USE_UPPER:
        pytest.skip("HICGAT_NO_UPPER=1: the upper-triangle upload is off")
    full = _sym_matrix(n, seed=n + 9)
    coords = random_coords(n, seed=n + 10)
    coords_host = coords.pin_memory()
    c_mse, c_l1 = _coefs(n)
    pitch = hg.WishTarget.pitch_for(n)
    ranges = [(0, n), (n // 2, n // 2)] + ([(37, n - 5)] if n > 42 else [])
    big = n >= 10000
    for r0, r1 in ranges:
        dev = torch.zeros(r1 - r0, pitch, device="cuda")
        if r1 > r0:
            dev[:, :n] = full[r0:r1]
            if symmetric:
                ii = torch.arange(r0, r1, device="cuda").unsqueeze(1)
                jj = torch.arange(pitch, device="cuda").unsqueeze(0)
                dev.masked_fill_(jj < ii // 128 * 128, float("nan"))
        host = dev.cpu().pin_memory()
        refs = {}
        for mode in (("value", "mse_moments_full", "contrastive") if big else MODES):
            bits = ops._MODES[mode]
            refs[mode] = pair_block_reference(coords, full[r0:r1], r0, symmetric, bits, c_mse, c_l1, with_slack=True) if r1 > r0 else None
        for block_rows in ((1000, n + 1) if big else (64, 100, 1000, n + 1)):
            calls = []
            hp = ops.HostPairLoss(n, r0, r1, block_rows=block_rows, reduce=calls.append, symmetric=symmetric)
            for s in hp.stage:
                s.fill_(float("nan"))
            nblk = (r1 - r0 + block_rows - 1) // block_rows
            cuts = [(lo, min(lo + block_rows, r1 - r0)) for lo in range(0, r1 - r0, block_rows)]
            assert len(cuts) == nblk
            want_h2d = 12 * n + sum((hi - lo) * (pitch - ((r0 + lo) // 128 * 128 if symmetric else 0)) * 4 for lo, hi in cuts)
            try:
                for variant in VARIANTS:
                    N.set_pairloss_tuning(0, variant)
                    for mode, ref in refs.items():
                        bits = ops._MODES[mode]
                        calls.clear()
                        m1, g1 = (x.clone() for x in hp(coords_host, host, bits, c_mse, c_l1))
                        assert len(calls) == 1 and calls[0] is hp.acc
                        assert bool(torch.isfinite(m1).all()) and torch.equal(calls[0].cpu()[:N.PAIR_NMOM], m1)
                        assert hp.h2d_bytes == want_h2d
                        m2, g2 = hp(coords_host, host, bits, c_mse, c_l1)
                        assert torch.equal(m1, m2) and torch.equal(g1, g2), (variant, block_rows, mode)
                        # resident replay of the same cuts
                        am = torch.zeros(N.PAIR_NMOM, dtype=torch.float64, device="cuda")
                        ag = torch.zeros(n, 3, dtype=torch.float64, device="cuda")
                        for lo, hi in cuts:
                            blk = hg.WishTarget(dev[lo:hi], n, r0 + lo, r0 + hi, symmetric=True if symmetric else None)
                            m, gr = ops.pairloss_raw(coords.cuda(), blk, bits, c_mse, c_l1)
                            am += m
                            if gr is not None:
                                ag += gr.double()
                        assert torch.equal(m1, am.cpu()) and torch.equal(g1, ag.cpu()), (variant, block_rows, mode)
                        if ref is None:
                            assert float(m1.abs().sum()) == 0.0 and float(g1.abs().sum()) == 0.0
                            continue
                        tol = TOL if n > 3 else 1e-4
                        assert rel_err(m1, ref[0]) < tol, (variant, block_rows, mode)
                        if bits & 3:
                            assert grad_within(g1, ref[1], ref[2], tol), (variant, block_rows, mode)
                        else:
                            assert float(g1.abs().sum()) == 0.0
            finally:
                N.set_pairloss_tuning(0, 0)
