"""The implicit (sparse) target of the fused pair loss (``SparseWishTarget``: ``fill`` everywhere, 0 on the diagonal, ``tval`` at the
stored pairs of a symmetric CSR pattern) against an f64 evaluation of the same sums, without any N x N array on either side.

The reference is :func:`helpers.pair_block_reference` over slabs of ``SLAB`` rows whose target rows are built in f64 from the CSR.
What one row block returns: moments 1..7 are sums over its pairs i < j, comparable per block; the CSR correction adds moment 0 and
the gradient as ROW-side sums of every stored pair of the block's rows, so those two are only defined for the sum over a partition
of all rows.  Tolerances are the suite's: moments 1e-6 relative, gradients 1e-5 of the max norm (plus the sign ambiguity of the L1
weight, see :func:`_slack_at_fill`)."""
import functools

import pytest
import torch

from helpers import grad_within, pair_block_reference, random_coords, rel_err, small_map

pytestmark = pytest.mark.gpu
TOL = 1e-5
MTOL = 1e-6
SLAB = 512
MODES = list(range(1, 10))  # every combination of GRAD_MSE (1), GRAD_L1 (2), MOMENTS (4), MOMENTS_D (8) the kernels instantiate
F32_EPS = 2.0 ** -24


@pytest.fixture(params=[True, False], ids=["upper", "fullrow"])
def upper(request, monkeypatch):
    from hic_gnn_b200 import ops

    monkeypatch.setattr(ops, "_USE_UPPER", request.param)
    return request.param


@pytest.fixture
def tuning():
    from hic_gnn_b200 import _native as N

    yield N.set_pairloss_tuning
    N.set_pairloss_tuning(0, 0)


def _coefs(n):
    return 4.0 / (float(n) * float(n)), 0.1 / max(n * (n - 1) / 2.0, 1.0)


def _target(n, a, b, fill=1.0, seed=0):
    """SparseWishTarget of the undirected pairs {a_k, b_k} (a_k != b_k, repeats allowed): t_ij = t_ji drawn from [0.05, 3] (above
    and below every fill used here), every fifth pair exactly ``fill``."""
    from hic_gnn_b200 import ops

    a = torch.as_tensor(a, dtype=torch.int64).cuda().reshape(-1)
    b = torch.as_tensor(b, dtype=torch.int64).cuda().reshape(-1)
    assert bool((a != b).all()) and (a.numel() == 0 or (int(a.min()) >= 0 and int(torch.maximum(a, b).max()) < n))
    key = torch.unique(torch.minimum(a, b) * n + torch.maximum(a, b))
    lo, hi = key // n, key % n
    g = torch.Generator(device="cuda").manual_seed(seed)
    t = 0.05 + 2.95 * torch.rand(key.numel(), generator=g, device="cuda", dtype=torch.float64)
    t[::5] = fill
    t = t.float()
    row, col, val = torch.cat([lo, hi]), torch.cat([hi, lo]), torch.cat([t, t])
    order = torch.argsort(row * n + col)
    rowptr = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    rowptr[1:] = torch.cumsum(torch.bincount(row, minlength=n), 0)
    return ops.SparseWishTarget(n, rowptr.int(), col[order].int(), val[order].contiguous(), fill)


@functools.lru_cache(maxsize=None)
def _pattern(n, fill=1.0, seed=0):
    """Hand-built map: rows with exactly 0, 1, 31, 32, 33 and 64 stored pairs (the CSR correction's lane-strided loop: one warp per
    row, 32 lanes), a hub row paired with ~7/8 of all loci, pairs at j = i +- 1, on the column-strip boundaries 127/128 and 255/256,
    and random pairs.  Returns the target and {designed row: its number of pairs}."""
    g = torch.Generator().manual_seed(1000 + n)
    pairs = []
    designed = {}
    if n >= 400:
        degrees = [0, 1, 31, 32, 33, 64]
        special = [n // 5 + 7 * k for k in range(len(degrees))]
        hub = n // 3
        pool = torch.tensor([j for j in range(n) if j not in special and j != hub])
        for r, deg in zip(special, degrees):
            partners = pool[torch.randperm(pool.numel(), generator=g)[:deg]]
            pairs += [(r, int(j)) for j in partners]
            designed[r] = deg
        free = [j for j in range(n) if j not in special]
    else:
        hub, free = (n // 3 if n >= 3 else None), list(range(n))
    fs = set(free)
    pairs += [(i, i + 1) for i in free[::3] if i + 1 in fs]                       # j = i + 1 (and i - 1 from the other side)
    for a, b in [(127, 128), (255, 256), (126, 128), (127, 255), (128, 256), (0, 127), (0, 128), (0, 255), (0, 256), (129, 383)]:
        if b < n and a in fs and b in fs:
            pairs.append((a, b))
    if hub is not None:
        pairs += [(hub, j) for j in free if j != hub and j % 8 != 5]
    if len(free) >= 2:
        fr = torch.tensor(free)
        a = fr[torch.randint(len(free), (2 * n,), generator=g)]
        b = fr[torch.randint(len(free), (2 * n,), generator=g)]
        keep = a != b
        pairs += list(zip(a[keep].tolist(), b[keep].tolist()))
    a = [p[0] for p in pairs]
    b = [p[1] for p in pairs]
    tgt = _target(n, a, b, fill, seed)
    rp = tgt.rowptr.long().cpu()
    for r, deg in designed.items():
        assert int(rp[r + 1] - rp[r]) == deg, (r, deg)
    return tgt, designed


def _rows_f64(tgt, s0, s1):
    """Target rows [s0, s1) in f64: fill, 0 on the diagonal, tval at the stored pairs."""
    n = tgt.n
    rows = torch.full((s1 - s0, n), tgt.fill, dtype=torch.float64, device="cuda")
    ar = torch.arange(s1 - s0, device="cuda")
    rows[ar, s0 + ar] = 0.0
    rp = tgt.rowptr.long()
    k0, k1 = int(rp[s0]), int(rp[s1])
    if k1 > k0:
        row_of = torch.repeat_interleave(torch.arange(s0, s1, device="cuda"), rp[s0 + 1:s1 + 1] - rp[s0:s1])
        rows[row_of - s0, tgt.col[k0:k1].long()] = tgt.tval[k0:k1].double()
    return rows


def _reference(coords, tgt, r0, r1, upper, mode, c_mse, c_l1, absum=False):
    """f64 (moments, grad, slack[, absum]) of rows [r0, r1), summed over slabs of SLAB rows.  ``absum`` (per gradient element):
    sum |w| |x_j - x_i| over the terms the element adds, the size of what an f32 evaluation rounds."""
    n = tgt.n
    c = coords.double().cuda()
    m = torch.zeros(8, dtype=torch.float64, device="cuda")
    grad = torch.zeros(n, 3, dtype=torch.float64, device="cuda")
    slack = torch.zeros_like(grad)
    size = torch.zeros_like(grad)
    for s0 in range(r0, r1, SLAB):
        s1 = min(s0 + SLAB, r1)
        rows = _rows_f64(tgt, s0, s1)
        mb, gb, sb = pair_block_reference(c, rows, s0, upper, mode, c_mse, c_l1, chunk=SLAB, with_slack=True)
        m += mb
        grad += gb
        slack += sb
        if absum:
            ci = c[s0:s1]
            d = torch.cdist(ci, c, compute_mode="donot_use_mm_for_euclid_dist")
            ii = torch.arange(s0, s1, device="cuda").unsqueeze(1)
            live = ((ii < torch.arange(n, device="cuda").unsqueeze(0)) if upper else torch.ones_like(d, dtype=torch.bool)) & (d > 0)
            w = torch.where(live, (c_mse * (d - rows).abs() * (mode & 1) + c_l1 * (mode & 2)) / d.clamp(min=1e-300), torch.zeros_like(d))
            del rows
            for q in range(3):
                term = w * (c[:, q].unsqueeze(0) - ci[:, q].unsqueeze(1)).abs()
                size[:, q] += term.sum(0)
                if upper:
                    size[s0:s1, q] += term.sum(1)
    return (m, grad, slack, size) if absum else (m, grad, slack)


def _slack_at_fill(coords, tgt, c_l1):
    """L1 sign ambiguity the dense reference does not see: at a stored pair whose d is within the f32 error of its distance
    (2e-6 d) of ``fill``, the background kernel and the CSR correction each take their own sign of d - fill.  Every stored pair
    is held in both directions, so a row-side sum over the CSR covers both of its loci."""
    c = coords.double().cuda()
    rp = tgt.rowptr.long()
    row = torch.repeat_interleave(torch.arange(tgt.n, device="cuda"), rp[1:] - rp[:-1])
    col = tgt.col.long()
    diff = (c[col] - c[row]).abs()
    d = diff.norm(dim=1)
    amb = torch.where((d - tgt.fill).abs() <= 2e-6 * d, 2 * c_l1 / d.clamp(min=1e-300), torch.zeros_like(d))
    out = torch.zeros(tgt.n, 3, dtype=torch.float64, device="cuda")
    out.index_add_(0, row, amb.unsqueeze(1) * diff)
    return out


def _check_moments(got, want, scale, what):
    """Per moment: 1e-6 relative, never tighter than 1e-6 of 1e-3 of the (sum d^2 + sum t^2) scale (n <= 3: one to three pairs,
    where d ~ t makes a moment of e = d - t a cancellation of two f32 numbers)."""
    got, want = got.double().cpu(), want.double().cpu()
    for k in range(8):
        assert abs(float(got[k] - want[k])) <= MTOL * max(abs(float(want[k])), 1e-3 * scale, 1e-12), (what, k, float(got[k]), float(want[k]))


def _check_full(coords, tgt, upper, mode, got_m, got_g, tol=TOL):
    n = tgt.n
    c_mse, c_l1 = _coefs(n)
    want_m, want_g, slack = _reference(coords, tgt, 0, n, upper, mode, c_mse, c_l1)
    full, _, _ = _reference(coords, tgt, 0, n, upper, 4, 0.0, 0.0) if not mode & 4 else (want_m, None, None)
    _check_moments(got_m, want_m, float(full[3] + full[5]), (n, upper, mode))
    if mode & 3:
        if mode & 2:
            slack = slack + _slack_at_fill(coords, tgt, c_l1)
        assert grad_within(got_g, want_g, slack, tol), (n, upper, mode, rel_err(got_g, want_g))


@pytest.mark.parametrize("n", [1, 2, 3, 127, 128, 129, 1000, 2493])
def test_every_mode_matches_f64(n, upper):
    from hic_gnn_b200 import ops

    tgt, _ = _pattern(n)
    coords = random_coords(n, seed=n + 5)
    c_mse, c_l1 = _coefs(n)
    for mode in MODES:
        m, g = ops.pairloss_raw(coords.cuda(), tgt, mode, c_mse, c_l1)
        _check_full(coords, tgt, upper, mode, m, g, TOL if n > 3 else 1e-4)


@pytest.mark.parametrize("fill", [0.5, 2.0])
def test_fill_other_than_one(fill, upper):
    from hic_gnn_b200 import ops

    n = 1000
    tgt, _ = _pattern(n, fill=fill, seed=1)
    coords = random_coords(n, seed=11)
    c_mse, c_l1 = _coefs(n)
    for mode in (1, 2, 5, 6, 7, 9):
        m, g = ops.pairloss_raw(coords.cuda(), tgt, mode, c_mse, c_l1)
        _check_full(coords, tgt, upper, mode, m, g)


@pytest.mark.parametrize("mode", [6, 7, 9])
def test_row_partitions_sum_to_f64(mode, upper):
    """Blocks with an empty block, a one-row block and cuts off the multiples of 8 / 64 / 128: moments 1..7 per block, moment 0
    and the gradient over the partition."""
    from hic_gnn_b200 import ops

    n = 1000
    tgt, _ = _pattern(n, seed=2)
    coords = random_coords(n, seed=12)
    c_mse, c_l1 = _coefs(n)
    m_sum = torch.zeros(8, dtype=torch.float64, device="cuda")
    g_sum = torch.zeros(n, 3, dtype=torch.float64, device="cuda")
    _, want_g, slack = _reference(coords, tgt, 0, n, upper, mode, c_mse, c_l1)
    want_m0 = 0.0
    for r0, r1 in [(0, 0), (0, 1), (1, 9), (9, 70), (70, 201), (201, 201), (201, 643), (643, 999), (999, 1000)]:
        m, g = ops.pairloss_raw(coords.cuda(), tgt.rows(r0, r1), mode, c_mse, c_l1)
        want, _, _ = _reference(coords, tgt, r0, r1, upper, mode | 4, c_mse, c_l1)
        ref, _, _ = _reference(coords, tgt, r0, r1, upper, mode, c_mse, c_l1)
        got = m.clone()
        got[0] = ref[0]  # moment 0 of one block is not defined (see the module docstring): checked on the sum below
        _check_moments(got, ref, float(want[3] + want[5]), (r0, r1, mode))
        want_m0 += float(ref[0])
        m_sum += m
        if g is not None:
            g_sum += g.double()
    assert abs(float(m_sum[0]) - want_m0) <= MTOL * abs(want_m0)
    if mode & 2:
        slack = slack + _slack_at_fill(coords, tgt, c_l1)
    assert grad_within(g_sum, want_g, slack, TOL), rel_err(g_sum, want_g)


@pytest.mark.parametrize("n,density", [(600, 0.05), (1500, 0.02)])
def test_synthetic_maps_from_both_loaders(n, density, upper):
    """Targets of ``load_input`` (dense map) and ``load_input_sparse`` (its contact list) against f64."""
    import numpy as np

    from hic_gnn_b200 import ops, utils

    adj = small_map(n, density, seed=n)
    iu = np.triu_indices(n)
    a = adj.numpy()
    keep = a[iu] != 0
    lst = np.stack([iu[0][keep], iu[1][keep], a[iu][keep]], axis=1)
    targets = [utils.sparse_wish_target(utils.load_input(a.copy(), np.zeros((n, 4))), 1.0),
               utils.sparse_wish_target(utils.load_input_sparse(lst), 1.0)]
    for tgt in targets:
        coords = random_coords(tgt.n, seed=n + 3)
        c_mse, c_l1 = _coefs(tgt.n)
        for mode in (5, 6, 9):
            m, g = ops.pairloss_raw(coords.cuda(), tgt, mode, c_mse, c_l1)
            _check_full(coords, tgt, upper, mode, m, g)


@pytest.mark.parametrize("rb", [0, 8, 64, 1024, 1512, 2048, 4096])
def test_per_lane_tunings(rb, upper, tuning):
    """``set_pairloss_tuning(rb, 1)`` at 5 000 loci: row chunks of up to 4 096 rows for the implicit target and for a dense target
    on the per-lane-load kernel (x_i of a chunk longer than 1 024 rows is staged in pieces), against f64.  The Pearson second pass
    against its default-tuning result (pinned to f64 by test_gpu_pearson_grad.py)."""
    import hic_gnn_b200 as hg
    from hic_gnn_b200 import _native as N
    from hic_gnn_b200 import ops

    n = 5000
    tgt, _ = _pattern(n, seed=3)
    dense = hg.WishTarget.from_dense(_rows_f64(tgt, 0, n).float(), symmetric=True)
    coords = random_coords(n, seed=13).cuda()
    c_mse, c_l1 = _coefs(n)
    targets = {"sparse": tgt, "dense": dense}
    mom, _ = ops.pairloss_raw(coords, tgt, N.PAIR_MOMENTS, 0.0, 0.0)
    pearson = {(name, w): ops.pearson_grad_raw(coords, t, mom, w) for name, t in targets.items() for w in (False, True)}
    tuning(rb, 1)
    for mode in (5, 6):
        want_m, want_g, slack = _reference(coords, tgt, 0, n, upper, mode, c_mse, c_l1)
        for name, t in targets.items():
            m, g = ops.pairloss_raw(coords, t, mode, c_mse, c_l1)
            _check_moments(m, want_m, float(want_m[3] + want_m[5]), (rb, name, mode))
            s = slack + _slack_at_fill(coords, tgt, c_l1) if (mode & 2 and name == "sparse") else slack
            assert grad_within(g, want_g, s, TOL), (rb, name, mode, rel_err(g, want_g))
    for (name, w), g0 in pearson.items():
        g = ops.pearson_grad_raw(coords, targets[name], mom, w)
        assert rel_err(g, g0) < TOL, (rb, name, w, rel_err(g, g0))


def _large(n, hub_every=8):
    """n loci, 16 stored pairs per row (offsets +-1, 2, 3, 5, 8, 13, 64, 128) and a hub paired with 7/8 of all loci."""
    i = torch.arange(n, device="cuda")
    a, b = [], []
    for o in (1, 2, 3, 5, 8, 13, 64, 128):
        a.append(i[: n - o])
        b.append(i[o:])
    hub = n // 3
    j = i[(i % hub_every != 5) & (i != hub)]
    a.append(torch.full_like(j, hub))
    b.append(j)
    return _target(n, torch.cat(a), torch.cat(b), 1.0, seed=n)


@pytest.mark.parametrize("n,cut", [(110592, 50000), (110593, 60001), (120000, 64000)])
def test_large_maps(n, cut, upper):
    """Maps whose row block gets chunks longer than 1 024 rows (above 110 592 loci, to stay within the chunk table): the full launch
    against f64, against the sum of two row blocks of at most 110 592 rows (the bounds of
    test_row_sharded_blocks_sum_to_full_and_are_deterministic), and bit-identical on a second call.  Gradient elements may also be
    off by a few f32 unit roundoffs of the size of their terms (sum |w (x_j - x_i)|): the ratio of the largest error to the max
    norm is printed."""
    from hic_gnn_b200 import ops

    tgt = _large(n)
    coords = random_coords(n, seed=17).cuda()
    c_mse, c_l1 = _coefs(n)
    mode = 7
    m, g = ops.pairloss_raw(coords, tgt, mode, c_mse, c_l1)
    m2, g2 = ops.pairloss_raw(coords, tgt, mode, c_mse, c_l1)
    assert torch.equal(m, m2) and torch.equal(g, g2)
    m_sum = torch.zeros_like(m)
    g_sum = torch.zeros(n, 3, dtype=torch.float64, device="cuda")
    for r0, r1 in [(0, cut), (cut, n)]:
        mb, gb = ops.pairloss_raw(coords, tgt.rows(r0, r1), mode, c_mse, c_l1)
        m_sum += mb
        g_sum += gb.double()
    assert rel_err(m_sum, m) < 1e-8
    assert rel_err(g_sum, g) < 1e-6
    want_m, want_g, slack, size = _reference(coords, tgt, 0, n, upper, mode, c_mse, c_l1, absum=True)
    _check_moments(m, want_m, float(want_m[3] + want_m[5]), (n, upper))
    slack = slack + _slack_at_fill(coords, tgt, c_l1)
    err = (g.double() - want_g).abs()
    print(f"n={n} upper={upper}: max |g - f64| / max |g| = {float(err.max() / want_g.abs().max()):.3e}, "
          f"beyond 1e-5 max|g| + L1 slack in units of eps32 * sum|w dx|: {float(((err - TOL * want_g.abs().max() - slack) / (F32_EPS * size).clamp(min=1e-300)).max()):.3f}")
    assert bool((err <= TOL * want_g.abs().max() + slack + 4 * F32_EPS * size).all())
