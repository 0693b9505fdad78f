"""GPU parity of the fused pairwise-distance loss (called through the C ABI) against the
oracle's torch.cdist + MSELoss / L1 / scipy glue.  Tolerance: 1e-5 relative on loss values and
gradients (north_star), written next to each assert."""
import numpy as np
import pytest
import torch

from helpers import pair_block_reference, poison_lower, random_coords, rel_err, small_map, wish_from_map

pytestmark = pytest.mark.gpu
TOL = 1e-5


def _oracle_mse(coords, truth):
    from oracle import loss as oloss

    c = coords.clone().requires_grad_(True)
    l = oloss.mse_loss(c, truth)
    (g,) = torch.autograd.grad(l, c)
    return l.detach(), g


def _oracle_contrastive(coords, truth):
    from oracle import loss as oloss

    c = coords.clone().requires_grad_(True)
    l = oloss.contrastive_loss(c, truth)
    (g,) = torch.autograd.grad(l, c)
    return l.detach(), g


def _gpu_loss(coords, truth, mode):
    import hic_gnn_b200 as hg

    tgt = hg.WishTarget.from_dense(truth.cuda())
    c = coords.cuda().requires_grad_(True)
    loss, moments = hg.pairwise_loss(c, tgt, mode)
    (g,) = torch.autograd.grad(loss, c)
    return loss.detach().cpu(), g.cpu(), moments.cpu()


@pytest.mark.parametrize("tag", ["1mb", "500kb"])
def test_mse_on_reference_maps(golden, tag):
    g, _ = golden
    truth = wish_from_map(torch.tensor(g[f"{tag}_kr_oracle"]), 1.0)
    coords = random_coords(truth.shape[0], seed=1)
    want_l, want_g = _oracle_mse(coords, truth)
    got_l, got_g, _ = _gpu_loss(coords, truth, "mse")
    assert got_l.dtype == torch.float32
    assert abs(float(got_l) - float(want_l)) / float(want_l) < TOL
    assert rel_err(got_g, want_g) < TOL


@pytest.mark.parametrize("n,density", [(1, 1.0), (2, 1.0), (3, 1.0), (31, 0.9), (127, 0.5), (128, 0.5), (129, 0.5), (300, 0.95), (1000, 0.3), (2493, 0.95)])
def test_mse_random_maps(n, density):
    # n <= 3: seeded, and scaled away from the typical distance (~0.7) so that d - t is not a cancellation of two f32 numbers
    truth = wish_from_map(small_map(n, density, seed=n), 1.0) if n > 3 else 0.25 * torch.rand(n, n, dtype=torch.float64, generator=torch.Generator().manual_seed(n))
    truth = (truth + truth.t()) / 2
    truth.fill_diagonal_(0)
    coords = random_coords(n, seed=n + 1)
    want_l, want_g = _oracle_mse(coords, truth)
    got_l, got_g, _ = _gpu_loss(coords, truth, "mse")
    # relative to the loss, but never tighter than 1e-5 of 1e-3 * mean(t^2): with one or three pairs the
    # random coordinates can land on d ~ t, where the loss is a cancellation of two f32 distances
    floor = 1e-3 * float((truth.float() ** 2).mean())
    assert abs(float(got_l) - float(want_l)) <= TOL * max(float(want_l), floor, 1e-12)
    if n > 1:
        # n <= 3: one to three pairs, no averaging; a coincidental d ~ t makes (d - t)/d a cancellation
        assert rel_err(got_g, want_g) < (TOL if n > 3 else 1e-4)


@pytest.mark.parametrize("n", [58, 300, 1000])
def test_moments_match_scipy_and_contrastive(n):
    from scipy.stats import pearsonr

    from hic_gnn_b200.ops import pearson_from_moments
    from oracle import loss as oloss

    truth = wish_from_map(small_map(n, 0.6, seed=5), 1.0)
    coords = random_coords(n, seed=2)
    dist_truth, dist_out = oloss.triu_pairs(truth, coords)
    want_r = pearsonr(dist_truth.numpy(), dist_out.numpy())[0]
    npairs = n * (n - 1) / 2
    want_l, want_g = _oracle_mse(coords, truth)
    # per-step training mode (coordinate-dependent moments from the kernel + cached target moments)
    got_l, got_g, m_light = _gpu_loss(coords, truth, "mse_moments")
    assert abs(float(pearson_from_moments(m_light, npairs)) - want_r) < 1e-6
    assert abs(float(got_l) - float(want_l)) / float(want_l) < TOL and rel_err(got_g, want_g) < TOL
    # all moments in one pass
    got_l, got_g, m = _gpu_loss(coords, truth, "mse_moments_full")
    assert abs(float(pearson_from_moments(m, npairs)) - want_r) < 1e-6
    assert abs(float(got_l) - float(want_l)) / float(want_l) < TOL and rel_err(got_g, want_g) < TOL
    for k in (0, 2, 3, 4, 5, 6, 7):
        assert abs(float(m_light[k]) - float(m[k])) <= 1e-6 * abs(float(m[k])), k
    # raw moments
    d, t = dist_out.double(), dist_truth.double()
    for k, want in [(1, (d - t).abs().sum()), (2, d.sum()), (3, (d * d).sum()), (4, t.sum()), (5, (t * t).sum()), (6, (d * t).sum()), (7, ((d - t) ** 2).sum())]:
        assert abs(float(m[k]) - float(want)) / float(want) < TOL, k
    # contrastive mode: value (f64 like the reference) and gradient
    want_l, want_g = _oracle_contrastive(coords, truth)
    got_l, got_g, _ = _gpu_loss(coords, truth, "contrastive")
    assert got_l.dtype == torch.float64
    assert abs(float(got_l) - float(want_l)) / float(want_l) < TOL
    assert rel_err(got_g, want_g) < TOL


def test_row_sharded_blocks_sum_to_full_and_are_deterministic():
    import hic_gnn_b200 as hg
    from hic_gnn_b200 import ops

    n = 777
    truth = wish_from_map(small_map(n, 0.4, seed=8), 1.0).cuda()
    coords = random_coords(n, seed=3).cuda()
    full = hg.WishTarget.from_dense(truth)
    mode = ops._MODES["mse_moments_full"]
    m_full, g_full = ops.pairloss_raw(coords, full, mode, 4.0 / n**2, 0.0)
    m_full2, g_full2 = ops.pairloss_raw(coords, full, mode, 4.0 / n**2, 0.0)
    assert torch.equal(m_full, m_full2) and torch.equal(g_full, g_full2)  # bit-reproducible
    m_sum = torch.zeros_like(m_full)
    g_sum = torch.zeros_like(g_full)
    for r0, r1 in [(0, 200), (200, 200), (200, 601), (601, 777)]:  # includes an empty block
        blk = hg.WishTarget.from_dense(truth, r0, r1)
        m, g = ops.pairloss_raw(coords, blk, mode, 4.0 / n**2, 0.0)
        m_sum += m
        g_sum += g
    assert rel_err(m_sum, m_full) < 1e-8  # f32 per-thread partials are grouped differently per block
    assert rel_err(g_sum, g_full) < 1e-6


def test_tuning_variants_agree():
    """Row-chunk sizes and the two load mechanisms (TMA tile ring / per-lane streaming loads)
    compute the same sums, up to f32 partial-sum grouping."""
    import hic_gnn_b200 as hg
    from hic_gnn_b200 import _native as N
    from hic_gnn_b200 import ops

    n = 1500
    truth = wish_from_map(small_map(n, 0.5, seed=4), 1.0).cuda()
    coords = random_coords(n, seed=5).cuda()
    tgt = hg.WishTarget.from_dense(truth)
    ref = None
    try:
        for variant in (0, 1, 2, 3, 4):
            for rb in (0, 8, 64, 256, 1024):
                N.set_pairloss_tuning(rb, variant)
                for mode in ("mse_moments_full", "contrastive"):
                    m, g = ops.pairloss_raw(coords, tgt, ops._MODES[mode], 4.0 / n**2, 0.1 / (n * (n - 1) / 2))
                    if ref is None:
                        ref = {}
                    if mode not in ref:
                        ref[mode] = (m.clone(), g.clone())
                    assert rel_err(m, ref[mode][0]) < 1e-7 and rel_err(g, ref[mode][1]) < 1e-5, (variant, rb, mode)
    finally:
        N.set_pairloss_tuning(0, 0)


@pytest.mark.parametrize("variant", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("n,r0,r1,rb", [(130, 0, 130, 0), (777, 3, 500, 0), (1000, 999, 1000, 0), (513, 64, 449, 0), (19500, 100, 1000, 128), (19300, 0, 700, 64),
                                        (40000, 5, 205, 0), (80000, 17, 60, 0)])
def test_row_blocks_any_alignment_both_variants(variant, n, r0, r1, rb):
    """Row blocks that start / end at rows that are not multiples of the tile height, single-row
    blocks and blocks shorter than one tile, against an f64 torch evaluation of the same sums."""
    import hic_gnn_b200 as hg
    from hic_gnn_b200 import _native as N
    from hic_gnn_b200 import ops

    g = torch.Generator().manual_seed(n + r0)
    # only the block's rows are needed: the column-side sums of ONE block do not rely on symmetry
    rows = torch.rand(r1 - r0, n, generator=g, dtype=torch.float64)
    rows[torch.arange(r1 - r0), torch.arange(r0, r1)] = 0.0
    coords = random_coords(n, seed=r1)
    c = coords.double()
    d = torch.cdist(c[r0:r1], c)
    t = rows.float().double()
    e = d - t
    up = torch.arange(r0, r1).unsqueeze(1) < torch.arange(n).unsqueeze(0)
    want = torch.tensor([(e * e).sum(), e[up].abs().sum(), d[up].sum(), (d[up] ** 2).sum(), t[up].sum(), (t[up] ** 2).sum(), (d[up] * t[up]).sum(), (e[up] ** 2).sum()])
    w = torch.where(d > 0, e / d.clamp(min=1e-30), torch.zeros_like(d))
    gwant = (4.0 / n**2) * (w.unsqueeze(-1) * (c.unsqueeze(0) - c[r0:r1].unsqueeze(1))).sum(0)
    try:
        N.set_pairloss_tuning(rb, variant)  # n > 148*128 with several chunks exercises the staggered strips
        blk = hg.WishTarget.empty(n, r0, r1)
        blk.data[:, :n].copy_(rows.cuda())
        m, gr = ops.pairloss_raw(coords.cuda(), blk, ops._MODES["mse_moments_full"], 4.0 / n**2, 0.0)
    finally:
        N.set_pairloss_tuning(0, 0)
    assert rel_err(m, want) < TOL
    assert rel_err(gr, gwant) < TOL


def test_pairdist_forward_backward_match_cdist():
    import hic_gnn_b200 as hg

    n = 200
    coords = random_coords(n, seed=6)
    w = torch.rand(n, n)
    c = coords.clone().requires_grad_(True)
    d_ref = torch.cdist(c, c, compute_mode="donot_use_mm_for_euclid_dist")
    (g_ref,) = torch.autograd.grad((d_ref * w).sum(), c)
    cg = coords.cuda().requires_grad_(True)
    d = hg.pairdist(cg)
    (g,) = torch.autograd.grad((d * w.cuda()).sum(), cg)
    assert rel_err(d, d_ref) < 1e-6
    assert rel_err(g, g_ref) < TOL


@pytest.mark.parametrize("n", [9970])
def test_full_size_closed_form_properties(n):
    """Size-independent properties at a BASELINE.json size (10k loci, 1e8 pairs): with
    target = pairwise distances of points y, coords = s*y gives MSE = (s-1)^2 mean(t^2),
    gradient = 4(s-1)/n^2 * sum_j t_ij (y_i-y_j)/|y_i-y_j| ... checked through its closed-form
    contraction <grad, y> = 2 s ... and Pearson r = 1; coords = y gives loss 0 and grad 0."""
    import hic_gnn_b200 as hg
    from hic_gnn_b200.ops import pearson_from_moments

    y = random_coords(n, seed=11).cuda()
    t = hg.pairdist(y)
    tgt = hg.WishTarget.from_dense(t)
    loss0, m0 = hg.pairwise_loss(y.clone().requires_grad_(True), tgt, "mse_moments")
    assert float(loss0.detach()) < 1e-12
    s = 1.25
    c = (s * y).requires_grad_(True)
    loss, m = hg.pairwise_loss(c, tgt, "mse_moments")
    (g,) = torch.autograd.grad(loss, c)
    mean_t2 = float((t.double() ** 2).mean())
    assert abs(float(loss.detach()) - (s - 1) ** 2 * mean_t2) / ((s - 1) ** 2 * mean_t2) < TOL
    # dL/ds = 2 (s-1) mean(t^2)  and  dL/ds = <grad, y>
    assert abs(float((g.double() * y.double()).sum()) - 2 * (s - 1) * mean_t2) / (2 * (s - 1) * mean_t2) < TOL
    assert abs(float(pearson_from_moments(m, n * (n - 1) / 2)) - 1.0) < 1e-6
    assert abs(float(g.double().sum(0).abs().max())) < 1e-6  # translation invariance: sum_i grad_i = 0


def test_full_size_c5_properties_and_row_sharding():
    """BASELINE.json's largest configuration (49 850 loci, 2.5e9 ordered pairs, 9.9 GB f32 target) through
    size-independent properties: target = pairwise distances of points y; coords = y gives loss 0 and gradient
    0; coords = s*y gives MSE = (s-1)^2 mean(t^2), <grad, y> = 2 (s-1) mean(t^2), Pearson r = 1 and a
    translation-free gradient; and the 8 row blocks of an 8-GPU run add up to the full-matrix launch."""
    import hic_gnn_b200 as hg
    from hic_gnn_b200 import ops, sharding
    from hic_gnn_b200.ops import pearson_from_moments

    n = 49850
    if torch.cuda.get_device_properties(0).total_memory < 60e9:
        pytest.skip("needs ~25 GB of device memory")
    y = random_coords(n, seed=21).cuda()
    tgt = hg.WishTarget.empty(n)
    for r0 in range(0, n, 4096):  # target rows = exact f32 distances of y, written block-wise
        r1 = min(r0 + 4096, n)
        tgt.data[r0:r1, :n] = torch.cdist(y[r0:r1].double(), y.double()).float()
    tgt.data[:, :n].fill_diagonal_(0)
    mean_t2 = 0.0
    for r0 in range(0, n, 4096):
        mean_t2 += float((tgt.data[r0:r0 + 4096, :n].double() ** 2).sum())
    mean_t2 /= float(n) * float(n)
    loss0, _ = hg.pairwise_loss(y.clone().requires_grad_(True), tgt, "mse_moments")
    assert float(loss0) < 1e-12 * mean_t2 + 1e-14
    s = 1.25
    c = (s * y).requires_grad_(True)
    loss, m = hg.pairwise_loss(c, tgt, "mse_moments")
    (g,) = torch.autograd.grad(loss, c)
    want = (s - 1) ** 2 * mean_t2
    assert abs(float(loss) - want) / want < TOL
    assert abs(float((g.double() * y.double()).sum()) - 2 * (s - 1) * mean_t2) / (2 * (s - 1) * mean_t2) < TOL
    assert abs(float(pearson_from_moments(m, n * (n - 1) / 2)) - 1.0) < 1e-6
    assert float(g.double().sum(0).abs().max()) < 1e-6 * float(g.abs().max()) * n
    # row blocks of an 8-way split, each through its own launch (what 8 ranks compute), against the full launch
    mode = ops._MODES["mse_moments_full"]
    m_full, g_full = ops.pairloss_raw(c.detach(), tgt, mode, 4.0 / n**2, 0.0)
    m_sum, g_sum = torch.zeros_like(m_full), torch.zeros(n, 3, dtype=torch.float64, device="cuda")
    for rank in range(8):
        r0, r1 = sharding.row_block(n, rank, 8)
        blk = hg.WishTarget(tgt.data[r0:r1], n, r0, r1)
        mb, gb = ops.pairloss_raw(c.detach(), blk, mode, 4.0 / n**2, 0.0)
        m_sum += mb
        g_sum += gb.double()
    assert rel_err(m_sum, m_full) < 1e-7
    assert rel_err(g_sum, g_full) < TOL


# ------------------------------------------------------------------------------ non-symmetric targets
def _asym_truth(n, seed):
    """Wish matrix with t_ij != t_ji, as the reference can produce one (utils.load_input keeps `y` as
    given, utils.py:29-35; convert_to_matrix's triu + tril(mat.T, 1), utils.py:21, is asymmetric on the
    first off-diagonal for lists with lower-triangle records)."""
    truth = wish_from_map(small_map(n, 0.6, seed=seed), 1.0)
    g = torch.Generator().manual_seed(seed)
    noise = 0.2 * torch.rand(n, n, generator=g, dtype=torch.float64)
    truth = truth + torch.triu(noise, 1)      # upper triangle only: T != T^T
    idx = torch.arange(n - 1)
    truth[idx + 1, idx] *= 0.5                # and the first sub-diagonal, like the reference's list quirk
    return truth


@pytest.mark.parametrize("n", [5, 129, 700])
def test_mse_asymmetric_target_matches_autograd(n):
    """The column-side sum is the complete gradient only for t_ij = t_ji.  For an asymmetric truth the target
    build detects it and the row-side term is added: loss, gradient AND the i<j moments must match the
    oracle's autograd / scipy on the same matrix (1e-5)."""
    import hic_gnn_b200 as hg
    from hic_gnn_b200 import ops
    from oracle import loss as oloss

    truth = _asym_truth(n, seed=n)
    assert float((truth - truth.t()).abs().max()) > 1e-3
    coords = random_coords(n, seed=n + 7)
    want_l, want_g = _oracle_mse(coords, truth)
    tgt = hg.WishTarget.from_dense(truth.cuda())
    assert tgt.symmetric is False
    c = coords.cuda().requires_grad_(True)
    loss, moments = hg.pairwise_loss(c, tgt, "mse_moments_full")
    (g,) = torch.autograd.grad(loss, c)
    assert abs(float(loss) - float(want_l)) / float(want_l) < TOL
    assert rel_err(g.cpu(), want_g) < TOL
    # what the symmetric fast path would have produced is measurably wrong here (the test has teeth)
    tgt_wrong = hg.WishTarget.from_dense(truth.cuda(), symmetric=True)
    _, g_wrong = ops.pairloss_raw(coords.cuda(), tgt_wrong, ops._MODES["mse"], 4.0 / n**2, 0.0)
    assert rel_err(g_wrong.cpu(), want_g) > 1e-3
    # moments follow the reference's triu gathers: t_ij with i < j
    dist_truth, dist_out = oloss.triu_pairs(truth, coords)
    d, t = dist_out.double(), dist_truth.double()
    m = moments.cpu()
    for k, want in [(4, t.sum()), (6, (d * t).sum()), (7, ((d - t) ** 2).sum())]:
        assert abs(float(m[k]) - float(want)) / float(want) < TOL, k
    # row blocks: every block adds its own row-side term
    c_mse = 4.0 / n**2
    g_sum = torch.zeros(n, 3, device="cuda")
    cuts = [0, n // 3, n // 3, n]
    for r0, r1 in zip(cuts[:-1], cuts[1:]):
        blk = hg.WishTarget.from_dense(truth.cuda(), r0, r1)
        assert blk.symmetric is False or r0 == r1
        _, gb = ops.pairloss_raw(coords.cuda(), blk, ops._MODES["mse"], c_mse, 0.0)
        g_sum += gb
    assert rel_err(g_sum.cpu(), want_g) < TOL
    with pytest.raises(NotImplementedError, match="symmetric"):
        hg.pairwise_loss(c, tgt, "contrastive")


def test_symmetry_check_on_reference_outputs(golden):
    """Outputs of the reference's own code: cont2dist of the (symmetric) chr19 map is symmetric; the wish matrix of
    the asymmetric `load_input` case and convert_to_matrix's `dup_matrix` are not (max |M - M^T| = 9 for the latter)."""
    import hic_gnn_b200 as hg
    from hic_gnn_b200 import ops, utils

    g, _ = golden
    assert hg.WishTarget.from_dense(torch.tensor(g["1mb_wish_1.0"]).cuda()).symmetric is True
    assert ops.asymmetry(torch.tensor(g["dup_matrix"]).cuda()) == 9.0
    asym = torch.tensor(g["asym_y"]).cuda()
    want = float((asym - asym.t()).abs().max())
    assert want > 0 and ops.asymmetry(asym) == want
    assert utils.wish_target(asym, 1.0).symmetric is False
    # an empty row block is trivially symmetric
    assert ops.asymmetry(asym, 2, 2) == 0.0


# ------------------------------------------------------------------------------ upper-triangle (symmetric) kernel
def _sym_truth(n, seed):
    g = torch.Generator().manual_seed(seed)
    t = torch.rand(n, n, generator=g, dtype=torch.float64)
    t = (t + t.t()) / 2
    d = 0.05 * torch.rand(n, generator=g, dtype=torch.float64)
    t[torch.arange(n), torch.arange(n)] = d  # a NON-zero diagonal: MSELoss over the full matrix counts t_ii^2
    return t.float().double()


@pytest.mark.parametrize("n", [1, 2, 7, 64, 127, 128, 129, 257, 1000, 2493])
@pytest.mark.parametrize("mode", ["mse", "mse_moments_full", "contrastive"])
def test_upper_triangle_kernel_matches_oracle(n, mode):
    """HICGAT_PAIR_SYMMETRIC streams only column >= row and evaluates every unordered pair once (column-side sum for j,
    row-side sum for i).  Loss, gradient and moments against the oracle's autograd on the full symmetric matrix: 1e-5."""
    import hic_gnn_b200 as hg
    from hic_gnn_b200 import ops

    truth = _sym_truth(n, n)
    coords = random_coords(n, seed=n + 3)
    tgt = hg.WishTarget.from_dense(truth.cuda())
    assert tgt.symmetric is True and ops.uses_upper_triangle(tgt)
    c = coords.cuda().requires_grad_(True)
    loss, moments = hg.pairwise_loss(c, tgt, mode)
    if mode == "contrastive":
        if n < 2:
            return
        want_l, want_g = _oracle_contrastive(coords, truth)
    else:
        want_l, want_g = _oracle_mse(coords, truth)
    (g,) = torch.autograd.grad(loss, c)
    floor = 1e-3 * float((truth.float() ** 2).mean())
    assert abs(float(loss) - float(want_l)) <= TOL * max(abs(float(want_l)), floor, 1e-12), (float(loss), float(want_l))
    if n > 3:
        assert rel_err(g.cpu(), want_g) < TOL
    # the full-matrix path of the same target gives the same numbers (f32 grouping only)
    plain = hg.WishTarget.from_dense(truth.cuda(), symmetric=None)
    plain.symmetric = None
    assert not ops.uses_upper_triangle(plain)
    loss2, moments2 = hg.pairwise_loss(c, plain, mode)
    (g2,) = torch.autograd.grad(loss2, c)
    assert abs(float(loss) - float(loss2)) <= 1e-6 * max(abs(float(loss2)), floor)
    if n > 3:
        assert rel_err(g, g2) < 2e-6
        assert rel_err(moments, moments2) < 1e-6
    # bit-reproducible
    loss3, moments3 = hg.pairwise_loss(c, tgt, mode)
    (g3,) = torch.autograd.grad(loss3, c)
    assert torch.equal(g, g3) and torch.equal(moments, moments3)


@pytest.mark.parametrize("variant", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("n,cuts,rb", [(777, [0, 200, 200, 601, 777], 0), (1000, [0, 999, 1000], 0), (513, [0, 64, 449, 513], 0), (3001, [0, 5, 1000, 1003, 3001], 64)])
def test_upper_triangle_row_blocks_sum_to_full(n, cuts, rb, variant):
    """Row blocks of any alignment (incl. empty ones and blocks that start inside a column strip): per block, f64 torch evaluation
    of the block's share (t_ii^2 + 2 sum_{j>i} e^2; column- plus row-side gradient of the pairs i in block, j > i).  Left of the
    diagonal the block holds what the contract allows there (NaN left of the diagonal strip, finite garbage inside it)."""
    import hic_gnn_b200 as hg
    from hic_gnn_b200 import _native as N
    from hic_gnn_b200 import ops

    coords = random_coords(n, seed=n)
    g = torch.Generator().manual_seed(n)
    mode = ops._MODES["mse_moments_full"]
    try:
        N.set_pairloss_tuning(rb, variant)  # 1 = per-lane loads, 2 = unstaggered, 3 = persistent CTAs with an item queue, 4 = static warp partition
        for r0, r1 in zip(cuts[:-1], cuts[1:]):
            rows = torch.rand(r1 - r0, n, generator=g, dtype=torch.float64).float().double()
            blk = hg.WishTarget.empty(n, r0, r1, symmetric=True)
            if r1 > r0:
                blk.data[:, :n].copy_(poison_lower(rows.float().cuda(), r0, seed=r0))
            m, gr = ops.pairloss_raw(coords.cuda(), blk, mode, 4.0 / n**2, 0.0)
            if r1 == r0:
                assert float(m.abs().sum()) == 0.0 and float(gr.abs().sum()) == 0.0
                continue
            want_m, want_g = pair_block_reference(coords, rows, r0, True, mode, c_mse=4.0 / n**2)
            assert rel_err(m, want_m) < TOL, (r0, r1)
            assert rel_err(gr, want_g) < TOL, (r0, r1)
    finally:
        N.set_pairloss_tuning(0, 0)


@pytest.mark.parametrize("n,cuts,groups,min_strips", [(3001, [0, 5, 1000, 1003, 3001], 8, 1), (3001, [0, 5, 1000, 1003, 3001], 5, 3), (777, [0, 200, 601, 777], 8, 1),
                                                      (777, [0, 200, 601, 777], 2, 1), (1300, [130, 1290], 5, 3), (30000, [0, 1900], 4, 96), (30000, [2000, 4100], 4, 96)])
def test_upper_triangle_segmented_combine_matches_one_cta_per_strip(n, cuts, groups, min_strips):
    """``hicgat_pairloss_set_combine``: the row-side sums of a strip of loci cut into segments (one combine CTA each, joined by the
    last arrival) against one CTA per strip: same moments bit for bit, gradients equal up to the order of the f64 adds; repeated
    calls bit-identical (the tickets return to zero); a workspace of unknown content (no HICGAT_PAIR_WS_CLEAN) is cleared first."""
    import hic_gnn_b200 as hg
    from hic_gnn_b200 import _native as N
    from hic_gnn_b200 import ops

    coords = random_coords(n, seed=n).cuda()
    g = torch.Generator().manual_seed(n)
    mode = ops._MODES["mse_moments_full"]
    try:
        for r0, r1 in zip(cuts[:-1], cuts[1:]):
            blk = hg.WishTarget.empty(n, r0, r1, symmetric=True)
            blk.data[:, :n].copy_(torch.rand(r1 - r0, n, generator=g).cuda())
            N.set_pairloss_combine(1, 96)
            m1, g1 = (t.clone() for t in ops.pairloss_raw(coords, blk, mode, 4.0 / n**2, 0.0))
            N.set_pairloss_combine(groups, min_strips)
            m2, g2 = (t.clone() for t in ops.pairloss_raw(coords, blk, mode, 4.0 / n**2, 0.0))
            m3, g3 = ops.pairloss_raw(coords, blk, mode, 4.0 / n**2, 0.0)
            assert torch.equal(m1, m2) and torch.equal(m2, m3) and torch.equal(g2, g3)
            assert rel_err(g2, g1) < 1e-6
            # raw call, workspace filled with ones, no WS_CLEAN bit
            lib = N.lib()
            bits = mode | N.PAIR_SYMMETRIC
            ws = torch.full((lib.hicgat_pairloss_workspace_bytes_mode(n, r0, r1, bits),), 1, dtype=torch.uint8, device="cuda")
            m4 = torch.empty(N.PAIR_NMOM, dtype=torch.float64, device="cuda")
            g4 = torch.empty(n, 3, dtype=torch.float32, device="cuda")
            for _ in range(2):
                N.check(lib.hicgat_pairloss_fwd_bwd(coords.data_ptr(), blk.data.data_ptr(), blk.pitch, n, r0, r1, bits, 4.0 / n**2, 0.0, m4.data_ptr(), g4.data_ptr(),
                                                    ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream), "hicgat_pairloss_fwd_bwd")
                assert torch.equal(m4, m2) and torch.equal(g4, g2)
    finally:
        N.set_pairloss_combine()
    with pytest.raises(RuntimeError):
        N.set_pairloss_combine(0, 24)


@pytest.mark.parametrize("variant", [0, 3, 4])
@pytest.mark.parametrize("n,cuts,rb", [(19500, [0, 100, 6016, 19500], 0), (19300, [0, 700, 19300], 128), (30000, [0, 30000], 0)])
def test_upper_triangle_large_maps_match_full_matrix_kernel(n, cuts, rb, variant):
    """More than 148 column strips (staggered chunk tables, several waves): the upper-triangle kernel over row blocks of a
    symmetric matrix must reproduce the full-matrix kernel's result on the same matrix (1e-6 moments / 1e-5 gradient), and the
    implicit-target kernels (upper and full) must agree with each other."""
    import hic_gnn_b200 as hg
    from hic_gnn_b200 import _native as N
    from hic_gnn_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(n)
    t = torch.rand(n, n, generator=g, device="cuda", dtype=torch.float32)
    t = torch.triu(t) + torch.triu(t, 1).t()
    coords = random_coords(n, seed=n).cuda()
    full = hg.WishTarget.from_dense(t, symmetric=None)
    full.symmetric = None
    mode = ops._MODES["mse_moments_full"]
    m_ref, g_ref = ops.pairloss_raw(coords, full, mode, 4.0 / n**2, 0.0)
    m_sum, g_sum = torch.zeros_like(m_ref), torch.zeros_like(g_ref)
    try:
        N.set_pairloss_tuning(rb, variant)
        for r0, r1 in zip(cuts[:-1], cuts[1:]):
            blk = hg.WishTarget(full.data[r0:r1], n, r0, r1, symmetric=True)
            m, gr = ops.pairloss_raw(coords, blk, mode, 4.0 / n**2, 0.0)
            m_sum += m
            g_sum += gr
    finally:
        N.set_pairloss_tuning(0, 0)
    assert rel_err(m_sum, m_ref) < 1e-6
    assert rel_err(g_sum, g_ref) < TOL
