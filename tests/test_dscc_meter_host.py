"""Per-step dSCC (``hicgat_dscc_*``, ``metrics.DsccMeter``, ``TrainStep(track_dscc=True)``) without a GPU: the argument checks of the
C entry points (made before any CUDA call), the Python refusals, and a numpy restatement of histogram mid-rank Spearman -- the
oracle of tests/test_gpu_dscc_meter.py -- against scipy on hand cases with heavy ties."""
import numpy as np
import pytest
import torch
from scipy.stats import spearmanr


# ----------------------------------------------------------------------------- numpy oracle
def midranks(hist):
    """Average 1-based rank of the members of every bin, the bin being one tie group."""
    h = np.asarray(hist, dtype=np.float64)
    return np.cumsum(h) - h + (h + 1.0) / 2.0


def spearman_from_bins(bd, bt, nbins):
    """Pearson of the histogram mid-ranks of two integer bin vectors (the rule of ``hicgat_dscc_*``); NaN for constant input."""
    hd, ht = np.bincount(bd, minlength=nbins), np.bincount(bt, minlength=nbins)
    rd, rt = midranks(hd), midranks(ht)
    p = float(len(bd))
    mean = (p + 1.0) / 2.0
    var_d, var_t = float((hd * (rd - mean) ** 2).sum()), float((ht * (rt - mean) ** 2).sum())
    cross = float((rd[bd] * rt[bt]).sum())
    vv = var_d * var_t
    return (cross - p * mean * mean) / np.sqrt(vv) if vv > 0 and np.isfinite(vv) else float("nan")


def spearman_implicit(bd_stored, t_stored, bd_all, fill):
    """The same with the target given as its stored values plus a fill group (the other pairs), as ``hicgat_dscc_implicit`` sums it:
    cross = sum_stored r_t r_d + r_fill (sum_all r_d - sum_stored r_d)."""
    p = float(len(bd_all))
    hd = np.bincount(bd_all)
    rd = midranks(hd)
    vals, inv, counts = np.unique(np.append(t_stored, fill), return_inverse=True, return_counts=True)
    counts = counts.astype(np.float64)
    counts[inv[-1]] += p - len(t_stored) - 1.0
    rank_vals = np.cumsum(counts) - counts + (counts + 1.0) / 2.0
    mean = (p + 1.0) / 2.0
    rs = rd[bd_stored]
    cross = float((rank_vals[inv[:-1]] * rs).sum()) + rank_vals[inv[-1]] * (float((hd * rd).sum()) - float(rs.sum()))
    var_d, var_t = float((hd * (rd - mean) ** 2).sum()), float((counts * (rank_vals - mean) ** 2).sum())
    return (cross - p * mean * mean) / np.sqrt(var_d * var_t)


def test_midrank_spearman_equals_scipy_on_exact_bins():
    """Values that are bin indices already (one value per bin): histogram mid-ranks ARE scipy's average ranks."""
    rng = np.random.default_rng(0)
    for size, levels in [(7, 3), (50, 4), (400, 12), (1000, 2)]:
        a, b = rng.integers(0, levels, size), rng.integers(0, levels, size)
        assert abs(spearman_from_bins(a, b, levels) - spearmanr(a, b)[0]) < 1e-12


def test_hand_case_with_one_dominant_tie_group():
    # 10 pairs, 7 of them in the fill group (t == 1.0 -> the top bin), distances with two ties
    t = np.array([1, 1, 1, 0, 1, 1, 2, 1, 1, 3]) / 3.0
    d = np.array([0.5, 0.1, 0.5, 0.2, 0.9, 0.9, 0.3, 0.7, 0.8, 0.05])
    bt, bd = (t * 3).astype(int), (d * 20).astype(int)       # distinct values never share a bin at this scale
    assert abs(spearman_from_bins(bd, bt, 21) - spearmanr(d, t)[0]) < 1e-12


def test_implicit_fill_identity_equals_dense():
    rng = np.random.default_rng(1)
    n = 40
    iu = np.triu_indices(n, 1)
    p = len(iu[0])
    stored = rng.random(p) < 0.15
    t = np.where(stored, rng.integers(1, 6, p) / 6.0, 1.0)
    t[np.flatnonzero(stored)[:3]] = 1.0                      # stored pairs whose value equals the fill join its tie group
    bd = rng.integers(0, 30, p)                               # distance bins with heavy ties
    want = spearmanr(bd, t)[0]
    assert abs(spearman_implicit(bd[stored], t[stored], bd, 1.0) - want) < 1e-12
    assert abs(spearman_from_bins(bd, (t * 6).astype(int), 31) - want) < 1e-12


def test_constant_input_gives_nan():
    assert np.isnan(spearman_from_bins(np.zeros(10, dtype=int), np.arange(10), 16))
    assert np.isnan(spearman_from_bins(np.array([3]), np.array([5]), 16))     # n = 2: one pair


# ----------------------------------------------------------------------------- C entry points
@pytest.fixture(scope="module")
def lib():
    from hic_gnn_b200 import _native as N
    from hic_gnn_b200 import build

    build.build()
    return N.lib()


def _fake():
    return 256  # a non-null address that is never dereferenced: every check below fails before any CUDA call


def test_workspace_bytes_rejects_bad_sizes(lib):
    assert lib.hicgat_dscc_workspace_bytes(0, 16) == 0
    assert lib.hicgat_dscc_workspace_bytes(-3, 16) == 0
    assert lib.hicgat_dscc_workspace_bytes(100, 0) == 0
    assert lib.hicgat_dscc_workspace_bytes(65535 * 32 + 1, 16) == 0
    assert lib.hicgat_dscc_workspace_bytes(100, 16) > 2 * 16 * 8


@pytest.mark.parametrize("n,nbins,pitch", [(0, 16, 8), (-1, 16, 8), (65535 * 32 + 1, 16, 65535 * 32 + 4), (8, 0, 8), (8, -4, 8), (8, 16, 4)])
def test_entry_points_reject_bad_sizes(lib, n, nbins, pitch):
    f, ws = _fake(), 1 << 30
    assert lib.hicgat_dscc_target_ranks(f, pitch, n, 1.0, nbins, f, f, f, ws, None) == -1
    assert b"hicgat_dscc_target_ranks" in lib.hicgat_last_error()
    assert lib.hicgat_dscc_dense(f, f, pitch, n, 1.0, nbins, f, f, f, f, ws, None) == -1
    assert b"hicgat_dscc_dense" in lib.hicgat_last_error()
    if pitch >= n:  # the implicit call takes no pitch
        assert lib.hicgat_dscc_implicit(f, f, f, f, n, f, f, nbins, f, f, ws, None) == -1
        assert b"hicgat_dscc_implicit" in lib.hicgat_last_error()


@pytest.mark.parametrize("null_at", range(6))
def test_dense_rejects_null_pointers(lib, null_at):
    ptrs = [_fake()] * 6
    ptrs[null_at] = None
    coords, target, rank_t, var_t, rho, ws = ptrs
    assert lib.hicgat_dscc_dense(coords, target, 8, 8, 1.0, 16, rank_t, var_t, rho, ws, 1 << 30, None) == -1
    assert b"null pointer" in lib.hicgat_last_error()


@pytest.mark.parametrize("null_at", range(8))
def test_implicit_rejects_null_pointers(lib, null_at):
    ptrs = [_fake()] * 8
    ptrs[null_at] = None
    coords, rowptr, col, rank_t, rank_fill, var_t, rho, ws = ptrs
    assert lib.hicgat_dscc_implicit(coords, rowptr, col, rank_t, 8, rank_fill, var_t, 16, rho, ws, 1 << 30, None) == -1
    assert b"null pointer" in lib.hicgat_last_error()


@pytest.mark.parametrize("null_at", range(4))
def test_target_ranks_rejects_null_pointers(lib, null_at):
    ptrs = [_fake()] * 4
    ptrs[null_at] = None
    target, rank_t, var_t, ws = ptrs
    assert lib.hicgat_dscc_target_ranks(target, 8, 8, 1.0, 16, rank_t, var_t, ws, 1 << 30, None) == -1
    assert b"null pointer" in lib.hicgat_last_error()


def test_entry_points_reject_short_workspace(lib):
    f = _fake()
    need = lib.hicgat_dscc_workspace_bytes(100, 64)
    assert lib.hicgat_dscc_dense(f, f, 100, 100, 1.0, 64, f, f, f, f, need - 1, None) == -1
    assert b"workspace" in lib.hicgat_last_error()
    assert lib.hicgat_dscc_implicit(f, f, f, f, 100, f, f, 64, f, f, need - 1, None) == -1
    assert lib.hicgat_dscc_target_ranks(f, 100, 100, 1.0, 64, f, f, f, need - 1, None) == -1


# ----------------------------------------------------------------------------- Python refusals
class _FakeDense:
    """Stands in for a WishTarget row block without device memory (the refusal comes before any allocation)."""


def _row_block(cls, n, r0, r1):
    t = cls.__new__(cls)
    t.n, t.r0, t.r1 = n, r0, r1
    return t


@pytest.mark.parametrize("r0,r1", [(0, 50), (10, 100), (50, 100)])
def test_meter_refuses_row_blocks(lib, r0, r1):
    from hic_gnn_b200 import metrics, ops

    for cls in (ops.WishTarget, ops.SparseWishTarget):
        with pytest.raises(ValueError, match="full target"):
            metrics.DsccMeter(_row_block(cls, 100, r0, r1))


def test_meter_refuses_other_targets_and_bins(lib):
    from hic_gnn_b200 import metrics, ops

    with pytest.raises(TypeError):
        metrics.DsccMeter(torch.zeros(4, 4))
    with pytest.raises(ValueError, match="nbins"):
        metrics.DsccMeter(_row_block(ops.WishTarget, 100, 0, 100), nbins=0)


def test_meter_refuses_cpu_and_misshapen_coords(lib):
    from hic_gnn_b200 import metrics

    meter = metrics.DsccMeter.__new__(metrics.DsccMeter)
    meter.n = 10
    with pytest.raises(RuntimeError, match="CUDA"):
        meter(torch.zeros(10, 3))
    if torch.cuda.is_available():
        for bad in (torch.zeros(9, 3, device="cuda"), torch.zeros(10, 3, dtype=torch.float64, device="cuda"), torch.zeros(3, 10, device="cuda").t()):
            with pytest.raises(RuntimeError, match="coords"):
                meter(bad)


def test_track_dscc_refuses_a_sharded_reducer(lib):
    from hic_gnn_b200 import train

    with pytest.raises(ValueError, match="track_dscc"):
        train.TrainStep(torch.nn.Linear(2, 2), None, None, _row_block(_FakeDense, 10, 0, 5), mode="mse", reducer=object(), track_dscc=True)
