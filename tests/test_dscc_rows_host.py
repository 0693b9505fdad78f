"""Row-block phases of the per-step dSCC without a GPU: the argument checks of ``hicgat_dscc_*_rows``, ``hicgat_dscc_hist_ranks``,
``hicgat_dscc_finish`` and ``hicgat_allreduce_u64_twoshot`` (made before any CUDA call), the refusals of ``metrics.ShardedDsccMeter``,
and those of ``TrainStep`` with a per-step dSCC meter."""
import pytest
import torch


@pytest.fixture(scope="module")
def lib():
    from hic_gnn_b200 import _native as N
    from hic_gnn_b200 import build

    build.build()
    return N.lib()


F = 256          # a non-null address that is never dereferenced: every check below fails before any CUDA call
WS = 1 << 30


def _calls(lib, n=8, r0=0, r1=8, nbins=16, pitch=8, ws=WS):
    """Every row-block entry point with its arguments: (name, pointer positions, call(ptrs))."""
    return {
        "hicgat_dscc_dist_hist_rows": (3, lambda p: lib.hicgat_dscc_dist_hist_rows(p[0], n, r0, r1, nbins, p[1], p[2], ws, None)),
        "hicgat_dscc_target_hist_rows": (2, lambda p: lib.hicgat_dscc_target_hist_rows(p[0], pitch, n, r0, r1, 1.0, nbins, p[1], None)),
        "hicgat_dscc_cross_dense_rows": (6, lambda p: lib.hicgat_dscc_cross_dense_rows(p[0], p[1], pitch, n, r0, r1, 1.0, nbins, p[2], p[3], p[4], p[5],
                                                                                       ws, None)),
        "hicgat_dscc_cross_implicit_rows": (7, lambda p: lib.hicgat_dscc_cross_implicit_rows(p[0], p[1], p[2], p[3], n, r0, r1, nbins, p[4], p[5], p[6],
                                                                                             ws, None)),
    }


@pytest.mark.parametrize("r0,r1", [(-1, 4), (5, 4), (0, 9), (9, 9), (3, -2)])
def test_row_entry_points_reject_bad_rows(lib, r0, r1):
    for name, (k, call) in _calls(lib, r0=r0, r1=r1).items():
        assert call([F] * k) == -1, name
        assert name.encode() in lib.hicgat_last_error() and b"r0/r1" in lib.hicgat_last_error()


@pytest.mark.parametrize("n,nbins", [(0, 16), (-1, 16), (65535 * 32 + 1, 16), (8, 0), (8, -4)])
def test_entry_points_reject_bad_sizes(lib, n, nbins):
    for name, (k, call) in _calls(lib, n=n, r0=0, r1=max(n, 0), nbins=nbins, pitch=max(n, 8)).items():
        assert call([F] * k) == -1, name
        assert name.encode() in lib.hicgat_last_error()
    assert lib.hicgat_dscc_hist_ranks(F, n, nbins, F, F, F, WS, None) == -1
    assert b"hicgat_dscc_hist_ranks" in lib.hicgat_last_error()
    assert lib.hicgat_dscc_finish(F, n, nbins, 1, F, F, F, F, WS, None) == -1
    assert b"hicgat_dscc_finish" in lib.hicgat_last_error()


def test_row_entry_points_reject_null_pointers(lib):
    for name, (k, call) in _calls(lib).items():
        for at in range(k):
            p = [F] * k
            p[at] = None
            assert call(p) == -1, (name, at)
            assert b"null pointer" in lib.hicgat_last_error(), (name, at)
    for at in range(4):
        p = [F] * 4
        p[at] = None
        assert lib.hicgat_dscc_hist_ranks(p[0], 8, 16, p[1], p[2], p[3], WS, None) == -1
        assert b"null pointer" in lib.hicgat_last_error()
    for at in range(4):
        p = [F] * 4
        p[at] = None
        assert lib.hicgat_dscc_finish(p[0], 8, 16, 0, None, p[1], p[2], p[3], WS, None) == -1
        assert b"null pointer" in lib.hicgat_last_error()
    assert lib.hicgat_dscc_finish(F, 8, 16, 1, None, F, F, F, WS, None) == -1       # the implicit finish reads rank_fill
    assert b"null pointer" in lib.hicgat_last_error()


def test_entry_points_reject_bad_pitch(lib):
    for name in ("hicgat_dscc_target_hist_rows", "hicgat_dscc_cross_dense_rows"):
        k, call = _calls(lib, n=8, pitch=4)[name]
        assert call([F] * k) == -1
        assert b"pitch" in lib.hicgat_last_error()


def test_entry_points_reject_short_workspace(lib):
    need = lib.hicgat_dscc_workspace_bytes(100, 64)
    for name, (k, call) in _calls(lib, n=100, r0=10, r1=60, nbins=64, pitch=100, ws=need - 1).items():
        if name == "hicgat_dscc_target_hist_rows":
            continue  # takes no workspace
        assert call([F] * k) == -1, name
        assert b"workspace" in lib.hicgat_last_error()
    assert lib.hicgat_dscc_hist_ranks(F, 100, 64, F, F, F, need - 1, None) == -1
    assert b"workspace" in lib.hicgat_last_error()
    assert lib.hicgat_dscc_finish(F, 100, 64, 0, None, F, F, F, need - 1, None) == -1
    assert b"workspace" in lib.hicgat_last_error()


def test_u64_allreduce_rejects_bad_arguments(lib):
    import ctypes as C

    tab = lambda *v: (C.c_uint64 * len(v))(*v)
    ok = tab(256, 512)
    assert lib.hicgat_allreduce_u64_twoshot(None, ok, ok, 0, 2, 10, 0, F, None) == -1
    assert b"null pointer" in lib.hicgat_last_error()
    assert lib.hicgat_allreduce_u64_twoshot(ok, ok, ok, 0, 2, 10, 0, None, None) == -1
    for rank, world in ((2, 2), (-1, 2), (0, 0), (0, 17)):
        assert lib.hicgat_allreduce_u64_twoshot(ok, ok, ok, rank, world, 10, 0, F, None) == -1
        assert b"rank/world" in lib.hicgat_last_error()
    assert lib.hicgat_allreduce_u64_twoshot(ok, ok, ok, 0, 2, 0, 0, F, None) == -1
    assert b"count" in lib.hicgat_last_error()
    assert lib.hicgat_allreduce_u64_twoshot(ok, ok, ok, 0, 2, 10, -1, F, None) == -1
    assert lib.hicgat_allreduce_u64_twoshot(tab(256, 0), ok, ok, 0, 2, 10, 0, F, None) == -1
    assert b"null peer pointer" in lib.hicgat_last_error()
    assert lib.hicgat_allreduce_u64_twoshot(tab(256, 520), ok, ok, 0, 2, 10, 0, F, None) == -1
    assert b"aligned" in lib.hicgat_last_error()


# ----------------------------------------------------------------------------- Python refusals
def _row_block(cls, n, r0, r1):
    t = cls.__new__(cls)
    t.n, t.r0, t.r1 = n, r0, r1
    return t


def test_sharded_meter_refusals(lib):
    from hic_gnn_b200 import metrics, ops

    with pytest.raises(TypeError):
        metrics.ShardedDsccMeter(torch.zeros(4, 4))
    for cls in (ops.WishTarget, ops.SparseWishTarget):
        for nbins in (0, -3):
            with pytest.raises(ValueError, match="nbins"):
                metrics.ShardedDsccMeter(_row_block(cls, 100, 0, 100), nbins=nbins)
        with pytest.raises(ValueError, match="transport"):
            metrics.ShardedDsccMeter(_row_block(cls, 100, 0, 100), transport="mpi")
        for r0, r1 in ((0, 50), (10, 100), (50, 50)):  # a block of a process group that does not exist
            with pytest.raises(ValueError, match="process group"):
                metrics.ShardedDsccMeter(_row_block(cls, 100, r0, r1))


def test_dscc_exchange_refuses_a_bad_transport():
    from hic_gnn_b200 import sharding

    with pytest.raises(ValueError, match="transport"):
        sharding.DsccExchange(16, "cpu", transport="gloo")


class _Meter:
    def __init__(self, capturable):
        self.capturable, self.transport = capturable, "nccl"


def _step(**kw):
    from hic_gnn_b200 import train

    target = _row_block(type("Block", (), {}), 10, 0, 5)
    return train.TrainStep(torch.nn.Linear(2, 2), None, None, target, **kw)


def test_train_step_refusals(lib):
    with pytest.raises(ValueError, match="track_dscc") as e:
        _step(mode="mse", reducer=object(), track_dscc=True)
    assert "dscc_meter" in str(e.value)
    with pytest.raises(ValueError, match="dscc_meter"):
        _step(mode="mse", track_dscc=True, dscc_meter=_Meter(True))
    with pytest.raises(ValueError, match="capturable dSCC meter"):
        _step(mode="mse", use_cuda_graph=True, reducer=type("R", (), {"capturable": True})(), dscc_meter=_Meter(False))


def test_mse_spearman_with_a_reducer_needs_a_meter(lib):
    """Without a meter each rank would add its own block-local dSCC to the total, and the stop rule would see different totals."""
    with pytest.raises(ValueError, match="mse_spearman"):
        _step(mode="mse_spearman", reducer=object())
    from hic_gnn_b200 import train

    with pytest.raises(ValueError, match="mse_spearman"):
        train._loss_of_coords(torch.zeros(10, 3), _row_block(type("Block", (), {}), 10, 0, 5), "mse_spearman", object(), 1.0)
