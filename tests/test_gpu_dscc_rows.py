"""Row-block phases of the per-step dSCC (``hicgat_dscc_*_rows``, ``hicgat_dscc_finish``) and ``metrics.ShardedDsccMeter`` on one GPU.
A W-way row-sharded evaluation is emulated block by block: block histograms summed in int64 (exact), block cross sums added in block
order from 0.0 (the order of the exchange), then the finish.  Checked: the summed histograms equal the (0, n) ones bit for bit, rho is
within 1e-12 of ``metrics.DsccMeter`` and within 1e-5 of scipy at small n, the old entry points are the (0, n) phases bit for bit, and
a graph replay equals the eager call."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

NBINS = 1 << 22


def _coords(n, seed, collapsed=False):
    g = torch.Generator().manual_seed(seed)
    t = torch.linspace(0, 6.0, n)
    c = torch.stack([torch.cos(t) * (1 + 0.1 * t), torch.sin(t) * (1 + 0.1 * t), 0.2 * t], dim=1)
    c = c + 0.05 * torch.randn(n, 3, generator=g)
    if collapsed:  # 90 % of the loci at one point: one distance bin holds 81 % of the pairs (the warp-aggregated atomics)
        c[torch.randperm(n, generator=g)[: (9 * n) // 10]] = 0.5
    return c.float().cuda().contiguous()


def _targets(n, seed):
    """(dense WishTarget, implicit SparseWishTarget) of a random sparse symmetric contact map: identical values at every pair."""
    from hic_gnn_b200 import ops
    from hic_gnn_b200.graph import CSRGraph

    g = torch.Generator().manual_seed(seed)
    a = torch.rand(n, n, generator=g, dtype=torch.float64)
    keep = torch.rand(n, n, generator=g) < max(0.15, 3.0 / n)
    adj = torch.triu(torch.where(keep, 1.0 + 9.0 * a, torch.zeros_like(a)), 1)
    if n > 1:
        adj[0, 1] = 2.0
    adj = (adj + adj.t()).cuda()
    _, dense = ops.cont2dist(adj, 1.0, want_f64=False, want_f32=True, symmetric=True)
    rowptr, col, val = ops.csr_from_dense(adj)
    sparse = ops.SparseWishTarget.from_graph(CSRGraph(rowptr, col, val, n), adj, 1.0)
    return dense, sparse


def _partitions(n):
    from hic_gnn_b200 import sharding

    parts = [sharding.all_blocks(n, w, bal) for w in (2, 3, 8) for bal in ("rows", "upper")]
    a, b = min(1, n), min(n, max(1, n // 3) + 1)
    parts.append([(0, 0), (0, a), (a, b), (b, n)])  # an empty block, a one-row block, odd boundaries
    return parts


class _Phases:
    """The C phases with one workspace, as one rank calls them."""

    def __init__(self, n, nbins=NBINS):
        from hic_gnn_b200 import _native as N

        self.N, self.lib, self.n, self.nbins = N, N.lib(), n, nbins
        self.wsb = self.lib.hicgat_dscc_workspace_bytes(n, nbins)
        self.ws = torch.empty(self.wsb, dtype=torch.uint8, device="cuda")
        self.st = torch.cuda.current_stream().cuda_stream

    def dist_hist(self, coords, r0, r1):
        h = torch.empty(self.nbins, dtype=torch.int64, device="cuda")
        self.N.check(self.lib.hicgat_dscc_dist_hist_rows(coords.data_ptr(), self.n, r0, r1, self.nbins, h.data_ptr(), self.ws.data_ptr(), self.wsb,
                                                         self.st), "dist_hist_rows")
        return h

    def target_hist(self, dense, t_scale, r0, r1):
        h = torch.empty(self.nbins, dtype=torch.int64, device="cuda")
        ptr = dense.data.data_ptr() + 4 * r0 * dense.pitch
        self.N.check(self.lib.hicgat_dscc_target_hist_rows(ptr, dense.pitch, self.n, r0, r1, t_scale, self.nbins, h.data_ptr(), self.st),
                     "target_hist_rows")
        return h

    def cross(self, coords, tgt, meter, hist_d, r0, r1):
        from hic_gnn_b200 import ops

        out = torch.full((2,), float("nan"), dtype=torch.float64, device="cuda")
        if isinstance(tgt, ops.WishTarget):
            rc = self.lib.hicgat_dscc_cross_dense_rows(coords.data_ptr(), tgt.data.data_ptr() + 4 * r0 * tgt.pitch, tgt.pitch, self.n, r0, r1,
                                                       meter._t_scale, self.nbins, hist_d.data_ptr(), meter._rank_t.data_ptr(), out.data_ptr(),
                                                       self.ws.data_ptr(), self.wsb, self.st)
        else:
            rc = self.lib.hicgat_dscc_cross_implicit_rows(coords.data_ptr(), tgt.rowptr.data_ptr(), ops._addr(tgt.col), meter._rank_t.data_ptr(),
                                                          self.n, r0, r1, self.nbins, hist_d.data_ptr(), out.data_ptr(), self.ws.data_ptr(),
                                                          self.wsb, self.st)
        self.N.check(rc, "cross_rows")
        return out

    def finish(self, cross, meter):
        rho = torch.empty((), dtype=torch.float64, device="cuda")
        implicit = getattr(meter, "_rank_fill", None) is not None
        self.N.check(self.lib.hicgat_dscc_finish(cross.data_ptr(), self.n, self.nbins, int(implicit), meter._rank_fill.data_ptr() if implicit else None,
                                                 meter._var_t.data_ptr(), rho.data_ptr(), self.ws.data_ptr(), self.wsb, self.st), "finish")
        return rho


def _emulate(ph, coords, tgt, meter, blocks):
    """rho of a row-sharded evaluation over ``blocks``, and the summed distance histogram."""
    hist = torch.zeros(ph.nbins, dtype=torch.int64, device="cuda")
    for r0, r1 in blocks:
        hist += ph.dist_hist(coords, r0, r1)
    crosses = [ph.cross(coords, tgt, meter, hist, r0, r1) for r0, r1 in blocks]
    total = torch.zeros(2, dtype=torch.float64, device="cuda")
    for c in crosses:  # block order from 0.0: the exchange's order
        total += c
    return ph.finish(total, meter), hist


def _close(a, b, tol=1e-12):
    a, b = float(a), float(b)
    if np.isnan(b):
        return np.isnan(a)
    return abs(a - b) <= tol * max(1.0, abs(b))


def _scipy(coords, dense):
    from scipy.stats import spearmanr

    n = dense.n
    iu = np.triu_indices(n, 1)
    t = dense.dense().cpu().double().numpy()[iu]
    c = coords.cpu().double()
    d = torch.cdist(c, c, compute_mode="donot_use_mm_for_euclid_dist").numpy()[iu]
    return float(spearmanr(t, d)[0])


@pytest.mark.parametrize("n", [2, 3, 777, 3001, 9973])
@pytest.mark.parametrize("collapsed", [False, True])
def test_block_phases_sum_to_the_full_evaluation(n, collapsed):
    from hic_gnn_b200 import metrics

    if collapsed and n < 777:
        pytest.skip("collapse needs loci to collapse")
    dense, sparse = _targets(n, seed=n)
    coords = _coords(n, seed=n + 1, collapsed=collapsed)
    ph = _Phases(n)
    full_hist = ph.dist_hist(coords, 0, n)
    assert int(full_hist.sum()) == n * (n - 1) // 2
    want_scipy = _scipy(coords, dense) if 2 < n <= 3001 else None
    for tgt in (dense, sparse):
        meter = metrics.DsccMeter(tgt)
        want = meter(coords).clone()
        if isinstance(tgt, type(dense)):  # the target side over blocks: histograms and rank table bit for bit
            full_t = ph.target_hist(dense, meter._t_scale, 0, n)
            rank_t = torch.empty(NBINS, dtype=torch.float64, device="cuda")
            var_t = torch.empty((), dtype=torch.float64, device="cuda")
            for blocks in _partitions(n)[:2]:
                ht = sum(ph.target_hist(dense, meter._t_scale, r0, r1) for r0, r1 in blocks)
                assert torch.equal(ht, full_t), blocks
            ph.N.check(ph.lib.hicgat_dscc_hist_ranks(full_t.data_ptr(), n, NBINS, rank_t.data_ptr(), var_t.data_ptr(), ph.ws.data_ptr(), ph.wsb,
                                                     ph.st), "hist_ranks")
            assert torch.equal(rank_t, meter._rank_t) and torch.equal(var_t, meter._var_t)
        for blocks in _partitions(n):
            rho, hist = _emulate(ph, coords, tgt, meter, blocks)
            assert torch.equal(hist, full_hist), blocks
            assert _close(rho, want), (type(tgt).__name__, blocks, float(rho), float(want))
            if want_scipy is not None and not collapsed:
                assert abs(float(rho) - want_scipy) < 1e-5, (float(rho), want_scipy)
        if n < 3:
            assert bool(torch.isnan(want))


@pytest.mark.parametrize("n", [3, 777, 3001])
def test_old_entry_points_are_the_full_block_phases(n):
    from hic_gnn_b200 import metrics

    dense, sparse = _targets(n, seed=7 * n)
    coords = _coords(n, seed=3)
    ph = _Phases(n)
    for tgt in (dense, sparse):
        meter = metrics.DsccMeter(tgt)
        want = meter(coords).clone()
        hist = ph.dist_hist(coords, 0, n)
        got = ph.finish(ph.cross(coords, tgt, meter, hist, 0, n), meter)
        assert got.view(torch.int64).item() == want.view(torch.int64).item(), (float(got), float(want))
        one = metrics.ShardedDsccMeter(tgt)  # one rank, no process group: the full target
        assert one.capturable
        assert one(coords).view(torch.int64).item() == want.view(torch.int64).item()


def test_constant_coordinates_give_nan():
    from hic_gnn_b200 import metrics

    n = 300
    dense, sparse = _targets(n, seed=1)
    same = torch.full((n, 3), 0.25, device="cuda")
    ph = _Phases(n)
    for tgt in (dense, sparse):
        meter = metrics.DsccMeter(tgt)
        rho, _ = _emulate(ph, same, tgt, meter, _partitions(n)[-1])
        assert bool(torch.isnan(rho)) and bool(torch.isnan(metrics.ShardedDsccMeter(tgt)(same)))


@pytest.mark.parametrize("kind", ["dense", "implicit"])
def test_sharded_meter_replays_in_a_graph(kind):
    from hic_gnn_b200 import metrics

    n = 2493
    dense, sparse = _targets(n, seed=11)
    meter = metrics.ShardedDsccMeter(dense if kind == "dense" else sparse)
    ref = metrics.DsccMeter(dense if kind == "dense" else sparse)
    sets = [_coords(n, s) for s in (1, 2, 3)]
    sets[2] = (sets[2] * torch.linspace(0.2, 3.0, n, device="cuda").unsqueeze(1)).contiguous()
    eager = [meter(c).clone() for c in sets]
    for c, e in zip(sets, eager):
        assert torch.equal(e, ref(c))
    assert len({float(e) for e in eager}) == 3
    static = sets[0].clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        meter(static)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = meter(static)
    for c, want in zip(sets, eager):
        static.copy_(c)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, want), (float(out), float(want))


def test_one_rank_training_step_with_a_sharded_meter():
    """``TrainStep(dscc_meter=ShardedDsccMeter(full target))`` on one rank tracks what ``track_dscc=True`` tracks, graphed, bit for bit."""
    from hic_gnn_b200 import metrics, models, ops, synth, train
    from hic_gnn_b200.graph import CSRGraph

    n = 777
    adj = synth.synthetic_map(n, 0.3, seed=5).cuda()
    x = synth.synthetic_features(n, seed=3).cuda()
    _, target = ops.cont2dist(adj, 1.0, want_f64=False, want_f32=True)
    graph = CSRGraph(*ops.csr_from_dense(adj), n)
    runs = []
    for kw in ({"track_dscc": True}, {"dscc_meter": metrics.ShardedDsccMeter(target)}):
        torch.manual_seed(42)
        model = models.GATNetSelectiveResidualsUpdated().cuda()
        out = []
        train.fit(model, x, graph, target, mode="mse_pearson", lr=1e-3, thresh=0.0, max_steps=5, use_cuda_graph=True, dscc_out=out,
                  **({} if "track_dscc" in kw else kw))
        runs.append(out)
    assert runs[0] == runs[1] and len(runs[0]) == 5
