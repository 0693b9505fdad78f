"""GPU parity of the differentiable Pearson modes (``pairwise_loss(..., "pearson" / "mse_pearson_grad")``, two passes) against
the f64 reference of tests/pearson_ref.py.  Tolerance: 1e-5 relative on loss values and gradients."""
import numpy as np
import pytest
import torch

import pearson_ref as R
from helpers import random_coords, rel_err, small_map, wish_from_map

pytestmark = pytest.mark.gpu
TOL = 1e-5
MODES = ["pearson", "mse_pearson_grad"]


def _ref(coords, truth, mode):
    c = coords.double().clone().requires_grad_(True)
    out = R.pearson_loss(c, truth.double()) if mode == "pearson" else R.mse_pearson_grad_loss(c, truth.double())[0]
    (g,) = torch.autograd.grad(out, c)
    return float(out.detach()), g


def _gpu(coords, target, mode, reducer=None):
    import hic_gnn_b200 as hg

    c = coords.cuda().float().requires_grad_(True)
    loss, moments = hg.pairwise_loss(c, target, mode, reducer)
    (g,) = torch.autograd.grad(loss, c)
    return float(loss), g, moments


def _sym(truth):
    truth = (truth + truth.t()) / 2
    truth.fill_diagonal_(0)
    return truth


@pytest.fixture(params=[True, False], ids=["upper", "fullrow"])
def upper(request, monkeypatch):
    from hic_gnn_b200 import ops

    monkeypatch.setattr(ops, "_USE_UPPER", request.param)
    return request.param


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("tag", ["1mb", "500kb"])
def test_reference_maps(golden, tag, mode, upper):
    import hic_gnn_b200 as hg

    g, _ = golden
    truth = _sym(wish_from_map(torch.tensor(g[f"{tag}_kr_oracle"]), 1.0))
    coords = random_coords(truth.shape[0], seed=1)
    want_l, want_g = _ref(coords, truth, mode)
    got_l, got_g, _ = _gpu(coords, hg.WishTarget.from_dense(truth.cuda(), symmetric=True), mode)
    assert abs(got_l - want_l) / abs(want_l) < TOL
    assert rel_err(got_g, want_g) < TOL


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("n", [3, 127, 128, 129, 1000, 2493])
def test_random_maps(n, mode, upper):
    import hic_gnn_b200 as hg

    truth = _sym(wish_from_map(small_map(n, 0.9, seed=n), 1.0) if n > 3 else torch.rand(n, n, dtype=torch.float64, generator=torch.Generator().manual_seed(n)))
    coords = random_coords(n, seed=n + 1)
    want_l, want_g = _ref(coords, truth, mode)
    got_l, got_g, _ = _gpu(coords, hg.WishTarget.from_dense(truth.cuda(), symmetric=True), mode)
    assert abs(got_l - want_l) / abs(want_l) < TOL
    # n = 3: three pairs, the regression residual of t on d is a cancellation of f32 numbers
    assert rel_err(got_g, want_g) < (TOL if n > 3 else 1e-4)


@pytest.mark.parametrize("variant", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("mode", MODES)
def test_variants_on_row_blocks(variant, mode, upper):
    """Pass 2 over row blocks whose edges cut strips and tiles: the per-block contributions add up to the full gradient."""
    import hic_gnn_b200 as hg
    from hic_gnn_b200 import _native as N
    from hic_gnn_b200 import ops

    n = 1000
    truth = _sym(wish_from_map(small_map(n, 0.7, seed=21), 1.0))
    coords = random_coords(n, seed=22)
    want_l, want_g = _ref(coords, truth, mode)
    full = hg.WishTarget.from_dense(truth.cuda(), symmetric=True)
    c = coords.cuda().float()
    m, _ = ops.pairloss_raw(c, full, N.PAIR_MOMENTS, 0.0, 0.0)
    N.set_pairloss_tuning(0, variant)
    try:
        grad = torch.zeros(n, 3, dtype=torch.float64, device="cuda")
        for r0, r1 in [(0, 1), (1, 127), (127, 129), (129, 500), (500, 1000)]:
            blk = hg.WishTarget.from_dense(truth.cuda(), r0, r1, symmetric=True)
            grad += ops.pearson_grad_raw(c, blk, m, mode == "mse_pearson_grad").double()
        got_l, got_g, _ = _gpu(coords, full, mode)
    finally:
        N.set_pairloss_tuning(0, 0)
    assert abs(float(ops.pearson_loss_from_moments(m, n, mode == "mse_pearson_grad")) - want_l) / abs(want_l) < TOL
    assert rel_err(grad, want_g) < TOL
    assert rel_err(got_g, want_g) < TOL


@pytest.mark.parametrize("mode", MODES)
def test_near_fit(mode, upper):
    """Coordinates = a 3-D embedding of a Euclidean target plus noise (r ~ 0.99): the regime training ends in."""
    import hic_gnn_b200 as hg

    n = 1500
    g = torch.Generator().manual_seed(3)
    y = torch.randn(n, 3, generator=g, dtype=torch.float64)
    truth = _sym(torch.cdist(y, y))
    coords = (y + 0.08 * torch.randn(n, 3, generator=g, dtype=torch.float64)).float()
    want_l, want_g = _ref(coords, truth, mode)
    r = 1.0 - float(R.pearson_loss(coords.double(), truth))
    assert 0.985 < r < 0.995, r
    got_l, got_g, _ = _gpu(coords, hg.WishTarget.from_dense(truth.cuda(), symmetric=True), mode)
    assert abs(got_l - want_l) / abs(want_l) < TOL
    assert rel_err(got_g, want_g) < TOL


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("n,density", [(58, 1.0), (777, 0.2), (3001, 0.01)])
def test_sparse_target_matches_dense(n, density, mode, upper):
    from hic_gnn_b200 import utils

    adj = small_map(n, density, seed=n)
    data = utils.load_input(adj.numpy().copy(), torch.zeros(n, 4).numpy())
    dense = utils.wish_target(data.y, 1.0)
    sparse = utils.sparse_wish_target(data, 1.0)
    coords = random_coords(n, seed=n + 1)
    l1, g1, m1 = _gpu(coords, dense, mode)
    l2, g2, m2 = _gpu(coords, sparse, mode)
    assert abs(l1 - l2) <= 1e-6 * abs(l1)
    assert rel_err(m2, m1) < 1e-6
    assert rel_err(g2, g1) < TOL
    want_l, want_g = _ref(coords, dense.dense().cpu().double(), mode)
    assert abs(l2 - want_l) / abs(want_l) < TOL
    assert rel_err(g2, want_g) < TOL


@pytest.mark.parametrize("mode", MODES)
def test_deterministic(mode, upper):
    import hic_gnn_b200 as hg

    n = 2493
    truth = _sym(wish_from_map(small_map(n, 0.9, seed=4), 1.0))
    tgt = hg.WishTarget.from_dense(truth.cuda(), symmetric=True)
    coords = random_coords(n, seed=5)
    l1, g1, m1 = _gpu(coords, tgt, mode)
    l2, g2, m2 = _gpu(coords, tgt, mode)
    assert l1 == l2 and torch.equal(g1, g2) and torch.equal(m1, m2)


@pytest.mark.parametrize("n", [9970, 49850])
def test_closed_form_checks_at_scale(n):
    """Translation and scale invariance of the gradient, and a central finite difference of 1 - r from f64 moments."""
    import hic_gnn_b200 as hg
    from hic_gnn_b200 import _native as N
    from hic_gnn_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(7)
    y = torch.randn(n, 3, generator=g, device="cuda")
    t = torch.cdist(y, y) + 0.5 * torch.rand(n, n, generator=g, device="cuda")
    t = t + t.t()
    t.fill_diagonal_(0)
    tgt = hg.WishTarget.from_dense(t, symmetric=True)
    del t
    x = y + 0.7 * torch.randn(n, 3, generator=g, device="cuda")
    _, gp, _ = _gpu(x, tgt, "pearson")
    _, gm, _ = _gpu(x, tgt, "mse_pearson_grad")
    gp, gm = gp.double(), gm.double()
    for grad in (gp, gm):
        assert float(grad.sum(0).abs().max()) < 1e-4 * float(grad.abs().sum(0).max())
    xd = x.double()
    assert abs(float((gp * xd).sum())) < 1e-4 * float(gp.norm() * xd.norm())

    def one_minus_r(c):
        m, _ = ops.pairloss_raw(c, tgt, N.PAIR_MOMENTS, 0.0, 0.0)
        return float(ops.pearson_loss_from_moments(m, n, False))

    v = torch.randn(n, 3, generator=g, device="cuda")
    h = 1e-2
    fd = (one_minus_r(x + h * v) - one_minus_r(x - h * v)) / (2 * h)
    an = float((gp * v.double()).sum())
    assert abs(fd - an) < 2e-3 * abs(an), (fd, an)
    del tgt
    torch.cuda.empty_cache()


def _gat(n, seed=4):
    from hic_gnn_b200 import utils as gutils

    adj = small_map(n, 1.0, seed=seed)
    x = 0.25 * torch.randn(n, 512, generator=torch.Generator().manual_seed(seed + 100))
    gdata = gutils.load_input(adj.numpy().copy(), x.numpy())
    return adj, x, gdata


def test_cuda_graph_matches_eager():
    from hic_gnn_b200 import models, train, utils

    n = 300
    _, _, gdata = _gat(n)
    target = utils.wish_target(gdata.y, 1.0)
    torch.manual_seed(42)
    init = models.GATNetSelectiveResidualsUpdated().state_dict()
    runs = []
    for graphed in (False, True):
        gm = models.GATNetSelectiveResidualsUpdated().cuda()
        gm.load_state_dict(init)
        step = train.TrainStep(gm, gdata.x.float(), gdata.edge_index, target, mode="mse_pearson_grad", lr=1e-3, use_cuda_graph=graphed)
        if not graphed:  # the same optimizer arithmetic as the captured step
            step.optimizer = torch.optim.Adam(gm.parameters(), lr=1e-3, capturable=True)
        totals = []
        for _ in range(20):
            total, _ = step()
            totals.append(total.clone())
        runs.append((torch.stack(totals), {k: v.detach().clone() for k, v in gm.state_dict().items()}))
    (t_e, p_e), (t_g, p_g) = runs
    assert torch.equal(t_e, t_g), (t_e - t_g).abs().max()
    assert all(torch.equal(p_e[k], p_g[k]) for k in p_e)
    assert torch.isfinite(t_e).all() and float(t_e[-1]) < float(t_e[0])


def test_training_parity_teacher_forced():
    """Teacher-forced GAT-net steps at 58 loci against the reference loop body (tests/pearson_ref.py): the step's loss within
    1e-5 of the f64 reference, every parameter gradient within max(2e-5, the error of the reference's own f32 evaluation) of its
    tensor's max -- the acceptance of the mse_pearson trajectory test of test_gpu_conv (steps with a unit at its activation
    kink may be off by a kink-sized amount, at least half of the steps are exact)."""
    from test_gpu_conv import _KinkWatch, _param_grads, _setup

    from hic_gnn_b200 import models as gmodels
    from hic_gnn_b200 import train as gtrain
    from hic_gnn_b200 import utils as gutils
    from oracle import models as omodels
    from oracle import wish as owish

    n, steps, cls = 58, 10, "GATNetSelectiveResidualsUpdated"
    _, _, odata, gdata = _setup(n, 1.0, seed=4)
    torch.manual_seed(42)
    om = getattr(omodels, cls)()
    gm = getattr(gmodels, cls)().cuda()
    truth = owish.cont2dist(odata.y.clone(), 1.0)
    target = gutils.wish_target(gdata.y, 1.0)
    opt = torch.optim.Adam(om.parameters(), lr=1e-3)
    watch = _KinkWatch(om, cls)
    ok_steps, violations = 0, []
    for s in range(steps):
        gm.load_state_dict(om.state_dict())
        opt.zero_grad()
        watch.reset()
        coords_o = om.get_model(odata.x.float(), odata.edge_index)
        lo32, _, _ = R.mse_pearson_grad_loss(coords_o, truth.float())  # the formula evaluated in f32, as a reference loop would
        lo32.backward(retain_graph=True)
        g32 = _param_grads(om)
        opt.zero_grad()
        lo64, _, _ = R.mse_pearson_grad_loss(coords_o.double(), truth)
        lo64.backward()
        g64 = _param_grads(om)
        gm.zero_grad(set_to_none=True)
        lg, total, _ = gtrain.step_loss(gm, gdata.x.float(), gdata.edge_index, target, "mse_pearson_grad")
        lg.backward()
        assert abs(float(lg) - float(lo64)) / abs(float(lo64)) < TOL, (s, float(lg), float(lo64))
        assert float(total) == float(lg)
        top = max(float(v.abs().max()) for v in g64.values() if v is not None)
        step_ok = True
        for name, p in gm.named_parameters():
            want = g64[name]
            # translation invariance: the last layer's bias has an exact 0 gradient, both sides hold rounding noise only
            if want is None or float(want.abs().max()) < 1e-6 * top:
                continue
            e, e_ref = rel_err(p.grad, want), rel_err(g32[name], want)
            if not e < max(2e-5, e_ref):
                step_ok = False
                violations.append((s, name, e, e_ref, watch.gap))
        ok_steps += step_ok
        opt.step()
    watch.close()
    assert all(v[2] < 1e-1 for v in violations), violations
    assert ok_steps >= steps // 2, (ok_steps, violations)


def test_refusals():
    import hic_gnn_b200 as hg
    from hic_gnn_b200 import ops

    n = 64
    t = torch.rand(n, n, device="cuda")
    t.fill_diagonal_(0)
    tgt = hg.WishTarget.from_dense(t)
    assert tgt.symmetric is False
    c = random_coords(n).cuda().requires_grad_(True)
    for mode in MODES:
        with pytest.raises(NotImplementedError, match="symmetric"):
            hg.pairwise_loss(c, tgt, mode)
    sym = hg.WishTarget.from_dense(_sym(t.double()).float())
    with pytest.raises(NotImplementedError, match="one-shot"):
        ops.sharded_reducer(sym, "pearson", transport="p2p_oneshot")


def _p2p_world1_worker(rank, port, tmpdir):
    """One-rank NCCL group: the capturable p2p two-pass reducer (both two-shot exchanges) against the unsharded step, eager and
    inside a captured training step."""
    import os

    import torch.distributed as dist

    import hic_gnn_b200 as hg
    from hic_gnn_b200 import models, ops, sharding, train, utils

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(0)
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
    try:
        n = 300
        adj = small_map(n, 1.0, seed=4)
        x = 0.25 * torch.randn(n, 512, generator=torch.Generator().manual_seed(104))
        gdata = utils.load_input(adj.numpy().copy(), x.numpy())
        target = utils.wish_target(gdata.y, 1.0)
        coords = random_coords(n, seed=3).cuda().requires_grad_(True)
        for mode in MODES:
            red = ops.sharded_reducer(target, mode, transport="p2p")
            assert isinstance(red, sharding.P2PTwoPassShardedPairLoss) and red.capturable
            for _ in range(3):  # several steps: the device-side epochs of both exchanges advance
                loss_s, mom_s = hg.pairwise_loss(coords, target, mode, reducer=red)
            (g_s,) = torch.autograd.grad(loss_s, coords)
            loss_1, mom_1 = hg.pairwise_loss(coords, target, mode)
            (g_1,) = torch.autograd.grad(loss_1, coords)
            assert abs(float(loss_s) - float(loss_1)) <= 1e-12 * abs(float(loss_1)), (mode, float(loss_s), float(loss_1))
            assert rel_err(mom_s, mom_1) < 1e-12 and rel_err(g_s, g_1) < 1e-7, (mode, rel_err(g_s, g_1))
        torch.manual_seed(42)
        init = models.GATNetSelectiveResidualsUpdated().state_dict()
        totals = []
        for graphed in (False, True):
            gm = models.GATNetSelectiveResidualsUpdated().cuda()
            gm.load_state_dict(init)
            red = ops.sharded_reducer(target, "mse_pearson_grad", transport="p2p")
            step = train.TrainStep(gm, gdata.x.float(), gdata.edge_index, target, mode="mse_pearson_grad", use_cuda_graph=graphed, reducer=red)
            if not graphed:
                step.optimizer = torch.optim.Adam(gm.parameters(), lr=1e-3, capturable=True)
            totals.append(torch.stack([step()[0].clone() for _ in range(10)]))
        assert torch.isfinite(totals[0]).all()
        assert float(((totals[1] - totals[0]) / totals[0]).abs().max()) < 1e-6, totals
        open(os.path.join(tmpdir, "ok0"), "w").write("ok")
    finally:
        dist.destroy_process_group()


def test_p2p_two_pass_reducer_one_rank(tmp_path):
    import os

    import torch.multiprocessing as mp

    port = 35500 + os.getpid() % 2000
    mp.spawn(_p2p_world1_worker, args=(port, str(tmp_path)), nprocs=1, join=True)
    assert (tmp_path / "ok0").exists()
