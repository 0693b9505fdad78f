"""Per-step dSCC on the device (``metrics.DsccMeter``, ``hicgat_dscc_*``) and its use in the training loop
(``TrainStep(track_dscc=True)``, ``fit(dscc_out=...)``): against scipy.stats.spearmanr (what the reference calls every iteration,
HiC_GAT_generalize_directly.py:242), against ``metrics.dscc_streamed`` (same bins: only the order of the cross sum differs), against the
exact sort-based evaluation, bit-reproducibility, CUDA-graph replay and degenerate inputs."""
import numpy as np
import pytest
import torch

from helpers import small_map

pytestmark = pytest.mark.gpu


def _structured_coords(n, seed):
    """A noisy helix: distances correlate with genomic distance, so rho is far from 0."""
    g = torch.Generator().manual_seed(seed)
    t = torch.linspace(0, 6.0, n)
    c = torch.stack([torch.cos(t) * (1 + 0.1 * t), torch.sin(t) * (1 + 0.1 * t), 0.2 * t], dim=1)
    return (c + 0.05 * torch.randn(n, 3, generator=g)).float()


def _targets(adj):
    """(dense WishTarget, implicit SparseWishTarget) of a contact matrix: identical values at every pair."""
    from hic_gnn_b200 import utils

    adj = np.asarray(adj, dtype=np.float64)
    data = utils.load_input(adj.copy(), np.zeros((adj.shape[0], 4), dtype=np.float32))
    return utils.wish_target(data.y, 1.0), utils.sparse_wish_target(data, 1.0)


def _scipy_dscc(coords, dense):
    from scipy.stats import spearmanr

    n = dense.n
    iu = np.triu_indices(n, 1)
    t = dense.dense().cpu().double().numpy()[iu]
    c = coords.cpu().double()
    d = torch.cdist(c, c, compute_mode="donot_use_mm_for_euclid_dist").numpy()[iu]
    return float(spearmanr(t, d)[0])


def _golden_map(golden, tag):
    g, _ = golden
    adj = np.array(g[f"{tag}_kr_oracle"], dtype=np.float64)
    np.fill_diagonal(adj, 0.0)
    return adj


@pytest.mark.parametrize("case", ["1mb", "500kb", "300", "1500"])
def test_meter_matches_scipy(golden, case):
    from hic_gnn_b200 import metrics

    if case in ("1mb", "500kb"):
        adj = _golden_map(golden, case)
    else:
        n = int(case)
        adj = small_map(n, 0.3 if n == 300 else 0.1, seed=n).numpy()
    dense, sparse = _targets(adj)
    coords = _structured_coords(dense.n, 3).cuda()
    want = _scipy_dscc(coords, dense)
    for tgt in (dense, sparse):
        got = float(metrics.DsccMeter(tgt)(coords))
        assert abs(got - want) < 1e-5, (type(tgt).__name__, got, want)


def _synthetic(n, density):
    from hic_gnn_b200 import ops, synth
    from hic_gnn_b200.graph import CSRGraph

    adj = synth.synthetic_map_chunked(n, density, device="cuda")
    _, dense = ops.cont2dist(adj, 1.0, want_f64=False, want_f32=True)
    rowptr, col, val = ops.csr_from_dense(adj)
    sparse = ops.SparseWishTarget.from_graph(CSRGraph(rowptr, col, val, n), adj, 1.0)
    return dense, sparse


@pytest.mark.parametrize("n,density", [(2493, 0.95), (9970, 0.07)])
def test_meter_matches_streamed_and_exact(n, density):
    from hic_gnn_b200 import metrics

    dense, sparse = _synthetic(n, density)
    coords = _structured_coords(n, 5).cuda()
    for tgt in (dense, sparse):
        got = float(metrics.DsccMeter(tgt)(coords))
        want = metrics.dscc_streamed(coords, tgt)
        assert abs(got - want) < 1e-12, (type(tgt).__name__, got, want)
    if n == 9970:
        t, d = metrics.upper_pairs(coords, dense)
        exact = float(metrics._pearson(metrics.average_ranks(t.double()), metrics.average_ranks(d.double())))
        assert abs(got - exact) < 1e-5, (got, exact)


@pytest.mark.parametrize("kind", ["dense", "implicit"])
def test_meter_is_deterministic_and_replays_in_a_graph(kind):
    from hic_gnn_b200 import metrics

    dense, sparse = _synthetic(2493, 0.3)
    meter = metrics.DsccMeter(dense if kind == "dense" else sparse)
    sets = [_structured_coords(2493, s).cuda() for s in (1, 2, 3)]
    sets[2] = (sets[2] * torch.linspace(0.2, 3.0, 2493, device="cuda").unsqueeze(1)).contiguous()
    eager = []
    for c in sets:
        a = meter(c).clone()
        b = meter(c).clone()
        assert a.dtype == torch.float64 and a.dim() == 0 and a.is_cuda
        assert torch.equal(a, b)
        eager.append(a)
    assert len({float(e) for e in eager}) == 3
    static = torch.empty_like(sets[0])
    static.copy_(sets[0])
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


def test_degenerate_inputs_give_nan():
    from hic_gnn_b200 import metrics, ops

    dense, sparse = _synthetic(300, 0.3)
    same = torch.full((300, 3), 0.25, device="cuda")
    for tgt in (dense, sparse):
        assert bool(torch.isnan(metrics.DsccMeter(tgt)(same)))
    two = ops.WishTarget.from_dense(torch.tensor([[0.0, 1.0], [1.0, 0.0]], device="cuda"))
    assert bool(torch.isnan(metrics.DsccMeter(two)(torch.tensor([[0.0, 0.0, 0.0], [1.0, 2.0, 3.0]], device="cuda"))))


def _chr19_setup(golden):
    from hic_gnn_b200 import models as gmodels, utils as gutils
    from oracle import graph as ograph, models as omodels, wish as owish

    g, _ = golden
    adj = g["1mb_kr_oracle"]
    n = adj.shape[0]
    x = 0.25 * torch.randn(n, 512, generator=torch.Generator().manual_seed(7))
    odata = ograph.load_input(adj.copy(), x.numpy())
    gdata = gutils.load_input(adj.copy(), x.numpy())
    truth = owish.cont2dist(odata.y.clone(), 1.0)
    target = gutils.wish_target(gdata.y, 1.0)
    torch.manual_seed(42)
    om = omodels.GATNetSelectiveResidualsUpdated()
    gm = gmodels.GATNetSelectiveResidualsUpdated().cuda()
    gm.load_state_dict(om.state_dict())
    return om, gm, odata, gdata, truth, target


def test_graphed_training_tracks_the_dscc_of_every_step(golden):
    from hic_gnn_b200 import metrics, train
    from oracle import loop as oloop, loss as oloss

    om, gm, odata, gdata, truth, target = _chr19_setup(golden)
    x = gdata.x.float()
    with torch.no_grad():
        exact64 = oloss.dscc(om.get_model(odata.x.float(), odata.edge_index).double(), truth)   # f64 distances of the oracle's start
    # the oracle's as-written loop records spearmanr of the pre-update structure (extras["dscc"]) from the same start
    _, extras = oloop.train(om, odata.x.float(), odata.edge_index, truth, mode="mse_pearson", lr=1e-3, thresh=0.0, max_steps=1, as_written=True)
    step = train.TrainStep(gm, x, gdata.edge_index, target, mode="mse_pearson", lr=1e-3, use_cuda_graph=True, track_dscc=True)
    got = []
    for s in range(20):
        with torch.no_grad():
            want = metrics.dscc(gm.get_model(x, gdata.edge_index), target)      # exact average ranks of this step's forward
        step()
        got.append(float(step.dscc))
        assert abs(got[-1] - want) < 1e-5, (s, got[-1], want)
    # step 0 against the oracle.  The reference's own value is spearmanr of f32 matmul-form cdist distances; its distance from the f64
    # value of the same coordinates is allowed on top of 1e-5
    noise = abs(extras[0]["dscc"] - exact64)
    print(f"step-0 dSCC: meter {got[0]!r}, oracle as written {extras[0]['dscc']!r}, oracle f64 {exact64!r}")
    assert abs(got[0] - exact64) < 1e-5, (got[0], exact64)
    assert abs(got[0] - extras[0]["dscc"]) < 1e-5 + noise, (got[0], extras[0]["dscc"], exact64)


def test_fit_fills_one_dscc_per_step(golden):
    from hic_gnn_b200 import train

    _, gm, _, gdata, _, target = _chr19_setup(golden)
    lst = []
    hist = train.fit(gm, gdata.x.float(), gdata.edge_index, target, mode="mse_pearson", lr=1e-3, thresh=0.0, max_steps=25, check_every=10,
                     use_cuda_graph=True, dscc_out=lst)
    assert len(hist) == 25 and len(lst) == 25 and all(np.isfinite(lst))
    assert lst[-1] != lst[0]


def test_graphed_c4_run_with_tracking():
    from hic_gnn_b200 import metrics, models, ops, synth, train
    from hic_gnn_b200.graph import CSRGraph

    n = 9970
    adj = synth.synthetic_map_chunked(n, 0.07, device="cuda")
    _, target = ops.cont2dist(adj, 1.0, want_f64=False, want_f32=True, symmetric=True)
    rowptr, col, val = ops.csr_from_dense(adj)
    graph = CSRGraph(rowptr, col, val, n)
    del adj
    x = synth.synthetic_features(n, device="cuda")
    torch.manual_seed(42)
    model = models.GATNetSelectiveResidualsUpdated().cuda()
    step = train.TrainStep(model, x, graph, target, mode="mse_pearson", lr=1e-3, use_cuda_graph=True, track_dscc=True)
    for _ in range(3):
        with torch.no_grad():
            want = metrics.dscc_streamed(model.get_model(x, graph), target)
        total, _ = step()
        got = float(step.dscc)
        assert np.isfinite(float(total)) and abs(got - want) < 1e-6, (got, want)


def test_generalize_example_tracks_dscc(monkeypatch, capsys):
    """examples/chr19_generalize.py --track-dscc: the per-step curve is printed every 50 steps and at the end."""
    import importlib.util
    import os
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("chr19_generalize", os.path.join(root, "examples", "chr19_generalize.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    monkeypatch.setattr(sys, "argv", ["chr19_generalize.py", "--steps", "60", "-thresh", "-1", "--track-dscc"])
    mod.main()
    lines = [ln for ln in capsys.readouterr().out.splitlines() if ln.startswith("step ")]
    assert [int(ln.split()[1].rstrip(":")) for ln in lines] == [0, 50, 59]
