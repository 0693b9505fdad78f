"""Row-block message passing (one GPU): GAT forward / fused backward and SAGE aggregation on target rows [g0, g1), the three
models on a row-block graph, and a one-rank sharded training step, against the full-graph calls and the f64 GAT reference of
tests/test_gpu_conv_shapes.py.  Partitions: one block, edge-balanced and equal-row blocks for 2, 3 and 8 ranks, and a hand-made
one with a one-row block, an empty block and boundaries that are not multiples of 8 or 16."""
import pytest
import torch

from helpers import rel_err, small_map
from test_gpu_conv_shapes import SHAPES, SLOPE, _check, _make_case, _self_loop_csr, gat_reference

pytestmark = pytest.mark.gpu


def _sparse_map(n: int, per_row: int = 12, seed: int = 0) -> torch.Tensor:
    """Symmetric f64 contact map with ~2 x per_row contacts per locus, mostly near the diagonal (a 10k-locus map without
    balancing a dense random matrix)."""
    g = torch.Generator().manual_seed(seed)
    i = torch.arange(n).repeat_interleave(per_row)
    d = (torch.rand(i.numel(), generator=g) ** 3 * n / 4).long() + 1
    j = (i + d) % n
    adj = torch.zeros(n, n, dtype=torch.float64)
    v = torch.rand(i.numel(), generator=g, dtype=torch.float64) + 0.1
    adj[i, j] = v
    adj[j, i] = v
    adj.fill_diagonal_(0)
    return adj


MAPS = {"n777": lambda: small_map(777, 0.05, seed=11), "n3001": lambda: small_map(3001, 0.02, seed=12), "n9973": lambda: _sparse_map(9973)}


def _partitions(graph):
    from hic_gnn_b200 import sharding

    n = graph.n
    parts = {"whole": [(0, n)]}
    for w in (2, 3, 8):
        parts[f"edges{w}"] = sharding.gnn_blocks(graph.rowptr, w)
        parts[f"rows{w}"] = sharding.all_blocks(n, w)
    h = n // 2 + 5
    parts["odd"] = [(0, 1), (1, 1), (1, 13), (13, h), (h, n)]
    for blocks in parts.values():
        assert blocks[0][0] == 0 and blocks[-1][1] == n and all(a1 == b0 for (_, a1), (b0, _) in zip(blocks, blocks[1:]))
    return parts


def _tuning(rows):
    from hic_gnn_b200 import _native as N

    N.check(N.lib().hicgat_gat_set_tuning(rows, 0), "hicgat_gat_set_tuning")


def _raw_fwd(graph, xl, gc, block=None):
    """hicgat_gat_fwd (block None) or hicgat_gat_fwd_rows: (out, alpha)."""
    from hic_gnn_b200 import _native as N
    from hic_gnn_b200.ops import _addr, _stream

    H, C = gc.heads, gc.out_channels
    r32, c32, _ = graph.with_self_loops()
    n = graph.n
    a_src, a_dst = torch.empty(n, H, device="cuda"), torch.empty(n, H, device="cuda")
    args = (xl.data_ptr(), gc.att_l.data_ptr(), gc.att_r.data_ptr(), gc.bias.data_ptr(), SLOPE, a_src.data_ptr(), a_dst.data_ptr())
    if block is None:
        alpha, out = torch.empty(c32.numel(), H, device="cuda"), torch.empty(n, H * C, device="cuda")
        N.check(N.lib().hicgat_gat_fwd(r32.data_ptr(), c32.data_ptr(), n, H, C, *args, alpha.data_ptr(), out.data_ptr(), _stream()), "hicgat_gat_fwd")
    else:
        (g0, g1), (e0, e1) = block, graph.row_block(*block).block_entries()
        alpha, out = torch.empty(e1 - e0, H, device="cuda"), torch.empty(g1 - g0, H * C, device="cuda")
        N.check(N.lib().hicgat_gat_fwd_rows(r32.data_ptr(), c32.data_ptr(), n, g0, g1, e0, H, C, *args, _addr(alpha), _addr(out), _stream()),
                "hicgat_gat_fwd_rows")
    return out, alpha


def _block_grads(graph, xl, gc, w, block):
    """Forward + backward of the row-block autograd function: (out rows, dxl partial, datt_l, datt_r, dbias)."""
    from hic_gnn_b200.layers import _GatAttendRows

    g0, g1 = block
    xg = xl.detach().clone().requires_grad_(True)
    out = _GatAttendRows.apply(xg, gc.att_l, gc.att_r, gc.bias, graph.row_block(g0, g1), gc.heads, gc.out_channels, SLOPE)
    grads = torch.autograd.grad(out, [xg, gc.att_l, gc.att_r, gc.bias], grad_outputs=w[g0:g1].contiguous(), allow_unused=True)
    return (out.detach(),) + tuple(torch.zeros_like(p) if g is None else g for g, p in zip(grads, [xg, gc.att_l, gc.att_r, gc.bias]))


@pytest.mark.parametrize("name", list(MAPS))
@pytest.mark.parametrize("H,C", SHAPES)
def test_gat_row_blocks(H, C, name):
    """Forward rows and alpha bit-identical to the full-graph call; block-summed backward against the f64 reference (the suite's
    tolerances, test_gpu_conv_shapes._check); both gather tunings give bit-identical results."""
    adj = MAPS[name]()
    f_in = (128, 256, 512)[(SHAPES.index((H, C)) + list(MAPS).index(name)) % 3]
    gc, x, graph, csr, w = _make_case(H, C, f_in, adj, seed=3)
    rowptr, col, deg = csr
    with torch.no_grad():
        xl = gc.lin_l(x).contiguous()
    eye = torch.eye(H * C, device="cuda")
    want = gat_reference(xl, eye, gc.att_l, gc.att_r, gc.bias, rowptr, col, H, w)  # "x" = dxl, "W" = dxl^T xl
    first = None
    try:
        for rows_per_cta in (8, 16):
            _tuning(rows_per_cta)
            out_full, alpha_full = _raw_fwd(graph, xl, gc)
            for pname, blocks in _partitions(graph).items():
                label = f"{name} H={H} C={C} {pname} rows/CTA={rows_per_cta}"
                for g0, g1 in blocks:
                    out_b, alpha_b = _raw_fwd(graph, xl, gc, (g0, g1))
                    e0, e1 = int(rowptr[g0]), int(rowptr[g1])
                    assert torch.equal(out_b, out_full[g0:g1]) and torch.equal(alpha_b, alpha_full[e0:e1]), (label, g0, g1)
                parts = [_block_grads(graph, xl, gc, w, b) for b in blocks]
                y = torch.cat([p[0] for p in parts])
                assert torch.equal(y, out_full), label
                dxl, datt_l, datt_r, dbias = (sum(p[k] for p in parts) for k in range(1, 5))
                got = (y, {"x": dxl, "W": dxl.double().t() @ xl.double(), "att_l": datt_l, "att_r": datt_r, "bias": dbias})
                _check(label, got, want, H, C, deg)
                if pname == "edges3":
                    if first is None:
                        first = got
                    else:  # 16 rows per CTA: same arithmetic per row as 8
                        for k in got[1]:
                            assert torch.equal(got[1][k], first[1][k]), (label, k)
    finally:
        _tuning(8)


@pytest.mark.parametrize("f", [128, 512, 1024])
@pytest.mark.parametrize("name", ["n777", "n3001"])
def test_sage_row_blocks_bit_identical(name, f):
    from hic_gnn_b200 import layers
    from hic_gnn_b200 import utils as gutils

    adj = MAPS[name]()
    n = adj.shape[0]
    x = 0.25 * torch.randn(n, f, generator=torch.Generator().manual_seed(f)).cuda()
    graph = gutils.load_input(adj.numpy().copy(), x.cpu().numpy()).edge_index
    full = layers._SageAggregate.apply(x, graph)
    for pname, blocks in _partitions(graph).items():
        got = torch.cat([layers._sage_aggregate_rows(x, graph.row_block(*b)) for b in blocks])
        assert torch.equal(got, full), (name, f, pname)
    with pytest.raises(NotImplementedError):
        layers._sage_aggregate_rows(x.clone().requires_grad_(True), graph.row_block(0, 5))


MODELS = ["Net", "GATNetSelectiveResidualsUpdated", "GATNetHeadsChanged3LayersLeakyReLUv2"]


@pytest.mark.parametrize("model_name", MODELS)
@pytest.mark.parametrize("name", ["n777", "n3001"])
def test_models_on_row_blocks(name, model_name):
    """get_model on row blocks: the block's rows of the full forward (1e-6; small blocks may take another GEMM path), and, given
    the full coordinate gradient, block-summed parameter gradients equal the full backward (1e-5)."""
    from hic_gnn_b200 import models, sharding, synth
    from hic_gnn_b200 import utils as gutils

    adj = MAPS[name]()
    n = adj.shape[0]
    x = synth.synthetic_features(n, seed=4).cuda()
    graph = gutils.load_input(adj.numpy().copy(), x.cpu().numpy()).edge_index
    torch.manual_seed(0)
    model = getattr(models, model_name)().cuda()
    params = list(model.parameters())
    gcoord = torch.randn(n, 3, generator=torch.Generator().manual_seed(5)).cuda()
    full = model.get_model(x, graph)
    g_full = torch.autograd.grad(full, params, grad_outputs=gcoord)
    h = n // 2 + 5
    for pname, blocks in {"edges3": sharding.gnn_blocks(graph.rowptr, 3), "rows8": sharding.all_blocks(n, 8),
                          "odd": [(0, 1), (1, 1), (1, 13), (13, h), (h, n)]}.items():
        acc = [torch.zeros_like(p) for p in params]
        rows = []
        for g0, g1 in blocks:
            y = model.get_model(x, graph.row_block(g0, g1))
            assert y.shape == (g1 - g0, 3)
            rows.append(y.detach())
            if g1 > g0:
                for a, g in zip(acc, torch.autograd.grad(y, params, grad_outputs=gcoord[g0:g1], allow_unused=True)):
                    if g is not None:
                        a += g
        assert rel_err(torch.cat(rows), full) < 1e-6, (model_name, pname)
        for (pn, _), a, g in zip(model.named_parameters(), acc, g_full):
            assert rel_err(a, g) < 1e-5, (model_name, pname, pn, rel_err(a, g))


def test_row_block_refusals():
    from hic_gnn_b200 import layers, models, synth
    from hic_gnn_b200 import utils as gutils

    adj = MAPS["n777"]()
    n = adj.shape[0]
    x = synth.synthetic_features(n, seed=4).cuda()
    graph = gutils.load_input(adj.numpy().copy(), x.cpu().numpy()).edge_index
    for g0, g1 in ((-1, 3), (5, 4), (0, n + 1)):
        with pytest.raises(ValueError):
            graph.row_block(g0, g1)
    blk = graph.row_block(3, 40)
    assert blk.rows == (3, 40) and graph.rows == (0, n) and blk._cache is graph._cache
    model = models.GATNetSelectiveResidualsUpdated().cuda()
    model.conv.path = "dense"
    with pytest.raises(ValueError, match="dense"):
        model.get_model(x, blk)
    model.conv.path = "auto"
    old = layers.GAT_BACKWARD
    layers.GAT_BACKWARD = "split"
    try:
        with pytest.raises(ValueError, match="split"):
            model.get_model(x, blk)
    finally:
        layers.GAT_BACKWARD = old
    # the C ABI refuses a bad block too
    from hic_gnn_b200 import _native as N

    r32, c32 = graph.i32()
    out = torch.empty(4, 512, device="cuda")
    assert N.lib().hicgat_spmm_csr_rows_f32(r32.data_ptr(), c32.data_ptr(), graph.sage_weights()[0].data_ptr(), x.data_ptr(), n, 5, 4, 512, out.data_ptr(), None) != 0
    assert N.lib().hicgat_spmm_csr_rows_f32(r32.data_ptr(), c32.data_ptr(), graph.sage_weights()[0].data_ptr(), x.data_ptr(), n, 0, n + 1, 512, out.data_ptr(), None) != 0


@pytest.mark.parametrize("graphed", [False, True])
def test_train_step_one_rank_shard_matches_replicated(graphed):
    """A one-rank GnnRowShard (block = all rows, local exchanges) follows the replicated step."""
    from hic_gnn_b200 import models, ops, sharding, synth, train
    from hic_gnn_b200 import utils as gutils

    n = 777
    adj = MAPS["n777"]()
    x = synth.synthetic_features(n, seed=3).cuda()
    data = gutils.load_input(adj.numpy().copy(), x.cpu().numpy())
    _, tgt = ops.cont2dist(adj.cuda(), 1.0, want_f64=False, want_f32=True)
    hist = {}
    for sharded in (False, True):
        torch.manual_seed(42)
        model = models.GATNetSelectiveResidualsUpdated().cuda()
        shard = sharding.GnnRowShard.for_rank(data.edge_index, model.parameters(), "cuda") if sharded else None
        if sharded:
            assert (shard.g0, shard.g1) == (0, n) and shard.capturable
        step = train.TrainStep(model, x, data.edge_index, tgt, mode="mse_pearson", use_cuda_graph=graphed, gnn_shard=shard)
        hist[sharded] = [float(step()[0]) for _ in range(4)]
    assert all(abs(a - b) <= 1e-6 * abs(b) for a, b in zip(hist[True], hist[False])), hist
