"""Row-sharded per-step dSCC on two GPUs (``metrics.ShardedDsccMeter`` over p2p and NCCL): the meter is bit-identical on both ranks and
within 1e-12 of the single-GPU ``DsccMeter``; ``fit(reducer=..., dscc_out=..., dscc_meter=...)`` eager and graphed keeps identical
histories on both ranks that follow the single-GPU ``track_dscc`` run; sharded ``mse_spearman`` gives both ranks the same totals.
Skipped on a 1-GPU box; the exchange's host logic is covered on CPU by tests/test_dscc_rows_gloo.py."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu


def _same_on_all_ranks(t, world):
    import torch.distributed as dist

    t = t.reshape(-1).double().cuda()
    everyone = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(everyone, t)
    return all(torch.equal(everyone[0], e) for e in everyone)


def _worker(rank, world, port, n, tmpdir):
    import torch.distributed as dist

    from hic_gnn_b200 import metrics, models, ops, sharding, synth, train
    from hic_gnn_b200.graph import CSRGraph

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        adj = synth.synthetic_map(n, 0.3, seed=5).cuda()
        x = synth.synthetic_features(n, seed=3).cuda()
        graph = CSRGraph(*ops.csr_from_dense(adj), n)
        r0, r1 = sharding.row_block(n, rank, world, balance="upper")
        _, tgt = ops.cont2dist(adj[r0:r1].contiguous(), 1.0, want_f64=False, want_f32=True, r0=r0, r1=r1, max_reduce=sharding.allreduce_max_)
        _, full = ops.cont2dist(adj, 1.0, want_f64=False, want_f32=True)
        sparse = ops.SparseWishTarget.from_graph(graph, adj, 1.0)
        g = torch.Generator().manual_seed(1)
        coords = (0.3 * torch.randn(n, 3, generator=g)).cuda()

        # the meter on the same coordinates
        for transport in ("p2p", "nccl"):
            for block, whole in ((tgt, full), (sparse.rows(r0, r1), sparse)):
                m = metrics.ShardedDsccMeter(block, transport=transport)
                assert m.transport == transport and m.capturable == (transport == "p2p")
                got = m(coords).clone()
                want = metrics.DsccMeter(whole)(coords)
                assert _same_on_all_ranks(got, world), transport
                assert abs(float(got) - float(want)) <= 1e-12 * max(1.0, abs(float(want))), (transport, float(got), float(want))
                assert torch.equal(m(coords), got)

        # training: single-GPU track_dscc history against the sharded meter's, eager and graphed
        torch.manual_seed(42)
        ref = []
        want_loss = train.fit(models.GATNetSelectiveResidualsUpdated().cuda(), x, graph, full, mode="mse_pearson", lr=1e-3, thresh=0.0,
                              max_steps=6, dscc_out=ref)
        for transport, graphed in (("nccl", False), ("p2p", False), ("p2p", True)):
            torch.manual_seed(42)
            model = models.GATNetSelectiveResidualsUpdated().cuda()
            red = ops.sharded_reducer(tgt, "mse_moments", transport="p2p" if graphed else transport)
            meter = metrics.ShardedDsccMeter(tgt, transport=transport)
            got = []
            loss = train.fit(model, x, graph, tgt, mode="mse_pearson", lr=1e-3, thresh=0.0, max_steps=6, use_cuda_graph=graphed, reducer=red,
                             dscc_out=got, dscc_meter=meter)
            assert _same_on_all_ranks(torch.tensor(got), world) and _same_on_all_ranks(torch.tensor(loss), world)
            assert abs(got[0] - ref[0]) <= 1e-12 * abs(ref[0]), (transport, graphed, got[0], ref[0])
            assert all(abs(a - b) <= 1e-2 * abs(b) for a, b in zip(got, ref)), (transport, graphed, got, ref)
            assert all(abs(a - b) <= 1e-2 * abs(b) for a, b in zip(loss, want_loss))

        # sharded mse_spearman: the same totals on both ranks; the first one is the single-GPU total
        torch.manual_seed(42)
        one = train.fit(models.GATNetSelectiveResidualsUpdated().cuda(), x, graph, full, mode="mse_spearman", lr=1e-3, thresh=0.0, max_steps=3)
        torch.manual_seed(42)
        red = ops.sharded_reducer(tgt, "mse_moments", transport="nccl")
        tot = train.fit(models.GATNetSelectiveResidualsUpdated().cuda(), x, graph, tgt, mode="mse_spearman", lr=1e-3, thresh=0.0, max_steps=3,
                        reducer=red, dscc_meter=metrics.ShardedDsccMeter(tgt, transport="nccl"))
        assert _same_on_all_ranks(torch.tensor(tot), world)
        assert abs(tot[0] - one[0]) < 1e-5, (tot, one)

        # histogram mid-ranks of the summed distance histogram against exact average ranks (distinct distances: one per bin)
        m = metrics.ShardedDsccMeter(tgt, transport="p2p")
        m(coords)
        hist = m._x.hist_sum.clone()
        d = metrics.upper_pairs(coords, full)[1].double()
        exact = metrics.average_ranks(d)
        assert int(hist.sum()) == d.numel()
        mid = metrics._midranks(hist)
        if int((hist > 1).sum()) == 0:
            bins = torch.nonzero(hist).reshape(-1)
            assert torch.equal(mid[bins], torch.sort(exact).values)
        open(os.path.join(tmpdir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("n", [777, 3001])
def test_sharded_dscc_matches_single_gpu(tmp_path, n):
    import torch.multiprocessing as mp

    world = 2
    port = 29700 + os.getpid() % 2000
    mp.spawn(_worker, args=(world, port, n, str(tmp_path)), nprocs=world, join=True)
    assert all((tmp_path / f"ok{r}").exists() for r in range(world))
