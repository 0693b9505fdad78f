"""Row-sharded differentiable Pearson modes on real GPUs over NCCL (two all_reduce calls per step) and over the capturable p2p
exchange (two two-shot exchanges): the sharded result must equal the single-GPU result, and a graph-captured sharded training
step must follow the eager one.  Skipped on a 1-GPU box; the host-side logic of the
two-exchange reducer is covered on CPU by tests/test_pearson_grad_host.py."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, n, tmpdir):
    import torch.distributed as dist

    import hic_gnn_b200 as hg
    from hic_gnn_b200 import ops, sharding, synth, utils
    from helpers import random_coords, rel_err

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        adj = synth.synthetic_map(n, 0.3, seed=5).cuda()
        coords = random_coords(n, seed=9).cuda().requires_grad_(True)
        balance = "upper" if ops._USE_UPPER else "rows"
        r0, r1 = sharding.row_block(n, rank, world, balance)
        _, tgt = ops.cont2dist(adj[r0:r1].contiguous(), 1.0, want_f64=False, want_f32=True, r0=r0, r1=r1, max_reduce=sharding.allreduce_max_,
                               symmetric=True)
        _, full = ops.cont2dist(adj, 1.0, want_f64=False, want_f32=True)
        data = utils.load_input(adj.cpu().numpy().copy(), torch.zeros(n, 4).numpy(), device=f"cuda:{rank}")
        sp_full = utils.sparse_wish_target(data, 1.0)
        for local, whole in ((tgt, full), (sp_full.rows(r0, r1), sp_full)):
            for mode, transport in (("pearson", "nccl"), ("mse_pearson_grad", "nccl"), ("pearson", "p2p"), ("mse_pearson_grad", "p2p")):
                red = ops.sharded_reducer(local, mode, transport=transport)
                for _ in range(2):
                    loss_s, mom_s = hg.pairwise_loss(coords, local, mode, reducer=red)
                (g_s,) = torch.autograd.grad(loss_s, coords)
                loss_1, mom_1 = hg.pairwise_loss(coords, whole, mode)
                (g_1,) = torch.autograd.grad(loss_1, coords)
                assert abs(float(loss_s) - float(loss_1)) <= 1e-6 * abs(float(loss_1)), (mode, float(loss_s), float(loss_1))
                assert rel_err(mom_s, mom_1) < 1e-7
                assert rel_err(g_s, g_1) < 1e-6, (mode, rel_err(g_s, g_1))
                gathered = [torch.empty_like(g_s) for _ in range(world)]
                dist.all_gather(gathered, g_s.contiguous())
                assert all(torch.equal(gathered[0], t) for t in gathered)
        # the graph-captured sharded training step over the p2p exchange against the eager one
        from hic_gnn_b200 import models, train

        x = 0.25 * torch.randn(n, 512, generator=torch.Generator().manual_seed(104))
        gdata = utils.load_input(adj.cpu().numpy().copy(), x.numpy(), device=f"cuda:{rank}")
        torch.manual_seed(42)
        init = models.GATNetSelectiveResidualsUpdated().state_dict()
        totals = []
        for graphed in (False, True):
            gm = models.GATNetSelectiveResidualsUpdated().cuda()
            gm.load_state_dict(init)
            red = ops.sharded_reducer(tgt, "mse_pearson_grad", transport="p2p")
            assert red.capturable
            step = train.TrainStep(gm, gdata.x.float(), gdata.edge_index, tgt, mode="mse_pearson_grad", use_cuda_graph=graphed, reducer=red)
            if not graphed:
                step.optimizer = torch.optim.Adam(gm.parameters(), lr=1e-3, capturable=True)
            totals.append(torch.stack([step()[0].clone() for _ in range(10)]))
        assert float(((totals[1] - totals[0]) / totals[0]).abs().max()) < 1e-6, totals
        open(os.path.join(tmpdir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_sharded_pearson_matches_single_gpu(tmp_path):
    import torch.multiprocessing as mp

    world = min(torch.cuda.device_count(), 8)
    port = 33500 + os.getpid() % 2000
    mp.spawn(_worker, args=(world, port, 1500, str(tmp_path)), nprocs=world, join=True)
    assert all((tmp_path / f"ok{r}").exists() for r in range(world))
