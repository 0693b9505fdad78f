"""Row-sharded GNN training on two GPUs: each rank runs the GAT net on its edge-balanced row block, the coordinates are
all-gathered and the parameter gradients all-reduced (sharding.GnnRowShard), the loss is row-sharded too.  The sharded step must
follow the single-GPU replicated step and keep the replicas bit-identical.  Skipped on a 1-GPU box; the host-side logic is
covered on CPU by tests/test_gnn_rows_gloo.py."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, n, tmpdir):
    import torch.distributed as dist

    from hic_gnn_b200 import models, ops, sharding, synth, train, utils

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        adj = synth.synthetic_map(n, 0.3, seed=5).cuda()
        x = synth.synthetic_features(n, seed=3).cuda()
        data = utils.load_input(adj.cpu().numpy().copy(), torch.zeros(n, 4).numpy(), device=f"cuda:{rank}")
        r0, r1 = sharding.row_block(n, rank, world)
        _, tgt = ops.cont2dist(adj[r0:r1].contiguous(), 1.0, want_f64=False, want_f32=True, r0=r0, r1=r1, max_reduce=sharding.allreduce_max_)
        _, full = ops.cont2dist(adj, 1.0, want_f64=False, want_f32=True)

        torch.manual_seed(42)
        ref_model = models.GATNetSelectiveResidualsUpdated().cuda()
        ref = train.TrainStep(ref_model, x, data.edge_index, full, mode="mse_pearson", lr=1e-3)
        want = [float(ref()[0]) for _ in range(6)]

        for transport, graphed in (("nccl", False), ("p2p", False), ("p2p", True)):
            torch.manual_seed(42)
            model = models.GATNetSelectiveResidualsUpdated().cuda()
            shard = sharding.GnnRowShard.for_rank(data.edge_index, model.parameters(), "cuda", transport=transport)
            assert shard.transport == transport
            red = ops.sharded_reducer(tgt, "mse_moments", transport="p2p" if graphed else transport)
            step = train.TrainStep(model, x, data.edge_index, tgt, mode="mse_pearson", lr=1e-3, use_cuda_graph=graphed, reducer=red, gnn_shard=shard)
            got = []
            for _ in range(6):
                got.append(float(step()[0]))
                sd = torch.cat([p.detach().reshape(-1) for p in model.parameters()])
                gathered = [torch.empty_like(sd) for _ in range(world)]
                dist.all_gather(gathered, sd)
                assert all(torch.equal(gathered[0], t) for t in gathered), (transport, graphed, "replicas diverged")
            assert abs(got[0] - want[0]) <= 1e-6 * abs(want[0]), (transport, graphed, got, want)
            assert all(abs(a - b) <= 1e-2 * abs(b) for a, b in zip(got, want)), (transport, graphed, got, want)
        with pytest.raises(ValueError, match="capturable"):
            shard = sharding.GnnRowShard.for_rank(data.edge_index, model.parameters(), "cuda", transport="nccl")
            train.TrainStep(model, x, data.edge_index, tgt, mode="mse_pearson", use_cuda_graph=True,
                            reducer=ops.sharded_reducer(tgt, "mse_moments", transport="p2p"), gnn_shard=shard)
        open(os.path.join(tmpdir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("n", [777, 3001])
def test_sharded_gnn_matches_single_gpu(tmp_path, n):
    import torch.multiprocessing as mp

    world = 2
    port = 29900 + os.getpid() % 2000
    mp.spawn(_worker, args=(world, port, n, str(tmp_path)), nprocs=world, join=True)
    assert all((tmp_path / f"ok{r}").exists() for r in range(world))
