"""Row-sharded pairwise loss on real GPUs over NCCL (world_size 2): the sharded result must equal
the single-GPU result of the same kernel and the oracle's loss.  Skipped on a 1-GPU box; the
host-side sharding logic is covered on CPU by tests/test_sharding_gloo.py."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, n, tmpdir):
    import torch.distributed as dist

    import hic_gnn_b200 as hg
    from hic_gnn_b200 import ops, sharding, synth
    from helpers import random_coords, rel_err

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        adj = synth.synthetic_map(n, 0.3, seed=5).cuda()
        coords = random_coords(n, seed=9).cuda().requires_grad_(True)
        r0, r1 = sharding.row_block(n, rank, world)
        # sharded wish-distance build: local max -> all-reduce(max) -> apply
        _, tgt = ops.cont2dist(adj[r0:r1].contiguous(), 1.0, want_f64=False, want_f32=True, r0=r0, r1=r1, max_reduce=sharding.allreduce_max_)
        _, full = ops.cont2dist(adj, 1.0, want_f64=False, want_f32=True)
        assert torch.equal(tgt.dense(), full.dense()[r0:r1])
        for mode, transport in [("mse", "nccl"), ("mse_moments", "nccl"), ("contrastive", "nccl"),
                                ("mse", "p2p"), ("mse_moments", "p2p"), ("contrastive", "p2p"), ("mse_moments", "p2p_oneshot")]:
            red = ops.sharded_reducer(tgt, mode, transport=transport)
            if transport != "nccl":  # several steps: exercises the (device-side) epoch / barrier protocol
                for _ in range(5):
                    hg.pairwise_loss(coords, tgt, mode, reducer=red)
            loss_s, mom_s = hg.pairwise_loss(coords, tgt, mode, reducer=red)
            (g_s,) = torch.autograd.grad(loss_s, coords)
            loss_1, mom_1 = hg.pairwise_loss(coords, full, mode)
            (g_1,) = torch.autograd.grad(loss_1, coords)
            assert abs(float(loss_s) - float(loss_1)) <= 1e-6 * abs(float(loss_1)), (mode, float(loss_s), float(loss_1))
            assert rel_err(mom_s, mom_1) < 1e-7
            assert rel_err(g_s, g_1) < 1e-5
            # every rank holds the identical reduced result (replicated GNN stays in lock step)
            gathered = [torch.empty_like(g_s) for _ in range(world)]
            dist.all_gather(gathered, g_s.contiguous())
            assert all(torch.equal(gathered[0], t) for t in gathered)
        # implicit (sparse) target, row-sharded over the same two transports
        from hic_gnn_b200 import utils

        data = utils.load_input(adj.cpu().numpy().copy(), torch.zeros(n, 4).numpy(), device=f"cuda:{rank}")
        sp_full = utils.sparse_wish_target(data, 1.0)
        sp_loc = sp_full.rows(r0, r1)
        for transport in ("nccl", "p2p"):
            red = ops.sharded_reducer(sp_loc, "mse_moments", transport=transport)
            loss_s, mom_s = hg.pairwise_loss(coords, sp_loc, "mse_moments", reducer=red)
            (g_s,) = torch.autograd.grad(loss_s, coords)
            loss_1, mom_1 = hg.pairwise_loss(coords, full, "mse_moments")
            (g_1,) = torch.autograd.grad(loss_1, coords)
            assert abs(float(loss_s) - float(loss_1)) <= 1e-6 * abs(float(loss_1)), (transport, float(loss_s), float(loss_1))
            assert rel_err(mom_s, mom_1) < 1e-6 and rel_err(g_s, g_1) < 1e-5
        # whole sharded training step (replicated GAT net, row-sharded loss, two-shot exchange) captured in ONE CUDA graph:
        # the exchange takes its epoch from device memory, so replays stay in step; must follow the eager sharded loop
        from hic_gnn_b200 import models, train

        x = synth.synthetic_features(n, seed=3).cuda()
        hist = {}
        for graphed in (False, True):
            torch.manual_seed(42)
            model = models.GATNetSelectiveResidualsUpdated().cuda()
            red = ops.sharded_reducer(tgt, "mse_moments", transport="p2p")
            step = train.TrainStep(model, x, data.edge_index, tgt, mode="mse_pearson", lr=1e-3, use_cuda_graph=graphed, reducer=red)
            hist[graphed] = [float(step()[0]) for _ in range(6)]
            sd = torch.cat([p.detach().reshape(-1) for p in model.parameters()])
            gathered = [torch.empty_like(sd) for _ in range(world)]
            dist.all_gather(gathered, sd)
            assert all(torch.equal(gathered[0], t) for t in gathered), "replicas diverged"
        assert abs(hist[True][0] - hist[False][0]) <= 1e-6 * abs(hist[False][0]), hist
        assert all(abs(a - b) <= 1e-2 * abs(b) for a, b in zip(hist[True], hist[False])), hist  # capturable Adam rounds its bias corrections differently
        with pytest.raises(ValueError, match="capturable"):
            train.TrainStep(model, x, data.edge_index, tgt, mode="mse_pearson", use_cuda_graph=True, reducer=ops.sharded_reducer(tgt, "mse_moments", transport="nccl"))
        open(os.path.join(tmpdir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("n", [777, 3001])
def test_sharded_loss_nccl_matches_single_gpu(tmp_path, n):
    import torch.multiprocessing as mp

    world = 2
    port = 29700 + os.getpid() % 2000
    mp.spawn(_worker, args=(world, port, n, str(tmp_path)), nprocs=world, join=True)
    assert all((tmp_path / f"ok{r}").exists() for r in range(world))
