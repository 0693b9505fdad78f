"""Host-side logic of the row-sharded GNN on CPU: the edge-balanced partition, and both exchanges of
``sharding.GnnRowShard`` over world_size-2 and -3 gloo process groups (the collective transport on CPU tensors)."""
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from hic_gnn_b200 import sharding


def _check_cover(blocks, n, world):
    assert len(blocks) == world and blocks[0][0] == 0 and blocks[-1][1] == n
    assert all(a0 <= a1 == b0 for (a0, a1), (b0, _) in zip(blocks, blocks[1:]))


def test_gnn_blocks_balance_edges_plus_one():
    g = torch.Generator().manual_seed(3)
    for n in (1, 2, 7, 100, 3001):
        deg = torch.randint(0, 40, (n,), generator=g)
        rowptr = torch.zeros(n + 1, dtype=torch.int64)
        rowptr[1:] = torch.cumsum(deg, 0)
        for world in (1, 2, 3, 8):
            blocks = sharding.gnn_blocks(rowptr, world)
            _check_cover(blocks, n, world)
            assert blocks == sharding.gnn_blocks(rowptr.tolist(), world)  # tensor or list, same arithmetic
            mass = [int(rowptr[b] - rowptr[a]) + (b - a) for a, b in blocks]
            total, heaviest = int(rowptr[-1]) + n, int(deg.max()) + 1
            # every cut sits within half a row of its ideal prefix weight
            assert all(abs(m - total / world) <= heaviest for m in mass), (n, world, mass)


def test_gnn_blocks_empty_and_one_row_blocks():
    assert sharding.gnn_blocks([0], 3) == [(0, 0)] * 3                    # no rows: all blocks empty
    assert sharding.gnn_blocks([0, 5], 2) == [(0, 0), (0, 1)]             # one row: ties go to the lower cut
    assert sharding.gnn_blocks([0, 100, 101, 102], 3) == [(0, 0), (0, 1), (1, 3)]  # a hub row outweighs a share
    assert sharding.gnn_blocks([0, 0, 0, 0, 0], 4) == [(0, 1), (1, 2), (2, 3), (3, 4)]  # edgeless: equal rows
    assert sharding.gnn_blocks([0, 1, 2], 1) == [(0, 2)]
    with pytest.raises(ValueError):
        sharding.gnn_blocks([0, 1], 0)


def _worker(rank, world, port, n, tmpdir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        g = torch.Generator().manual_seed(0)
        deg = torch.randint(0, 9, (n,), generator=g)
        rowptr = torch.zeros(n + 1, dtype=torch.int64)
        rowptr[1:] = torch.cumsum(deg, 0)
        blocks = sharding.gnn_blocks(rowptr, world)
        g0, g1 = blocks[rank]
        params = [torch.nn.Parameter(torch.zeros(5, 3)), torch.nn.Parameter(torch.zeros(7)), torch.nn.Parameter(torch.zeros(2, 2, 2))]
        shard = sharding.GnnRowShard(n, (g0, g1), params, "cpu", transport="auto")
        assert shard.transport == "nccl" and not shard.capturable

        # coordinate gather: exact in both directions
        full = torch.randn(n, 3, generator=g)
        local = full[g0:g1].clone().requires_grad_(True)
        got = shard.gather_coords(local)
        assert torch.equal(got, full)
        up = torch.randn(n, 3, generator=g)  # the (already reduced) coordinate gradient, the same on every rank
        (got * up).sum().backward()
        assert torch.equal(local.grad, up[g0:g1])
        with pytest.raises(ValueError):
            shard.gather_coords(torch.zeros(g1 - g0 + 1, 3))

        # parameter gradients: pack, reduce, unpack; identical on every rank; a missing gradient counts as zero
        per_rank = [[torch.randn(p.shape, generator=g) for p in params] for _ in range(world)]
        for p, v in zip(params, per_rank[rank]):
            p.grad = v.clone()
        params[1].grad = None if rank == 0 else params[1].grad
        shard.reduce_grads()
        for k, p in enumerate(params):
            want = sum(per_rank[r][k].double() for r in range(world) if not (k == 1 and r == 0)).float()
            assert torch.allclose(p.grad, want, rtol=1e-6, atol=1e-6), k
            everyone = [torch.empty_like(p.grad) for _ in range(world)]
            dist.all_gather(everyone, p.grad)
            assert all(torch.equal(everyone[0], t) for t in everyone)
        with pytest.raises(ValueError):
            shard.reduce_grads(params[:2])
        open(os.path.join(tmpdir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,n", [(2, 37), (3, 10), (3, 2)])
def test_gnn_row_shard_gloo(tmp_path, world, n):
    port = 30500 + os.getpid() % 2000 + 10 * world + n % 10
    mp.spawn(_worker, args=(world, port, n, str(tmp_path)), nprocs=world, join=True)
    assert all((tmp_path / f"ok{r}").exists() for r in range(world))


def test_gnn_row_shard_rejects_bad_arguments():
    p = [torch.nn.Parameter(torch.zeros(3))]
    with pytest.raises(ValueError):
        sharding.GnnRowShard(10, (4, 2), p, "cpu")
    with pytest.raises(ValueError):
        sharding.GnnRowShard(10, (0, 11), p, "cpu")
    with pytest.raises(ValueError):
        sharding.GnnRowShard(10, (0, 5), p, "cpu", transport="mpi")
    solo = sharding.GnnRowShard(10, (0, 10), p, "cpu")  # no process group: a local no-op exchange, capturable
    assert solo.capturable
    x = torch.randn(10, 3)
    assert torch.equal(solo.gather_coords(x), x)
