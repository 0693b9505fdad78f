"""The collective transport of ``sharding.DsccExchange`` (the exchanges of a row-sharded per-step dSCC) over world-size-2 and -3 gloo
process groups on CPU tensors: the u64 histogram is summed exactly, and the f64[2] cross sums are added in rank order from 0.0, so every
rank holds the same bits."""
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from hic_gnn_b200 import sharding


def _worker(rank, world, port, nbins, tmpdir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        x = sharding.DsccExchange(nbins, "cpu", transport="auto")
        assert x.transport == "nccl" and not x.capturable
        g = torch.Generator().manual_seed(0)
        hists = [torch.randint(0, 1 << 40, (nbins,), generator=g, dtype=torch.int64) for _ in range(world)]
        hists[1][: nbins // 2] = (1 << 62) + 12345          # counts whose sum needs every bit of an int64
        # partial cross sums of very different sizes: the grouping changes the f64 sum
        crosses = [torch.tensor([1e16 * (r + 1) + 1.25, (-1) ** r * 3.0 ** r / 7.0], dtype=torch.float64) for r in range(world)]
        for step in range(2):
            x.hist.copy_(hists[rank] + step)
            x.cross.copy_(crosses[rank] * (step + 1))
            got = x.sum_hist()
            want = sum(h + step for h in hists)
            assert torch.equal(got, want)
            c = x.sum_cross()
            ref = torch.zeros(2, dtype=torch.float64)
            for r in range(world):
                ref += crosses[r] * (step + 1)
            assert torch.equal(c, ref), (c, ref)
            everyone = [torch.empty(2, dtype=torch.float64) for _ in range(world)]
            dist.all_gather(everyone, c)
            assert all(torch.equal(everyone[0], t) for t in everyone)
        open(os.path.join(tmpdir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,nbins", [(2, 37), (3, 16), (3, 1)])
def test_dscc_exchange_gloo(tmp_path, world, nbins):
    port = 31500 + os.getpid() % 2000 + 10 * world + nbins % 10
    mp.spawn(_worker, args=(world, port, nbins, str(tmp_path)), nprocs=world, join=True)
    assert all((tmp_path / f"ok{r}").exists() for r in range(world))


def test_one_rank_exchange_is_a_no_op():
    x = sharding.DsccExchange(8, "cpu")
    assert x.capturable and x.transport == "nccl"
    x.hist.copy_(torch.arange(8))
    x.cross.copy_(torch.tensor([2.5, -1.0], dtype=torch.float64))
    assert torch.equal(x.sum_hist(), torch.arange(8)) and torch.equal(x.sum_cross(), torch.tensor([2.5, -1.0], dtype=torch.float64))
