#!/usr/bin/env python
"""Row-sharded per-step dSCC (``metrics.ShardedDsccMeter``, ``hicgat_dscc_*_rows``).

    python scripts/bench_dscc_rows.py [--sizes 9970:0.07,49850:0.01] [--out profiles/r8_dscc_rows.json]
    torchrun --nproc-per-node G scripts/bench_dscc_rows.py [--out ...]

On one GPU (bench.py's c4 / c5 synthetic maps, dense WishTarget and implicit SparseWishTarget of the same map, helix coordinates,
2^22 bins): the row-sharded evaluation is emulated.  For W in {1, 2, 4, 8} blocks from ``sharding.row_block(..., balance="upper")``,
each block's local work -- the block distance histogram (``hicgat_dscc_dist_hist_rows``, with the scale kernel) and the block cross sum
(``hicgat_dscc_cross_*_rows``, with the mid-rank scan of the summed histogram) -- is timed by CUDA events over ``--calls`` back-to-back
calls, alternating with ``metrics.DsccMeter``; the slowest block is reported against the meter.  The exchanges, the finish and rank skew
are not in it.

Under torchrun with G >= 2 ranks: the full ``ShardedDsccMeter`` call (both exchanges) over p2p and over NCCL, alternating, and the
graphed GAT step (GATNetSelectiveResidualsUpdated, mse_pearson, sharded loss over p2p) with and without the p2p meter.
The GPU name, power limit and maximum SM clock are read in the same run.  Needs a GPU; there is no CPU path.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch
import torch.distributed as dist

from hic_gnn_b200 import _native as N
from hic_gnn_b200 import metrics, models, ops, sharding, synth, train
from hic_gnn_b200.graph import CSRGraph


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"name": torch.cuda.get_device_name(), "nvidia_smi": out.stdout.strip().splitlines() if out.returncode == 0 else None}


def helix(n, seed=5):
    g = torch.Generator().manual_seed(seed)
    t = torch.linspace(0, 6.0, n)
    c = torch.stack([torch.cos(t) * (1 + 0.1 * t), torch.sin(t) * (1 + 0.1 * t), 0.2 * t], dim=1)
    return (c + 0.05 * torch.randn(n, 3, generator=g)).float().cuda().contiguous()


def events(fn, calls):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(calls):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / calls


def maps(n, density, device="cuda"):
    adj = synth.synthetic_map_chunked(n, density, device=device)
    _, dense = ops.cont2dist(adj, 1.0, want_f64=False, want_f32=True, symmetric=True)
    rowptr, col, val = ops.csr_from_dense(adj)
    graph = CSRGraph(rowptr, col, val, n)
    sparse = ops.SparseWishTarget.from_graph(graph, adj, 1.0)
    return adj, dense, sparse, graph


def block_work(meter, tgt, coords, r0, r1, hist_sum, ws, cross):
    """The local work of one rank's block: its distance histogram, then its cross sum against the summed histogram."""
    lib, st, n, nb = N.lib(), ops._stream(), tgt.n, meter.nbins
    hist = torch.empty(nb, dtype=torch.int64, device="cuda")

    def run():
        N.check(lib.hicgat_dscc_dist_hist_rows(coords.data_ptr(), n, r0, r1, nb, hist.data_ptr(), ws.data_ptr(), ws.numel(), st), "dist_hist_rows")
        if isinstance(tgt, ops.WishTarget):
            rc = lib.hicgat_dscc_cross_dense_rows(coords.data_ptr(), tgt.data.data_ptr() + 4 * r0 * tgt.pitch, tgt.pitch, n, r0, r1, meter._t_scale, nb,
                                                  hist_sum.data_ptr(), meter._rank_t.data_ptr(), cross.data_ptr(), ws.data_ptr(), ws.numel(), st)
        else:
            rc = lib.hicgat_dscc_cross_implicit_rows(coords.data_ptr(), tgt.rowptr.data_ptr(), ops._addr(tgt.col), meter._rank_t.data_ptr(), n, r0, r1,
                                                     nb, hist_sum.data_ptr(), cross.data_ptr(), ws.data_ptr(), ws.numel(), st)
        N.check(rc, "cross_rows")

    return run, hist


def bench_one_gpu(n, density, rounds, calls):
    adj, dense, sparse, _ = maps(n, density)
    del adj
    coords = helix(n)
    out = {"n": n, "density": density, "pairs": n * (n - 1) // 2}
    for name, tgt in (("dense", dense), ("implicit", sparse)):
        meter = metrics.DsccMeter(tgt)
        ws = torch.empty(N.lib().hicgat_dscc_workspace_bytes(n, meter.nbins), dtype=torch.uint8, device="cuda")
        cross = torch.empty(2, dtype=torch.float64, device="cuda")
        rho_full = float(meter(coords))
        rows = {"meter_ms": [], "rho_meter": rho_full}
        for w in (1, 2, 4, 8):
            blocks = sharding.all_blocks(n, w, "upper")
            hist_sum = torch.zeros(meter.nbins, dtype=torch.int64, device="cuda")
            runs = []
            for r0, r1 in blocks:
                run, h = block_work(meter, tgt, coords, r0, r1, hist_sum, ws, cross)
                run()
                hist_sum += h
                runs.append(run)
            times = [[] for _ in blocks]
            for _ in range(rounds):
                rows["meter_ms"].append(events(lambda: meter(coords), calls))
                for k, run in enumerate(runs):
                    run()
                    times[k].append(events(run, calls))
            med = [statistics.median(t) for t in times]
            rows[f"W{w}"] = {"blocks": blocks, "block_ms": med, "slowest_ms": max(med)}
        rows["meter_ms"] = statistics.median(rows["meter_ms"])
        for w in (1, 2, 4, 8):
            rows[f"W{w}"]["slowest_over_meter"] = rows[f"W{w}"]["slowest_ms"] / rows["meter_ms"]
        out[name] = rows
        print(json.dumps({n: {name: {k: (v["slowest_ms"] if isinstance(v, dict) else v) for k, v in rows.items()}}}), flush=True)
    return out


def bench_multi(n, density, rounds, calls, steps):
    rank, world = dist.get_rank(), dist.get_world_size()
    adj, full, sparse, graph = maps(n, density)
    r0, r1 = sharding.row_block(n, rank, world, "upper")
    _, tgt = ops.cont2dist(adj[r0:r1].contiguous(), 1.0, want_f64=False, want_f32=True, r0=r0, r1=r1, max_reduce=sharding.allreduce_max_)
    del adj
    coords = helix(n)
    out = {"n": n, "world": world}
    for name, block in (("dense", tgt), ("implicit", sparse.rows(r0, r1))):
        meters = {t: metrics.ShardedDsccMeter(block, transport=t) for t in ("p2p", "nccl")}
        ms = {t: [] for t in meters}
        for _ in range(rounds):
            for t, m in meters.items():
                m(coords)
                dist.barrier()
                ms[t].append(events(lambda: m(coords), calls))
        rho = {t: float(m(coords)) for t, m in meters.items()}
        out[name] = {f"call_ms_{t}": statistics.median(v) for t, v in ms.items()} | {"rho": rho}
        del meters
    x = synth.synthetic_features(n, device="cuda")
    red = ops.sharded_reducer(tgt, "mse_moments", transport="p2p")
    stepper = {}
    for with_meter in (False, True):
        torch.manual_seed(42)
        model = models.GATNetSelectiveResidualsUpdated().cuda()
        kw = {"dscc_meter": metrics.ShardedDsccMeter(tgt, transport="p2p")} if with_meter else {}
        stepper[with_meter] = train.TrainStep(model, x, graph, tgt, mode="mse_pearson", lr=1e-3, use_cuda_graph=True, reducer=red, **kw)
    st = {False: [], True: []}
    for _ in range(rounds):
        for k, s in stepper.items():
            s()
            dist.barrier()
            st[k].append(events(s, steps))
    out["train_step_ms"] = {"without_meter": statistics.median(st[False]), "with_meter": statistics.median(st[True])}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="9970:0.07,49850:0.01")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    sizes = [(int(s.split(":")[0]), float(s.split(":")[1])) for s in a.sizes.split(",")]
    multi = int(os.environ.get("WORLD_SIZE", "1")) > 1
    if multi:
        local = int(os.environ["LOCAL_RANK"])
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    res = {"gpu": gpu_info(), "nbins": metrics.NBINS}
    if multi:
        res["multi_gpu"] = [bench_multi(n, d, a.rounds, a.calls, a.steps) for n, d in sizes]
    else:
        res["one_gpu"] = [bench_one_gpu(n, d, a.rounds, a.calls) for n, d in sizes]
        res["multi_gpu"] = "not measured: one GPU (run under torchrun with >= 2 ranks)"
    if not multi or dist.get_rank() == 0:
        text = json.dumps(res, indent=1)
        print(text)
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            open(a.out, "w").write(text + "\n")
    if multi:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
