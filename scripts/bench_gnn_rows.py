"""Row-sharded GNN (sharding.GnnRowShard) against the replicated GNN on the synthetic C4 / C5 maps.

    torchrun --nproc_per_node G scripts/bench_gnn_rows.py [--workloads c5,c4] [--steps 50] [--rounds 3] [--out profiles/r7_gnn_rows.json]
    python scripts/bench_gnn_rows.py [--workloads c5,c4] [--worlds 2,4,8] [--out ...]

Under torchrun (G > 1): graphed training steps/s of the GAT net (mode mse_pearson, row-sharded loss over the two-shot p2p
exchange) with the GNN replicated and with the GNN row-sharded, measured in the same run, alternating ``--rounds`` times.

On one GPU (no torchrun): an EMULATION of one rank's local GNN work for G ranks -- the GAT net's forward and backward
(projection GEMMs, GAT kernels, head) on every rank's edge-balanced row block in turn, given a coordinate gradient, and the
GAT message-passing kernels alone (forward + fused backward) on the block; the slowest block is the per-rank time.  The
exchanges and the sharded loss are not part of it.  The replicated full-map forward + backward and the graphed replicated
training step are timed alongside.  CUDA events, after warm-ups."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch


def timed(fn, reps=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def card():
    dev = torch.cuda.current_device()
    out = {"gpu": torch.cuda.get_device_name(dev)}
    try:  # read-only query
        q = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        out["power_limit"] = q.stdout.strip() or "unknown"
    except Exception:
        out["power_limit"] = "unknown"
    return out


def setup(name, dev):
    import bench
    from hic_gnn_b200 import ops, synth
    from hic_gnn_b200.graph import CSRGraph

    w = bench.WORKLOADS[name]
    n = w["n"]
    adj = synth.synthetic_map_chunked(n, w["density"], device=dev)
    rowptr, col, val = ops.csr_from_dense(adj)
    graph = CSRGraph(rowptr, col, val, n)
    x = synth.synthetic_features(n).to(dev)
    return w, n, adj, graph, x


def emulate(name, worlds, reps):
    from hic_gnn_b200 import layers, models, sharding

    w, n, adj, graph, x = setup(name, "cuda")
    del adj
    torch.manual_seed(0)
    model = models.GATNetSelectiveResidualsUpdated().cuda()
    params = list(model.parameters())
    gcoord = 1e-3 * torch.randn(n, 3, device="cuda")

    def fwd_bwd(view, g0, g1):
        y = model.get_model(x, view)
        torch.autograd.grad(y, params, grad_outputs=gcoord[g0:g1])

    conv = model.conv
    with torch.no_grad():
        xl = conv.lin_l(x).contiguous()
    xl.requires_grad_(True)
    gout = torch.randn(n, 512, device="cuda")

    def gat_only(view, g0, g1):
        out = layers._GatAttendRows.apply(xl, conv.att_l, conv.att_r, conv.bias, view, 2, 256, 0.2)
        torch.autograd.grad(out, [xl, conv.att_l, conv.att_r, conv.bias], gout[g0:g1])

    full = graph.row_block(0, n)
    entry = {"n": n, "edges": graph.nnz, "replicated": {"gnn_fwd_bwd_ms": timed(lambda: fwd_bwd(graph, 0, n), reps),
                                                         "gat_fwd_bwd_ms": timed(lambda: gat_only(full, 0, n), reps)}}
    entry["per_rank_emulated"] = {}
    for G in worlds:
        blocks = sharding.gnn_blocks(graph.rowptr, G)
        t_all, t_gat = [], []
        for g0, g1 in blocks:
            view = graph.row_block(g0, g1)
            t_all.append(timed(lambda: fwd_bwd(view, g0, g1), reps))
            t_gat.append(timed(lambda: gat_only(view, g0, g1), reps))
        entry["per_rank_emulated"][str(G)] = {"blocks": blocks, "gnn_fwd_bwd_ms": [round(t, 4) for t in t_all], "gat_fwd_bwd_ms": [round(t, 4) for t in t_gat],
                                              "slowest_gnn_fwd_bwd_ms": round(max(t_all), 4), "slowest_gat_fwd_bwd_ms": round(max(t_gat), 4)}
        print(name, G, entry["per_rank_emulated"][str(G)]["slowest_gnn_fwd_bwd_ms"], flush=True)
    return entry


def distributed(name, steps, rounds):
    import torch.distributed as dist

    from hic_gnn_b200 import models, ops, sharding, train

    rank, world = dist.get_rank(), dist.get_world_size()
    w, n, adj, graph, x = setup(name, "cuda")
    r0, r1 = sharding.row_block(n, rank, world, "upper" if ops._USE_UPPER else "rows")
    tgt = ops.cont2dist(adj[r0:r1], w["factor"], want_f64=False, want_f32=True, r0=r0, r1=r1, max_reduce=sharding.allreduce_max_, symmetric=True)[1]
    del adj
    torch.cuda.empty_cache()
    runs = {}
    for kind in ("replicated", "sharded"):
        torch.manual_seed(0)
        model = models.GATNetSelectiveResidualsUpdated().cuda()
        shard = sharding.GnnRowShard.for_rank(graph, model.parameters(), "cuda", transport="p2p") if kind == "sharded" else None
        red = ops.sharded_reducer(tgt, w["mode"] if w["mode"] != "mse_pearson" else "mse_moments", transport="p2p")
        runs[kind] = train.TrainStep(model, x, graph, tgt, mode=w["mode"], use_cuda_graph=True, reducer=red, gnn_shard=shard)
    res = {k: [] for k in runs}
    for _ in range(rounds):
        for kind, step in runs.items():
            for _ in range(3):
                step()
            torch.cuda.synchronize()
            dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step()
            e1.record()
            e1.synchronize()
            t = torch.tensor([e0.elapsed_time(e1) / steps], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            res[kind].append(round(1000.0 / float(t), 2))
    blocks = sharding.gnn_blocks(graph.rowptr, world)
    return {"n": n, "world": world, "gnn_blocks": blocks, "steps_per_s": res, "median_steps_per_s": {k: sorted(v)[len(v) // 2] for k, v in res.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c5,c4")
    ap.add_argument("--worlds", default="2,4,8", help="emulated rank counts (one GPU)")
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        import torch.distributed as dist

        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    out = {"card": card(), "mode": "torchrun" if world > 1 else "one-GPU emulation", "workloads": {}}
    for name in args.workloads.split(","):
        if world > 1:
            out["workloads"][name] = distributed(name, args.steps, args.rounds)
        else:
            out["workloads"][name] = emulate(name, [int(g) for g in args.worlds.split(",")], args.reps)
    if world > 1:
        import torch.distributed as dist

        rank = dist.get_rank()
        dist.destroy_process_group()
        if rank != 0:
            return
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
