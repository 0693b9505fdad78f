#!/usr/bin/env python
"""Per-step dSCC on one GPU: ``metrics.DsccMeter`` (``hicgat_dscc_*``) against ``metrics.dscc_streamed`` (``hicgat_rank_*``), and the
cost of ``TrainStep(track_dscc=True)`` in graphed GAT training.

    python scripts/bench_dscc.py [--sizes 2493:0.95,9970:0.07,49850:0.01] [--out profiles/r5_dscc.json]

Per size (bench.py's c3 / c4 / c5 synthetic maps), dense WishTarget and implicit SparseWishTarget of the same map:
  * per-call time, alternating the two paths after a warm-up: ``dscc_streamed`` by the host clock around the call and a device
    synchronise (it reads values back), the meter by CUDA events over ``--calls`` back-to-back calls; results of both are recorded;
  * kernel times of one call of each path from torch.profiler (run after the timed section), with pair counts and bytes computed from
    the shapes: every pass visits P = n (n - 1) / 2 pairs; the dense cross pass streams 4 P bytes of target;
  * the same kernels on a collapsed structure (90 % of the loci at one point: 81 % of the pairs in distance bin 0), where per-pair
    atomics (``dist_hist_kernel``) serialise on one address and ``dscc_hist_kernel`` adds once per warp whose pairs share a bin;
  * graphed GAT training (GATNetSelectiveResidualsUpdated, mse_pearson, dense target) with and without track_dscc, alternating,
    steps/s by CUDA events (``--train-sizes``).
The GPU name, power limit and maximum SM clock are read in the same run.  Needs a GPU; there is no CPU path.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch

from hic_gnn_b200 import metrics, models, ops, synth, train
from hic_gnn_b200.graph import CSRGraph


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": out.stdout.strip().splitlines()[0] if out.returncode == 0 else None}


def helix(n, seed=5):
    g = torch.Generator().manual_seed(seed)
    t = torch.linspace(0, 6.0, n)
    c = torch.stack([torch.cos(t) * (1 + 0.1 * t), torch.sin(t) * (1 + 0.1 * t), 0.2 * t], dim=1)
    return (c + 0.05 * torch.randn(n, 3, generator=g)).float().cuda()


def collapsed(n, seed=6):
    g = torch.Generator().manual_seed(seed)
    c = torch.zeros(n, 3)
    k = n // 10
    c[:k] = torch.randn(k, 3, generator=g)
    return c.cuda()


def time_streamed(coords, tgt):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    v = metrics.dscc_streamed(coords, tgt)
    torch.cuda.synchronize()
    return time.perf_counter() - t0, v


def time_meter(meter, coords, calls):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(calls):
        r = meter(coords)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3 / calls, float(r)


def kernel_times(fn):
    """{kernel name: (total µs, launches)} of one call of ``fn`` (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile

    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if e.device_type.name == "CUDA" and getattr(e, "device_time_total", 0) > 0:
            m = re.search(r"(\w+_kernel\w*(?:<[^>(]*>)?)", e.key)
            name = m.group(1) if m else e.key[:60]
            slot = out.setdefault(name, {"us": 0.0, "calls": 0})
            slot["us"] = round(slot["us"] + e.device_time_total, 1)
            slot["calls"] += e.count
    return out


def bench_size(n, density, rounds, calls):
    adj = synth.synthetic_map_chunked(n, density, device="cuda")
    _, dense = ops.cont2dist(adj, 1.0, want_f64=False, want_f32=True, symmetric=True)
    rowptr, col, val = ops.csr_from_dense(adj)
    sparse = ops.SparseWishTarget.from_graph(CSRGraph(rowptr, col, val, n), adj, 1.0)
    del adj
    torch.cuda.empty_cache()
    pairs = n * (n - 1) // 2
    stored_upper = int(sparse.col.numel()) // 2
    res = {"n": n, "density": density, "pairs": pairs, "stored_pairs_upper": stored_upper, "nbins": metrics.NBINS}
    coords = helix(n)
    for kind, tgt in (("dense", dense), ("implicit", sparse)):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        meter = metrics.DsccMeter(tgt)
        torch.cuda.synchronize()
        setup = time.perf_counter() - t0
        time_streamed(coords, tgt)
        time_meter(meter, coords, 2)
        old, new = [], []
        for _ in range(rounds):
            t, v_old = time_streamed(coords, tgt)
            old.append(t)
            t, v_new = time_meter(meter, coords, calls)
            new.append(t)
        k_new = kernel_times(lambda: meter(coords))
        k_old = kernel_times(lambda: metrics.dscc_streamed(coords, tgt))
        med_old, med_new = sorted(old)[len(old) // 2], sorted(new)[len(new) // 2]
        entry = {"meter_setup_s": round(setup, 4), "streamed_ms": [round(x * 1e3, 3) for x in old], "meter_ms": [round(x * 1e3, 4) for x in new],
                 "streamed_ms_median": round(med_old * 1e3, 3), "meter_ms_median": round(med_new * 1e3, 4), "speedup": round(med_old / med_new, 1),
                 "rho_streamed": v_old, "rho_meter": v_new, "abs_diff": abs(v_old - v_new),
                 "meter_kernels": k_new, "streamed_kernels": k_old}
        hist_us = sum(v["us"] for k, v in k_new.items() if "dscc_hist_kernel" in k)
        entry["meter_dist_hist_pairs_per_s"] = pairs / (hist_us * 1e-6) if hist_us else None
        cross_us = sum(v["us"] for k, v in k_new.items() if "dscc_cross" in k)
        if kind == "dense":
            entry["meter_cross_target_bytes"] = 4 * pairs
            entry["meter_cross_target_TB_per_s"] = 4 * pairs / (cross_us * 1e-6) / 1e12 if cross_us else None
        entry["meter_cross_pairs_per_s"] = (pairs if kind == "dense" else stored_upper) / (cross_us * 1e-6) if cross_us else None
        if kind == "implicit":
            # atomic scheme on a collapsed structure: per-pair atomics (dscc_streamed's dist_hist_kernel) vs the warp-uniform fast path
            cc = collapsed(n)
            entry["collapsed"] = {"meter_kernels": kernel_times(lambda: meter(cc)), "streamed_kernels": kernel_times(lambda: metrics.dscc_streamed(cc, tgt)),
                                  "rho_meter": float(meter(cc)), "rho_streamed": metrics.dscc_streamed(cc, tgt)}
        res[kind] = entry
        print(json.dumps({"n": n, kind: {k: entry[k] for k in ("streamed_ms_median", "meter_ms_median", "speedup", "abs_diff")}}), flush=True)
        del meter
        torch.cuda.empty_cache()
    return res


def bench_train(n, density, steps, rounds):
    adj = synth.synthetic_map_chunked(n, density, device="cuda")
    _, target = ops.cont2dist(adj, 1.0, want_f64=False, want_f32=True, symmetric=True)
    rowptr, col, val = ops.csr_from_dense(adj)
    graph = CSRGraph(rowptr, col, val, n)
    del adj
    x = synth.synthetic_features(n, device="cuda")
    runs = {}
    for track in (False, True):
        torch.manual_seed(42)
        model = models.GATNetSelectiveResidualsUpdated().cuda()
        runs[track] = train.TrainStep(model, x, graph, target, mode="mse_pearson", lr=1e-3, use_cuda_graph=True, track_dscc=track)
    times = {False: [], True: []}
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for st in runs.values():
        for _ in range(3):
            st()
    for _ in range(rounds):
        for track, st in runs.items():
            a.record()
            for _ in range(steps):
                st()
            b.record()
            torch.cuda.synchronize()
            times[track].append(a.elapsed_time(b) / steps)
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    out = {"n": n, "steps_per_round": steps, "ms_per_step": {"plain": [round(t, 4) for t in times[False]], "track_dscc": [round(t, 4) for t in times[True]]},
           "steps_per_s_plain": round(1e3 / med[False], 1), "steps_per_s_track_dscc": round(1e3 / med[True], 1),
           "tracking_ms_per_step": round(med[True] - med[False], 4), "tracking_over_step": round((med[True] - med[False]) / med[False], 3),
           "last_dscc": float(runs[True].dscc)}
    print(json.dumps(out), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="2493:0.95,9970:0.07,49850:0.01")
    ap.add_argument("--train-sizes", default="9970:0.07,49850:0.01")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--out", default="profiles/r5_dscc.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_dscc needs a GPU")
    res = {"gpu": gpu_info(), "sizes": [], "train": []}
    for spec in args.sizes.split(","):
        if spec:
            n, d = spec.split(":")
            res["sizes"].append(bench_size(int(n), float(d), args.rounds, args.calls))
            torch.cuda.empty_cache()
    for spec in args.train_sizes.split(","):
        if spec:
            n, d = spec.split(":")
            res["train"].append(bench_train(int(n), float(d), 20 if int(n) < 20000 else 10, args.rounds))
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
