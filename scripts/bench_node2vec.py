#!/usr/bin/env python
"""node2vec on one GPU at the reference's parameters (Node2Vec(dimensions=512, walk_length=150, num_walks=50, p=1.75, q=0.4),
gensim's fit defaults: window 5, negative 5, sample 1e-3).

    python scripts/bench_node2vec.py [--sizes 9970:5,49850:1] [--out profiles/r4_node2vec.json]

Per size (C4 = 9 970 loci at 7 % density, C5 = 49 850 loci at 1 %: the synthetic maps of bench.py through load_input), with
``size:epochs`` skip-gram epochs:
  * walks: CUDA-event time of ``hicgat_node2vec_walks`` over all num_walks * n starts, transitions/s, and the expected
    number of proposals per second-order step, max(1/p, 1, 1/q) / E[alpha], evaluated exactly on a sample of 4 096 of the
    walks' steps (the kernel does not count its attempts);
  * skip-gram: CUDA-event time of each Hogwild ``hicgat_sgns_epoch``, raw tokens/s, and (centre, context) pairs/s against the
    expected pair count (expected kept tokens from gensim's keep probabilities x the mean context count 2 (window - E[b]),
    walk-edge effects ignored); FLOP/s (2 x 3 x dim per target, 1 + negative targets per pair) and the bytes/s the pair
    loop moves at L2 (each of the 1 + 1 + negative rows read once and added once, 4 B per element) over the HBM peak.
The GPU name and power limit are read in the same run.  Needs a GPU; there is no CPU path, and no CPU baseline is run
(gensim and node2vec are not installed).
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np
import torch

from hic_gnn_b200 import node2vec as n2v
from hic_gnn_b200 import synth, utils

DENSITY = {2493: 0.95, 9970: 0.07, 49850: 0.01}  # bench.py's c3 / c4 / c5


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": out.stdout.strip().splitlines()[0] if out.returncode == 0 else None}


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    r = fn()
    b.record()
    torch.cuda.synchronize()
    return r, a.elapsed_time(b) / 1e3


def expected_proposals(g, walks, p, q, samples=4096, seed=0):
    """Mean over sampled second-order steps (t -> v) of max(1/p, 1, 1/q) / sum_x w(v,x) alpha(t,x) / sum_x w(v,x)."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    rows = torch.randint(0, walks.shape[0], (samples,), generator=gen, device="cuda")
    cols = torch.randint(1, walks.shape[1] - 1, (samples,), generator=gen, device="cuda")
    t, v = walks[rows, cols - 1].long(), walks[rows, cols].long()
    ok = (t >= 0) & (v >= 0)
    t, v = t[ok], v[ok]
    deg = g.rowptr[v + 1] - g.rowptr[v]
    ctx = torch.repeat_interleave(torch.arange(t.numel(), device="cuda"), deg)
    first = torch.repeat_interleave(g.rowptr[v], deg)
    entry = first + torch.arange(ctx.numel(), device="cuda") - torch.repeat_interleave(torch.cumsum(deg, 0) - deg, deg)
    x, w = g.col[entry], g.value[entry].double()
    keys = g.storage.row() * g.n + g.col                       # CSR order is row-major: globally sorted
    probe = t[ctx] * g.n + x
    pos = torch.searchsorted(keys, probe).clamp(max=keys.numel() - 1)
    alpha = torch.where(x == t[ctx], 1.0 / p, torch.where(keys[pos] == probe, 1.0, 1.0 / q))
    num = torch.zeros(t.numel(), dtype=torch.float64, device="cuda").index_add_(0, ctx, w * alpha)
    den = torch.zeros(t.numel(), dtype=torch.float64, device="cuda").index_add_(0, ctx, w)
    return float((max(1.0 / p, 1.0, 1.0 / q) / (num / den)).mean())


def run_size(n, epochs, args, hbm_peak):
    adj = synth.synthetic_map_chunked(n, DENSITY[n], device="cuda")
    g = utils.load_input(adj, torch.zeros(n, 1)).edge_index
    del adj
    torch.cuda.empty_cache()
    res = {"n": n, "density": DENSITY[n], "nnz": g.nnz, "mean_degree": g.nnz / n}
    m = n2v.Node2Vec(g, dimensions=args.dim, walk_length=2, num_walks=1, p=args.p, q=args.q, seed=1)  # warm-up: module load, CDF
    gen = torch.Generator(device="cuda").manual_seed(42)
    starts = torch.cat([torch.randperm(n, generator=gen, device="cuda") for _ in range(args.num_walks)])
    walks, t_walk = timed(lambda: n2v.random_walks(g, starts, args.walk_length, args.p, args.q, 42))
    transitions = int((walks[:, 1:] >= 0).sum())
    res["walks"] = {"seconds": t_walk, "walks": walks.shape[0], "transitions": transitions, "transitions_per_s": transitions / t_walk,
                    "expected_proposals_per_step": expected_proposals(g, walks, args.p, args.q)}
    sg = n2v.SkipGram(walks, n, args.dim, window=5, negative=5, sample=1e-3, epochs=epochs, seed=1)
    counts = sg.counts.astype(np.float64)
    kept = float((counts * np.minimum(n2v.keep_thresholds(counts, 1e-3).astype(np.float64) / (2**32 - 1), 1.0)).sum())
    pairs = kept * 2 * (5 - 2.0)                                # E[b] = 2 for b uniform in [0, 5)
    flop = pairs * 6 * 3 * args.dim * 2
    bytes_ = pairs * (1 + 6) * 2 * args.dim * 4
    per_epoch = []
    for e in range(epochs):
        _, t = timed(lambda: sg.epoch(e))
        per_epoch.append(t)
    t_ep = float(np.median(per_epoch))
    assert bool(torch.isfinite(sg.syn0).all())
    res["skipgram"] = {"epochs_run": epochs, "epoch_seconds": per_epoch, "median_epoch_seconds": t_ep, "tokens": sg.total_tokens,
                       "tokens_per_s": sg.total_tokens / t_ep, "expected_kept_tokens": kept, "expected_pairs": pairs,
                       "pairs_per_s": pairs / t_ep, "flop_per_epoch": flop, "tflop_per_s": flop / t_ep / 1e12,
                       "l2_bytes_per_epoch": bytes_, "l2_tb_per_s": bytes_ / t_ep / 1e12,
                       "l2_bytes_over_hbm_peak": bytes_ / t_ep / hbm_peak,
                       "syn_bytes": 2 * n * args.dim * 4}
    print(json.dumps(res), flush=True)
    del m, walks, sg, g
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="9970:5,49850:1", help="n:epochs,...")
    ap.add_argument("--dim", type=int, default=512)
    ap.add_argument("--walk-length", type=int, default=150)
    ap.add_argument("--num-walks", type=int, default=50)
    ap.add_argument("--p", type=float, default=1.75)
    ap.add_argument("--q", type=float, default=0.4)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_node2vec.py needs a GPU")
    hbm_peak = 7.7e12
    out = {"gpu": gpu_info(), "params": {"dim": args.dim, "walk_length": args.walk_length, "num_walks": args.num_walks, "p": args.p, "q": args.q,
                                         "window": 5, "negative": 5, "sample": 1e-3}, "hbm_peak_datasheet_bytes_per_s": hbm_peak, "sizes": []}
    for item in args.sizes.split(","):
        n, e = (int(x) for x in item.split(":"))
        out["sizes"].append(run_size(n, e, args, hbm_peak))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(out["gpu"]))


if __name__ == "__main__":
    main()
