#!/usr/bin/env python
"""Cost of the differentiable Pearson loss (two passes) against the one-pass MSE + moments step, on one GPU.

    python scripts/bench_pearson_grad.py [--sizes 9970,49850] [--iters 50] [--train-steps 20] [--out profiles/r3_pearson_grad.json]

Per size (C4 = 9 970 loci, C5 = 49 850 loci, synthetic maps of bench.py), for the dense target streamed as its upper
triangle and for the implicit (sparse) target: CUDA-event times of pass 1 (moments), pass 2 (gradient), the whole
``pairwise_loss(..., "mse_pearson_grad")`` step and the one-pass ``mse_moments`` step; pair rates; and the algorithmic
HBM traffic of the dense two-pass step (2 passes x 4 B per ordered pair) over the HBM bandwidth measured in the same run
by a device-to-device copy.  Then GAT-net training steps/s for ``mse_pearson`` vs ``mse_pearson_grad``.  The GPU name
and power limit are recorded beside the numbers.  Needs a GPU; there is no CPU path.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch

from hic_gnn_b200 import _native as N
from hic_gnn_b200 import models, ops, synth, train, utils


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": out.stdout.strip().splitlines()[0] if out.returncode == 0 else None}


def time_ms(fn, iters, warm=5):
    for _ in range(warm):
        fn()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    t = sorted(a.elapsed_time(b) for a, b in ev)
    return {"mean_ms": sum(t) / len(t), "median_ms": t[len(t) // 2], "min_ms": t[0]}


def hbm_copy_gbs(nbytes=8 << 30, iters=20):
    src = torch.empty(nbytes // 4, dtype=torch.float32, device="cuda")
    dst = torch.empty_like(src)
    r = time_ms(lambda: dst.copy_(src), iters)
    del src, dst
    torch.cuda.empty_cache()
    return 2 * nbytes / (r["median_ms"] * 1e-3) / 1e9  # read + write


def loss_legs(n, target, coords, iters, hbm):
    c_mse = 4.0 / (float(n) * n)
    moments = {}

    def pass1():
        m, _ = ops.pairloss_raw(coords, target, N.PAIR_MOMENTS_D, 0.0, 0.0)
        moments["m"] = m + target.t_moments()

    pass1()
    grad = torch.empty(n, 3, dtype=torch.float32, device="cuda")
    c = coords.clone().requires_grad_(True)

    def step():
        loss, _ = ops.pairwise_loss(c, target, "mse_pearson_grad")
        loss.backward()

    legs = {
        "pass1_moments": time_ms(pass1, iters),
        "pass2_gradient": time_ms(lambda: ops.pearson_grad_raw(coords, target, moments["m"], True, grad=grad), iters),
        "mse_pearson_grad_step": time_ms(step, iters),
        "mse_moments_one_pass": time_ms(lambda: ops.pairloss_raw(coords, target, ops._MODES["mse_moments"], c_mse, 0.0), iters),
    }
    pairs = float(n) * float(n)
    for v in legs.values():
        v["gpairs_per_s"] = pairs / (v["median_ms"] * 1e-3) / 1e9
    if isinstance(target, ops.WishTarget):
        byt = 2 * 4 * pairs  # two passes x 4 B per ordered pair
        legs["mse_pearson_grad_step"]["algorithmic_bytes"] = byt
        legs["mse_pearson_grad_step"]["share_of_measured_hbm"] = byt / (legs["mse_pearson_grad_step"]["median_ms"] * 1e-3) / (hbm * 1e9)
    legs["pass2_over_mse_moments"] = legs["pass2_gradient"]["median_ms"] / legs["mse_moments_one_pass"]["median_ms"]
    legs["step_over_mse_moments"] = legs["mse_pearson_grad_step"]["median_ms"] / legs["mse_moments_one_pass"]["median_ms"]
    return legs


def train_rates(gdata, target, steps):
    out = {}
    torch.manual_seed(42)
    init = models.GATNetSelectiveResidualsUpdated().state_dict()
    for mode in ("mse_pearson", "mse_pearson_grad"):
        gm = models.GATNetSelectiveResidualsUpdated().cuda()
        gm.load_state_dict(init)
        st = train.TrainStep(gm, gdata.x.float(), gdata.edge_index, target, mode=mode, lr=1e-3, use_cuda_graph=True)
        r = time_ms(lambda: st(), steps, warm=3)
        out[mode] = {"steps_per_s": 1e3 / r["median_ms"], **r}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="9970,49850")
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--train-steps", type=int, default=20)
    ap.add_argument("--out", default="profiles/r3_pearson_grad.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_pearson_grad.py needs a GPU")
    torch.cuda.set_device(0)
    res = {"gpu": gpu_info(), "hbm_copy_gbs": hbm_copy_gbs(), "upper_triangle": ops._USE_UPPER, "sizes": {},
           "sharded_8gpu_c5": "not measured (one GPU)"}
    for n in [int(s) for s in args.sizes.split(",")]:
        adj = synth.synthetic_map_chunked(n, 0.01, device="cuda")
        gdata = utils.load_input(adj, synth.synthetic_features(n, device="cuda"))
        del adj
        dense = utils.wish_target(gdata.y, 1.0)
        sparse = utils.sparse_wish_target(gdata, 1.0)
        coords = (0.3 * torch.randn(n, 3, generator=torch.Generator().manual_seed(n))).cuda()
        row = {"dense_upper": loss_legs(n, dense, coords, args.iters, res["hbm_copy_gbs"]),
               "implicit_sparse": loss_legs(n, sparse, coords, args.iters, res["hbm_copy_gbs"])}
        if args.train_steps > 0:
            row["gat_train_dense"] = train_rates(gdata, dense, args.train_steps)
        res["sizes"][str(n)] = row
        print(json.dumps({n: row}), flush=True)
        del gdata, dense, sparse
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
