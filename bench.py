#!/usr/bin/env python
"""Benchmark of the HiC-GNN / GAT-HiC training hot path on B200 (BASELINE.json metric:
"train steps/s & pairwise-loss Gpairs/s vs N loci, % HBM roofline, 1/2/4/8 B200").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c5|c4|c3|c2|c1] [--impl reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

One JSON line on rank 0.  What is measured (definitions in DESIGN.md, "Measurement"):

* ``value`` -- pairwise-loss throughput of the PRIMARY workload (default c5 = BASELINE.json configs[4]) in
  Gpairs/s, pairs = ORDERED pairs = N^2 per fused forward+backward loss evaluation (SURVEY.md 8d).  One step =
  the fused sm_100a kernel over this rank's row block of the resident f32 wish-distance matrix + ONE exchange of
  the partials over NVLink.  Strong scaling: N^2 is fixed, the rows are sharded over the ranks.
* ``roofline`` -- the fused kernel alone: N_local*N*4 B per launch / CUDA-event duration of the launches inside
  the timed region, against the measured HBM copy bandwidth.
* ``e2e`` -- the same evaluation through the C ABI from HOST buffers: coordinates and this rank's target rows are
  copied from pinned host memory every step (double-buffered against the kernel), the result is read back.
* ``train`` -- the whole fused training step (GNN forward, fused loss, backward, Adam; GNN replicated, loss
  row-sharded) in steps/s, with ``train.cpu_baseline`` = the reference's CPU training loop (oracle restatement of
  HiC-GNN_main.py:123-132 / HiC_GAT_generalize_directly.py:202-243) timed on this box's host cores in the same run.
* ``cpu_baseline`` -- the reference formulation of the loss (torch.cdist + MSELoss + autograd) on a bounded row
  sample of the same workload, all host cores ("port").
* ``configs`` -- the other BASELINE.json configurations in the same run: c1 (chr19 1 Mb, Net), c2 (chr19 1 Mb ->
  500 kb, GAT net), c3 (2 493 loci), c4 (9 970 loci) at 1 GPU; c4 row-sharded at N > 1.  Each entry: loss Gpairs/s,
  kernel time / HBM fraction, train steps/s and the CPU training-loop baseline beside it.

``--impl reference`` runs only the CPU formulation of the loss (rank 0, no GPU, no native library), K timed steps.

``--dump-outputs DIR`` writes, after the timed steps, what the last timed step returned as ``DIR/<name>.npy`` (f32 / f64
as computed): ``loss_moments`` and ``loss_grad`` of the loss step, and ``train_total`` / ``train_moments`` of the last
training step when that leg runs (reference arm: ``loss`` and ``loss_grad``).  The inputs are pure functions of fixed
seeds, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[0..4]; chr1 = 249 Mb for the synthetic maps
    "c1": dict(kind="fixture", tag="1mb", n=58, density=1.0, model="net", mode="mse", factor=0.5,
               desc="GM12878 chr19 1 Mb (58 loci, Data/GM12878_1mb_chr19_list.txt) HiC-GNN_main.py: Net (SAGEConv) + MSE, conversion 0.5"),
    "c2": dict(kind="fixture", tag="1mb", gen_tag="500kb", n=58, density=1.0, model="gat", mode="mse_pearson", factor=1.0,
               desc="GM12878 chr19 1 Mb (58 loci) -> 500 kb (114 loci) GAT generalisation (HiC_GAT_generalize_directly.py)"),
    "c3": dict(kind="synthetic", n=2493, density=0.95, model="gat", mode="mse_pearson", factor=1.0,
               desc="synthetic chr1 100 kb (2493 loci, near-dense) GAT + combined MSE/Pearson loss"),
    "c4": dict(kind="synthetic", n=9970, density=0.07, model="gat", mode="mse_pearson", factor=1.0,
               desc="synthetic chr1 25 kb (9970 loci, ~1e8 pairs) sparse CSR GAT"),
    "c5": dict(kind="synthetic", n=49850, density=0.01, model="gat", mode="mse_pearson", factor=1.0,
               desc="synthetic chr1 5 kb (49850 loci, ~2.5e9 pairs) row-sharded pairwise loss"),
}
METRIC = "pairwise_loss_gpairs_per_s"
UNIT = "Gpairs/s"
MODEL_CLASSES = {"gat": "GATNetSelectiveResidualsUpdated", "net": "Net", "gat_v2": "GATNetHeadsChanged3LayersLeakyReLUv2"}


def workload_config(name: str, loss_mode: str) -> dict:
    """The workload-defining part of the JSON line: identical in the native and the reference arm."""
    w = WORKLOADS[name]
    n = w["n"]
    return {"workload": w["desc"], "name": name, "n_loci": n, "density": w["density"], "pairs_per_step": float(n) * float(n), "loss_mode": loss_mode,
            "target": "dense f32 wish-distance matrix, 4 B per ordered pair"}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=["native", "reference", "cpu-train"],
                    help="cpu-train: internal -- the CPU training-loop baseline of --workload in a child process (an out-of-memory kill must not take the bench down)")
    ap.add_argument("--workload", default="c5", choices=sorted(WORKLOADS))
    ap.add_argument("--configs", default="auto", help="other workloads reported in the `configs` block: auto (c1-c4 at 1 GPU, c4 at N>1 when the primary is c5), none, or a comma list")
    ap.add_argument("--loss-mode", default="mse", choices=["mse", "mse_moments", "mse_moments_full", "contrastive"])
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = min(steps, 10)")
    ap.add_argument("--train-steps", type=int, default=0, help="0 = min(steps, 10) for the primary workload")
    ap.add_argument("--variant", type=int, default=0, help="pair-loss kernel: 0 = TMA tile ring (default), 1 = per-lane streaming loads")
    ap.add_argument("--rows-per-cta", type=int, default=0, help="pair-loss row-chunk override (0 = library default)")
    ap.add_argument("--transport", default="auto", choices=["auto", "p2p", "p2p_oneshot", "nccl"], help="exchange of the sharded loss partials")
    ap.add_argument("--emulate-world", type=int, default=0, help="profiling aid: on ONE GPU run one rank's row block of a W-way split (not a bench line)")
    ap.add_argument("--emulate-rank", type=int, default=0, help="which rank's block --emulate-world runs")
    ap.add_argument("--no-rebalance", action="store_true", help="multi-GPU: keep the area-balanced row blocks (skip the measured rebalancing at setup)")
    ap.add_argument("--no-measure-copy", dest="measure_copy", action="store_false", help="skip the same-process copy-bandwidth control")
    ap.add_argument("--no-cuda-graph", action="store_true", help="run the training step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--no-sparse", action="store_true", help="skip the implicit-target (row f-4) leg")
    ap.add_argument("--model", default="", choices=["", "gat", "net", "gat_v2"], help="network of the training-step leg (default: the workload's own)")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-sample-pairs", type=float, default=1e8, help="ordered pairs per CPU-baseline loss step")
    ap.add_argument("--cpu-train-budget", type=float, default=1.0, help="scale of the CPU training-loop baseline's work (1 = default samples)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def dump_outputs(path: str, arrays: dict) -> None:
    """``DIR/<name>.npy`` for every (host) array, in the f32 / f64 it was computed in."""
    import numpy as np

    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(path, f"{name}.npy"), a)


# ------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Polls SM clock + clock-event reasons of one GPU through NVML on a thread; samples carry
    a wall-clock stamp so the timed regions can be cut out afterwards."""

    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, torch_index: int, period_s: float = 0.02):
        self.samples = []  # (t, sm_mhz, reasons_mask)
        self.period = period_s
        self.sm_max = None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            import torch

            pynvml.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(torch_index).uuid)
            if not uuid.startswith("GPU-"):
                uuid = "GPU-" + uuid
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(torch_index)
            self.nv = pynvml
            self.sm_max = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # no NVML: report that instead of inventing clocks
            self.nv = None
            self.err = repr(e)

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                clk = int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.samples.append((time.time(), clk, mask))
            except Exception:
                pass
            self._stop.wait(self.period)

    def start(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join(timeout=2)

    def summary(self, windows):
        """windows: {name: (t0, t1)} wall-clock; primary window first."""
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "error": getattr(self, "err", "nvml unavailable")}
        import statistics

        def cut(t0, t1):
            return [s for s in self.samples if t0 <= s[0] <= t1]

        names = list(windows)
        prim = cut(*windows[names[0]])
        allw = [s for n in names for s in cut(*windows[n])]
        use, scope = (prim, names[0]) if len(prim) >= 3 else (allw, "+".join(names))
        mask = 0
        for s in allw:
            mask |= s[2]
        out = {
            "sm_mhz": statistics.median([s[1] for s in use]) if use else None,
            "sm_max_mhz": self.sm_max,
            "reasons": sorted(v for k, v in self.REASONS.items() if mask & k),
            "samples": len(use),
            "window": scope,
        }
        for n in names[1:]:
            w = cut(*windows[n])
            if w:
                out[f"sm_mhz_{n}"] = statistics.median([s[1] for s in w])
        return out


# ------------------------------------------------------------------------------ CPU formulation of the loss
def cpu_sample_step(coords, truth_rows, sample_rows):
    """One reference-formulation loss evaluation on rows [0, sample_rows): torch.cdist ->
    MSELoss(out.float(), truth.float()) -> backward (HiC-GNN_main.py:126-129)."""
    from oracle import loss as oloss

    coords.grad = None
    l = oloss.mse_loss_rows(coords, truth_rows, 0, sample_rows)
    l.backward()
    return float(l.detach())


def time_cpu_sample(n, truth_rows_f64, sample_rows, warmup, steps, outputs=None):
    """``outputs``: a dict that receives the loss and the coordinate gradient of the last timed step."""
    import torch

    torch.set_num_threads(os.cpu_count() or 1)
    g = torch.Generator().manual_seed(7)
    coords = (0.3 * torch.randn(n, 3, generator=g)).requires_grad_(True)
    truth = truth_rows_f64[:sample_rows].contiguous()
    for _ in range(warmup):
        cpu_sample_step(coords, truth, sample_rows)
    t0 = time.perf_counter()
    for _ in range(steps):
        loss = cpu_sample_step(coords, truth, sample_rows)
    dt = time.perf_counter() - t0
    if outputs is not None:
        outputs.update(loss=torch.tensor([loss], dtype=torch.float64), loss_grad=coords.grad.clone())
    return sample_rows * n * steps / dt / 1e9, dt / steps, torch.get_num_threads()


def fixture_arrays():
    import numpy as np

    return np.load(os.path.join(ROOT, "tests", "golden", "reference_golden.npz"))


def cpu_truth_rows(name: str, sample_rows: int):
    """f64 wish-distance rows [0, sample_rows) as the reference holds them (``truth`` is f64 and cast per
    iteration), generated on the CPU: the reference arm never touches the GPU or the native library.  Synthetic
    maps: from the unbalanced counts (the balancing changes values, not the timing of cdist + MSELoss)."""
    import torch

    w = WORKLOADS[name]
    n = w["n"]
    if w["kind"] == "fixture":
        from oracle import wish as owish

        adj = torch.tensor(fixture_arrays()[f"{w['tag']}_kr_oracle"], dtype=torch.float64)
        return owish.cont2dist(adj, w["factor"])[:sample_rows].contiguous()
    from hic_gnn_b200 import synth  # pure torch, no native code

    raw = synth.raw_block(n, 0, sample_rows, synth.solve_c0(n, w["density"]), 1234 + n)
    d = 1.0 / raw
    d[torch.arange(sample_rows), torch.arange(sample_rows)] = 0
    mx = d[torch.isfinite(d)].max()
    return torch.nan_to_num(d, posinf=float(mx)) / mx


def sample_rows_for(n: int, pairs: float) -> int:
    return max(min(8, n), min(n, int(pairs // n)))


# ------------------------------------------------------------------------------ reference arm
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = WORKLOADS[args.workload]
    n = w["n"]
    sample_rows = sample_rows_for(n, args.cpu_sample_pairs)
    truth = cpu_truth_rows(args.workload, sample_rows)
    outputs = {}
    gps, sec_per_step, threads = time_cpu_sample(n, truth, sample_rows, max(args.warmup, 1), args.steps, outputs)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    sample = f"oracle torch.cdist+MSELoss+autograd on rows [0,{sample_rows}) x {n} cols ({sample_rows * n:.3g} ordered pairs) per step"
    line = {
        "impl": "reference", "metric": METRIC, "value": gps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": max(args.warmup, 1), "ms_per_step": sec_per_step * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic" if w["kind"] == "synthetic" else "reference fixture (chr19)",
        "config": workload_config(args.workload, "mse"),
        "run": {"sample": f"rows [0,{sample_rows}) x {n} columns per step", "host_threads": threads},
        "cpu_baseline": {"value": gps, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": gps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------ CPU training-loop baseline
def _time_call(fn, repeat=1):
    best = float("inf")
    for _ in range(repeat):
        t0 = time.perf_counter()
        fn()
        best = min(best, time.perf_counter() - t0)
    return best


def cpu_train_full(model_name, adj_np, x_np, factor, mode, steps, warm, with_as_written=True):
    """The reference's training loop on the CPU (oracle/loop.py restates HiC-GNN_main.py:117-132 and
    HiC_GAT_generalize_directly.py:186-243 op for op): ``as_written`` replays every op of the script body (second
    forward, per-iteration triu_indices gathers, scipy pearsonr / spearmanr), ``kernel_equivalent`` keeps only what
    determines the parameter trajectory (one forward, loss, backward, Adam) -- the work the fused GPU step does."""
    import torch

    from oracle import graph as ograph
    from oracle import loop as oloop
    from oracle import models as omodels
    from oracle import wish as owish

    torch.set_num_threads(os.cpu_count() or 1)
    data = ograph.load_input(adj_np, x_np)
    truth = owish.cont2dist(data.y.clone(), factor)
    out = {}
    variants = [("kernel_equivalent", False)] + ([("as_written", True)] if mode != "mse" and with_as_written else [])
    for key, as_written in variants:
        torch.manual_seed(42)
        model = getattr(omodels, model_name)()
        if warm:
            oloop.train(model, data.x.float(), data.edge_index, truth, mode=mode, thresh=-1.0, max_steps=warm, as_written=as_written)
        t0 = time.perf_counter()
        hist, _ = oloop.train(model, data.x.float(), data.edge_index, truth, mode=mode, thresh=-1.0, max_steps=steps, as_written=as_written)
        dt = (time.perf_counter() - t0) / len(hist)
        out[key] = {"steps_per_s": 1.0 / dt, "s_per_step": dt, "steps": len(hist)}
    if mode == "mse":  # HiC-GNN_main.py's loop body has no per-iteration logging: as written == kernel-equivalent
        out["as_written"] = dict(out["kernel_equivalent"])
    out.setdefault("as_written", None)  # not timed: two live autograd graphs of E x H x C messages do not fit this host
    out.update({"unit": "steps/s", "cores": torch.get_num_threads(), "kind": "port", "extrapolated": False,
                "sample": f"oracle loop ({model_name}, {mode}), full map, {steps} timed steps after {warm} warm-up"})
    return out


def cpu_train_sliced(model_name, csr, x_cpu, truth_rows_f64, sample_rows, n, mode, edge_budget):
    """Same baseline for maps the reference formulation cannot hold in host memory (PyG materialises an
    E x H x C message tensor: 12.8 GB per intermediate at 6 M edges; the N x N f64 truth alone is 20 GB at 50k loci):
    each part of ONE kernel-equivalent step is timed on a slice and scaled by its unit of work --
    the GATConv edge work on the target rows [0, R) (scaled by edges), the projection / set_diag / MLP head on all N rows,
    cdist + MSELoss (+ the Pearson term) + backward on a row sample (scaled by rows)."""
    import numpy as np
    import torch
    from scipy.stats import pearsonr

    from oracle import graph as ograph
    from oracle import models as omodels

    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(42)
    model = getattr(omodels, model_name)()
    conv = model.conv
    x = x_cpu.float()
    parts = {}
    if hasattr(conv, "forward_rows"):  # GATConv
        edges_total = int(csr.rowptr[-1]) + n
        cum = csr.rowptr + torch.arange(n + 1)
        R = int(torch.searchsorted(cum, torch.tensor(int(edge_budget))).clamp(min=1, max=n))
        edges_slice = int(cum[R])
        gsel = torch.randn(R, conv.heads * conv.out_channels)

        def fixed():  # per-step costs that do not depend on the slice: projection fwd+bwd, set_diag (re-done every forward)
            model.zero_grad()
            x_l, a_l, a_r = conv._project(x)
            ograph.set_diag(csr)
            (x_l.sum() + a_l.sum() + a_r.sum()).backward()

        def sliced():
            model.zero_grad()
            (conv.forward_rows(x, csr, R) * gsel).sum().backward()

        t_fixed = _time_call(fixed)
        t_slice = _time_call(sliced)
        t_conv = t_fixed + max(t_slice - t_fixed, 0.0) * edges_total / edges_slice
        parts["conv"] = {"s": t_conv, "fixed_s": t_fixed, "slice_s": t_slice, "rows": R, "edges_slice": edges_slice, "edges_total": edges_total}
    else:  # SAGEConv: cheap enough to run in full
        def sage():
            model.zero_grad()
            conv(x, csr).sum().backward()

        t_conv = _time_call(sage)
        parts["conv"] = {"s": t_conv}
    # MLP head on all N rows (fwd + bwd); get_model minus the conv = feed the head a conv-shaped tensor
    h_in = torch.randn(n, 512)

    class _Id(torch.nn.Module):
        def forward(self, x, *_a, **_k):
            return h_in

    real_conv, model.conv = model.conv, _Id()

    def head():
        model.zero_grad()
        model.get_model(x, csr).sum().backward()

    t_head = _time_call(head)
    model.conv = real_conv
    parts["mlp_head"] = {"s": t_head}
    # loss on a row sample
    g = torch.Generator().manual_seed(7)
    coords = (0.3 * torch.randn(n, 3, generator=g)).requires_grad_(True)
    truth = truth_rows_f64[:sample_rows].contiguous()

    def loss():
        cpu_sample_step(coords, truth, sample_rows)

    loss()
    t_loss = _time_call(loss, 2) * n / sample_rows
    parts["loss"] = {"s": t_loss, "sample_rows": sample_rows}
    t_step = t_conv + t_head + t_loss
    if mode == "mse_pearson":  # the Pearson term of the combined loss: triu gathers + scipy pearsonr (HiC_GAT_generalize_directly.py:210-220)
        def pear():
            d = torch.cdist(coords[:sample_rows].detach(), coords.detach())
            iu = torch.triu_indices(sample_rows, n, 1)
            pearsonr(truth[iu[0], iu[1]].numpy(), d[iu[0], iu[1]].numpy())

        t_p = _time_call(pear) * (n * (n - 1) / 2.0) / (sample_rows * n - sample_rows * (sample_rows + 1) / 2.0)
        parts["pearson"] = {"s": t_p}
        t_step += t_p
    return {"kernel_equivalent": {"steps_per_s": 1.0 / t_step, "s_per_step": t_step}, "as_written": None, "unit": "steps/s",
            "cores": torch.get_num_threads(), "kind": "port", "extrapolated": True, "parts": parts,
            "sample": f"oracle ops of one kernel-equivalent step ({model_name}, {mode}), each part timed on a slice and scaled (conv: edges of {parts['conv'].get('rows', n)} target rows; "
                      f"loss: {sample_rows} rows); as-written (second forward + per-iteration spearmanr over {n * (n - 1) // 2:.3g} pairs) not timed at this size"}


def run_cpu_train_child(args):
    """Child process of the native arm: the as-written / kernel-equivalent oracle loop on a map generated on the CPU."""
    import torch

    from hic_gnn_b200 import synth

    w = WORKLOADS[args.workload]
    n = w["n"]
    adj = fixture_arrays()[f"{w['tag']}_kr_oracle"] if w["kind"] == "fixture" else synth.synthetic_map(n, w["density"]).numpy()
    x = synth.synthetic_features(n).numpy()
    # library warm-up (thread pools, scipy import, allocator) on the 58-locus fixture: the timed loop below runs few steps
    cpu_train_full(MODEL_CLASSES[args.model or w["model"]], fixture_arrays()["1mb_kr_oracle"], synth.synthetic_features(58).numpy(), 1.0, w["mode"], 2, warm=0)
    out = cpu_train_full(MODEL_CLASSES[args.model or w["model"]], adj, x, w["factor"], w["mode"], max(1, args.steps), warm=0)
    print(json.dumps(out), flush=True)


def cpu_train_in_child(name: str, model_key: str, steps: int, timeout_s: float):
    import subprocess

    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "cpu-train", "--workload", name, "--steps", str(steps)] + (["--model", model_key] if model_key else [])
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(k, None)
    try:
        p = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout_s, env=env)
        if p.returncode != 0:
            return {"error": f"child exited with {p.returncode}: {p.stderr[-300:]}"}
        return json.loads(p.stdout.strip().splitlines()[-1])
    except Exception as e:  # timeout, parse error
        return {"error": repr(e)[:300]}


# ------------------------------------------------------------------------------ native arm
def profile_region(name: str, on: bool) -> None:
    """cudaProfilerStart/Stop around one timed region when HICGAT_PROFILE_REGION names it, so that
    `ncu --profile-from-start off` lists exactly the launches of that region (every thread:
    autograd's backward kernels are launched from its own thread, outside any NVTX range)."""
    if os.environ.get("HICGAT_PROFILE_REGION") == name:
        import torch

        torch.cuda.synchronize()
        (torch.cuda.profiler.start if on else torch.cuda.profiler.stop)()


class Env:
    """Process-wide state of the native arm (rank, device, collectives, timers)."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist

        self.torch, self.dist, self.args = torch, dist, args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py (native arm) needs a B200: there is no CPU fallback for the hot path")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.numa = None
        if self.world > 1:
            # pin this rank to the CPUs next to its GPU BEFORE any pinned host buffer is allocated: first touch
            # then places the staging memory on the GPU's NUMA node (matters for the host-buffer e2e legs)
            try:
                import pynvml

                pynvml.nvmlInit()
                uuid = str(torch.cuda.get_device_properties(self.local).uuid)
                h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid if not uuid.startswith("GPU-") else uuid).encode())
                words = (os.cpu_count() + 63) // 64
                mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
                cpus = {64 * w + b for w in range(words) for b in range(64) if (int(mask[w]) >> b) & 1}
                cpus &= os.sched_getaffinity(0)
                if cpus:
                    os.sched_setaffinity(0, cpus)
                    self.numa = len(cpus)
            except Exception:
                self.numa = None
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)
        if self.world != args.gpus and self.rank == 0:
            print(f"[bench] note: --gpus {args.gpus} but WORLD_SIZE={self.world}; using WORLD_SIZE", file=sys.stderr)
        self.sampler = ClockSampler(self.local)
        self.windows = {}
        self.start, self.stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t)


def peak_hbm():
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(peaks["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback 6650 GB/s (B200_PROFILING.md)"


def build_inputs(env: Env, name: str, want_graph: bool, want_cpu_rows: int):
    """Contact map -> (this rank's f32 target rows, CSR graph, features, CPU-side pieces for the baselines).
    Outside every timed region."""
    import numpy as np

    torch = env.torch
    from hic_gnn_b200 import ops, sharding, synth
    from hic_gnn_b200.graph import CSRGraph

    w = WORKLOADS[name]
    n, dev = w["n"], env.dev
    out = {"adj_cpu": None, "cpu_truth": None}
    if w["kind"] == "fixture":
        adj = torch.tensor(fixture_arrays()[f"{w['tag']}_kr_oracle"], dtype=torch.float64, device=dev)
        adj.fill_diagonal_(0)
    else:
        adj = synth.synthetic_map_chunked(n, w["density"], device=dev)
    balance = "upper" if ops._USE_UPPER else "rows"  # symmetric targets stream only the upper triangle: balance the blocks by its area
    world_eff, rank_eff = (env.args.emulate_world, env.args.emulate_rank) if (env.args.emulate_world and env.world == 1) else (env.world, env.rank)
    cuts = [sharding.row_block(n, r, world_eff, balance)[0] for r in range(world_eff)] + [n]
    rebalanced = []

    def build_target(r0, r1):
        # the maps are symmetric by construction (synth) / checked by the tests (fixtures): stated, not re-checked per rank
        return ops.cont2dist(adj[r0:r1], w["factor"], want_f64=False, want_f32=True, r0=r0, r1=r1, max_reduce=sharding.allreduce_max_, symmetric=True)[1]

    r0, r1 = cuts[rank_eff], cuts[rank_eff + 1]
    target = build_target(r0, r1)
    if balance == "upper" and env.world > 1 and n >= 4096 and not env.args.no_rebalance:
        # MEASURED load balancing (setup, outside every timed region): equal-area blocks do not take equal time, and the exchange waits
        # for the slowest rank.  Three rounds of: time this rank's kernel, all-gather the times, move the cuts (sharding.rebalance_cuts).
        g = torch.Generator().manual_seed(7)
        c_probe = (0.3 * torch.randn(n, 3, generator=g)).to(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ROUNDS = 3
        for it in range(ROUNDS + 1):
            for _w in range(3):
                ops.pairloss_raw(c_probe, target, ops._MODES["mse"], 4.0 / n**2, 0.0)
            env.barrier()
            e0.record()
            for _w in range(20):
                ops.pairloss_raw(c_probe, target, ops._MODES["mse"], 4.0 / n**2, 0.0)
            e1.record()
            e1.synchronize()
            t = torch.tensor([e0.elapsed_time(e1) / 20], dtype=torch.float64, device=dev)
            times = [torch.zeros_like(t) for _ in range(env.world)]
            env.dist.all_gather(times, t)
            times = [float(x) for x in times]
            rebalanced.append({"cuts": list(cuts), "kernel_ms": [round(x, 4) for x in times]})
            if it < ROUNDS:
                new_cuts = sharding.rebalance_cuts(n, cuts, times)
            else:  # the model is piecewise linear, the kernel's schedule is not: keep the best partition that was MEASURED
                new_cuts = min(rebalanced, key=lambda h: max(h["kernel_ms"]))["cuts"]
            if list(new_cuts) != list(cuts):
                cuts = list(new_cuts)
                r0, r1 = cuts[rank_eff], cuts[rank_eff + 1]
                del target
                torch.cuda.empty_cache()
                target = build_target(r0, r1)
        del c_probe
    graph = None
    if want_graph:
        rowptr, col, val = ops.csr_from_dense(adj)
        graph = CSRGraph(rowptr, col, val, n)
    if want_cpu_rows:
        rows = min(want_cpu_rows, n)

        def global_max(m):  # max over finite (1/a)^f = (1 / smallest non-zero contact)^f
            lo = float("inf")
            for a in range(0, n, 2048):
                blk = adj[a:a + 2048]
                pos = blk[blk > 0]
                if pos.numel():
                    lo = min(lo, float(pos.min()))
            m.copy_(torch.tensor([(1.0 / lo) ** w["factor"]], dtype=torch.float64, device=dev))

        cpu_truth, _ = ops.cont2dist(adj[:rows].contiguous(), w["factor"], want_f64=True, want_f32=False, r0=0, r1=rows, max_reduce=global_max)
        out["cpu_truth"] = cpu_truth.cpu()
        if n <= 3000:
            out["adj_cpu"] = adj.cpu().numpy()
    out.update({"adj": adj, "target": target, "graph": graph, "r0": r0, "r1": r1, "balance": balance + ("+measured" if rebalanced else ""), "rebalance": rebalanced, "cuts": cuts})
    return out


def measure_workload(env: Env, name: str, primary: bool):
    """All GPU legs of one workload.  ``primary``: every leg (loss, e2e, implicit target, train, CPU baselines) with the
    caller's step counts; otherwise the compact `configs` entry (loss + train + CPU baselines)."""
    torch, args, dev, world, rank = env.torch, env.args, env.dev, env.world, env.rank
    from hic_gnn_b200 import _native as N
    from hic_gnn_b200 import models, ops, sharding, synth, train

    w = WORKLOADS[name]
    n = w["n"]
    K = args.steps if primary else max(20, min(args.steps, 100))
    W = max(args.warmup, 3)
    want_train = not args.no_train
    want_cpu = (not args.no_cpu_baseline) and world == 1 and rank == 0
    sample_rows = sample_rows_for(n, args.cpu_sample_pairs if primary else min(args.cpu_sample_pairs, 5e7))
    t_setup = time.time()
    inp = build_inputs(env, name, want_graph=want_train, want_cpu_rows=sample_rows if want_cpu else 0)
    target, graph, r0, r1 = inp["target"], inp["graph"], inp["r0"], inp["r1"]
    sparse_tgt = None
    if primary and graph is not None and not args.no_sparse and w["kind"] == "synthetic":  # row f-4: the same target in implicit form
        sparse_tgt = ops.SparseWishTarget.from_graph(graph, inp["adj"], w["factor"], r0, r1)
    x = synth.synthetic_features(n, device=dev) if want_train else None
    csr_cpu = None
    if want_cpu and want_train and graph is not None and inp["adj_cpu"] is None:
        from oracle import graph as ograph  # CPU-baseline leg only

        csr_cpu = ograph.CSR(graph.rowptr.cpu(), graph.col.cpu(), graph.value.cpu(), n)
    inp["adj"] = None
    torch.cuda.empty_cache()
    g = torch.Generator().manual_seed(7)
    coords = (0.3 * torch.randn(n, 3, generator=g)).to(dev)
    nloc = r1 - r0
    loss_mode = args.loss_mode
    mode = ops._MODES[loss_mode]
    c_mse, c_l1 = 4.0 / (float(n) * float(n)), 0.1 / max(n * (n - 1) / 2.0, 1.0)
    target_bytes = nloc * target.pitch * 4
    t_setup = time.time() - t_setup
    start, stop = env.start, env.stop
    barrier, max_over_ranks = env.barrier, env.max_over_ranks

    # ---- (1) resident loss step: fused kernel on the local rows + ONE exchange of the partials
    # The kernel is bracketed by CUDA events INSIDE the timed region, but only on every EVERY-th step: an event record between two
    # launches costs a few microseconds of stream time and breaks their programmatic (PDL) chaining, which at 8 GPUs (0.2 ms steps)
    # would be 5 % of the number being measured.
    EVERY = 1 if K < 8 else (4 if K < 32 else 8)
    sampled = [k for k in range(K) if k % EVERY == 0]
    ev = {k: (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for k in sampled}
    ev_end = {k: torch.cuda.Event(enable_timing=True) for k in sampled}
    cursor = {"k": None}

    def timed(raw):  # the fused kernel, bracketed by events inside the timed region
        def fn(*a):
            k = cursor["k"]
            if k in ev:
                ev[k][0].record()
            raw(*a)
            if k in ev:
                ev[k][1].record()
        return fn

    def make_loss_fn(mode_bits, tgt, with_events=True):
        wrap = timed if with_events else (lambda f: f)
        if world == 1:  # one GPU: the library call itself, results in place (no packed buffer, no unpack kernels)
            m_out = torch.empty(N.PAIR_NMOM, dtype=torch.float64, device=dev)
            g_out = torch.empty(n, 3, dtype=torch.float32, device=dev)
            raw = wrap(lambda c: ops.pairloss_raw(c, tgt, mode_bits, c_mse, c_l1, moments=m_out, grad=g_out))

            def single(c):
                raw(c)
                return m_out, g_out

            return single
        const = None
        if mode_bits & N.PAIR_MOMENTS_D and not mode_bits & N.PAIR_MOMENTS:
            const = sharding.allreduce_packed(tgt.t_moments().clone())
        fn = sharding.make_sharded_pair_loss(n, wrap(sharding.cuda_local_fn(tgt, mode_bits, c_mse, c_l1)), dev, moment_const=const, transport=args.transport,
                                             local_split_fn=wrap(sharding.cuda_local_split_fn(tgt, mode_bits, c_mse, c_l1)))
        return fn

    loss_fn = make_loss_fn(mode, target)
    transport = "none" if world == 1 else ("nccl_allreduce" if not isinstance(loss_fn, sharding.P2PShardedPairLoss) else ("p2p_oneshot" if loss_fn.oneshot else "p2p_twoshot"))

    def loss_step(k=None):
        cursor["k"] = k
        out = loss_fn(coords)
        if k in ev_end:
            ev_end[k].record()  # kernel end -> here = the exchange (barrier wait on the slowest rank + reduction) / nothing at 1 GPU
        return out

    for _ in range(W):
        loss_step()
    attempts = 0
    while True:
        attempts += 1
        barrier()
        launches0 = N.launch_count()
        w0 = time.time()
        if primary:
            profile_region("loss", True)
        torch.cuda.nvtx.range_push(f"hicgat_loss_{name}")
        start.record()
        for k in range(K):
            moments, grad = loss_step(k)
        stop.record()
        barrier()
        torch.cuda.nvtx.range_pop()
        if primary:
            profile_region("loss", False)
        w1 = time.time()
        launches = N.launch_count() - launches0
        elapsed_ms = max_over_ranks(start.elapsed_time(stop))
        kern_ms = sum(a.elapsed_time(b) for a, b in ev.values()) / len(ev)
        exch_ms = sum(ev[k][1].elapsed_time(ev_end[k]) for k in sampled) / len(sampled)
        # A host-side stall (noisy neighbour, GC) leaves the GPU queue empty and shows up as step time far above
        # the kernel time; like a throttled run it is re-measured ONCE and the fact is reported.
        stalled = max_over_ranks(1.0 if elapsed_ms / K > 1.25 * kern_ms + 0.1 else 0.0) > 0
        if not stalled or attempts == 2:
            break
    # copied now: the legs below run the same loss function into the same device buffers
    outputs = {"loss_moments": moments.cpu(), "loss_grad": grad.reshape(n, 3).cpu()} if primary and args.dump_outputs else None
    value = float(n) * float(n) * K / (elapsed_ms * 1e-3) / 1e9
    mse = float(moments[0]) / (float(n) * float(n))
    env.windows[f"loss_{name}" if not primary else "loss"] = (w0, w1)
    peak, peak_src = peak_hbm()
    upper = ops.uses_upper_triangle(target)
    shards = args.emulate_world if (args.emulate_world and world == 1) else world
    # algorithmic bytes (SURVEY.md 8d): 4 B per ordered pair of this rank's share; in upper-triangle mode the share is 1/shards of
    # the pairs (blocks are balanced by area) and the kernel actually streams about half of that (2 B per ordered pair)
    alg_bytes = (float(n) * float(n) / shards if upper else float(nloc) * n) * 4.0
    streamed = (sum(n - i for i in (r0, r1 - 1)) / 2.0 * (r1 - r0) if r1 > r0 else 0.0) * 4.0 if upper else float(nloc) * n * 4.0
    achieved = alg_bytes / (kern_ms * 1e-3) / 1e9
    res = {"name": name, "n": n, "K": K, "W": W, "value": value, "ms_per_step": elapsed_ms / K, "kernel_ms": kern_ms, "exchange_ms": exch_ms, "launches": int(launches),
           "attempts": attempts, "kernel_samples": len(sampled), "mse": mse, "nloc": nloc, "target_bytes": target_bytes, "transport": transport, "setup_s": round(t_setup, 1),
           "achieved": achieved, "peak": peak, "peak_src": peak_src, "loss_mode": loss_mode, "upper": upper, "alg_bytes": alg_bytes, "streamed_bytes": streamed,
           "rows": [r0, r1], "balance": inp["balance"], "rebalance": inp["rebalance"], "cuts": inp["cuts"], "outputs": outputs}

    # ---- (1b) the other per-step mode of the training loops (MSE + Pearson moments in the same pass), briefly
    if primary and loss_mode == "mse":
        alt_fn = make_loss_fn(ops._MODES["mse_moments"], target, with_events=False)
        cursor["k"] = None
        for _ in range(3):
            alt_fn(coords)
        Ka = min(K, 50)
        barrier()
        start.record()
        for _ in range(Ka):
            alt_fn(coords)
        stop.record()
        barrier()
        a_ms = max_over_ranks(start.elapsed_time(stop))
        res["loss_modes"] = {"mse_moments": {"value": float(n) * float(n) * Ka / (a_ms * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": a_ms / Ka, "steps": Ka,
                                             "note": "MSE gradient + the Pearson moments of the GAT loops in the same pass (what the training step launches)"}}
        del alt_fn

    # ---- (2) end to end from host buffers (pinned), copies inside the timed region
    e2e = None
    if primary and not args.no_e2e:
        Ke = args.e2e_steps or min(K, 10)
        host_target = torch.empty(nloc, target.pitch, dtype=torch.float32, pin_memory=True)
        host_target.copy_(target.data)
        host_coords = torch.empty(n, 3, dtype=torch.float32, pin_memory=True)
        host_coords.copy_(coords)
        hp = ops.HostPairLoss(n, r0, r1, block_rows=max(64, min(4096, (256 << 20) // (target.pitch * 4))), device=dev,
                              reduce=sharding.allreduce_packed if world > 1 else None,  # host-buffer path: NCCL exchange
                              symmetric=upper)  # symmetric target: only the upper-triangle columns of every row block cross PCIe
        for _ in range(2):
            hm, hgrad = hp(host_coords, host_target, mode, c_mse, c_l1)
        barrier()
        w0 = time.time()
        start.record()
        for _ in range(Ke):
            hm, hgrad = hp(host_coords, host_target, mode, c_mse, c_l1)
        stop.record()
        barrier()
        env.windows["e2e"] = (w0, time.time())
        e_ms = max_over_ranks(start.elapsed_time(stop))
        h2d = max_over_ranks(float(hp.h2d_bytes))
        assert abs(float(hm[0]) - float(moments[0])) <= 1e-5 * abs(float(moments[0])), (float(hm[0]), float(moments[0]))
        # the host-buffer path walks ~1 300-row blocks (another schedule, the segmented combine): its gradient must be the resident one
        g_res = grad.detach().double().cpu().reshape(n, 3)
        e2e_grad_err = float((hgrad.double() - g_res).abs().max() / g_res.abs().max().clamp(min=1e-300))
        assert e2e_grad_err < 1e-5, e2e_grad_err
        e2e = {"value": float(n) * float(n) * Ke / (e_ms * 1e-3) / 1e9, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(hp.d2h_bytes), "steps": Ke, "ms_per_step": e_ms / Ke,
               "h2d_gbs": h2d / (e_ms / Ke * 1e-3) / 1e9, "grad_rel_err_vs_resident": e2e_grad_err,
               "note": "per rank: coords + this rank's f32 target rows from pinned host memory every step (PCIe-bound by construction)"
                       + ("; the target is symmetric, so only the columns at or right of each row block's diagonal are copied" if upper else "")}
        del host_target, hp
        torch.cuda.empty_cache()
        # (2b) the training-loop variant of the same call: the target stays resident (uploaded once, like
        # utils.wish_target does), only the step's coordinates go up and its loss moments + gradient come back
        out_host = torch.empty(N.PAIR_NMOM + 3 * n, dtype=torch.float64, pin_memory=True)
        coords_dev = torch.empty_like(coords)

        def resident_step():
            coords_dev.copy_(host_coords, non_blocking=True)
            m_, g_ = loss_fn(coords_dev)
            out_host[: N.PAIR_NMOM].copy_(m_, non_blocking=True)
            out_host[N.PAIR_NMOM:].copy_(g_.reshape(-1), non_blocking=True)
            torch.cuda.current_stream().synchronize()

        cursor["k"] = None
        for _ in range(3):
            resident_step()
        barrier()
        start.record()
        for _ in range(K):
            resident_step()
        stop.record()
        barrier()
        r_ms = max_over_ranks(start.elapsed_time(stop))
        e2e["resident_target"] = {"value": float(n) * float(n) * K / (r_ms * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": r_ms / K,
                                  "h2d_bytes_per_step": int(host_coords.numel() * 4), "d2h_bytes_per_step": int(out_host.numel() * 8),
                                  "note": "same call with the f32 target resident in HBM (how the training loop uses it): per step coords H2D, moments+gradient D2H, host sync"}
    res["e2e"] = e2e

    # ---- (2c) row f-4: the same loss against the implicit (sparse) target -- no N x N array, compute-bound
    sparse_out = None
    if sparse_tgt is not None:
        sp_fn = make_loss_fn(mode, sparse_tgt, with_events=False)
        cursor["k"] = None
        for _ in range(W):
            sm_, sg_ = sp_fn(coords)
        barrier()
        start.record()
        for _ in range(K):
            sm_, sg_ = sp_fn(coords)
        stop.record()
        barrier()
        s_ms = max_over_ranks(start.elapsed_time(stop))
        k0, k1 = int(sparse_tgt.rowptr[r0]), int(sparse_tgt.rowptr[r1])
        sparse_out = {"value": float(n) * float(n) * K / (s_ms * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": s_ms / K, "nnz_this_rank": k1 - k0,
                      "target_bytes_this_rank": (k1 - k0) * 8 + (n + 1) * 4, "bound": "fp32/mufu (no target stream)",
                      "mse_matches_dense": abs(float(sm_[0]) - float(moments[0])) <= 1e-6 * abs(float(moments[0]))}
        if not args.no_e2e:  # from host buffers: the CSR slice of this rank + coords go up every step, the result comes back
            Ke = args.e2e_steps or min(K, 10)
            h_col = torch.empty(k1 - k0, dtype=torch.int32, pin_memory=True); h_col.copy_(sparse_tgt.col[k0:k1])
            h_val = torch.empty(k1 - k0, dtype=torch.float32, pin_memory=True); h_val.copy_(sparse_tgt.tval[k0:k1])
            h_ptr = torch.empty(n + 1, dtype=torch.int32, pin_memory=True); h_ptr.copy_(sparse_tgt.rowptr)
            h_xyz = torch.empty(n, 3, dtype=torch.float32, pin_memory=True); h_xyz.copy_(coords)
            h_out = torch.empty(N.PAIR_NMOM + 3 * n, dtype=torch.float64, pin_memory=True)
            d_xyz = torch.empty_like(coords)

            def sparse_e2e_step():
                sparse_tgt.col[k0:k1].copy_(h_col, non_blocking=True)
                sparse_tgt.tval[k0:k1].copy_(h_val, non_blocking=True)
                sparse_tgt.rowptr.copy_(h_ptr, non_blocking=True)
                d_xyz.copy_(h_xyz, non_blocking=True)
                m_, g_ = sp_fn(d_xyz)
                h_out[: N.PAIR_NMOM].copy_(m_, non_blocking=True)
                h_out[N.PAIR_NMOM:].copy_(g_.reshape(-1), non_blocking=True)
                torch.cuda.current_stream().synchronize()

            for _ in range(2):
                sparse_e2e_step()
            barrier()
            start.record()
            for _ in range(Ke):
                sparse_e2e_step()
            stop.record()
            barrier()
            se_ms = max_over_ranks(start.elapsed_time(stop))
            sparse_out["e2e"] = {"value": float(n) * float(n) * Ke / (se_ms * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": se_ms / Ke,
                                 "h2d_bytes_per_step": int((k1 - k0) * 8 + (n + 1) * 4 + n * 12), "d2h_bytes_per_step": int(h_out.numel() * 8),
                                 "note": "host CSR slice (col, wish value) + rowptr + coords up, moments + gradient down, every step"}
        del sp_fn
    res["sparse"] = sparse_out
    del loss_fn

    # ---- (3) whole training step: GNN forward, fused loss, backward, Adam
    train_out = None
    if want_train:
        Kt = (args.train_steps or min(K, 10)) if primary else (10 if n > 20000 else 50)
        torch.manual_seed(42)
        model_key = args.model or w["model"]
        model_cls = getattr(models, MODEL_CLASSES[model_key])
        model = model_cls().to(dev)
        tmode = w["mode"]
        kmode = train._KERNEL_MODE[tmode]
        reducer = ops.sharded_reducer(target, kmode, transport=args.transport) if world > 1 else None
        graphed = (not args.no_cuda_graph) and (reducer is None or getattr(reducer, "capturable", False))
        lc0 = N.launch_count()
        tstep = train.TrainStep(model, x, graph, target, mode=tmode, lr=1e-3, use_cuda_graph=graphed, reducer=reducer)
        graph_kernels = (N.launch_count() - lc0) / 4.0 if graphed else None  # 3 warm-up steps + 1 captured step
        for _ in range(3):
            total, _m = tstep()
        barrier()
        l0 = N.launch_count()
        w0 = time.time()
        if primary:
            profile_region("train", True)
        torch.cuda.nvtx.range_push(f"hicgat_train_{name}")
        start.record()
        for _ in range(Kt):
            total, _m = tstep()
        stop.record()
        barrier()
        torch.cuda.nvtx.range_pop()
        if primary:
            profile_region("train", False)
        env.windows["train" if primary else f"train_{name}"] = (w0, time.time())
        if outputs is not None:
            outputs.update(train_total=total.reshape(1).cpu(), train_moments=_m.cpu())
        t_ms = max_over_ranks(start.elapsed_time(stop))
        train_out = {"steps_per_s": Kt / (t_ms * 1e-3), "ms_per_step": t_ms / Kt, "steps": Kt, "model": model_cls.__name__,
                     "loss": {"mse": "mse", "mse_pearson": "mse + alpha*(1-pearson)"}.get(tmode, tmode), "nnz": graph.nnz, "total_loss": float(total),
                     "hicgat_launches_per_step": graph_kernels if graphed else (N.launch_count() - l0) / Kt, "gnn": "replicated",
                     "loss_rows": "sharded" if world > 1 else "all", "cuda_graph": bool(graphed)}
        if w.get("gen_tag"):  # c2: the generalisation pass (HiC_GAT_generalize_directly.py:312-335): 500 kb structure from the 1 Mb model
            from hic_gnn_b200 import utils as hutils

            adj2 = torch.tensor(fixture_arrays()[f"{w['gen_tag']}_kr_oracle"], dtype=torch.float64, device=dev)
            data2 = hutils.load_input(adj2, synth.synthetic_features(adj2.shape[0], device=dev))
            model.eval()
            with torch.no_grad():
                for _ in range(3):
                    c2 = model.get_model(data2.x.float(), data2.edge_index)
                barrier()
                start.record()
                for _ in range(20):
                    c2 = model.get_model(data2.x.float(), data2.edge_index)
                stop.record()
                barrier()
            train_out["generalize"] = {"n_loci": int(adj2.shape[0]), "forward_ms": start.elapsed_time(stop) / 20,
                                       "note": "get_model of the trained net on the 500 kb graph (coords for cdist / dSCC / WritePDB)"}
        del tstep, model
    res["train"] = train_out

    # ---- (4) CPU baselines on this box's host cores (rank 0, N=1 only): the loss formulation and the training loop
    cpu = None
    if want_cpu:
        gps, sec, threads = time_cpu_sample(n, inp["cpu_truth"], sample_rows, 1, 5 if primary else 3)
        cpu = {"value": gps, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"oracle torch.cdist+MSELoss+autograd on rows [0,{sample_rows}) x {n} cols ({sample_rows * n:.3g} ordered pairs) per step, {sec * 1e3:.1f} ms/step"}
        if train_out is not None:
            model_name = MODEL_CLASSES[args.model or w["model"]]
            try:
                import psutil

                avail_gb = psutil.virtual_memory().available / 1e9
            except Exception:
                avail_gb = 0.0
            budget = args.cpu_train_budget
            edges = (graph.nnz + n) if graph is not None else 0
            need_gb = edges * 512 * 4 * 8 / 1e9  # E x H x C f32 message tensor: ~4 live copies per autograd graph, two graphs as written
            if n <= 300:
                tb = cpu_train_full(model_name, inp["adj_cpu"], x.cpu().numpy(), w["factor"], w["mode"], max(1, int(40 * budget)), warm=3)
            elif inp["adj_cpu"] is not None and need_gb < 0.5 * avail_gb:
                # in a child process: the as-written loop keeps two autograd graphs of E x H x C messages alive; if the host
                # cannot hold them the child dies, not the bench
                tb = cpu_train_in_child(name, args.model, max(1, int(budget)), timeout_s=600)
                if "error" in tb:
                    tb = {"kernel_equivalent": {"steps_per_s": None}, "as_written": None, "unit": "steps/s", "kind": "port", "error": tb["error"]}
            else:
                if csr_cpu is None:
                    from oracle import graph as ograph

                    csr_cpu = ograph.CSR(graph.rowptr.cpu(), graph.col.cpu(), graph.value.cpu(), n)
                tb = cpu_train_sliced(model_name, csr_cpu, x.cpu(), inp["cpu_truth"], sample_rows, n, w["mode"], edge_budget=1.0e6 * budget)
            tb["host_mem_available_gb"] = round(avail_gb, 1)
            train_out["cpu_baseline"] = tb
            ke = tb["kernel_equivalent"]["steps_per_s"]
            train_out["vs_cpu_kernel_equivalent"] = train_out["steps_per_s"] / ke if ke else None
    res["cpu"] = cpu
    del target, graph, x, coords, inp
    torch.cuda.empty_cache()
    return res


def compact(res):
    """`configs` entry of a secondary workload."""
    peak = res["peak"]
    n = res["n"]
    l2_note = "target is L2-resident (126 MB L2): HBM fraction not meaningful, judge the time" if res["target_bytes"] < 100e6 else None
    out = {"workload": WORKLOADS[res["name"]]["desc"], "n_loci": n, "pairs_per_step": float(n) * float(n),
           "loss": {"value": res["value"], "unit": UNIT, "ms_per_step": res["ms_per_step"], "kernel_ms": res["kernel_ms"], "exchange_ms": res["exchange_ms"],
                    "steps": res["K"], "loss_mode": res["loss_mode"], "rows_per_rank": res["nloc"],
                    "rows": res["rows"], "upper_triangle_only": res["upper"],
                    "roofline": {"bound": "hbm", "achieved": res["achieved"], "peak": peak, "unit": "GB/s", "frac": res["achieved"] / peak, "algorithmic_bytes": res["alg_bytes"],
                                 "streamed_bytes": res["streamed_bytes"], "note": l2_note}},
           "train": res["train"], "cpu_baseline": res["cpu"], "check": {"mse": res["mse"]}}
    return out


def run_native(args):
    env = Env(args)
    torch, world, rank, dev = env.torch, env.world, env.rank, env.dev
    from hic_gnn_b200 import _native as N

    if args.variant or args.rows_per_cta:
        N.set_pairloss_tuning(args.rows_per_cta, args.variant)
    env.sampler.start()

    # ---- (0) this box's copy bandwidth right now (same recipe as MEASURED_PEAKS.json: b.copy_(a), bytes read +
    # written, best of 10): a same-process control for box-to-box variation, reported beside the roofline
    copy_gbs = None
    if args.measure_copy:
        a_ = torch.empty(1 << 30, dtype=torch.bfloat16, device=dev)
        b_ = torch.empty_like(a_)
        best = float("inf")
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(12):
            e0.record()
            b_.copy_(a_)
            e1.record()
            e1.synchronize()
            best = min(best, e0.elapsed_time(e1))
        copy_gbs = 2 * a_.numel() * 2 / (best * 1e-3) / 1e9
        del a_, b_
        torch.cuda.empty_cache()

    name = args.workload
    res = measure_workload(env, name, primary=True)
    if args.configs == "auto":
        others = [] if args.emulate_world else (["c1", "c2", "c3", "c4"] if world == 1 else (["c4"] if name == "c5" else []))
        others = [o for o in others if o != name]
    elif args.configs in ("none", ""):
        others = []
    else:
        others = [o for o in args.configs.split(",") if o in WORKLOADS and o != name]
    configs = {}
    for o in others:
        t0 = time.time()
        configs[o] = compact(measure_workload(env, o, primary=False))
        configs[o]["wall_s"] = round(time.time() - t0, 1)
    env.sampler.stop()

    if rank == 0:
        w = WORKLOADS[name]
        n, nloc, kern_ms = res["n"], res["nloc"], res["kernel_ms"]
        peak, achieved = res["peak"], res["achieved"]
        traffic = None  # DRAM bytes per launch from the committed ncu capture of this exact shape, if there is one
        try:
            t = json.load(open(os.path.join(ROOT, "profiles", "pairloss_traffic.json"))).get(f"{nloc}x{n}" + ("_upper" if res["upper"] else ""))
            if t and args.variant == 0:
                traffic = float(t["dram_bytes_read"] + t["dram_bytes_write"] + t.get("combine_dram_bytes_read", 0))
        except Exception:
            pass
        line = {
            "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": res["K"], "warmup": res["W"], "ms_per_step": res["ms_per_step"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic" if w["kind"] == "synthetic" else "reference fixture (chr19)",
            "config": workload_config(name, res["loss_mode"]),
            "run": {"parallelism": f"rows{world}" if world > 1 else ("single" if not args.emulate_world else f"rank0-of-{args.emulate_world} (emulated, NOT a bench line)"),
                    "rows_per_rank": nloc, "rows": res["rows"], "row_balance": res["balance"], "row_cuts": res["cuts"], "rebalance_rounds": res["rebalance"], "upper_triangle_only": res["upper"], "cpus_near_gpu": env.numa, "exchange": res["transport"], "exchange_ms": res["exchange_ms"],
                    "timed_attempts": res["attempts"], "l2": f"no flush: each step streams {res['target_bytes'] / 1e6:.0f} MB of target per rank (L2 is 126 MB)",
                    "setup_s": res["setup_s"]},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "kernel": ("pairloss_tma_kernel" if args.variant == 0 else "pairloss_ldg_kernel") + " + pairloss_combine_kernel", "kernel_ms": kern_ms,
                         "kernel_samples": res["kernel_samples"],
                         "note": "kernel_ms = CUDA events around the two launches of one loss evaluation, on every 4th (K < 32) or 8th step of the timed region; peak is a COPY bandwidth (half reads, half writes): a read-only stream can exceed it slightly; "
                                 "traffic = dram bytes of the committed ncu capture of this shape (profiles/pairloss_traffic.json), not re-measured in this run",
                         "algorithmic_bytes": res["alg_bytes"], "streamed_bytes": res["streamed_bytes"],
                         "streamed_note": "upper-triangle mode: the target is symmetric, the kernel reads ~2 B per ordered pair (column >= row only) and evaluates every unordered pair once; "
                                          "`achieved` stays the ALGORITHMIC 4 B per ordered pair / kernel time (SURVEY.md 8d), so frac > 1 is the symmetry gain; streamed_bytes / kernel time is the DRAM-side rate" if res["upper"] else None,
                         "streamed_gbs": res["streamed_bytes"] / (kern_ms * 1e-3) / 1e9,
                         "peak_source": res["peak_src"], "frac_of_spec_8000": achieved / 8000.0,
                         "copy_gbs_this_run": copy_gbs, "frac_of_copy_this_run": (achieved / copy_gbs) if copy_gbs else None},
            "cpu_baseline": res["cpu"],
            "e2e": res["e2e"],
            "train": res["train"],
            "loss_modes": res.get("loss_modes"),
            "sparse_target": res["sparse"],
            "configs": configs,
            "gpu_launches": res["launches"],
            "clocks": env.sampler.summary(env.windows),
            "check": {"mse": res["mse"]},
        }
        print(json.dumps(line), flush=True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, res["outputs"])
    if world > 1:
        env.dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "cpu-train":
        run_cpu_train_child(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
