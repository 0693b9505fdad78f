"""The reference's full-batch training loops with the loop body replaced by the fused step.

Loop semantics kept (same flags/defaults): Adam(lr), ``while abs(old - new) > thresh``
(HiC-GNN_main.py:117-132, HiC_GAT_generalize_directly.py:186-243,
train_and_test_same_res_GAT_node2vec.py:93-143) or a fixed epoch count
(combined_loss_training.py:106).  Per step: ONE forward to N x 3 coordinates, ONE fused
loss+gradient launch over the f32 target, backward through the conv kernels, Adam.

``mode``:
  ``"mse"``          total = MSE                                       (HiC-GNN_main.py:127)
  ``"mse_pearson"``  total = MSE + min(1, 0.1 + 1/(MSE+1e-6)) (1 - r)  (HiC_GAT_generalize_directly.py:219-225;
                     r is a constant w.r.t. autograd in the reference, so the gradient is MSE's)
  ``"mse_pearson_grad"``  the same total as ``"mse_pearson"``, but the (1 - r) term carries its gradient (alpha held
                     constant): two passes per step (moments, then the gradient from the global moments), no host read,
                     graph-capturable, also sharded over the p2p exchange (ops.sharded_reducer, transport "p2p" / "auto")
  ``"contrastive"``  total = 0.1 mean_{i<j} |t - d|                    (train_and_test_same_res_GAT_node2vec.py:131-134)
  ``"mse_spearman"`` total = MSE + alpha (1 - dSCC), fixed alpha       (combined_loss_training.py:119-142; the Spearman
                     term is a scipy value in the reference, i.e. a constant for autograd: the gradient is MSE's.  The
                     rank transform runs on the GPU (metrics.dscc) but costs a host read per step: no CUDA graph.  With a
                     sharded ``reducer`` the dSCC comes from a ``dscc_meter`` (metrics.ShardedDsccMeter), identical on every rank)
"""
from __future__ import annotations

import torch
from torch.optim import Adam

from .ops import WishTarget, pairwise_loss, pearson_from_moments

_KERNEL_MODE = {"mse": "mse", "mse_pearson": "mse_moments", "mse_pearson_grad": "mse_pearson_grad", "contrastive": "contrastive",
                "mse_spearman": "mse_moments"}


def drmsd_from_moments(moments: torch.Tensor, n: int) -> torch.Tensor:
    """``calculate_dRMSD`` (combined_loss_training.py:22-26) from the fused kernel's upper-triangle ``sum (d-t)^2``."""
    return torch.sqrt(moments[7] / (n * (n - 1) / 2.0))


def step_loss(model, x, graph, target: WishTarget, mode: str, reducer=None, alpha: float = 1.0):
    """Forward + fused loss; returns (differentiable loss, total value tensor, moments)."""
    return _loss_of_coords(model.get_model(x, graph), target, mode, reducer, alpha)


def _loss_of_coords(coords, target, mode: str, reducer, alpha: float, rho=None):
    """``rho``: the dSCC of ``coords`` from a meter (0-d tensor), for ``mse_spearman``; needed with a sharded ``reducer``, whose ``target``
    is a row block: a block-local rank correlation would differ from rank to rank, and so would the totals the stop rule compares."""
    if mode == "mse_spearman" and rho is None and reducer is not None:
        raise ValueError("mse_spearman with a sharded reducer needs dscc_meter= (metrics.ShardedDsccMeter): "
                         "the dSCC of a row block differs from rank to rank")
    loss, moments = pairwise_loss(coords, target, _KERNEL_MODE[mode], reducer)
    total = loss.detach()  # mse_pearson_grad: the f64 total from the same moments as the gradient
    if mode == "mse_spearman":
        from . import metrics

        rho = metrics.dscc(coords.detach(), target) if rho is None else float(rho)   # spearmanr of the i<j distances (:137)
        if rho != rho:                                        # NaN -> 0 (:138-140)
            rho = 0.0
        total = total.double() + alpha * (1.0 - rho)
    if mode == "mse_pearson":
        n = target.n
        r = pearson_from_moments(moments, n * (n - 1) / 2.0)
        mse = total.double()
        alpha = torch.clamp(0.1 + 1.0 / (mse + 1e-6), max=1.0)
        total = mse + alpha * (1.0 - r)
    return loss, total, moments


class TrainStep:
    """One training iteration, optionally captured in a CUDA graph (small N is launch-bound:
    ~40 kernels per step).  ``total`` / ``moments`` are static device tensors when graphed.

    ``track_dscc=True`` also evaluates the dSCC of every step's forward coordinates -- the structure before that step's update, whose
    ``spearmanr`` the reference records every iteration (HiC_GAT_generalize_directly.py:242) -- with a :class:`metrics.DsccMeter`, on
    the device and inside the graph.  The value is ``step.dscc`` (0-d f64, overwritten by the next step).  Needs the full target:
    refused with a sharded ``reducer``.

    ``dscc_meter``: a caller-built :class:`metrics.DsccMeter` or :class:`metrics.ShardedDsccMeter` in place of ``track_dscc``; it is
    evaluated on the same (gathered, pre-update) coordinates every step into ``step.dscc``, inside the graph when the step is graphed
    (which needs ``dscc_meter.capturable``).  With a sharded ``reducer`` it is what gives per-step dSCC, and ``mode="mse_spearman"``
    takes its rho from it (without a meter that combination is refused; without a reducer ``mse_spearman`` keeps ``metrics.dscc``).

    ``gnn_shard`` (:class:`sharding.GnnRowShard`): the GNN runs on this rank's target rows only.  A step is: forward on the
    row-block view of ``graph`` -> ``gnn_shard.gather_coords`` (all N coordinates) -> the fused loss (sharded with ``reducer`` or
    not) -> backward -> ``gnn_shard.reduce_grads`` -> Adam; every rank ends the step with identical parameters.  With
    ``use_cuda_graph`` the exchange must be capturable (the p2p transport)."""

    def __init__(self, model, x, graph, target: WishTarget, mode: str = "mse", lr: float = 1e-3, use_cuda_graph: bool = False, reducer=None,
                 alpha: float = 1.0, track_dscc: bool = False, gnn_shard=None, dscc_meter=None):
        if mode not in _KERNEL_MODE:
            raise ValueError(mode)
        if track_dscc and dscc_meter is not None:
            raise ValueError("track_dscc and dscc_meter both ask for a per-step dSCC: pass one of them")
        if track_dscc and reducer is not None:
            raise ValueError("track_dscc needs the full target on one GPU: for a row-sharded target pass "
                             "dscc_meter=metrics.ShardedDsccMeter(target) instead")
        if mode == "mse_spearman" and reducer is not None and dscc_meter is None:
            raise ValueError("mse_spearman with a sharded reducer needs dscc_meter= (metrics.ShardedDsccMeter): "
                             "the dSCC of a row block differs from rank to rank")
        if use_cuda_graph and dscc_meter is not None and not getattr(dscc_meter, "capturable", True):
            raise ValueError("use_cuda_graph needs a capturable dSCC meter (the two-shot p2p exchange); "
                             f"the {getattr(dscc_meter, 'transport', '?')!r} exchange of {type(dscc_meter).__name__} is eager only")
        if mode == "mse_spearman" and use_cuda_graph:
            raise ValueError("mse_spearman reads the rank correlation back every step: it cannot be captured in a CUDA graph")
        if use_cuda_graph and reducer is not None and not getattr(reducer, "capturable", False):
            # a captured launch replays its arguments: an exchange that takes the epoch / buffer parity from the host (the
            # one-shot p2p kernel) or runs a NCCL collective outside torch's graph support would reuse one epoch forever
            raise ValueError("use_cuda_graph needs a capturable sharded reducer (the default two-shot p2p exchange); "
                             f"{type(reducer).__name__} takes per-step host arguments")
        if use_cuda_graph and gnn_shard is not None and not gnn_shard.capturable:
            # the NCCL exchange of the sharded GNN runs collectives outside torch's graph support
            raise ValueError("use_cuda_graph needs a capturable GNN row shard (the two-shot p2p exchange); "
                             f"the {gnn_shard.transport!r} exchange of {type(gnn_shard).__name__} is eager only")
        self.gnn_shard = gnn_shard
        if gnn_shard is not None:
            from .graph import as_graph

            graph = gnn_shard.graph(as_graph(graph, None, x.shape[0]))
        self.model, self.x, self.graph, self.target, self.mode, self.reducer, self.alpha = model, x, graph, target, mode, reducer, alpha
        self.optimizer = Adam(model.parameters(), lr=lr, capturable=use_cuda_graph)
        self.total = None
        self.moments = None
        self.dscc = None
        self._meter = dscc_meter
        if track_dscc:
            from .metrics import DsccMeter

            self._meter = DsccMeter(target)      # target-side tables and every buffer exist before a capture
        self._graph = None
        if use_cuda_graph:
            self._capture()

    def _eager(self):
        self.optimizer.zero_grad(set_to_none=True)
        coords = self.model.get_model(self.x, self.graph)
        if self.gnn_shard is not None:
            coords = self.gnn_shard.gather_coords(coords)
        if self._meter is not None:
            self.dscc = self._meter(coords.detach().contiguous())
        rho = self.dscc if self.reducer is not None and self.mode == "mse_spearman" else None  # one GPU: metrics.dscc, exact up to 4 096 loci
        loss, total, moments = _loss_of_coords(coords, self.target, self.mode, self.reducer, self.alpha, rho)
        loss.backward()
        if self.gnn_shard is not None:
            self.gnn_shard.reduce_grads(self.model.parameters())
        self.optimizer.step()
        return total, moments

    def _capture(self):
        # warm up on a side stream (allocator, lazy graph arrays, cuBLAS handles), then capture
        state = {k: v.detach().clone() for k, v in self.model.state_dict().items()}
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(3):
                self._eager()
        torch.cuda.current_stream().wait_stream(s)
        # undo the warm-up updates so that graphed and eager runs follow the same trajectory
        # (Adam state is zeroed IN PLACE: state created inside the capture would be re-zeroed
        # by every replay)
        self.model.load_state_dict(state)
        for st in self.optimizer.state.values():
            for v in st.values():
                if torch.is_tensor(v):
                    v.zero_()
        self.optimizer.zero_grad(set_to_none=True)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self.total, self.moments = self._eager()
        self._graph = g

    def __call__(self):
        if self._graph is not None:
            self._graph.replay()
            return self.total, self.moments
        self.total, self.moments = self._eager()
        return self.total, self.moments


def fit(model, x, graph, target: WishTarget, mode: str = "mse", lr: float = 1e-3, thresh: float = 1e-8, max_steps: int | None = None,
        check_every: int = 1, use_cuda_graph: bool = False, reducer=None, alpha: float = 1.0, dscc_out: list | None = None, gnn_shard=None,
        dscc_meter=None):
    """Reference loop.  Returns the list of per-step total losses (floats).

    ``check_every=1`` evaluates the stop rule every step exactly like the reference (one host
    read per step).  Larger values read the losses back in batches: same trajectory, but the
    loop may overrun the reference's stopping step by up to ``check_every-1`` iterations.

    ``dscc_out``: a list to which the dSCC of every step's (pre-update) structure is appended, like the reference's ``SpRho``
    history (``TrainStep(track_dscc=True)``); read back in the same batched reads as the losses.

    ``gnn_shard``: row-sharded GNN (:class:`TrainStep`).

    ``dscc_meter``: the meter that fills ``dscc_out`` (and gives ``mse_spearman`` its rho) instead of a :class:`metrics.DsccMeter` built
    here; with a sharded ``reducer`` a :class:`metrics.ShardedDsccMeter` of the same row block (:class:`TrainStep`)."""
    track = dscc_out is not None
    step = TrainStep(model, x, graph, target, mode, lr, use_cuda_graph, reducer, alpha, track_dscc=track and dscc_meter is None, gnn_shard=gnn_shard,
                     dscc_meter=dscc_meter)
    hist: list[float] = []
    pending: list[torch.Tensor] = []
    pending_dscc: list[torch.Tensor] = []
    old = 1.0
    done = False
    while not done and (max_steps is None or len(hist) + len(pending) < max_steps):
        model.train()
        total, _ = step()
        pending.append(total.clone() if use_cuda_graph else total)
        if track:
            pending_dscc.append(step.dscc.clone())
        if len(pending) >= check_every or (max_steps is not None and len(hist) + len(pending) >= max_steps):
            k = len(pending)
            vals = torch.stack([p.double().reshape(()) for p in pending + pending_dscc]).tolist()
            pending.clear()
            pending_dscc.clear()
            if track:
                dscc_out.extend(vals[k:])
            for v in vals[:k]:
                hist.append(v)
                if not (abs(old - v) > thresh):  # the reference loops `while lossdiff > thresh`: a NaN loss ends training
                    done = True
                old = v
    return hist
