"""Row-block sharding of the pairwise loss across the GPUs of one box (SURVEY.md section 8e).

Rank r owns target rows ``[r*ceil(N/G), (r+1)*ceil(N/G))`` x all N columns.  The GNN is
replicated, so every rank already holds identical N x 3 coordinates; per step each rank runs
the fused kernel on its block and ONE exchange combines the partials (latency-bound: <= 0.6 MB
per rank at 50k loci):

* :class:`P2PShardedPairLoss` (default on CUDA): the library's one-shot all-reduce kernel over
  NVLink peer memory (csrc/comm.cu), partials ``[8 x f64 moments | 3N x f32 gradient]`` in a
  symmetric buffer;
* :class:`ShardedPairLoss`: one NCCL / gloo ``all_reduce`` of the packed f64 buffer
  ``[8 moments | 3N gradient]``.  Backend-agnostic: the gloo tests run it on CPU tensors with a
  stand-in for the kernel.
"""
from __future__ import annotations

import torch
import torch.distributed as dist

from . import _native as N


def row_block(n: int, rank: int, world: int, balance: str = "rows") -> tuple[int, int]:
    """Contiguous row range of ``rank``; trailing ranks may be short or empty.

    ``balance="rows"``: equal row counts (the kernels stream the full row block).
    ``balance="upper"``: equal UPPER-TRIANGLE area (symmetric targets: row i costs n - i pairs, so the first rank gets
    few long rows and the last one many short ones); boundaries rounded to the kernel's 64-row tiles on big maps."""
    if balance == "rows":
        per = (n + world - 1) // world
        r0 = min(rank * per, n)
        return r0, min(r0 + per, n)
    if balance != "upper":
        raise ValueError(balance)

    def cut(r: int) -> int:
        if r <= 0:
            return 0
        if r >= world:
            return n
        # rows [0, c) hold a fraction 1 - (1 - c/n)^2 of the triangle
        c = n * (1.0 - (1.0 - r / world) ** 0.5)
        unit = 64 if n // world >= 2048 else 8  # big blocks: whole 64-row tiles; small ones: the rounding would unbalance them
        return max(0, min(n, int(round(c / unit)) * unit))

    return cut(rank), cut(rank + 1)


def all_blocks(n: int, world: int, balance: str = "rows") -> list[tuple[int, int]]:
    return [row_block(n, r, world, balance) for r in range(world)]


def rebalance_cuts(n: int, cuts: list[int], times: list[float], unit: int = 64) -> list[int]:
    """One step of MEASURED load balancing for the upper-triangle kernel: ``cuts`` (world + 1 row boundaries, cuts[0] = 0,
    cuts[-1] = n) were run and rank r's kernel took ``times[r]``.  Equal-area blocks do not take equal time (a wide, short
    block pays the per-item overhead more often than a tall triangle), so the cost per unit of triangle area is taken to be
    constant INSIDE each measured block and the boundaries are moved to where the cumulative cost reaches k / world of the total.
    Pure arithmetic (no GPU, no collectives): every rank calls it with the same gathered ``times`` and gets the same answer."""
    world = len(cuts) - 1
    if world < 2 or any(t <= 0 for t in times):
        return list(cuts)

    def frac(r):  # share of the upper triangle above row r
        return 1.0 - (1.0 - r / n) ** 2

    u = [frac(c) for c in cuts]
    total = sum(times)
    new = [0]
    acc, k = 0.0, 0
    for j in range(1, world):
        want = total * j / world
        while k < world - 1 and acc + times[k] < want:
            acc += times[k]
            k += 1
        width = u[k + 1] - u[k]
        uu = u[k] + (width * (want - acc) / times[k] if width > 0 else 0.0)
        row = n * (1.0 - max(0.0, 1.0 - uu) ** 0.5)
        uu_unit = unit if n // world >= 2048 else 8
        row = int(round(row / uu_unit)) * uu_unit
        new.append(max(new[-1], min(n, row)))
    new.append(n)
    return new


def unpack(packed: torch.Tensor, n: int):
    """packed f64[8+3n] -> (moments f64[8], grad f32[n,3])."""
    return packed[: N.PAIR_NMOM], packed[N.PAIR_NMOM:].view(n, 3).to(torch.float32)


def allreduce_packed(packed: torch.Tensor, group=None) -> torch.Tensor:
    """The single per-step collective.  No-op without an initialised process group."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(packed, op=dist.ReduceOp.SUM, group=group)
    return packed


def allreduce_max_(x: torch.Tensor, group=None) -> torch.Tensor:
    """Global max for the sharded wish-distance build (between cont2dist's two passes)."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(x, op=dist.ReduceOp.MAX, group=group)
    return x


class ShardedPairLoss:
    """Callable ``(coords) -> (moments, grad)`` over this rank's row block + one all-reduce.
    ``local_fn(coords, packed)`` fills the packed buffer for the local block (the CUDA kernel
    in production; tests inject a CPU stand-in)."""

    def __init__(self, n: int, local_fn, device, group=None, moment_const=None):
        self.n, self.local_fn, self.group = n, local_fn, group
        self.packed = torch.zeros(N.PAIR_NMOM + 3 * n, dtype=torch.float64, device=device)
        self.moment_const = moment_const  # f64[8] added after the reduction (target-only moments)

    def __call__(self, coords: torch.Tensor):
        self.local_fn(coords, self.packed)
        allreduce_packed(self.packed, self.group)
        moments, grad = unpack(self.packed, self.n)
        if self.moment_const is not None:
            moments = moments + self.moment_const
        return moments, grad


class TwoPassShardedPairLoss:
    """Same contract as :class:`ShardedPairLoss` for the differentiable Pearson modes, whose gradient needs the GLOBAL
    moments: ``moments_fn(coords, moments_f64[8])`` fills this block's pass-1 moments, one ``all_reduce`` sums them (plus
    ``moment_const``, the target-only sums), ``grad_fn(coords, global_moments) -> grad_f32[n,3]`` is this block's pass-2
    gradient, and a second ``all_reduce`` (f64) sums that.  Backend-agnostic (NCCL, or gloo with CPU stand-ins in the
    tests); not capturable in a CUDA graph."""

    capturable = False

    def __init__(self, n: int, moments_fn, grad_fn, device, group=None, moment_const=None):
        self.n, self.moments_fn, self.grad_fn, self.group = n, moments_fn, grad_fn, group
        self.moments = torch.zeros(N.PAIR_NMOM, dtype=torch.float64, device=device)
        self.gbuf = torch.zeros(3 * n, dtype=torch.float64, device=device)
        self.moment_const = moment_const

    def __call__(self, coords: torch.Tensor):
        self.moments_fn(coords, self.moments)
        allreduce_packed(self.moments, self.group)
        moments = self.moments if self.moment_const is None else self.moments + self.moment_const
        self.gbuf.copy_(self.grad_fn(coords, moments).reshape(-1))
        allreduce_packed(self.gbuf, self.group)
        return moments, self.gbuf.view(self.n, 3).to(torch.float32)


class P2PShardedPairLoss:
    """Same contract as :class:`ShardedPairLoss`, but the exchange is the hand-written two-shot all-reduce over
    NVLink peer memory (``hicgat_allreduce_partials_twoshot``, csrc/comm.cu): the fused loss kernel writes its partial
    ``[8 x f64 moments | 3n x f32 gradient]`` straight into a symmetric buffer that every rank maps; ONE kernel per rank
    then does barrier -> reduce slice ``rank`` of all partials (rank order, f64) -> store it into every rank's result
    buffer -> barrier.  The epoch counter lives in device memory, so every launch has identical arguments and the whole
    sharded step (loss kernel + exchange) can be captured in a CUDA graph (``capturable``).  The returned gradient is
    a view of this rank's result buffer: valid until the next call.
    ``local_fn(coords, moments_f64[8], grad_f32[n,3])`` fills the local partial.
    ``oneshot=True`` selects the older one-shot kernel (every rank reads all partials; host-side epoch, not capturable)."""

    SLOT_BASE = 256  # uint32 slot offset inside torch's signal pad (its own barriers use the low channels)

    def __init__(self, n: int, local_fn, device, group=None, moment_const=None, oneshot: bool = False):
        import ctypes as C

        import torch.distributed._symmetric_memory as symm

        group = group if group is not None else dist.group.WORLD
        self.n, self.local_fn, self.oneshot = n, local_fn, oneshot
        self.capturable = not oneshot
        grad_bytes = (12 * n + 15) // 16 * 16
        self.part_bytes = 64 + grad_bytes
        # layout: [partial 0 | partial 1 (one-shot only: epoch parity) | result]
        self.res_off = 2 * self.part_bytes
        self.buf = symm.empty(self.res_off + grad_bytes, dtype=torch.uint8, device=device)
        self.buf.zero_()
        self.hdl = symm.rendezvous(self.buf, group)
        self.world, self.rank = self.hdl.world_size, self.hdl.rank
        if self.hdl.signal_pad_size < 4 * (self.SLOT_BASE + 64):
            raise RuntimeError("symmetric-memory signal pad too small")
        ptrs = [int(p) for p in self.hdl.buffer_ptrs]
        self._bufs = (C.c_uint64 * self.world)(*ptrs)
        self._res = (C.c_uint64 * self.world)(*[p + self.res_off for p in ptrs])
        self._pads = (C.c_uint64 * self.world)(*[int(p) for p in self.hdl.signal_pad_ptrs])
        self.moment_const = moment_const
        # typed views of the local partial(s) and of the result
        self.part_m = [self.buf[h * self.part_bytes: h * self.part_bytes + 64].view(torch.float64) for h in range(2)]
        self.part_g = [self.buf[h * self.part_bytes + 64: h * self.part_bytes + 64 + 12 * n].view(torch.float32).view(n, 3) for h in range(2)]
        self.res_g = self.buf[self.res_off: self.res_off + 12 * n].view(torch.float32).view(n, 3)
        self.out_m = [torch.empty(N.PAIR_NMOM, dtype=torch.float64, device=device) for _ in range(2)]
        self.out_g = [torch.empty(n, 3, dtype=torch.float32, device=device) for _ in range(2)]
        self.state = torch.zeros(4, dtype=torch.int32, device=device)  # [epoch, ticket, ticket, -]: maintained by the kernel
        self.epoch = 0
        torch.cuda.synchronize(device)
        dist.barrier(group)  # every rank's buffer is zeroed and mapped before the first signal

    def __call__(self, coords: torch.Tensor):
        if not self.oneshot:
            self.local_fn(coords, self.part_m[0], self.part_g[0])
            rc = N.lib().hicgat_allreduce_partials_twoshot(
                self._bufs, self._res, self._pads, self.rank, self.world, self.n, self.SLOT_BASE + 32, self.state.data_ptr(),
                None if self.moment_const is None else self.moment_const.data_ptr(), self.out_m[0].data_ptr(), torch.cuda.current_stream().cuda_stream,
            )
            N.check(rc, "hicgat_allreduce_partials_twoshot")
            return self.out_m[0], self.res_g
        self.epoch += 1
        par = self.epoch & 1
        self.local_fn(coords, self.part_m[par], self.part_g[par])
        m, g = self.out_m[par], self.out_g[par]
        rc = N.lib().hicgat_allreduce_partials_p2p(
            self._bufs, self._pads, self.rank, self.world, self.n, par * self.part_bytes, self.SLOT_BASE, self.epoch & 0xFFFFFFFF,
            None if self.moment_const is None else self.moment_const.data_ptr(), m.data_ptr(), g.data_ptr(),
            torch.cuda.current_stream().cuda_stream,
        )
        N.check(rc, "hicgat_allreduce_partials_p2p")
        return m, g


class P2PTwoPassShardedPairLoss:
    """:class:`TwoPassShardedPairLoss` over NVLink peer memory: both exchanges are the two-shot kernel
    (``hicgat_allreduce_partials_twoshot``), so the whole sharded step -- pass 1, moments exchange, pass 2, gradient exchange --
    has identical launch arguments every step and can be captured in a CUDA graph (``capturable``).
    The moments exchange is a two-shot all-reduce of a moments-only partial (``n = 1``: the 16-byte gradient part stays zero);
    the gradient exchange reduces a partial whose moment part stays zero.  Each has its own state array and signal-slot range.
    ``moments_fn(coords, moments_f64[8])`` fills this block's pass-1 moments in place, ``grad_fn(coords, global_moments, grad_f32[n,3])``
    this block's pass-2 gradient in place.  The returned moments / gradient are views of the result buffers: valid until the next call."""

    SLOT_BASE = P2PShardedPairLoss.SLOT_BASE
    SLOTS_MOMENTS = SLOT_BASE + 64   # two-shot barriers use 2 x 16 slots from their base
    SLOTS_GRAD = SLOT_BASE + 96
    capturable = True

    def __init__(self, n: int, moments_fn, grad_fn, device, group=None, moment_const=None):
        import ctypes as C

        import torch.distributed._symmetric_memory as symm

        group = group if group is not None else dist.group.WORLD
        self.n, self.moments_fn, self.grad_fn = n, moments_fn, grad_fn
        grad_bytes = (12 * n + 15) // 16 * 16
        # layout: [moments partial: 64 + 16 | moments result: 16 | gradient partial: 64 + grad_bytes | gradient result: grad_bytes]
        self.m_part, self.m_res = 0, 80
        self.g_part = 96
        self.g_res = self.g_part + 64 + grad_bytes
        self.buf = symm.empty(self.g_res + grad_bytes, dtype=torch.uint8, device=device)
        self.buf.zero_()
        self.hdl = symm.rendezvous(self.buf, group)
        self.world, self.rank = self.hdl.world_size, self.hdl.rank
        if self.hdl.signal_pad_size < 4 * (self.SLOTS_GRAD + 32):
            raise RuntimeError("symmetric-memory signal pad too small")
        ptrs = [int(p) for p in self.hdl.buffer_ptrs]
        table = lambda off: (C.c_uint64 * self.world)(*[p + off for p in ptrs])
        self._m_bufs, self._m_res = table(self.m_part), table(self.m_res)
        self._g_bufs, self._g_res = table(self.g_part), table(self.g_res)
        self._pads = (C.c_uint64 * self.world)(*[int(p) for p in self.hdl.signal_pad_ptrs])
        self.moment_const = moment_const
        self.part_m = self.buf[self.m_part: self.m_part + 64].view(torch.float64)
        self.part_g = self.buf[self.g_part + 64: self.g_part + 64 + 12 * n].view(torch.float32).view(n, 3)
        self.res_g = self.buf[self.g_res: self.g_res + 12 * n].view(torch.float32).view(n, 3)
        self.out_m = torch.empty(N.PAIR_NMOM, dtype=torch.float64, device=device)
        self.scratch_m = torch.empty(N.PAIR_NMOM, dtype=torch.float64, device=device)  # the gradient exchange's (zero) moment sum
        self.state_m = torch.zeros(4, dtype=torch.int32, device=device)
        self.state_g = torch.zeros(4, dtype=torch.int32, device=device)
        torch.cuda.synchronize(device)
        dist.barrier(group)  # every rank's buffer is zeroed and mapped before the first signal

    def __call__(self, coords: torch.Tensor):
        lib, stream = N.lib(), torch.cuda.current_stream().cuda_stream
        self.moments_fn(coords, self.part_m)
        N.check(lib.hicgat_allreduce_partials_twoshot(self._m_bufs, self._m_res, self._pads, self.rank, self.world, 1, self.SLOTS_MOMENTS,
                                                      self.state_m.data_ptr(), None if self.moment_const is None else self.moment_const.data_ptr(),
                                                      self.out_m.data_ptr(), stream), "hicgat_allreduce_partials_twoshot")
        self.grad_fn(coords, self.out_m, self.part_g)
        N.check(lib.hicgat_allreduce_partials_twoshot(self._g_bufs, self._g_res, self._pads, self.rank, self.world, self.n, self.SLOTS_GRAD,
                                                      self.state_g.data_ptr(), None, self.scratch_m.data_ptr(), stream),
                "hicgat_allreduce_partials_twoshot")
        return self.out_m, self.res_g


def make_sharded_pair_loss(n: int, local_fn, device, group=None, moment_const=None, transport: str = "auto", local_split_fn=None):
    """``transport``: ``"p2p"`` (two-shot kernel over NVLink peer memory; needs ``local_split_fn``), ``"p2p_oneshot"``
    (the older one-shot kernel, A/B only), ``"nccl"`` (packed ``all_reduce``; uses ``local_fn``) or ``"auto"`` (p2p on CUDA
    with an initialised multi-rank NCCL group when the symmetric-memory rendezvous succeeds, else nccl)."""
    multi = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
    if local_split_fn is not None and (transport in ("p2p", "p2p_oneshot") or (transport == "auto" and multi and torch.device(device).type == "cuda")):
        try:
            return P2PShardedPairLoss(n, local_split_fn, device, group, moment_const, oneshot=transport == "p2p_oneshot")
        except Exception as e:  # no symmetric memory on this system: the NCCL exchange is equivalent
            if transport in ("p2p", "p2p_oneshot"):
                raise
            import warnings

            warnings.warn(f"symmetric-memory exchange unavailable ({e!r}); using the NCCL all-reduce")
    elif transport in ("p2p", "p2p_oneshot"):
        raise RuntimeError("transport='p2p' needs local_split_fn")
    return ShardedPairLoss(n, local_fn, device, group, moment_const)


def cuda_local_fn(target, mode: int, c_mse: float, c_l1: float):
    """The production ``local_fn`` of the NCCL exchange: fills the packed f64 buffer for this rank's
    target (dense: hicgat_pairloss_fwd_bwd_packed in one launch; implicit/sparse: the split call + a pack)."""
    from .ops import SparseWishTarget, _PairWorkspace, _cuda, _stream, pairloss_raw

    def sparse_fn_for(target, mode, c_mse, c_l1):
        def sparse_fn(coords: torch.Tensor, packed: torch.Tensor):
            m, g = pairloss_raw(coords, target, mode, c_mse, c_l1)
            packed[: N.PAIR_NMOM].copy_(m)
            packed[N.PAIR_NMOM:].copy_(g.reshape(-1))

        return sparse_fn

    if isinstance(target, SparseWishTarget):
        return sparse_fn_for(target, mode, c_mse, c_l1)

    if target.symmetric is False:  # needs the row-side pass: go through the split call (ops.pairloss_raw) and pack
        return sparse_fn_for(target, mode, c_mse, c_l1)

    from .ops import uses_upper_triangle

    sym = uses_upper_triangle(target)

    def fn(coords: torch.Tensor, packed: torch.Tensor):
        _cuda(coords, packed)
        ws = _PairWorkspace.get(coords.device, target.n, target.r0, target.r1, sym=sym)
        rc = N.lib().hicgat_pairloss_fwd_bwd_packed(
            coords.contiguous().data_ptr(), target.data.data_ptr(), target.pitch, target.n, target.r0, target.r1,
            mode | N.PAIR_WS_CLEAN | (N.PAIR_SYMMETRIC if sym else 0), c_mse, c_l1, packed.data_ptr(), ws.data_ptr(), ws.numel(), _stream(),
        )
        N.check(rc, "hicgat_pairloss_fwd_bwd_packed")

    return fn


def cuda_local_split_fn(target, mode: int, c_mse: float, c_l1: float):
    """``local_fn`` of :class:`P2PShardedPairLoss`: the loss kernel writes moments / grad straight into
    the symmetric partial (dense or implicit target)."""
    from .ops import pairloss_raw

    def fn(coords: torch.Tensor, moments: torch.Tensor, grad: torch.Tensor):
        pairloss_raw(coords, target, mode, c_mse, c_l1, moments=moments, grad=grad)

    return fn
