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


# ------------------------------------------------------------------------------ row-sharded GNN
def gnn_blocks(rowptr, world: int) -> list[tuple[int, int]]:
    """Partition of the GNN's target rows into ``world`` contiguous blocks of equal work.  The message-passing kernels cost one
    warp-row per locus plus one gather per edge, so row i weighs ``deg(i) + 1`` (its row of the self-loop pattern), and the rows
    ``[0, i)`` weigh ``rowptr[i] + i``.  Cut r is the row whose prefix weight is nearest to ``r / world`` of the total (ties to the
    lower row); blocks may be empty when one row outweighs a whole share.  Pure arithmetic on the host (one read of ``rowptr``
    if it is a device tensor); independent of the loss's :func:`row_block` cuts."""
    import bisect

    if world < 1:
        raise ValueError(f"gnn_blocks: world must be >= 1, got {world}")
    rp = [int(v) for v in (rowptr.tolist() if torch.is_tensor(rowptr) else rowptr)]
    n = len(rp) - 1
    if n < 0:
        raise ValueError("gnn_blocks: rowptr needs n + 1 >= 1 entries")
    mass = [(rp[i] + i) * world for i in range(n + 1)]  # prefix weights, scaled so that cut r aims at r * total
    total = rp[n] + n
    cuts = [0]
    for r in range(1, world):
        want = r * total
        i = bisect.bisect_left(mass, want)
        if i > 0 and want - mass[i - 1] <= mass[min(i, n)] - want:
            i -= 1
        cuts.append(max(cuts[-1], min(i, n)))
    cuts.append(n)
    return list(zip(cuts[:-1], cuts[1:]))


class _GatherCoords(torch.autograd.Function):
    """Block rows ``[g0, g1)`` of the coordinates -> all N rows (exchange); backward: rows ``[g0, g1)`` of the incoming gradient,
    which every rank already holds in full (a sharded loss reduces it, an unsharded one computes it on every rank alike)."""

    @staticmethod
    def forward(ctx, local, shard):
        ctx.block = (shard.g0, shard.g1)
        return shard._x.gather(local.detach(), shard.g0, shard.g1)

    @staticmethod
    def backward(ctx, g):
        g0, g1 = ctx.block
        return g[g0:g1], None


class _CollectiveExchange:
    """Both exchanges as ONE ``all_reduce`` each of an f64 buffer (NCCL, or gloo on CPU): the coordinate partial is zero outside
    the rank's rows, so the gather is exact; the gradient sum is rounded to f32 once.  Eager only: not capturable."""

    capturable = False

    def __init__(self, n: int, numel: int, device, group):
        self.n, self.numel, self.device, self.group = n, numel, device, group

    def gather(self, local, g0, g1):
        buf = torch.zeros(self.n, 3, dtype=torch.float64, device=self.device)
        buf[g0:g1] = local.double()
        return allreduce_packed(buf, self.group).to(torch.float32)

    def reduce(self, grads):
        flat = torch.cat([g.reshape(-1).double() for g in grads])
        allreduce_packed(flat, self.group)
        torch._foreach_copy_(grads, [v.view_as(g) for v, g in zip(flat.split([g.numel() for g in grads]), grads)])


class _P2PExchange:
    """Both exchanges over NVLink peer memory with the two-shot all-reduce of the sharded loss (``hicgat_allreduce_partials_twoshot``):
    an f32 buffer is reduced as the ``[k, 3]`` gradient part of a partial whose moment part stays zero (f64 accumulation in rank
    order, one rounding: bit-identical on every rank; the coordinate gather is exact, the other ranks add zeros).  Each exchange has
    its own state array and signal-slot range, beyond those of the sharded loss exchanges, so all of them can share a step and a
    CUDA graph (``capturable``)."""

    capturable = True
    SLOTS_COORDS = P2PShardedPairLoss.SLOT_BASE + 128  # the loss exchanges use SLOT_BASE + 0 .. + 127
    SLOTS_GRADS = P2PShardedPairLoss.SLOT_BASE + 160

    def __init__(self, n: int, numel: int, device, group):
        import ctypes as C

        import torch.distributed._symmetric_memory as symm

        group = group if group is not None else dist.group.WORLD
        self.n, self.numel = n, numel
        self.kg = (numel + 2) // 3  # rows of the [k, 3] view of the flat gradient
        cbytes, gbytes = (12 * n + 15) // 16 * 16, (12 * self.kg + 15) // 16 * 16
        # layout: [coords partial: 64 + cbytes | coords result: cbytes | grads partial: 64 + gbytes | grads result: gbytes]
        self.c_part, self.c_res = 0, 64 + cbytes
        self.g_part = self.c_res + cbytes
        self.g_res = self.g_part + 64 + gbytes
        self.buf = symm.empty(self.g_res + gbytes, dtype=torch.uint8, device=device)
        self.buf.zero_()
        self.hdl = symm.rendezvous(self.buf, group)
        self.world, self.rank = self.hdl.world_size, self.hdl.rank
        if self.hdl.signal_pad_size < 4 * (self.SLOTS_GRADS + 32):
            raise RuntimeError("symmetric-memory signal pad too small")
        ptrs = [int(p) for p in self.hdl.buffer_ptrs]
        table = lambda off: (C.c_uint64 * self.world)(*[p + off for p in ptrs])
        self._c_bufs, self._c_res = table(self.c_part), table(self.c_res)
        self._g_bufs, self._g_res = table(self.g_part), table(self.g_res)
        self._pads = (C.c_uint64 * self.world)(*[int(p) for p in self.hdl.signal_pad_ptrs])
        f32 = lambda off, k: self.buf[off: off + 4 * k].view(torch.float32)
        self.part_c = f32(self.c_part + 64, 3 * n).view(n, 3)   # rows outside the block stay zero forever
        self.res_c = f32(self.c_res, 3 * n).view(n, 3)
        self.part_g = f32(self.g_part + 64, numel)
        self.res_g = f32(self.g_res, numel)
        self.scratch_m = torch.empty(N.PAIR_NMOM, dtype=torch.float64, device=device)  # the (zero) moment sums
        self.state_c = torch.zeros(4, dtype=torch.int32, device=device)
        self.state_g = torch.zeros(4, dtype=torch.int32, device=device)
        torch.cuda.synchronize(device)
        dist.barrier(group)  # every rank's buffer is zeroed and mapped before the first signal

    def _twoshot(self, bufs, res, k, slots, state):
        N.check(N.lib().hicgat_allreduce_partials_twoshot(bufs, res, self._pads, self.rank, self.world, k, slots, state.data_ptr(), None,
                                                          self.scratch_m.data_ptr(), torch.cuda.current_stream().cuda_stream),
                "hicgat_allreduce_partials_twoshot")

    def gather(self, local, g0, g1):
        self.part_c[g0:g1].copy_(local)
        self._twoshot(self._c_bufs, self._c_res, self.n, self.SLOTS_COORDS, self.state_c)
        return self.res_c.clone()

    def reduce(self, grads):
        torch.cat([g.reshape(-1) for g in grads], out=self.part_g)
        self._twoshot(self._g_bufs, self._g_res, self.kg, self.SLOTS_GRADS, self.state_g)
        torch._foreach_copy_(grads, [v.view_as(g) for v, g in zip(self.res_g.split([g.numel() for g in grads]), grads)])


class GnnRowShard:
    """Row-sharded GNN across the ranks of a process group: this rank runs the message passing and the MLP head on its target
    rows ``block = (g0, g1)`` only (``graph.row_block(g0, g1)``, blocks from :func:`gnn_blocks`), and two exchanges keep every rank
    consistent:

    * :meth:`gather_coords` (autograd): the block's ``[g1 - g0, 3]`` coordinates -> all ``[n, 3]``; its backward hands the block's
      rows of the coordinate gradient back (no communication);
    * :meth:`reduce_grads`: sums the parameter gradients -- each rank's are partial sums over its rows -- over the ranks, in place,
      bit-identical on every rank, so that the replicated parameters stay in lock step.

    ``transport``: ``"p2p"`` (two-shot kernel over NVLink peer memory, capturable), ``"nccl"`` (one f64 ``all_reduce`` per
    exchange; with a gloo group on CPU tensors too; eager only) or ``"auto"`` (p2p on CUDA with an initialised multi-rank group
    when the symmetric-memory rendezvous succeeds, else nccl -- the rule of :func:`make_sharded_pair_loss`).  Without a multi-rank
    process group both exchanges are local no-ops around the one block."""

    def __init__(self, n: int, block: tuple[int, int], params, device, group=None, transport: str = "auto"):
        if transport not in ("auto", "p2p", "nccl"):
            raise ValueError(f"GnnRowShard: transport must be 'auto', 'p2p' or 'nccl', got {transport!r}")
        g0, g1 = int(block[0]), int(block[1])
        if not 0 <= g0 <= g1 <= n:
            raise ValueError(f"GnnRowShard: need 0 <= g0 <= g1 <= n = {n}, got [{g0}, {g1})")
        self.n, self.g0, self.g1, self.group = n, g0, g1, group
        self.params = list(params)
        numel = sum(p.numel() for p in self.params)
        multi = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
        self._x = None
        if transport == "p2p" or (transport == "auto" and multi and torch.device(device).type == "cuda"):
            try:
                self._x = _P2PExchange(n, numel, device, group)
            except Exception as e:  # no symmetric memory on this system: the collective exchange is equivalent
                if transport == "p2p":
                    raise
                import warnings

                warnings.warn(f"symmetric-memory exchange unavailable ({e!r}); using the NCCL all-reduce")
        if self._x is None:
            self._x = _CollectiveExchange(n, numel, device, group)
        self.transport = "p2p" if isinstance(self._x, _P2PExchange) else "nccl"
        # a single rank has nothing to exchange: its (local) collective exchange launches no collective and can be captured
        self.capturable = self._x.capturable or not multi

    @classmethod
    def for_rank(cls, graph, params, device, group=None, transport: str = "auto", rank: int | None = None, world: int | None = None):
        """The shard of this rank (or of ``rank`` of ``world``) with the edge-balanced blocks of :func:`gnn_blocks`."""
        multi = dist.is_available() and dist.is_initialized()
        world = world if world is not None else (dist.get_world_size(group) if multi else 1)
        rank = rank if rank is not None else (dist.get_rank(group) if multi else 0)
        return cls(graph.n, gnn_blocks(graph.rowptr, world)[rank], params, device, group, transport)

    def graph(self, graph):
        """This rank's row-block view of ``graph``."""
        return graph.row_block(self.g0, self.g1)

    def gather_coords(self, local: torch.Tensor) -> torch.Tensor:
        if local.shape != (self.g1 - self.g0, 3):
            raise ValueError(f"GnnRowShard.gather_coords: expected [{self.g1 - self.g0}, 3] block coordinates, got {list(local.shape)}")
        return _GatherCoords.apply(local, self)

    def reduce_grads(self, params=None) -> None:
        """Sum ``p.grad`` over the ranks for the shard's parameters (a missing gradient counts as zero and is created)."""
        params = self.params if params is None else list(params)
        if [p.numel() for p in params] != [p.numel() for p in self.params]:
            raise ValueError("GnnRowShard.reduce_grads: the parameters differ from those the shard was built for")
        for p in params:
            if p.grad is None:
                p.grad = torch.zeros_like(p)
        self._x.reduce([p.grad for p in params])


# ------------------------------------------------------------------------------ row-sharded per-step dSCC
class DsccExchange:
    """The two exchanges of a row-sharded dSCC evaluation (:class:`metrics.ShardedDsccMeter`):

    * :meth:`sum_hist`: ``hist_sum = sum over the ranks of hist`` (u64[nbins] distance or target histograms; integer counts, so exact
      and independent of the order);
    * :meth:`sum_cross`: ``cross_sum = sum over the ranks of cross`` (f64[2] block cross sums), added in rank order starting from 0.0,
      so the result is bit-identical on every rank and between the transports.

    The local buffers ``hist`` / ``cross`` are where this rank's block phases write; ``hist_sum`` / ``cross_sum`` hold the results.
    ``transport``: ``"p2p"`` (``hicgat_allreduce_u64_twoshot`` for the histogram; the two-shot partials kernel for the cross sums, which
    ride in its moment slot with a zero gradient part; both capturable), ``"nccl"`` (an int64 ``all_reduce`` of the histogram, and
    ``allreduce_packed`` of a ``[world, 2]`` buffer that is zero outside this rank's row, summed over the rows in rank order; with gloo
    on CPU tensors too; eager only) or ``"auto"`` (the rule of :class:`GnnRowShard`).  Without a multi-rank process group both steps
    are no-ops and the sums are the local buffers."""

    SLOTS_HIST = P2PShardedPairLoss.SLOT_BASE + 192   # the loss exchanges use SLOT_BASE + 0 .. + 127, the GNN exchanges + 128 .. + 191
    SLOTS_CROSS = P2PShardedPairLoss.SLOT_BASE + 224

    def __init__(self, nbins: int, device, group=None, transport: str = "auto"):
        if transport not in ("auto", "p2p", "nccl"):
            raise ValueError(f"DsccExchange: transport must be 'auto', 'p2p' or 'nccl', got {transport!r}")
        self.nbins, self.group = int(nbins), group
        multi = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
        self.world = dist.get_world_size(group) if multi else 1
        self.rank = dist.get_rank(group) if multi else 0
        self._p2p = False
        if transport == "p2p" or (transport == "auto" and multi and torch.device(device).type == "cuda"):
            try:
                self._init_p2p(device, group)
                self._p2p = True
            except Exception as e:  # no symmetric memory on this system: the collective exchange is equivalent
                if transport == "p2p":
                    raise
                import warnings

                warnings.warn(f"symmetric-memory exchange unavailable ({e!r}); using the NCCL all-reduce")
        if not self._p2p:
            self.hist = torch.zeros(self.nbins, dtype=torch.int64, device=device)
            self.cross = torch.zeros(2, dtype=torch.float64, device=device)
            self.hist_sum, self.cross_sum = self.hist, (self.cross if not multi else torch.zeros(2, dtype=torch.float64, device=device))
            self._rows = torch.zeros(self.world, 2, dtype=torch.float64, device=device) if multi else None
        self.multi = multi
        self.transport = "p2p" if self._p2p else "nccl"
        self.capturable = self._p2p or not multi

    def _init_p2p(self, device, group):
        import ctypes as C

        import torch.distributed._symmetric_memory as symm

        group = group if group is not None else dist.group.WORLD
        hbytes = (8 * self.nbins + 15) // 16 * 16
        # layout: [hist: hbytes | hist_sum: hbytes | cross partial: 64 moments + 16 zero gradient | cross result: 16]
        h_part, h_res, c_part = 0, hbytes, 2 * hbytes
        c_res = c_part + 80
        self.buf = symm.empty(c_res + 16, dtype=torch.uint8, device=device)
        self.buf.zero_()
        self.hdl = symm.rendezvous(self.buf, group)
        self.world, self.rank = self.hdl.world_size, self.hdl.rank
        if self.hdl.signal_pad_size < 4 * (self.SLOTS_CROSS + 32):
            raise RuntimeError("symmetric-memory signal pad too small")
        ptrs = [int(p) for p in self.hdl.buffer_ptrs]
        table = lambda off: (C.c_uint64 * self.world)(*[p + off for p in ptrs])
        self._h_part, self._h_res = table(h_part), table(h_res)
        self._c_part, self._c_res = table(c_part), table(c_res)
        self._pads = (C.c_uint64 * self.world)(*[int(p) for p in self.hdl.signal_pad_ptrs])
        self.hist = self.buf[h_part: h_part + 8 * self.nbins].view(torch.int64)
        self.hist_sum = self.buf[h_res: h_res + 8 * self.nbins].view(torch.int64)
        self.cross = self.buf[c_part: c_part + 16].view(torch.float64)    # moments 0, 1 of the partial; moments 2..7 stay zero
        self._moments = torch.zeros(N.PAIR_NMOM, dtype=torch.float64, device=device)
        self.cross_sum = self._moments[:2]
        self.state_h = torch.zeros(4, dtype=torch.int32, device=device)
        self.state_c = torch.zeros(4, dtype=torch.int32, device=device)
        torch.cuda.synchronize(device)
        dist.barrier(group)  # every rank's buffer is zeroed and mapped before the first signal

    def sum_hist(self) -> torch.Tensor:
        if self._p2p:
            N.check(N.lib().hicgat_allreduce_u64_twoshot(self._h_part, self._h_res, self._pads, self.rank, self.world, self.nbins, self.SLOTS_HIST,
                                                         self.state_h.data_ptr(), torch.cuda.current_stream().cuda_stream),
                    "hicgat_allreduce_u64_twoshot")
        elif self.multi:
            dist.all_reduce(self.hist, op=dist.ReduceOp.SUM, group=self.group)
        return self.hist_sum

    def sum_cross(self) -> torch.Tensor:
        if self._p2p:
            N.check(N.lib().hicgat_allreduce_partials_twoshot(self._c_part, self._c_res, self._pads, self.rank, self.world, 1, self.SLOTS_CROSS,
                                                              self.state_c.data_ptr(), None, self._moments.data_ptr(),
                                                              torch.cuda.current_stream().cuda_stream),
                    "hicgat_allreduce_partials_twoshot")
        elif self.multi:
            self._rows.zero_()
            self._rows[self.rank] = self.cross
            allreduce_packed(self._rows, self.group)   # x + 0 + ... + 0 = x: each row arrives exactly
            self.cross_sum.zero_()
            for r in range(self.world):                # rank order, from 0.0: the sum of the p2p kernel
                self.cross_sum += self._rows[r]
        return self.cross_sum
