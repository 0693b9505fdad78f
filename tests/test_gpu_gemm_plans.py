"""The tcgen05 3xTF32 GEMM (csrc/gemm.cu) at every branch of its tile plan, through the C ABI and ``ops``.

* Small-integer operands make every product and partial sum exact in fp32, whatever the order or truncation: a misplaced tile,
  row, column or k-block, or a write outside ``[m, n]``, changes an integer (``torch.equal`` against the exact product).
* Operands ``a = h + l 2^-20`` split into exactly ``hi = h``, ``lo = l 2^-20``: the main (hi.hi) sums and the cross sums are each
  exact in their own accumulator, so the result is pinned bit for bit to ``RN_f32(main + cross)`` per split and the f64 sum of
  the splits -- the two-accumulator routing and the split-K boundaries are checked exactly.
* Random operands whose rows span 10^-3..10^3 are bounded element by element on every production GEMM.
* ``hicgat_split_tf32`` is compared bit for bit with a host emulation of ``cvt.rna.tf32.f32``.
* The ``Linear`` layer against f64 autograd at the wide split-K dx shape, and the split memo of ``ops``.
"""
import numpy as np
import pytest
import torch

from gemm_plan import ALL_BRANCHES, ROWS, kpad, linear_gemms, plan_gemm

gpu = pytest.mark.gpu

# (m, n, K', kparts): together they reach every branch of plan_gemm (test_plans_cover_every_branch)
PLANS = [
    (129, 257, 96, 3),      # narrow, one split, m % 128 = 1, n % 32 and n % 4 tails (scalar epilogue)
    (33, 100, 96, 3),       # m < 128
    (127, 36, 96, 1),       # m < 128, plain TF32
    (4129, 300, 192, 3),    # m % 128 = 33
    (4223, 260, 288, 3),    # m % 128 = 127
    (1000, 512, 1536, 3),   # narrow split-K, split count by the tile rule, last split shorter (18, 18, 12 k-blocks)
    (4100, 256, 1536, 3),   # narrow split-K, equal splits
    (1000, 512, 1536, 1),   # plain TF32 split-K
    (50, 130, 1600, 1),     # plain TF32 split-K with a short last split, m < 128, n tails
    (9970, 1024, 1536, 3),  # wide, one split (GATConv H*C = 1024 forward at 9 970 loci)
    (9970, 512, 3072, 3),   # wide split-K, split count by the 16-main-block cap (its dx GEMM)
    (16385, 257, 192, 3),   # wide with an N tail of 1 column in the last 256-wide tile
    (16385, 257, 96, 1),    # same, plain TF32
    (2000, 500, 4800, 3),   # narrow, cap-set splits, last split shorter (48, 48, 48, 6)
]
PLAN_IDS = [f"{m}x{n}x{k}_kp{kp}" for m, n, k, kp in PLANS]


def test_plans_cover_every_branch():
    hit = set()
    for shape in PLANS:
        hit |= plan_gemm(*shape).branches()
    assert hit == ALL_BRANCHES, sorted(ALL_BRANCHES - hit)
    assert plan_gemm(9970, 512, 3072, 3).wide and plan_gemm(9970, 512, 3072, 3).ksplit == 2


def _lib():
    from hic_gnn_b200 import _native as N

    return N, N.lib()


def _gemm_raw(a, lda, b, ldb, m, n, k, kparts, bias, d_ptr, ldd, ws=None, ws_bytes=None):
    N, lib = _lib()
    if ws is None:
        need = lib.hicgat_gemm_tf32_workspace_bytes(m, n, k, kparts)
        ws = torch.empty(max(need, 16), dtype=torch.uint8, device="cuda")
    return lib.hicgat_gemm_tf32_tn(a, lda, b, ldb, m, n, k, kparts, None if bias is None else bias.data_ptr(), d_ptr, ldd, ws.data_ptr(),
                                   ws.numel() if ws_bytes is None else ws_bytes, torch.cuda.current_stream().cuda_stream)


def _padded(rows, cols, ld, fill, gen, lo=-4, hi=4):
    """[rows, ld] buffer: integers in [lo, hi] in the first ``cols`` columns, ``fill`` beyond."""
    buf = torch.full((rows, ld), fill, dtype=torch.float32, device="cuda")
    buf[:, :cols] = torch.randint(lo, hi + 1, (rows, cols), generator=gen, device="cuda").float()
    return buf


# ---------------------------------------------------------------------------------------------------- exact data movement
@gpu
@pytest.mark.parametrize("layout", ["dense", "padded", "padded_odd_ldd"])
@pytest.mark.parametrize("shape", PLANS, ids=PLAN_IDS)
def test_integer_operands_exact(shape, layout):
    """Exact integer product on every plan; ``lda``/``ldb`` > k with NaN in the unread columns; ``ldd`` > n with a NaN sentinel
    in columns n..ldd and around the output, which must survive; ``d`` 16 bytes into its allocation."""
    m, n, k, kparts = shape
    N, _ = _lib()
    g = torch.Generator(device="cuda").manual_seed(m * 7 + n * 3 + k + kparts)
    nan = float("nan")
    if layout == "dense":
        lda, ldb, ldd, off, with_bias = k, k, n, 0, False
    elif layout == "padded":
        lda, ldb, ldd, off, with_bias = k + 32, k + 4, (n + 3) // 4 * 4 + 4, 4, True
    else:  # ldd % 4 != 0: every row start but the first is misaligned, the epilogue must take its scalar path
        lda, ldb, ldd, off, with_bias = k + 4, k + 36, n + 1 if (n + 1) % 4 else n + 2, 4, True
    a = _padded(m, k, lda, nan, g)
    b = _padded(n, k, ldb, nan, g)
    bias = torch.randint(-100, 101, (n,), generator=g, device="cuda").float() if with_bias else None
    buf = torch.full((off + m * ldd + 64,), nan, dtype=torch.float32, device="cuda")
    d = buf[off:off + m * ldd].view(m, ldd)
    rc = _gemm_raw(a.data_ptr(), lda, b.data_ptr(), ldb, m, n, k, kparts, bias, d.data_ptr(), ldd)
    N.check(rc, "hicgat_gemm_tf32_tn")
    want = a[:, :k].double() @ b[:, :k].double().t()
    if bias is not None:
        want = want + bias.double()
    assert float(want.abs().max()) < 2 ** 24  # every partial sum is an integer below 2^24: exact in fp32
    assert torch.equal(d[:, :n], want.float())
    assert bool(torch.isnan(d[:, n:]).all()) and bool(torch.isnan(buf[:off]).all()) and bool(torch.isnan(buf[off + m * ldd:]).all())


# ---------------------------------------------------------------------------------------------------- accumulator routing
_S = 20  # lo = l * 2^-20 with |l| <= 255 stays below half a TF32 ulp of every h in [1, 15] (2^-12 for h = 1 - lo)


def _hl_source(rows, cols, gen):
    mag = torch.randint(1, 16, (rows, cols), generator=gen, device="cuda")
    sign = torch.randint(0, 2, (rows, cols), generator=gen, device="cuda") * 2 - 1
    h = (mag * sign).float()
    l = torch.randint(-255, 256, (rows, cols), generator=gen, device="cuda").float()
    return h, l * 2.0 ** -_S


def _parts(s, rows, k):
    kp = s.shape[1] // 3
    return s.view(rows, kp // 32, 3, 32).permute(2, 0, 1, 3).reshape(3, rows, kp)[:, :, :k]


@gpu
@pytest.mark.parametrize("shape", [(4223, 260, 288), (9970, 1024, 1536), (9970, 512, 3072), (1000, 512, 1536), (2000, 500, 4800)],
                         ids=["narrow", "wide", "wide_cap_split", "short_last_split", "cap_split_short_last"])
def test_accumulator_routing_exact(shape):
    """Per split, the main and cross accumulators are exact; the epilogue adds them round-to-nearest, the reduce sums the split
    partials in f64 in split order and adds the bias in fp32.  A cross-term block routed to the main accumulator (or a split
    boundary in the wrong place) rounds differently in most elements."""
    from hic_gnn_b200 import ops

    m, n, kk = shape
    k = kk // 3
    p = plan_gemm(m, n, kk, 3)
    g = torch.Generator(device="cuda").manual_seed(m + n + k)
    ha, la = _hl_source(m, k, g)
    hb, lb = _hl_source(n, k, g)
    a, b = ha + la, hb + lb
    assert torch.equal(a - ha, la) and torch.equal(b - hb, lb)  # the sources are exact in fp32
    bias = torch.randn(n, generator=g, device="cuda")
    As, Bs = ops.split_tf32(a, 0b100), ops.split_tf32(b, 0b010)
    pa, pb = _parts(As, m, k), _parts(Bs, n, k)
    assert torch.equal(pa[0], ha) and torch.equal(pa[1], ha) and torch.equal(pa[2], la)
    assert torch.equal(pb[0], hb) and torch.equal(pb[1], lb) and torch.equal(pb[2], hb)
    got = ops.gemm_tf32_tn(As, Bs, bias)

    blk = torch.arange(As.shape[1], device="cuda") // 32  # k-block of every column of the split operands
    total = torch.zeros(m, n, dtype=torch.float64, device="cuda")
    off_grid = 0.0
    for kb0, kb1 in p.split_ranges():
        sel = (blk >= kb0) & (blk < kb1)
        main_cols = sel & (blk % 3 == 0)
        cross_cols = sel & (blk % 3 != 0)
        main = As[:, main_cols].double() @ Bs[:, main_cols].double().t()
        cross = As[:, cross_cols].double() @ Bs[:, cross_cols].double().t()
        part = (main + cross).float()  # RN of the exact sum
        # how often one truncating accumulator would differ: the exact sum is not a float, and truncation != nearest
        rn = part.double()
        tr = torch.where(rn.abs() > (main + cross).abs(), torch.nextafter(part, torch.zeros_like(part)).double(), rn)
        off_grid = max(off_grid, float((tr != rn).double().mean()))
        total += rn
    want = total.float() + bias
    assert off_grid > 0.3, off_grid
    assert torch.equal(got, want), float((got.double() - want.double()).abs().max())


# ---------------------------------------------------------------------------------------------------- per-element accuracy
# Calibrated on a B200: max over the production shapes of |got - f64| / (2^-21 (1 + main k-blocks per accumulator) (|A| |B|^T)_ij).
# 2^-21 covers the 3xTF32 split (hi + lo and the dropped lo.lo), the main-block term the truncating accumulator (64 MMA steps of
# at most 2^-23 of the partial sum per 16 blocks).
C_ELEM = 1.0


def _bound_ratio(got, A, B, p):
    want = A.double() @ B.double().t()
    S = A.double().abs() @ B.double().abs().t()
    scale = 2.0 ** -21 * (1 + p.main_blocks_per_acc)
    err = (got.double() - want).abs()
    zero = S == 0
    assert bool((err[zero] == 0).all())
    return float((err[~zero] / (scale * S[~zero])).max())


def _rows_spanning(rows, cols, gen, zero_frac=0.0):
    x = torch.randn(rows, cols, generator=gen, device="cuda")
    x *= 10.0 ** (6 * torch.rand(rows, 1, generator=gen, device="cuda") - 3)
    if zero_frac:
        x[torch.rand(rows, generator=gen, device="cuda") < zero_frac] = 0.0  # rows a ReLU zeroed
    return x


_PRODUCTION = sorted({(rows, nin, nout) for rows in ROWS for nin, nout in ((512, 512), (512, 256), (512, 1024))})


@gpu
@pytest.mark.parametrize("rows,nin,nout", _PRODUCTION)
def test_production_gemms_elementwise(rows, nin, nout):
    """The three GEMMs of every Linear that runs on the tensor cores (weight >= 100 000 elements), including the wide split-K dx of
    512 -> 1024 at 9 970 and 49 850 loci, with the operands laid out as ``ops._Linear3xTF32`` splits them."""
    from hic_gnn_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(rows + nin + nout)
    x = _rows_spanning(rows, nin, g, zero_frac=0.1)
    w = _rows_spanning(nout, nin, g) * 0.05
    gy = _rows_spanning(rows, nout, g)
    ratios = {}
    for name, m, n, kk in linear_gemms(rows, nin, nout):
        p = plan_gemm(m, n, kk, 3)
        if name == "fwd":
            got, A, B = ops.gemm_tf32_tn(ops.split_tf32(x, 0b100), ops.split_tf32(w, 0b010)), x, w
        elif name == "dx":
            got, A, B = ops.gemm_tf32_tn(ops.split_tf32(gy, 0b100), ops.split_tf32(w, 0b010, transpose=True)), gy, w.t()
        else:
            got, A, B = ops.gemm_tf32_tn(ops.split_tf32(gy, 0b100, transpose=True), ops.split_tf32(x, 0b010, transpose=True)), gy.t(), x.t()
        ratios[name] = (_bound_ratio(got, A, B, p), p.wide, p.ksplit)
    print(f"elementwise ratio rows={rows} {nin}->{nout}: {ratios}")
    assert all(r <= C_ELEM for r, _, _ in ratios.values()), ratios


# ---------------------------------------------------------------------------------------------------- reproducibility, refusals
@gpu
@pytest.mark.parametrize("shape", PLANS, ids=PLAN_IDS)
def test_two_launches_bit_identical(shape):
    m, n, k, kparts = shape
    N, _ = _lib()
    g = torch.Generator(device="cuda").manual_seed(m + n + k)
    a = torch.randn(m, k, generator=g, device="cuda")
    b = torch.randn(n, k, generator=g, device="cuda")
    a, b = _rna(a), _rna(b)  # TF32-exact operands (what the ABI requires)
    bias = torch.randn(n, generator=g, device="cuda")
    outs = []
    for _ in range(2):
        d = torch.empty(m, n, dtype=torch.float32, device="cuda")
        N.check(_gemm_raw(a.data_ptr(), k, b.data_ptr(), k, m, n, k, kparts, bias, d.data_ptr(), n), "hicgat_gemm_tf32_tn")
        outs.append(d)
    assert torch.equal(outs[0], outs[1])
    assert bool(torch.isfinite(outs[0]).all())


@gpu
def test_abi_refusals():
    N, lib = _lib()
    m, n = 256, 256
    a = torch.zeros(m, 4 * 96, device="cuda")
    b = torch.zeros(n, 4 * 96, device="cuda")
    d = torch.zeros(m, n + 4, device="cuda")

    def refused(rc, text):
        assert rc != 0
        msg = lib.hicgat_last_error().decode()
        assert text in msg, msg

    refused(_gemm_raw(a.data_ptr(), 384, b.data_ptr(), 384, m, n, 48, 1, None, d.data_ptr(), n), "k must be a multiple of 32 * kparts")
    refused(_gemm_raw(a.data_ptr(), 384, b.data_ptr(), 384, m, n, 64, 3, None, d.data_ptr(), n), "k must be a multiple of 32 * kparts")
    refused(_gemm_raw(a.data_ptr(), 384, b.data_ptr(), 384, m, n, 96, 2, None, d.data_ptr(), n), "kparts 1 or 3")
    refused(_gemm_raw(a.data_ptr() + 4, 384, b.data_ptr(), 384, m, n, 96, 3, None, d.data_ptr(), n), "16-byte aligned")
    refused(_gemm_raw(a.data_ptr(), 384, b.data_ptr() + 8, 384, m, n, 96, 3, None, d.data_ptr(), n), "16-byte aligned")
    refused(_gemm_raw(a.data_ptr(), 384, b.data_ptr(), 384, m, n, 96, 3, None, d.data_ptr() + 4, n), "16-byte aligned")
    refused(_gemm_raw(a.data_ptr(), 383, b.data_ptr(), 384, m, n, 96, 3, None, d.data_ptr(), n), "multiples of 4")
    refused(_gemm_raw(a.data_ptr(), 384, b.data_ptr(), 386, m, n, 96, 3, None, d.data_ptr(), n), "multiples of 4")
    # a split-K plan: the workspace is checked against the plan's partial buffer
    m2, n2, k2 = 1000, 512, 1536
    need = lib.hicgat_gemm_tf32_workspace_bytes(m2, n2, k2, 3)
    assert need == plan_gemm(m2, n2, k2, 3).workspace_bytes > 0
    a2, b2, d2 = torch.zeros(m2, k2, device="cuda"), torch.zeros(n2, k2, device="cuda"), torch.zeros(m2, n2, device="cuda")
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    refused(_gemm_raw(a2.data_ptr(), k2, b2.data_ptr(), k2, m2, n2, k2, 3, None, d2.data_ptr(), n2, ws, need - 16), "workspace too small")
    N.check(_gemm_raw(a2.data_ptr(), k2, b2.data_ptr(), k2, m2, n2, k2, 3, None, d2.data_ptr(), n2, ws, need), "hicgat_gemm_tf32_tn")
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------- the split, bit for bit
def _rna_bits(bits: np.ndarray) -> np.ndarray:
    """cvt.rna.tf32.f32 on finite values: add half a TF32 ulp to the magnitude's bit pattern and clear the 13 low bits."""
    u = bits.astype(np.uint32)
    finite = (u & 0x7F800000) != 0x7F800000
    return np.where(finite, (u + 0x1000) & np.uint32(0xFFFFE000), u).astype(np.uint32)


def _rna(t: torch.Tensor) -> torch.Tensor:
    bits = t.contiguous().view(torch.int32)
    return ((bits + 0x1000) & -8192).view(torch.float32)


def _host_split(src: np.ndarray, pattern: int, transpose: bool) -> np.ndarray:
    a = src.astype(np.float32)
    hi = _rna_bits(a.view(np.uint32)).view(np.float32)
    with np.errstate(invalid="ignore", over="ignore"):
        lo = _rna_bits((a - hi).astype(np.float32).view(np.uint32)).view(np.float32)
    if transpose:
        hi, lo = hi.T, lo.T
    rows, red = hi.shape
    kp = kpad(red)
    out = np.zeros((rows, kp // 32, 3, 32), dtype=np.float32)
    for p in range(3):
        part = np.zeros((rows, kp), dtype=np.float32)
        part[:, :red] = lo if (pattern >> p) & 1 else hi
        out[:, :, p, :] = part.reshape(rows, kp // 32, 32)
    return out.reshape(rows, 3 * kp)


def _special_values(rows, cols, seed):
    """Random normals over 10^+-30, mantissa-all-ones carries, exact ties, subnormals, +-0 and values just below the TF32
    overflow threshold, mixed per element."""
    rng = np.random.default_rng(seed)
    n = rows * cols
    kind = rng.integers(0, 6, n)
    sign = np.where(rng.integers(0, 2, n) == 1, np.uint32(0x80000000), np.uint32(0))
    normal = (rng.standard_normal(n) * 10.0 ** rng.uniform(-30, 30, n)).astype(np.float32).view(np.uint32)
    ones = (rng.integers(1, 254, n).astype(np.uint32) << 23) | np.uint32(0x7FFFFF)
    tie = (rng.integers(1, 254, n).astype(np.uint32) << 23) | (rng.integers(0, 1 << 10, n).astype(np.uint32) << 13) | np.uint32(0x1000)
    sub = rng.integers(1, 1 << 23, n).astype(np.uint32)
    big = rng.choice(np.array([0x7F7FEFFF, 0x7F7FE000, 0x7F7FE001, 0x7F7FDFFF], dtype=np.uint32), n)
    bits = np.select([kind == 0, kind == 1, kind == 2, kind == 3, kind == 4], [normal, ones, tie, sub, np.zeros(n, np.uint32)], big)
    return (bits | sign).astype(np.uint32).view(np.float32).reshape(rows, cols)


@gpu
@pytest.mark.parametrize("transpose", [0, 1])
@pytest.mark.parametrize("cols", [1, 31, 32, 33, 1000])
@pytest.mark.parametrize("rows", [1, 31, 32, 33, 1000])
def test_split_matches_host_emulation(rows, cols, transpose):
    N, lib = _lib()
    src = _special_values(rows, cols, rows * 1009 + cols * 7 + transpose)
    for ld in (cols, cols + 3):
        buf = torch.full((rows, ld), float("nan"), dtype=torch.float32)
        buf[:, :cols] = torch.from_numpy(src)
        dev = buf.cuda()
        for pattern in range(8):
            want = _host_split(src, pattern, bool(transpose))
            out = torch.full(want.shape, float("nan"), dtype=torch.float32, device="cuda")
            N.check(lib.hicgat_split_tf32(dev.data_ptr(), rows, cols, ld, out.data_ptr(), pattern, transpose, torch.cuda.current_stream().cuda_stream),
                    "hicgat_split_tf32")
            got = out.cpu().numpy()
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (ld, pattern, int((got.view(np.uint32) != want.view(np.uint32)).sum()))


@gpu
def test_split_overflows_at_the_tf32_rounding_threshold():
    """|a| >= (2 - 2^-11) 2^127 rounds to a TF32 ``hi`` of inf (and ``lo`` = -inf): the 3xTF32 product of such an input is not
    finite where the fp32 GEMM is.  The domain the header documents is |a| < (2 - 2^-11) 2^127; just below it the split is exact."""
    from hic_gnn_b200 import ops

    bits = np.array([0x7F7FEFFF, 0x7F7FF000, 0x7F7FFFFF, 0xFF7FEFFF, 0xFF7FF000, 0xFF7FFFFF], dtype=np.uint32)
    src = bits.view(np.float32).reshape(1, -1)
    s = ops.split_tf32(torch.from_numpy(src.copy()).cuda(), 0b100).cpu().numpy()
    assert np.array_equal(s.view(np.uint32), _host_split(src, 0b100, False).view(np.uint32))
    hi, lo = s[0, :6], s[0, 64:70]
    assert hi[0] == np.float32(2.0 ** 127 * (2 - 2.0 ** -10)) and hi[3] == -hi[0] and np.isfinite(lo[[0, 3]]).all()
    assert (hi[[1, 2]] == np.inf).all() and (lo[[1, 2]] == -np.inf).all()
    assert (hi[[4, 5]] == -np.inf).all() and (lo[[4, 5]] == np.inf).all()


# ---------------------------------------------------------------------------------------------------- the Linear layer
def _f64_grads(x, weight, bias, gy):
    x64 = x.detach().double().requires_grad_(True)
    w64 = weight.detach().double().requires_grad_(True)
    b64 = None if bias is None else bias.detach().double().requires_grad_(True)
    y64 = torch.nn.functional.linear(x64, w64, b64)
    grads = torch.autograd.grad((y64 * gy.double()).sum(), [x64, w64] + ([b64] if b64 is not None else []))
    return y64, grads


@gpu
@pytest.mark.parametrize("variant", ["bias", "no_bias", "noncontiguous_x"])
def test_linear_512_1024_against_f64_autograd(variant):
    """``Linear(512, 1024)`` on 9 970 rows: its dx GEMM is the wide split-K plan (128 x 256 tiles, two cap-set splits)."""
    from hic_gnn_b200 import ops

    rows, nin, nout = 9970, 512, 1024
    assert plan_gemm(rows, nin, 3 * nout, 3).wide and plan_gemm(rows, nin, 3 * nout, 3).ksplit == 2
    g = torch.Generator(device="cuda").manual_seed(9970)
    torch.manual_seed(1)
    lin = ops.Linear(nin, nout, bias=variant != "no_bias").cuda()
    x0 = _rows_spanning(rows, nin, g, zero_frac=0.1)
    if variant == "noncontiguous_x":
        x = torch.empty(nin, rows, device="cuda").t()
        x.copy_(x0)
        assert not x.is_contiguous()
    else:
        x = x0.clone()
    x.requires_grad_(True)
    gy = _rows_spanning(rows, nout, g)
    y = lin(x)
    params = [x, lin.weight] + ([lin.bias] if lin.bias is not None else [])
    grads = torch.autograd.grad((y * gy).sum(), params)
    y64, grads64 = _f64_grads(x, lin.weight, lin.bias, gy)
    xd, wd = x.detach(), lin.weight.detach()
    checks = [("y", y, xd, wd, plan_gemm(rows, nout, 3 * kpad(nin), 3)), ("dx", grads[0], gy, wd.t(), plan_gemm(rows, nin, 3 * kpad(nout), 3)),
              ("dW", grads[1], gy.t(), xd.t(), plan_gemm(nout, nin, 3 * kpad(rows), 3))]
    for name, got, A, B, p in checks:
        if name == "y" and lin.bias is not None:  # the bias is added in fp32 to the rounded product: one more rounding of |y|
            S = A.double().abs() @ B.double().abs().t()
            err = (got.double() - y64.detach()).abs()
            tol = C_ELEM * 2.0 ** -21 * (1 + p.main_blocks_per_acc) * S + 2.0 ** -24 * got.detach().double().abs()
            assert bool((err <= tol).all()), (name, float((err / tol.clamp(min=1e-300)).max()))
        else:
            assert _bound_ratio(got, A, B, p) <= C_ELEM, name
    if lin.bias is not None:
        gb, gb64 = grads[2].double(), grads64[2]
        assert float(((gb - gb64).abs() / gy.double().abs().sum(0)).max()) < 1e-6


@gpu
def test_linear_dispatch_boundaries():
    """4 095 rows or a weight of 99 840 elements stay on the fp32 GEMM of torch, bit-identical with ``F.linear``; 4 096 rows with
    100 096 weight elements run the tensor-core GEMM."""
    from hic_gnn_b200 import _native as N
    from hic_gnn_b200 import ops

    torch.manual_seed(3)
    cases = [(4095, 391, 256, False), (4096, 391, 256, True), (4096, 390, 256, False), (4095, 390, 256, False)]
    for rows, nin, nout, tc in cases:
        lin = ops.Linear(nin, nout).cuda()
        assert (lin.weight.numel() >= 100000) == (nin == 391)
        x = torch.randn(rows, nin, device="cuda")
        l0 = N.launch_count()
        y = lin(x)
        torch.cuda.synchronize()
        assert (N.launch_count() > l0) == tc, (rows, nin)  # the splits and the GEMM count as library launches
        ref = torch.nn.functional.linear(x, lin.weight, lin.bias)
        if tc:
            assert float((y.double() - ref.double()).abs().max() / ref.double().abs().max()) < 5e-6
        else:
            assert torch.equal(y, ref), (rows, nin)


# ---------------------------------------------------------------------------------------------------- the split memo of ops
class _SplitCounter:
    """Wraps the ctypes entry ``hicgat_split_tf32`` and records ``(source address, transpose)`` of every launch."""

    def __init__(self, monkeypatch):
        N, lib = _lib()
        self.calls = []
        real = lib.hicgat_split_tf32

        def counted(src, rows, cols, ld, dst, pattern, transpose, stream):
            self.calls.append((src, transpose))
            return real(src, rows, cols, ld, dst, pattern, transpose, stream)

        monkeypatch.setattr(lib, "hicgat_split_tf32", counted)

    def of(self, t, transpose=0):
        return sum(1 for src, tr in self.calls if src == t.data_ptr() and tr == transpose)


@gpu
def test_memo_splits_constant_features_once(monkeypatch):
    from hic_gnn_b200 import ops

    torch.manual_seed(5)
    lin = ops.Linear(512, 256).cuda()
    x = torch.randn(4096, 512, device="cuda")  # constant input features
    count = _SplitCounter(monkeypatch)
    with torch.no_grad():
        y1 = lin(x)
        y2 = lin(x)
    assert torch.equal(y1, y2)
    assert count.of(x) == 1, count.calls
    for _ in range(2):  # training steps: the forward split and the transposed split of the weight-gradient GEMM, once each
        lin(x).sum().backward()
    assert count.of(x) == 1 and count.of(x, 1) == 1, count.calls


@gpu
def test_memo_shares_one_split_between_layers_reading_one_activation(monkeypatch):
    """densea / align_densea of the GAT net read the same activation: one split for both, with and without autograd."""
    from hic_gnn_b200 import models

    torch.manual_seed(6)
    model = models.GATNetSelectiveResidualsUpdated().cuda()
    w = torch.randn(512, 512, device="cuda", requires_grad=True)
    feats = torch.randn(4096, 512, device="cuda")
    count = _SplitCounter(monkeypatch)
    h = torch.relu(feats @ w)  # an activation that requires grad
    a, b = model.align_densea(h), model.densea(h)
    assert count.of(h) == 1, count.calls
    (a.sum() + b.sum()).backward()
    assert count.of(h, 1) == 1, count.calls  # and the two weight-gradient GEMMs share its transposed split
    with torch.no_grad():
        h2 = torch.relu(feats @ w)
        model.align_densea(h2), model.densea(h2)
    assert count.of(h2) == 1, count.calls


@gpu
def test_captured_backward_owns_its_splits():
    """A graph captured after an eager split of constant features must not read that split's buffer: after the memo is cleared
    and the block is handed to a NaN-filled tensor on the same stream, a replay still equals the eager result."""
    from hic_gnn_b200 import ops

    torch.manual_seed(7)
    lin = ops.Linear(512, 256).cuda()
    x = torch.randn(4096, 512, device="cuda")  # constant: the memo keeps its splits
    gy = torch.randn(4096, 256, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        # 1. eager forward + backward: the memo holds the transposed split of x (the weight-gradient operand)
        gw_eager = torch.autograd.grad(lin(x), lin.weight, gy)[0]
        before = {v[1].data_ptr(): tuple(v[1].shape) for v in ops._split_cache.values()}
        assert before, "the eager Linear left no split in the memo"
        # 2. capture the Linear forward + backward on the same stream
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            gw_static = torch.autograd.grad(lin(x), lin.weight, gy)[0]
        # 3. clear the memo and drop every reference to its buffers
        ops._split_cache.clear()
        # 4. same-size NaN tensors on the same stream: one of them must take a freed block
        fills = [torch.full(shape, float("nan"), device="cuda") for shape in before.values() for _ in range(2)]
        reused = {f.data_ptr() for f in fills} & set(before)
        assert reused, "inconclusive: no freed split buffer was reused"
        # 5. replay and compare with eager
        graph.replay()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    assert torch.equal(gw_static, gw_eager), float((gw_static - gw_eager).abs().max())
    del fills


@gpu
def test_graphed_training_gradients_with_eager_forwards_between_replays():
    """A graphed GAT-net training step at 5 000 loci (the GATConv projection runs its 3xTF32 GEMMs), with four eager no-grad
    forwards between replays: after each replay every parameter gradient equals an eager backward from the parameters the
    replay started from."""
    import copy

    from hic_gnn_b200 import models, ops, synth, train
    from hic_gnn_b200.graph import CSRGraph
    from helpers import rel_err

    n = 5000
    adj = synth.synthetic_map_chunked(n, 0.05, device="cuda")
    _, target = ops.cont2dist(adj, 1.0, want_f64=False, want_f32=True, symmetric=True)
    rowptr, col, val = ops.csr_from_dense(adj)
    graph = CSRGraph(rowptr, col, val, n)
    del adj
    x = synth.synthetic_features(n, device="cuda")
    torch.manual_seed(42)
    model = models.GATNetSelectiveResidualsUpdated().cuda()
    step = train.TrainStep(model, x, graph, target, mode="mse_pearson", lr=1e-3, use_cuda_graph=True)
    for it in range(3):
        for _ in range(4):
            with torch.no_grad():
                model.get_model(x, graph)
        ref = copy.deepcopy(model)  # the parameters this replay starts from
        step()
        torch.cuda.synchronize()
        ref.zero_grad(set_to_none=True)
        loss, _, _ = train.step_loss(ref, x, graph, target, "mse_pearson")
        loss.backward()
        for (name, p), q in zip(model.named_parameters(), ref.parameters()):
            assert p.grad is not None and q.grad is not None, name
            assert rel_err(p.grad, q.grad) <= 1e-6, (it, name, rel_err(p.grad, q.grad))
