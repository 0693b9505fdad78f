"""The hand-written tcgen05 TF32 GEMM (csrc/gemm.cu) and the 3xTF32 Linear built on it, against f64 matmul and against the cuBLAS
fp32 GEMM it replaces on large maps (torch.nn.Linear in the reference's MLP heads / GATConv projection, models.py:634-691)."""
import pytest
import torch

from helpers import rel_err

pytestmark = pytest.mark.gpu


# the last three are GATConv projections with H*C = 1024 (test_gpu_conv_shapes.py): the dx GEMM of 512 -> 1024 on 5 000 loci (K' = 3 072:
# two split-K partials over 40 M tiles), the forward of 512 -> 1024 at 9 970 loci (128 x 256 tiles, 4 N tiles) and of 128 -> 1024
@pytest.mark.parametrize("m,n,k", [(128, 128, 32), (300, 70, 100), (129, 257, 33), (1000, 512, 512), (4100, 256, 512), (49850, 512, 512), (20000, 3, 64),
                                   (5000, 512, 1024), (9970, 1024, 512), (5000, 1024, 128)])
def test_gemm_tf32x3_matches_f64(m, n, k):
    from hic_gnn_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(m + n + k)
    a = torch.randn(m, k, generator=g, device="cuda")
    b = torch.randn(n, k, generator=g, device="cuda") * 0.1
    bias = torch.randn(n, generator=g, device="cuda")
    got = ops.gemm_tf32_tn(ops.split_tf32(a, 0b100), ops.split_tf32(b, 0b010), bias)
    want = a.double() @ b.double().t() + bias.double()
    ref32 = torch.nn.functional.linear(a, b, bias)
    e, e32 = rel_err(got, want), rel_err(ref32, want)
    assert e < max(5e-6, 5 * e32), (e, e32)  # 3xTF32: ~2^-21 per product + the tensor core's accumulator rounding
    # the split itself: hi + lo reproduces the input to 2^-21, both parts are TF32-exact (13 low mantissa bits clear)
    s = ops.split_tf32(a, 0b100)
    kp = s.shape[1] // 3
    parts = s.view(m, kp // 32, 3, 32).permute(2, 0, 1, 3).reshape(3, m, kp)  # the three parts are interleaved per k-block of 32
    hi, lo = parts[0][:, :k], parts[2][:, :k]
    assert torch.equal(parts[1][:, :k], hi) and float(((hi + lo) - a).abs().max()) <= 2.0 ** -21 * float(a.abs().max())
    assert int((hi.contiguous().view(torch.int32) & 0x1FFF).abs().max()) == 0 and int((lo.contiguous().view(torch.int32) & 0x1FFF).abs().max()) == 0
    if kp > k:
        assert float(parts[:, :, k:].abs().max()) == 0.0  # reduction padding is zero


@pytest.mark.parametrize("rows,nout,nin", [(5000, 256, 512), (49850, 512, 512), (4096, 512, 256)])
def test_linear_tf32x3_forward_backward(rows, nout, nin):
    """All three GEMMs of a Linear layer (the weight gradient runs split-K over the rows) against f64 autograd."""
    from hic_gnn_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(rows)
    x = (0.5 * torch.randn(rows, nin, generator=g, device="cuda")).requires_grad_(True)
    lin = ops.Linear(nin, nout).cuda()
    gy = torch.randn(rows, nout, generator=g, device="cuda")
    assert rows >= ops.TF32X3_MIN_ROWS
    y = lin(x)
    gx, gw, gb = torch.autograd.grad((y * gy).sum(), [x, lin.weight, lin.bias])
    x64 = x.detach().double().requires_grad_(True)
    w64, b64 = lin.weight.detach().double().requires_grad_(True), lin.bias.detach().double().requires_grad_(True)
    y64 = torch.nn.functional.linear(x64, w64, b64)
    gx64, gw64, gb64 = torch.autograd.grad((y64 * gy.double()).sum(), [x64, w64, b64])
    y32 = torch.nn.functional.linear(x, lin.weight, lin.bias)
    gx32, gw32, gb32 = torch.autograd.grad((y32 * gy).sum(), [x, lin.weight, lin.bias])
    for name, got, want, ref in (("y", y, y64, y32), ("dx", gx, gx64, gx32), ("dW", gw, gw64, gw32), ("db", gb, gb64, gb32)):
        e, e32 = rel_err(got, want), rel_err(ref, want)
        assert e < max(5e-6, 5 * e32), (name, e, e32)
    # small maps keep the cuBLAS fp32 path (bit-identical with torch)
    xs = x[:100].detach()
    assert torch.equal(lin(xs), torch.nn.functional.linear(xs, lin.weight, lin.bias))
