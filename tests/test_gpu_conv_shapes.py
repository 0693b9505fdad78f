"""The GAT and SAGE message-passing kernels at every (heads, channels) and feature width they are compiled for, against an f64
reference of the same operation.

conv.cu instantiates the GAT kernels for eight (H, Q = H*C/128) pairs and gat_dense.cu maps heads and 128-column tiles onto its
grid; the rest of the suite only runs (2, 256).  The cases here cover all eight pairs with every input width, both backward
variants of the CSR path, its 16-rows-per-CTA launch and the dense-tile path with and without split-K, on patterns built to hit
the short-row tails of the 4-at-a-time gather (degrees 1-6, 32-34, 128-130 after ``set_diag``), an isolated locus, a hub, an
edgeless graph and tiny n.  Errors are measured per head and per degree class, each against its own slice's maximum, so that a
mistake confined to one head or to the short rows is not hidden under the largest values of the tensor."""
import pytest
import torch
import torch.nn.functional as F

from helpers import rel_err, small_map

pytestmark = pytest.mark.gpu
TOL, GTOL = 1e-5, 2e-5   # the suite's forward / gradient tolerances (test_gpu_conv.py)
SLOPE = 0.2
SHAPES = [(1, 128), (1, 256), (1, 512), (2, 128), (2, 256), (2, 512), (4, 128), (4, 256)]
F_INS = [128, 256, 512]
DEGREES = [1, 2, 3, 4, 5, 6, 32, 33, 34, 128, 129, 130]   # row lengths after set_diag


# ------------------------------------------------------------------------------------------------ graphs (dense f64 adjacency, CPU)
def degree_pattern(seed: int = 0) -> torch.Tensor:
    """Symmetric, duplicate-free contact map whose rows have, after ``set_diag``, exactly the lengths in ``DEGREES`` (at least 8 rows
    each), plus one hub adjacent to every locus that is not isolated.  A class of degree d >= 2 is the hub, the self loop and a
    (d - 2)-regular circulant on its own rows.  Loci are shuffled so that one CTA mixes row lengths; values are positive counts."""
    g = torch.Generator().manual_seed(seed)
    blocks, n = [], 0
    for d in DEGREES:
        k = max(d - 2, 0)
        m = max(8, k + 1)
        if k % 2 and m % 2:
            m += 1
        blocks.append((d, n, m, k))
        n += m
    hub = n
    n += 1
    a = torch.zeros(n, n, dtype=torch.float64)
    for d, r0, m, k in blocks:
        idx = torch.arange(m)
        offsets = list(range(1, k // 2 + 1)) + ([m // 2] if k % 2 else [])
        for o in offsets:
            a[r0 + idx, r0 + (idx + o) % m] = 1.0
            a[r0 + (idx + o) % m, r0 + idx] = 1.0
        if d >= 2:
            a[hub, r0:r0 + m] = a[r0:r0 + m, hub] = 1.0
    vals = 0.5 + torch.rand(n, n, generator=g, dtype=torch.float64)
    a = a * torch.triu(vals, 1) + (a * torch.triu(vals, 1)).t()
    perm = torch.randperm(n, generator=g)
    return a[perm][:, perm].contiguous()


def star(n: int) -> torch.Tensor:
    a = torch.zeros(n, n, dtype=torch.float64)
    a[0, 1:] = a[1:, 0] = 1.0
    return a


def banded(n: int, width: int) -> torch.Tensor:
    i = torch.arange(n)
    s = (i.unsqueeze(1) - i.unsqueeze(0)).abs()
    return ((s > 0) & (s <= width)).double()


GRAPHS = {
    "edgeless": lambda: torch.zeros(37, 37, dtype=torch.float64),
    "n1": lambda: torch.zeros(1, 1, dtype=torch.float64),
    "n2": lambda: star(2),
    "star7": lambda: star(7),            # a hub whose row holds all n loci
    "random1003": lambda: small_map(1003, 0.05, seed=5),
}


def _load(adj: torch.Tensor, x: torch.Tensor):
    from hic_gnn_b200 import utils as gutils

    return gutils.load_input(adj.numpy().copy(), x.numpy()).edge_index


def _self_loop_csr(graph):
    """(rowptr, col) int64 of set_diag(pattern) on the device and the row lengths (= degree classes) on the host."""
    r32, c32, _ = graph.with_self_loops()
    rowptr, col = r32.long(), c32.long()
    return rowptr, col, (rowptr[1:] - rowptr[:-1]).cpu()


def _degree_classes(deg: torch.Tensor) -> dict:
    """Row indices per row length; lengths outside ``DEGREES`` are grouped by power of two."""
    key = torch.where(torch.isin(deg, torch.tensor(DEGREES)), deg, 1000 + torch.log2(deg.double()).floor().long())
    return {int(k): torch.nonzero(key == k).flatten() for k in torch.unique(key)}


# ------------------------------------------------------------------------------------------------ f64 reference
def gat_reference(x, weight, att_l, att_r, bias, rowptr, col, heads: int, gout, slope: float = SLOPE, budget: int = 1 << 25):
    """torch-geometric 1.7.2 GATConv (concat, one shared projection, ``set_diag`` self loops, softmax ``exp(e - max) / (sum +
    1e-16)``) in f64 on the device, literal message/aggregate order over the self-loop edge list ``(rowptr, col)``, chunked over
    target rows so that no chunk holds more than ``budget`` message elements.  Returns ``out``, the gradients of
    ``(out * gout).sum()`` for x, the projection weight, att_l, att_r and bias, and the size of the terms the att gradients are
    summed from (see :func:`_check`).  The row max is a constant of the softmax and is detached (its derivative vanishes
    identically)."""
    n = x.shape[0]
    HC = weight.shape[0]
    H, C = heads, HC // heads
    f64 = dict(dtype=torch.float64, device=x.device)
    leaves = [t.detach().double().requires_grad_(True) for t in (x, weight, att_l.reshape(1, H, C), att_r.reshape(1, H, C), bias)]
    x64, w64, al64, ar64, b64 = leaves
    g64 = gout.double()
    out = torch.empty(n, HC, **f64)
    grads = [torch.zeros_like(t) for t in leaves]
    mag_src, mag_dst = torch.zeros(n, H, **f64), torch.zeros(n, H, **f64)
    per_chunk = max(budget // HC, 1)
    rp = rowptr.cpu()
    r0 = 0
    while r0 < n:
        r1 = int(torch.searchsorted(rp, rp[r0] + per_chunk, right=True)) - 1
        r1 = min(max(r1, r0 + 1), n)
        k0, k1 = int(rp[r0]), int(rp[r1])
        row = torch.repeat_interleave(torch.arange(r1 - r0, device=x.device), rowptr[r0 + 1:r1 + 1] - rowptr[r0:r1])
        c = col[k0:k1]
        xl = (x64 @ w64.t()).view(n, H, C)
        a_src, a_dst = (xl * al64).sum(-1), (xl * ar64).sum(-1)
        e = F.leaky_relu(a_src[c] + a_dst[r0 + row], slope)
        m = torch.full((r1 - r0, H), float("-inf"), **f64)
        m = m.scatter_reduce(0, row.unsqueeze(1).expand(-1, H), e.detach(), reduce="amax", include_self=True)
        p = (e - m[row]).exp()
        s = torch.zeros(r1 - r0, H, **f64).index_add(0, row, p)
        a = p / (s[row] + 1e-16)
        o = torch.zeros(r1 - r0, H, C, **f64).index_add(0, row, xl[c] * a.unsqueeze(-1))
        o = o.reshape(r1 - r0, HC) + b64
        out[r0:r1] = o.detach()
        for acc, gr in zip(grads, torch.autograd.grad(o, leaves, grad_outputs=g64[r0:r1])):
            acc += gr
        with torch.no_grad():  # dz_ij = a_ij (<g_i, xl_j> - <g_i, out_i - bias>) x slope, per head: the size of its terms
            ag = g64[r0:r1].abs().view(-1, H, C)
            rowterm = (ag * (o - b64).abs().view(-1, H, C)).sum(-1)
            terms = a * ((ag[row] * xl[c].abs()).sum(-1) + rowterm[row])
            mag_dst.index_add_(0, r0 + row, terms)
            mag_src.index_add_(0, c, terms)
        r0 = r1
    with torch.no_grad():
        xa = (x64 @ w64.t()).abs().view(n, H, C)
        scale = {"att_l": (mag_src.unsqueeze(-1) * xa).sum(0), "att_r": (mag_dst.unsqueeze(-1) * xa).sum(0)}   # [H, C]
    return out, dict(zip(["x", "W", "att_l", "att_r", "bias"], grads)), scale


# ------------------------------------------------------------------------------------------------ layer set-up and runs
def _make_case(H, C, f_in, adj, seed=0):
    """GATConv(f_in, C, heads=H) + inputs whose edge logits z_ij = a_src[j] + a_dst[i] all stay far from the LeakyReLU kink.

    With ~1e6 edges x 4 heads (the near-dense cases), the sharpened random parameters ``_gat_case`` scans put several logits within
    f32 rounding of 0 for almost every seed, and each such edge takes the other slope in f32 than in f64 and moves its rows'
    gradients by ~1e-4.  So the logits are built to keep away from 0 (the construction of ``_kink_free_gat``, with an independent
    sign per head): input feature h < H carries +-3 per locus and is routed, alone, into channel 0 of head h, where att_l picks it
    up; the rest of each head is random with a 0.2 spread.  Every row then mixes sources on the 0.2 slope (negative sign) with
    sources on slope 1, per head differently.  The minimum |z| over all edges and heads is checked in f64."""
    from hic_gnn_b200 import layers as glayers

    n = adj.shape[0]
    g = torch.Generator().manual_seed(1000 + seed)
    x = 0.25 * torch.randn(n, f_in, generator=g)
    sign = torch.where(torch.rand(n, H, generator=g) < 0.5, -1.0, 1.0)
    x[:, :H] = 3.0 * sign
    torch.manual_seed(seed)
    gc = glayers.GATConv(f_in, C, heads=H)
    with torch.no_grad():
        W = gc.lin_l.weight                       # [H*C, f_in]
        W[:, :H] = 0.0
        for h in range(H):
            W[h * C, :] = 0.0
            W[h * C, h] = 1.0
        gc.bias.uniform_(-0.1, 0.1, generator=g)
        xl = (x @ W.t()).view(n, H, C)
        for att, special in ((gc.att_l, 1.0), (gc.att_r, 0.0)):
            att.normal_(0.0, 1.0, generator=g)
            for h in range(H):
                att[0, h, 0] = 0.0
                rms = float((xl[:, h, 1:] * att[0, h, 1:]).sum(-1).pow(2).mean().sqrt())
                att[0, h, 1:] *= 0.2 / rms
                att[0, h, 0] = special
    gc = gc.cuda()
    graph = _load(adj, x)
    rowptr, col, deg = _self_loop_csr(graph)
    with torch.no_grad():
        xl64 = (x.cuda().double() @ gc.lin_l.weight.double().t()).view(n, H, C)
        a_src, a_dst = (xl64 * gc.att_l.double()).sum(-1), (xl64 * gc.att_r.double()).sum(-1)
        row = torch.repeat_interleave(torch.arange(n, device="cuda"), rowptr[1:] - rowptr[:-1])
        gap = float((a_src[col] + a_dst[row]).abs().min())
    assert gap > 0.5, gap
    w = torch.randn(n, H * C, generator=g).cuda()
    return gc, x.cuda(), graph, (rowptr, col, deg), w


def _run(gc, x, graph, w, path, backward="fused"):
    from hic_gnn_b200 import layers as glayers

    gc.path = path
    old = glayers.GAT_BACKWARD
    glayers.GAT_BACKWARD = backward
    try:
        xg = x.clone().requires_grad_(True)
        y = gc(xg, graph)
        grads = torch.autograd.grad((y * w).sum(), [xg, gc.lin_l.weight, gc.att_l, gc.att_r, gc.bias])
    finally:
        glayers.GAT_BACKWARD = old
    return y.detach(), dict(zip(["x", "W", "att_l", "att_r", "bias"], grads))


def _run_16_rows(gc, x, graph, w):
    from hic_gnn_b200 import _native as N

    try:
        N.check(N.lib().hicgat_gat_set_tuning(16, 0), "hicgat_gat_set_tuning")
        return _run(gc, x, graph, w, "csr", "fused")
    finally:
        N.check(N.lib().hicgat_gat_set_tuning(8, 0), "hicgat_gat_set_tuning")


def _slice_err(got, want, rows=None, cols=None):
    if rows is not None:
        got, want = got[rows], want[rows]
    if cols is not None:
        got, want = got[:, cols], want[:, cols]
    return rel_err(got, want) if want.numel() else 0.0


def _check(label, got, want, H, C, deg):
    """Output per (degree class, head), dx per degree class, dW / att / bias per head -- each slice against its own maximum.

    The att gradients sum, over edges, dz_ij = a_ij (<g_i, xl_j> - <g_i, out_i - bias>) x slope, whose row sums cancel (the
    softmax's sum_j de_ij is 0, and a_dst[i] shifts all of row i's logits alike, so d a_dst[i] keeps only the difference between
    the two LeakyReLU slopes; with self loops only, the gradient is exactly 0).  Their value can therefore sit far below the size
    of the terms, ``want[2]`` (300x to 6e4x on these cases), and no f32 evaluation comes closer to it than the rounding of those
    terms: their bound is 2e-5 of the slice's maximum plus 16 f32 unit roundoffs (2^-20) of the terms' size.  On one row the
    rounding of the two 512-channel dot products behind dz alone reaches 1.3 unit roundoffs."""
    y = got[0].detach().double().cpu()
    g = {k: v.detach().double().cpu() for k, v in got[1].items()}
    y64, g64 = want[0].cpu(), {k: v.cpu() for k, v in want[1].items()}
    heads = [slice(h * C, (h + 1) * C) for h in range(H)]
    errs = []
    for d, rows in _degree_classes(deg).items():
        for h, cs in enumerate(heads):
            errs.append((_slice_err(y, y64, rows, cs), TOL, "out", d, h))
        errs.append((_slice_err(g["x"], g64["x"], rows), GTOL, "x", d, None))
    for h, cs in enumerate(heads):
        errs.append((_slice_err(g["W"], g64["W"], cs), GTOL, "W", None, h))
        errs.append((_slice_err(g["bias"].view(1, -1), g64["bias"].view(1, -1), None, cs), GTOL, "bias", None, h))
        for name in ("att_l", "att_r"):
            err = float((g[name][0, h] - g64[name][0, h]).abs().max())
            allowed = GTOL * float(g64[name][0, h].abs().max()) + 2.0 ** -20 * float(want[2][name][h].max())
            errs.append((err / allowed, 1.0, name, None, h))
    bad = [e for e in errs if not e[0] < e[1]]
    assert not bad, (label, sorted(bad, key=lambda e: -e[0] / e[1])[:6])


def _selfloop_rows_exact(gc, x, y, deg, label):
    """A row whose only entry is its self loop has attention exactly 1 on both paths: its output is the f32 ``xl_i + bias`` of
    the layer's own projection, bit for bit."""
    iso = torch.nonzero(deg == 1).flatten().cuda()
    if iso.numel() == 0:
        return
    with torch.no_grad():
        want = (gc.lin_l(x) + gc.bias)[iso]
    assert torch.equal(y[iso], want), (label, float((y[iso] - want).abs().max()))


def _reference_for(gc, x, csr, w):
    rowptr, col, _ = csr
    return gat_reference(x, gc.lin_l.weight, gc.att_l, gc.att_r, gc.bias, rowptr, col, gc.heads, w)


def _all_paths(gc, x, graph, csr, w, label):
    """CSR (one-pass and two-pass backward), CSR with 16 rows per CTA (bit-identical to 8) and the dense-tile path, each against
    the f64 reference; rows made of their self loop alone are exact on both paths."""
    H, C = gc.heads, gc.out_channels
    deg = csr[2]
    want = _reference_for(gc, x, csr, w)
    fused = _run(gc, x, graph, w, "csr", "fused")
    runs = {"csr-fused": fused, "csr-split": _run(gc, x, graph, w, "csr", "split")}
    rows16 = _run_16_rows(gc, x, graph, w)
    assert torch.equal(rows16[0], fused[0]), label
    for k in fused[1]:
        assert torch.equal(rows16[1][k], fused[1][k]), (label, k)
    runs["dense"] = _run(gc, x, graph, w, "dense")
    for path, got in runs.items():
        _check(f"{label} {path}", got, want, H, C, deg)
        _selfloop_rows_exact(gc, x, got[0], deg, f"{label} {path}")


# ------------------------------------------------------------------------------------------------ tests
@pytest.mark.parametrize("H,C", SHAPES)
def test_reference_matches_oracle_dense_form(H, C):
    """The f64 reference above against ``oracle.conv.GATConv`` cast to double (masked-dense form) on a small random map."""
    from oracle import conv as oconv
    from oracle import graph as ograph

    n, f_in = 45, 128
    adj = small_map(n, 0.3, seed=2)
    g = torch.Generator().manual_seed(H * C)
    x = 0.25 * torch.randn(n, f_in, generator=g)
    torch.manual_seed(H + C)
    oc = oconv.GATConv(f_in, C, heads=H).double()
    with torch.no_grad():
        oc.bias.uniform_(-0.1, 0.1)
        oc.att_l.mul_(3.0)
        oc.att_r.mul_(3.0)
    odata = ograph.load_input(adj.numpy().copy(), x.numpy())
    w = torch.randn(n, H * C, generator=g, dtype=torch.float64)
    xo = x.double().requires_grad_(True)
    yo = oc(xo, odata.edge_index, dense=True)
    go = torch.autograd.grad((yo * w).sum(), [xo, oc.lin_l.weight, oc.att_l, oc.att_r, oc.bias])
    graph = _load(adj, x)
    rowptr, col, _ = _self_loop_csr(graph)
    y64, g64, _ = gat_reference(x.cuda(), oc.lin_l.weight.cuda(), oc.att_l.cuda(), oc.att_r.cuda(), oc.bias.cuda(), rowptr, col, H, w.cuda(),
                             budget=4096)   # several chunks
    assert rel_err(y64, yo) < 1e-12
    for name, want in zip(["x", "W", "att_l", "att_r", "bias"], go):
        assert rel_err(g64[name], want) < 1e-12, name


@pytest.mark.parametrize("f_in", F_INS)
@pytest.mark.parametrize("H,C", SHAPES)
def test_gat_degree_classes_every_shape(H, C, f_in):
    """Row lengths 1-6, 32-34, 128-130 and a hub (529 loci, not a multiple of 8 or 16), every path, every input width."""
    adj = degree_pattern()
    gc, x, graph, csr, w = _make_case(H, C, f_in, adj, seed=f_in)
    assert sorted(set(csr[2].tolist()))[: len(DEGREES)] == DEGREES
    _all_paths(gc, x, graph, csr, w, f"degrees H={H} C={C} F_in={f_in}")


@pytest.mark.parametrize("name", list(GRAPHS))
@pytest.mark.parametrize("H,C", SHAPES)
def test_gat_small_and_edgeless_graphs(H, C, name):
    """An edgeless graph (nnz = 0: self loops only), n = 1, 2, a 7-locus star and a sparse random map of 1 003 loci."""
    adj = GRAPHS[name]()
    f_in = F_INS[(SHAPES.index((H, C)) + list(GRAPHS).index(name)) % 3]
    gc, x, graph, csr, w = _make_case(H, C, f_in, adj, seed=7)
    _all_paths(gc, x, graph, csr, w, f"{name} H={H} C={C} F_in={f_in}")


@pytest.mark.parametrize("n,density,splits", [(1024, 0.95, 4), (200, 0.9, 1)])
@pytest.mark.parametrize("H,C", SHAPES)
def test_gat_dense_tiles_with_and_without_split_k(H, C, n, density, splits):
    """The dense-tile path on a near-dense map: at 1 024 loci every shape splits the k range in four (partials added by the combine
    kernels), at 200 loci none does.  The CSR path runs on the same inputs."""
    from hic_gnn_b200 import _native as N

    ws = N.lib().hicgat_gat_dense_workspace_bytes(n, H, C)
    if splits == 4:
        assert ws >= 4 * 4 * n * H * C       # the [nsplit][n][H*C] f32 partials
    else:
        assert 0 < ws < 4 * n * H * C       # no partial buffer
    f_in = F_INS[SHAPES.index((H, C)) % 3]
    gc, x, graph, csr, w = _make_case(H, C, f_in, small_map(n, density, seed=3), seed=11)
    want = _reference_for(gc, x, csr, w)
    for path in ("dense", "csr"):
        _check(f"n={n} H={H} C={C} {path}", _run(gc, x, graph, w, path), want, H, C, csr[2])


# ------------------------------------------------------------------------------------------------ the projection GEMM at GATConv shapes
@pytest.mark.parametrize("f_in,H,C", [(128, 4, 256), (256, 1, 512), (256, 2, 512), (512, 4, 256)])
def test_gat_projection_on_tensor_cores(monkeypatch, f_in, H, C):
    """5 000 loci on a banded pattern: the projection (F_in -> H*C, >= 100 000 weights) runs the three 3xTF32 GEMMs, the dx one
    with K = 3 * H*C (split-K over many M tiles when H*C = 1024).  y, dx and dW against f64 with test_gpu_gemm's bound
    max(5e-6, 5 x the cuBLAS fp32 error), given the kernels' own dL/dxl; the layer output and gradients against the f64 reference."""
    from hic_gnn_b200 import ops

    n = 5000
    assert n >= ops.TF32X3_MIN_ROWS and f_in * H * C >= 100000
    calls = []
    gemm = ops.gemm_tf32_tn
    monkeypatch.setattr(ops, "gemm_tf32_tn", lambda *a, **k: calls.append(a[0].shape) or gemm(*a, **k))
    gc, x, graph, csr, w = _make_case(H, C, f_in, banded(n, 8), seed=13)
    captured = []

    def keep_xl(mod, inp, out):
        out.retain_grad()
        captured.append(out)

    hook = gc.lin_l.register_forward_hook(keep_xl)
    try:
        got = _run(gc, x, graph, w, "csr")
    finally:
        hook.remove()
    assert len(calls) == 3, calls
    xl, dxl = captured[0].detach(), captured[0].grad
    W = gc.lin_l.weight.detach()
    x64, W64, dxl64 = x.double(), W.double(), dxl.double()
    for name, mine, want, ref32 in (("y", xl, x64 @ W64.t(), x @ W.t()), ("dx", got[1]["x"], dxl64 @ W64, dxl @ W),
                                    ("dW", got[1]["W"], dxl64.t() @ x64, dxl.t() @ x)):
        e, e32 = rel_err(mine, want), rel_err(ref32, want)
        assert e < max(5e-6, 5 * e32), (name, e, e32)
    _check(f"banded H={H} C={C} F_in={f_in}", got, _reference_for(gc, x, csr, w), H, C, csr[2])


# ------------------------------------------------------------------------------------------------ SAGE aggregation
@pytest.mark.parametrize("F_", [128, 256, 512, 1024])
def test_sage_aggregate_every_width(F_):
    """``hicgat_spmm_csr_f32`` (SAGEConv's D^-1 A x) at every feature width it dispatches, forward and backward, against f64 per
    degree class; rows of isolated loci are exactly zero, and an edgeless graph gives zeros both ways."""
    from hic_gnn_b200 import layers as glayers

    for adj in (degree_pattern(seed=1), torch.zeros(19, 19, dtype=torch.float64)):
        n = adj.shape[0]
        g = torch.Generator().manual_seed(F_ + n)
        x = torch.randn(n, F_, generator=g)
        graph = _load(adj, x)
        gout = torch.randn(n, F_, generator=g).cuda()
        xg = x.cuda().requires_grad_(True)
        y = glayers._SageAggregate.apply(xg, graph)
        dx, = torch.autograd.grad((y * gout).sum(), [xg])
        a = adj.double().clone()
        a.fill_diagonal_(0)
        a = a.float().double()                      # the graph stores float32(value)
        colsum = a.sum(0)
        M = torch.where(colsum.unsqueeze(1) > 0, a / colsum.clamp(min=1e-300).unsqueeze(1), torch.zeros_like(a)).cuda()
        want_y, want_dx = M @ x.cuda().double(), M.t() @ gout.double()
        deg = (a != 0).sum(1) + 1                   # the same classes as the GAT cases (self loop included)
        iso = torch.nonzero(deg == 1).flatten().cuda()
        assert torch.equal(y[iso], torch.zeros_like(y[iso])) and torch.equal(dx[iso], torch.zeros_like(dx[iso]))
        for d, rows in _degree_classes(deg).items():
            if d == 1:
                continue
            assert _slice_err(y.detach().double().cpu(), want_y.cpu(), rows) < TOL, (n, F_, d)
            assert _slice_err(dx.double().cpu(), want_dx.cpu(), rows) < TOL, (n, F_, d)


@pytest.mark.parametrize("n,density", [(58, 1.0), (200, 0.3)])
@pytest.mark.parametrize("f_in", [128, 256])
def test_sage_conv_input_widths(f_in, n, density):
    """``layers.SAGEConv(in, out)`` at the input widths below the suite's 512, against the oracle (test_sage_aggregate_forward_backward)."""
    from hic_gnn_b200 import layers as glayers
    from oracle import conv as oconv
    from oracle import graph as ograph

    adj = small_map(n, density, seed=1)
    x = 2.0 * torch.randn(n, f_in, generator=torch.Generator().manual_seed(f_in + n))   # |x| > 1 exercises x.long()
    odata = ograph.load_input(adj.numpy().copy(), x.numpy())
    graph = _load(adj, x)
    torch.manual_seed(0)
    oc = oconv.SAGEConv(f_in, 128)
    gc = glayers.SAGEConv(f_in, 128).cuda()
    gc.load_state_dict(oc.state_dict())
    xo = x.clone().requires_grad_(True)
    xg = x.cuda().requires_grad_(True)
    yo = oc(xo, odata.edge_index)
    yg = gc(xg, graph)
    assert rel_err(yg, yo) < TOL
    w = torch.randn_like(yo)
    go = torch.autograd.grad((yo * w).sum(), [xo, oc.lin_l.weight, oc.lin_r.weight])
    gg = torch.autograd.grad((yg * w.cuda()).sum(), [xg, gc.lin_l.weight, gc.lin_r.weight])
    for a, b in zip(gg, go):
        assert rel_err(a, b) < TOL
