"""The (heads, channels) pairs the GAT kernels accept, checked without a GPU: the C ABI's workspace-size functions (host
arithmetic only, no launch) and the ``GATConv`` constructor must agree on exactly the eight compiled instantiations."""
import pytest

from hic_gnn_b200 import _native as N
from hic_gnn_b200 import layers

# conv.cu HICGAT_DISPATCH_HQ: (H, Q = H*C/128) in {(1,1) (1,2) (1,4) (2,2) (2,4) (2,8) (4,4) (4,8)}
SUPPORTED = {(1, 128), (1, 256), (1, 512), (2, 128), (2, 256), (2, 512), (4, 128), (4, 256)}
HEADS = [1, 2, 3, 4, 5]
CHANNELS = [32, 64, 128, 192, 256, 384, 512, 1024]


@pytest.fixture(scope="module")
def lib():
    from hic_gnn_b200 import build

    build.build()
    return N.lib()


@pytest.mark.parametrize("heads", HEADS)
@pytest.mark.parametrize("channels", CHANNELS)
def test_workspace_sizes_are_nonzero_exactly_for_the_compiled_shapes(lib, heads, channels):
    ok = (heads, channels) in SUPPORTED
    for n, nnz in ((1, 1), (1003, 20000), (50000, 25_000_000)):
        sizes = {
            "bwd": lib.hicgat_gat_bwd_workspace_bytes(n, nnz, heads, channels),
            "dense": lib.hicgat_gat_dense_workspace_bytes(n, heads, channels),
            "param_grads": lib.hicgat_gat_param_grads_workspace_bytes(n, heads, channels),
        }
        assert all((s != 0) == ok for s in sizes.values()), (n, nnz, sizes)
        if ok:  # each holds at least the [3, H*C] parameter-gradient partials of one CTA, the CSR one also dz [nnz, H]
            assert sizes["param_grads"] >= 12 * heads * channels
            assert sizes["bwd"] >= 4 * nnz * heads + sizes["param_grads"] - 256
    assert lib.hicgat_gat_bwd_workspace_bytes(0, 0, heads, channels) == 0
    assert lib.hicgat_gat_dense_workspace_bytes(0, heads, channels) == 0
    assert lib.hicgat_gat_param_grads_workspace_bytes(0, heads, channels) == 0


@pytest.mark.parametrize("heads", HEADS)
@pytest.mark.parametrize("channels", CHANNELS)
def test_gatconv_constructs_exactly_for_the_compiled_shapes(heads, channels):
    assert set(layers.GAT_SHAPES) == SUPPORTED
    if (heads, channels) in SUPPORTED:
        conv = layers.GATConv(256, channels, heads=heads)
        assert conv.lin_l.weight.shape == (heads * channels, 256) and conv.att_l.shape == (1, heads, channels)
        return
    with pytest.raises(NotImplementedError) as err:
        layers.GATConv(256, channels, heads=heads)
    msg = str(err.value)
    assert all(str(p) in msg for p in sorted(SUPPORTED)), msg
    assert f"({heads}, {channels})" in msg
