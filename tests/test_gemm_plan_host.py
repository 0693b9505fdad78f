"""The GEMM tile plan, checked without a GPU: the Python mirror of ``plan_gemm`` (tests/gemm_plan.py), which the GEMM tests use
to choose shapes and split-K boundaries, must give the workspace size ``hicgat_gemm_tf32_workspace_bytes`` computes (host
arithmetic only, no launch) on every Linear GEMM of the three models and on a grid around the plan's thresholds."""
import itertools

import pytest

from gemm_plan import ROWS, linear_gemms, plan_gemm, production_linears
from hic_gnn_b200 import _native as N


@pytest.fixture(scope="module")
def lib():
    from hic_gnn_b200 import build

    build.build()
    return N.lib()


def _production_gemms():
    for layer, nin, nout in production_linears():
        for rows in ROWS:
            for name, m, n, k in linear_gemms(rows, nin, nout):
                yield f"{layer} {name} rows={rows}", m, n, k


def test_mirror_matches_workspace_on_production_gemms(lib):
    seen = set()
    for what, m, n, k in _production_gemms():
        for kparts in (1, 3):
            p = plan_gemm(m, n, k, kparts)
            assert lib.hicgat_gemm_tf32_workspace_bytes(m, n, k, kparts) == p.workspace_bytes, (what, kparts, p)
            seen.add((p.wide, p.ksplit > 1))
    # the production GEMMs themselves reach both tile widths, and split K on both
    assert seen == {(False, False), (False, True), (True, False), (True, True)}, seen


def test_wide_split_k_dx_of_gatconv_1024():
    """The dx GEMM of a GATConv with H*C = 1024 from 9 345 loci on: 128 x 256 tiles and two splits set by the 16-main-block cap."""
    for rows in (9345, 9970, 49850):
        p = plan_gemm(rows, 512, 3 * 1024, 3)
        assert p.wide and p.capped and p.ksplit == 2 and p.kb_per_split == 48, p
    assert not plan_gemm(9344, 512, 3 * 1024, 3).wide


def test_mirror_matches_workspace_on_a_grid(lib):
    ms = [1, 33, 127, 128, 129, 1000, 4095, 4096, 4097, 9344, 9345, 9970, 18943, 18944, 49850]
    ns = [1, 3, 4, 5, 127, 128, 129, 255, 256, 257, 300, 384, 500, 512, 1024]
    ks = [32, 96, 480, 512, 1536, 3072, 4800, 12288, 3 * 9984, 3 * 49856]
    for m, n, k in itertools.product(ms, ns, ks):
        for kparts in (1, 3):
            p = plan_gemm(m, n, k, kparts)
            assert lib.hicgat_gemm_tf32_workspace_bytes(m, n, k, kparts) == p.workspace_bytes, (m, n, k, kparts, p)
    assert lib.hicgat_gemm_tf32_workspace_bytes(0, 128, 96, 3) == 0
    assert lib.hicgat_gemm_tf32_workspace_bytes(128, 0, 96, 3) == 0
    assert lib.hicgat_gemm_tf32_workspace_bytes(128, 128, 0, 3) == 0
