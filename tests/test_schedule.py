"""Host logic of the pair-loss grid (no GPU): the row-chunk schedule every column strip is cut into.

The kernels trust these tables blindly (chunk c of a strip = rows [bounds[c], bounds[c+1]) of the row
block), so the CPU suite checks, through the C ABI's introspection entry point, that for any shape and
tuning they tile the block exactly once, in order, within the table size."""
import ctypes as C
import itertools

import numpy as np
import pytest

from hic_gnn_b200 import _native as N

MAX_CHUNKS = 128


def schedule(n, r0, r1, mode=0):
    buf = (C.c_int32 * 600)()
    k = N.lib().hicgat_pairloss_describe_schedule_mode(n, r0, r1, mode, C.addressof(buf), 600)
    assert k > 0, N.lib().hicgat_last_error()
    a = list(buf[:k])
    nstrips, stagger, c0, c1 = a[:4]
    b0 = a[4:4 + c0 + 1]
    b1 = a[4 + c0 + 1:4 + c0 + 1 + c1 + 1]
    assert 4 + len(b0) + len(b1) == k
    return nstrips, stagger, np.array(b0), np.array(b1)


@pytest.fixture(autouse=True)
def _reset_tuning():
    yield
    N.set_pairloss_tuning(0, 0)
    N.set_pairloss_schedule(-1, 256)


SHAPES = [(58, 0, 58), (130, 0, 130), (1000, 999, 1000), (2493, 0, 2493), (9970, 0, 9970), (9970, 4985, 9970), (19500, 100, 1000),
          (40000, 5, 205), (49850, 0, 49850), (49850, 43618, 49850), (49850, 0, 6232), (80000, 17, 60), (200000, 0, 200000)]


@pytest.mark.parametrize("variant", [0, 1, 2])
@pytest.mark.parametrize("rb", [0, 8, 64, 256, 1024, 4096])
@pytest.mark.parametrize("tail", [(-1, 256), (0, 256), (1, 256), (3, 128), (8, 64)])
def test_schedule_tiles_the_row_block(variant, rb, tail):
    """Full-row and upper-triangle (``PAIR_SYMMETRIC``) layouts: the launches of every variant, the implicit target's
    included, take the mode's schedule."""
    N.set_pairloss_tuning(rb, variant)
    N.set_pairloss_schedule(*tail)
    for (n, r0, r1), mode in itertools.product(SHAPES, (0, N.PAIR_SYMMETRIC)):
        nstrips, stagger, b0, b1 = schedule(n, r0, r1, mode)
        assert nstrips == (n + 127) // 128
        for b in (b0, b1):
            assert b[0] == 0 and b[-1] == r1 - r0, (n, r0, r1, mode, b)
            assert (np.diff(b) > 0).all(), (n, r0, r1, mode, b)
            assert len(b) - 1 <= MAX_CHUNKS
        if not stagger:
            assert (b0 == b1).all() if len(b0) == len(b1) else False
        if variant != 0:
            assert not stagger


def test_default_schedule_of_the_benchmark_shapes():
    """The shapes bench.py measures: equal chunks + half-chunk stagger on the 50k-locus blocks (390 strips),
    a shrinking tail on the 10k-locus map (78 strips)."""
    _, stagger, b0, b1 = schedule(49850, 0, 49850)
    assert stagger == 1
    d0, d1 = np.diff(b0), np.diff(b1)
    assert d0.max() - d0[:-1].min() == 0                  # equal chunks, the last one takes the remainder
    assert d1[0] * 2 == d0[0] and len(d1) == len(d0) + 1  # staggered strips start with half a chunk
    _, stagger, b0, _ = schedule(9970, 0, 9970)
    assert stagger == 0
    d = np.diff(b0)
    assert d.max() <= 1024 and list(d[-3:]) == [512, 256, 128]
    _, stagger, b0, _ = schedule(49850, 0, 6232)          # one rank's block of an 8-way split
    assert stagger == 1 and len(b0) - 1 <= 4


def test_schedule_argument_validation():
    lib = N.lib()
    assert lib.hicgat_pairloss_set_schedule(9, 256) == -1
    assert lib.hicgat_pairloss_set_schedule(2, 32) == -1
    buf = (C.c_int32 * 4)()
    assert lib.hicgat_pairloss_describe_schedule(9970, 0, 9970, C.addressof(buf), 4) == -3  # capacity too small
    assert lib.hicgat_pairloss_describe_schedule(0, 0, 0, C.addressof(buf), 4) == -1


def test_segmented_combine_workspace_and_validation():
    """``hicgat_pairloss_set_combine`` (host logic only): segments of the row-side sums need ticket + scratch space only for
    upper-triangle blocks whose strip chain is long enough; (1, x) switches them off; bad arguments are refused."""
    lib = N.lib()
    n = 49850
    sym = N.PAIR_SYMMETRIC

    def ws(r0, r1, mode):
        return lib.hicgat_pairloss_workspace_bytes_mode(n, r0, r1, mode)

    try:
        N.set_pairloss_combine(1, 96)
        base_shard, base_full, base_tail, base_plain = ws(0, 3200, sym), ws(0, n, sym), ws(32256, n, sym), ws(0, 3200, 0)
        N.set_pairloss_combine(4, 96)
        # rows 0..3199 = 25 strips of loci, chains of up to 390 strips: 4 segments -> 25 tickets + 25 * 4 * 384 f64
        assert ws(0, 3200, sym) - base_shard >= 25 * 4 * 384 * 8
        assert ws(0, 3200, sym) - base_shard <= 25 * 4 * 384 * 8 + 4096
        assert ws(0, n, sym) == base_full          # 390 strips of loci: more than one wave already, no segments
        assert ws(32256, n, sym) == base_tail      # chains of at most 138 strips: shorter than one 96-strip segment pair
        assert ws(0, 3200, 0) == base_plain        # full-matrix mode has no row-side sums
        N.set_pairloss_combine(8, 1)
        assert ws(32256, n, sym) > base_tail
        for bad in ((0, 96), (17, 96), (4, 0)):
            assert lib.hicgat_pairloss_set_combine(*bad) != 0
            assert b"set_combine" in lib.hicgat_last_error()
    finally:
        N.set_pairloss_combine()
