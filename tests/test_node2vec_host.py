"""node2vec contract pieces that need no GPU: the oracle's transition probabilities, gensim's count rules (against the
module's host glue and hand-computed values), the hash, the Python refusals and the C ABI's argument checks."""
import math

import numpy as np
import pytest

import node2vec_ref as R
from hic_gnn_b200 import _native as N
from hic_gnn_b200 import node2vec as n2v

# 0 - 1 - 2 - 3 path plus the chord 0 - 2 and a pendant 3 - 4, weighted, symmetric, sorted columns
_EDGES = {(0, 1): 2.0, (0, 2): 0.5, (1, 2): 1.0, (2, 3): 3.0, (3, 4): 1.5}


def _hand_csr():
    n = 5
    adj = np.zeros((n, n))
    for (i, j), w in _EDGES.items():
        adj[i, j] = adj[j, i] = w
    rowptr = np.concatenate(([0], np.cumsum((adj != 0).sum(1))))
    col = np.concatenate([np.nonzero(adj[i])[0] for i in range(n)])
    w = np.concatenate([adj[i][adj[i] != 0] for i in range(n)])
    return rowptr, col, w


@pytest.mark.parametrize("p,q", [(1.0, 1.0), (1.75, 0.4), (0.25, 4.0)])
def test_transition_probs_sum_to_one(p, q):
    rowptr, col, w = _hand_csr()
    for v in range(5):
        for t in [-1] + col[rowptr[v]:rowptr[v + 1]].tolist():
            pr = R.transition_probs(rowptr, col, w, t, v, p, q)
            assert math.isclose(sum(pr.values()), 1.0, rel_tol=1e-12)
            assert set(pr) == set(col[rowptr[v]:rowptr[v + 1]].tolist())


def test_transition_probs_first_order_at_p_q_one():
    rowptr, col, w = _hand_csr()
    for v in range(5):
        first = R.transition_probs(rowptr, col, w, -1, v, 1.0, 1.0)
        for t in col[rowptr[v]:rowptr[v + 1]].tolist():
            assert R.transition_probs(rowptr, col, w, t, v, 1.0, 1.0) == pytest.approx(first, rel=1e-12)


def test_transition_probs_hand_case():
    rowptr, col, w = _hand_csr()
    # from t = 1 at v = 2: x = 1 is the return (1/p), x = 0 is a neighbour of 1 (1), x = 3 is not (1/q)
    p, q = 2.0, 0.5
    pr = R.transition_probs(rowptr, col, w, 1, 2, p, q)
    raw = {0: 0.5 * 1.0, 1: 1.0 / p, 3: 3.0 / q}
    s = sum(raw.values())
    assert pr == pytest.approx({k: v / s for k, v in raw.items()}, rel=1e-12)


def test_cum_table_hand_cases():
    assert R.cum_table([1, 1]).tolist() == [1073741824, 2147483647]         # round(0.5 * (2^31 - 1)), half to even
    assert R.cum_table([16, 1]).tolist() == [round(8 / 9 * (2**31 - 1)), 2**31 - 1]  # 16^0.75 = 8
    counts = np.random.default_rng(0).integers(1, 5000, 777)
    assert np.array_equal(n2v.cum_table(counts), R.cum_table(counts))


def test_keep_probability_hand_cases():
    # T = 1010, sample 1e-3 -> threshold count 1.01
    pk = R.keep_probability([1000, 10], 1e-3)
    assert pk[0] == pytest.approx((math.sqrt(1000 / 1.01) + 1) * 1.01 / 1000, rel=1e-12)
    assert pk[1] == pytest.approx((math.sqrt(10 / 1.01) + 1) * 1.01 / 10, rel=1e-12)
    assert 0.0327 < pk[0] < 0.0329 and 0.418 < pk[1] < 0.420
    assert R.keep_probability([3, 1], 1.0).tolist() == [1.0, 1.0]           # capped at 1
    assert R.keep_thresholds([5, 7], 0.0).tolist() == [2**32 - 1] * 2        # sample 0 keeps every token
    counts = np.random.default_rng(1).integers(1, 5000, 777)
    for s in (0.0, 1e-3, 1e-5):
        assert np.array_equal(n2v.keep_thresholds(counts, s), R.keep_thresholds(counts, s))


def test_hash_is_splitmix64():
    assert R.mix64(0x9E3779B97F4A7C15) == 0xE220A8397B1DCDAF  # first output of splitmix64 seeded with 0
    assert R.n2v_hash(0, 0, 0, 0) == R.mix64(R.mix64(R.mix64(0xE220A8397B1DCDAF)))
    draws = {R.n2v_hash(42, w, s, a) for w in range(20) for s in range(20) for a in range(5)}
    assert len(draws) == 2000


def test_python_refusals():
    with pytest.raises(NotImplementedError, match="sg=1"):
        n2v.SkipGram(None, 10, sg=0)
    with pytest.raises(NotImplementedError, match="hs=1"):
        n2v.SkipGram(None, 10, hs=1)
    with pytest.raises(NotImplementedError, match="min_count"):
        n2v.SkipGram(None, 10, min_count=2)
    with pytest.raises(ValueError, match="multiple of 128"):
        n2v.SkipGram(None, 10, vector_size=100)
    with pytest.raises(ValueError, match="window"):
        n2v.SkipGram(None, 10, window=0)
    for p, q in [(0.0, 1.0), (1.0, -1.0), (float("nan"), 1.0)]:
        with pytest.raises(ValueError, match="p and q"):
            n2v.Node2Vec(None, p=p, q=q)
    with pytest.raises(ValueError, match="multiple of 128"):
        n2v.Node2Vec(None, dimensions=200)
    with pytest.raises(ValueError, match="walk_length"):
        n2v.Node2Vec(None, walk_length=n2v.MAX_WALK_LENGTH + 1)


@pytest.fixture(scope="module")
def lib():
    from hic_gnn_b200 import build

    build.build()
    return N.lib()


def _err(lib):
    return lib.hicgat_last_error().decode()


def test_abi_walks_validation(lib):
    fake = 256  # never dereferenced: every check below fails before any CUDA call
    assert lib.hicgat_node2vec_walks(None, fake, fake, fake, 4, 0, 8, 1.0, 1.0, 0, fake, None) == -1
    assert "null pointer" in _err(lib)
    for p, q in [(0.0, 1.0), (1.0, 0.0), (-1.0, 1.0)]:
        assert lib.hicgat_node2vec_walks(fake, fake, fake, fake, 4, 0, 8, p, q, 0, fake, None) == -1
        assert "p and q" in _err(lib)
    assert lib.hicgat_node2vec_walks(fake, fake, fake, fake, 4, 0, n2v.MAX_WALK_LENGTH + 1, 1.0, 1.0, 0, fake, None) == -1
    assert "walk_length" in _err(lib)


def test_abi_sgns_validation(lib):
    fake = 256

    def call(**kw):
        a = dict(walks=fake, off=fake, nw=4, L=8, cum=fake, thr=fake, n=10, dim=128, window=5, negative=5, epoch=0, epochs=1, s0=fake, s1=fake)
        a.update(kw)
        return lib.hicgat_sgns_epoch(a["walks"], a["off"], a["nw"], a["L"], a["cum"], a["thr"], a["n"], a["dim"], a["window"], a["negative"],
                                     0.025, 1e-4, a["epoch"], a["epochs"], 1, 1, a["s0"], a["s1"], None)

    assert call(s1=None) == -1 and "null pointer" in _err(lib)
    for d in (0, 100, 1152):
        assert call(dim=d) == -1 and "dim" in _err(lib)
    assert call(L=n2v.MAX_WALK_LENGTH + 1) == -1 and "walk_length" in _err(lib)
    assert call(window=0) == -1 and "window" in _err(lib)
    assert call(negative=-1) == -1 and "negative" in _err(lib)
    assert call(negative=32) == -1 and "negative" in _err(lib)
    assert call(epoch=1, epochs=1) == -1 and "epoch" in _err(lib)
    assert lib.hicgat_version() == 202
