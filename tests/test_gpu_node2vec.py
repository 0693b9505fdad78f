"""node2vec on the GPU: walk validity and determinism, the walk distribution against the oracle's P(x | t, v) (G-test), the
one-warp skip-gram epoch against the numpy replay, Hogwild quality against the serial run, a C4-sized smoke and the
generalisation example with node2vec features."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch
from scipy import stats

import node2vec_ref as R
from hic_gnn_b200 import synth, utils
from hic_gnn_b200 import node2vec as n2v
from hic_gnn_b200.graph import CSRGraph

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def sparse_graph():
    """A few hundred loci of a synthetic Hi-C map at ~10 % density: the q branch (x not a neighbour of t) occurs."""
    adj = synth.synthetic_map(240, 0.1, seed=5)
    g = utils.load_input(adj, np.zeros((240, 1), np.float32)).edge_index
    assert 0.05 < g.nnz / 240**2 < 0.2
    return g


@pytest.fixture(scope="module")
def hand_graph():
    edges = {(0, 1): 2.0, (0, 2): 0.5, (1, 2): 1.0, (2, 3): 3.0, (3, 4): 1.5, (4, 5): 1.0, (3, 5): 0.25, (5, 6): 2.5, (1, 6): 0.75}
    ij = [(i, j, w) for (i, j), w in edges.items()] + [(j, i, w) for (i, j), w in edges.items()]
    ei = torch.tensor([[a for a, _, _ in ij], [b for _, b, _ in ij]], device="cuda")
    return CSRGraph.from_edge_index(ei, torch.tensor([w for _, _, w in ij], device="cuda"), 7)


@pytest.fixture(scope="module")
def chr19_graph(golden):
    arrays, _ = golden
    return utils.load_input(arrays["1mb_kr_oracle"], np.zeros((58, 1), np.float32)).edge_index


def _host_csr(g):
    return g.rowptr.cpu().numpy(), g.col.cpu().numpy(), g.value.cpu().numpy()


def test_walks_are_valid_and_start_right(sparse_graph):
    g = sparse_graph
    m = n2v.Node2Vec(g, dimensions=128, walk_length=24, num_walks=3, p=1.75, q=0.4, seed=3)
    w = m.walks
    assert w.dtype == torch.int32 and w.is_cuda and tuple(w.shape) == (3 * g.n, 24)
    adj = torch.zeros(g.n, g.n, dtype=torch.bool, device="cuda")
    adj[g.storage.row(), g.col] = True
    assert bool((w >= 0).all())                                   # every locus has neighbours here
    a, b = w[:, :-1].long(), w[:, 1:].long()
    assert bool(adj[a, b].all()), "a step that is not an edge"
    for r in range(3):
        assert torch.equal(torch.sort(w[r * g.n:(r + 1) * g.n, 0]).values.cpu(), torch.arange(g.n, dtype=torch.int32))


def test_isolated_node_pads_with_minus_one():
    ei = torch.tensor([[0, 1, 1, 2], [1, 0, 2, 1]], device="cuda")
    g = CSRGraph.from_edge_index(ei, torch.tensor([1.0, 1.0, 2.0, 2.0], device="cuda"), 4)  # node 3 is isolated
    w = n2v.Node2Vec(g, walk_length=6, num_walks=2, seed=0).walks.cpu()
    iso = w[w[:, 0] == 3]
    assert iso.shape[0] == 2 and bool((iso[:, 1:] == -1).all())
    assert bool((w[w[:, 0] != 3] >= 0).all())
    sg = n2v.SkipGram(n2v.Node2Vec(g, walk_length=6, num_walks=2, seed=0).walks, 4, 128, sample=0.0, num_warps=1, epochs=1).train()
    assert int(sg.walk_offsets[-1]) == 3 * 2 * 6 + 2 and bool(torch.isfinite(sg.syn0).all())


def test_walks_are_bit_reproducible_across_runs_and_batchings(sparse_graph):
    g = sparse_graph
    starts = torch.cat([torch.randperm(g.n, device="cuda") for _ in range(4)])
    full = n2v.random_walks(g, starts, 30, 0.25, 4.0, seed=99)
    assert torch.equal(full, n2v.random_walks(g, starts, 30, 0.25, 4.0, seed=99))
    parts = [n2v.random_walks(g, starts[a:b], 30, 0.25, 4.0, seed=99, walk_id0=a) for a, b in [(0, 7), (7, 500), (500, starts.numel())]]
    assert torch.equal(full, torch.cat(parts))
    assert not torch.equal(full, n2v.random_walks(g, starts, 30, 0.25, 4.0, seed=100))


def _g_test(counts: dict, rowptr, col, w, p, q, min_visits):
    """Pooled G statistic and degrees of freedom over the contexts with >= min_visits visits.  Within a context the cells
    are merged in ascending order of expected count until each expects >= 10, and G carries Williams' correction
    q = 1 + (sum 1/pi - 1) / (6 n (k - 1))."""
    G, df, contexts = 0.0, 0, 0
    for (t, v), obs in counts.items():
        n = sum(obs.values())
        if n < min_visits:
            continue
        pr = R.transition_probs(rowptr, col, w, t, v, p, q)
        assert set(obs) <= set(pr), "a step that is not an edge"
        cells, acc_o, acc_e = [], 0, 0.0
        for x, px in sorted(pr.items(), key=lambda kv: kv[1]):
            acc_o, acc_e = acc_o + obs.get(x, 0), acc_e + n * px
            if acc_e >= 10:
                cells.append((acc_o, acc_e))
                acc_o, acc_e = 0, 0.0
        if acc_e > 0 and cells:
            cells[-1] = (cells[-1][0] + acc_o, cells[-1][1] + acc_e)
        k = len(cells)
        if k < 2:
            continue
        williams = 1.0 + (sum(n / e for _, e in cells) - 1.0) / (6.0 * n * (k - 1))
        G += 2 * sum(o * np.log(o / e) for o, e in cells if o > 0) / williams
        df += k - 1
        contexts += 1
    return G, df, contexts


def _transition_counts(walks: torch.Tensor, n: int):
    w = walks.long()
    first = torch.stack((torch.full_like(w[:, 0], -1), w[:, 0], w[:, 1]), 1)
    later = torch.stack((w[:, :-2], w[:, 1:-1], w[:, 2:]), 2).reshape(-1, 3)
    out = []
    for trip in (first, later):
        trip = trip[trip[:, 2] >= 0]
        key = ((trip[:, 0] + 1) * n + trip[:, 1]) * n + trip[:, 2]
        u, c = torch.unique(key, return_counts=True)
        u, c = u.cpu().numpy(), c.cpu().numpy()
        d = {}
        for k, cnt in zip(u.tolist(), c.tolist()):
            x, rest = k % n, k // n
            d.setdefault((rest // n - 1, rest % n), {})[x] = cnt
        out.append(d)
    return out


@pytest.mark.parametrize("p,q", [(1.0, 1.0), (1.75, 0.4), (0.25, 4.0)])
@pytest.mark.parametrize("which", ["sparse", "hand"])
def test_walk_distribution_g_test(which, p, q, sparse_graph, hand_graph):
    g = sparse_graph if which == "sparse" else hand_graph
    num_walks = 120 if which == "sparse" else 3000
    m = n2v.Node2Vec(g, walk_length=40, num_walks=num_walks, p=p, q=q, seed=2024)
    rowptr, col, w = _host_csr(g)
    first, later = _transition_counts(m.walks, g.n)
    for counts, min_visits in ((first, 50), (later, 100)):
        G, df, contexts = _g_test(counts, rowptr, col, w, p, q, min_visits)
        pval = stats.chi2.sf(G, df)
        print(f"{which} p={p} q={q}: {contexts} contexts, G={G:.1f}, df={df}, p-value={pval:.3g}")
        assert contexts >= (0.9 * g.n if counts is first else min(3 * g.n, g.nnz)) and df > 0
        # At tens of visits per context even exact multinomial draws leave the corrected, pooled G ~1 % above df, which over
        # ~5e4 degrees of freedom is a few standard deviations; so a large pooled test passes on a small relative excess
        # instead.  A wrong alpha class moves G / df by far more than 3 %.
        assert pval > 1e-4 or G / df < 1.03, (G, df)


def _chr19_walks(g, seed=7):
    return n2v.Node2Vec(g, dimensions=128, walk_length=16, num_walks=3, p=1.75, q=0.4, seed=seed).walks


@pytest.mark.parametrize("dim", [128, 512])
@pytest.mark.parametrize("sample", [0.0, 1e-3])
def test_serial_epoch_matches_numpy_replay(chr19_graph, dim, sample):
    walks = _chr19_walks(chr19_graph)
    sg = n2v.SkipGram(walks, 58, dim, window=5, negative=5, sample=sample, epochs=2, seed=11, num_warps=1)
    syn0_init = sg.syn0.cpu().numpy().copy()
    sg.train()
    ref0, ref1 = R.sgns_replay(walks.cpu().numpy(), syn0_init, 58, 5, 5, sample, 0.025, 1e-4, 2, 11)
    if sample:
        kept = np.mean([(R.n2v_hash(11, 0, r, 0) >> 32) <= t for r, t in enumerate(sg.keep_threshold.cpu().numpy().view(np.uint32)[walks.cpu().numpy().ravel()])])
        print(f"sample={sample}: {100 * (1 - kept):.0f} % of the tokens dropped in epoch 0")
    for got, ref in ((sg.syn0, ref0), (sg.syn1neg, ref1)):
        err = float(np.abs(got.cpu().numpy() - ref).max())
        scale = float(np.abs(ref).max())
        print(f"dim={dim} sample={sample}: max |gpu - replay| = {err:.3g} (max |ref| {scale:.3g})")
        # the only difference is the f32 order of the 1+K dot products per pair (lane partial sums + butterfly vs numpy)
        assert err <= 1e-4 * scale, (err, scale)


def _neighbour_quality(vec: torch.Tensor, k: int = 5) -> float:
    """Fraction of each node's top-k cosine neighbours that lie within k bins on the genome."""
    v = torch.nn.functional.normalize(vec.double(), dim=1)
    s = v @ v.t()
    s.fill_diagonal_(-2.0)
    top = s.topk(k, dim=1).indices
    idx = torch.arange(vec.shape[0], device=vec.device).unsqueeze(1)
    return float(((top - idx).abs() <= k).double().mean())


@pytest.mark.parametrize("which", ["chr19", "synthetic_2493"])
def test_hogwild_quality_against_serial(which, chr19_graph):
    if which == "chr19":
        g, walks = chr19_graph, n2v.Node2Vec(chr19_graph, walk_length=40, num_walks=10, p=1.75, q=0.4, seed=42).walks
    else:
        adj = synth.synthetic_map(2493, 0.3, seed=9, device="cuda")
        g = utils.load_input(adj, np.zeros((2493, 1), np.float32)).edge_index
        walks = n2v.Node2Vec(g, walk_length=40, num_walks=4, p=1.75, q=0.4, seed=42).walks
    serial = n2v.SkipGram(walks, g.n, 128, epochs=2, seed=3, num_warps=1).train()
    hog = n2v.SkipGram(walks, g.n, 128, epochs=2, seed=3)
    objective = [_objective_probe(hog, walks, g.n)]
    for e in range(hog.epochs):
        hog.epoch(e)
        objective.append(_objective_probe(hog, walks, g.n))
    q_serial, q_hog = _neighbour_quality(serial.syn0), _neighbour_quality(hog.syn0)
    q_rand = _neighbour_quality(synth.synthetic_features(g.n, 128).cuda())
    print(f"{which}: top-5 neighbours within 5 bins: serial {q_serial:.3f}, Hogwild {q_hog:.3f}, random {q_rand:.3f}; "
          f"objective {[round(x, 4) for x in objective]}")
    assert q_hog >= q_serial - 0.15
    assert q_serial >= q_rand + 0.15 and q_hog >= q_rand + 0.15
    assert all(a > b for a, b in zip(objective, objective[1:])), objective


def _objective_probe(sg, walks, n, pairs=4000, negative=5) -> float:
    """Mean SGNS objective -log s(c.o) - sum log s(-n.o) over a fixed sample of adjacent (centre, context) pairs."""
    gen = torch.Generator(device="cuda").manual_seed(123)
    rows = torch.randint(0, walks.shape[0], (pairs,), generator=gen, device="cuda")
    cols = torch.randint(0, walks.shape[1] - 1, (pairs,), generator=gen, device="cuda")
    c, o = walks[rows, cols].long(), walks[rows, cols + 1].long()
    neg = torch.randint(0, n, (pairs, negative), generator=gen, device="cuda")
    l1 = sg.syn0[o].double()
    pos = torch.nn.functional.logsigmoid((sg.syn1neg[c].double() * l1).sum(1))
    negs = torch.nn.functional.logsigmoid(-(sg.syn1neg[neg].double() * l1.unsqueeze(1)).sum(2)).sum(1)
    return float(-(pos + negs).mean())


def test_c4_scale_smoke():
    n = synth.CHR1_LOCI["25kb"]
    adj = synth.synthetic_map_chunked(n, 0.07, device="cuda")
    g = utils.load_input(adj, np.zeros((n, 1), np.float32)).edge_index
    del adj
    m = n2v.Node2Vec(g, dimensions=512, walk_length=150, num_walks=50, p=1.75, q=0.4, seed=42)
    model = m.fit(epochs=1)
    v = model.wv.vectors
    assert tuple(v.shape) == (n, 512) and v.dtype == torch.float32 and v.is_cuda
    assert bool(torch.isfinite(v).all()) and float(v.abs().max()) > 0
    assert torch.equal(model.wv["17"], v[17]) and torch.equal(model.wv[17], v[17])


def test_generalize_example_with_node2vec_features():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "chr19_generalize.py"), "--features", "node2vec", "--steps", "30"],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    print(out.stdout)
    d = [float(x) for x in re.findall(r"dSCC=([-\d.naninf]+)", out.stdout)]
    assert len(d) == 2 and all(np.isfinite(d))
