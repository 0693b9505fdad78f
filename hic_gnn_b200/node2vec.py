"""node2vec node features on the GPU: a drop-in for ``Node2Vec(graph, ...).fit(...)`` of node2vec 0.4.3 + gensim 4
(``HiC_GAT_generalize_directly.py:153-155``: ``Node2Vec(G, dimensions=512, walk_length=150, num_walks=50, p=1.75, q=0.4,
seed=42)``; ``train_and_test_same_res_GAT_node2vec.py:72``, ``combined_loss_training.py:90``,
``HiC-GNN_node2vec_conversion.py:118`` with other walk parameters), on the CSR graph ``load_input`` /
``load_input_sparse`` build.

Contract (the kernels are ``hicgat_node2vec_walks`` / ``hicgat_sgns_epoch``; ``include/hicgat.h`` states every rule,
``tests/node2vec_ref.py`` restates it in numpy):

* Walks follow node2vec 0.4.3 on the weighted, symmetric, diagonal-free graph (edge weight = the stored f32 value,
  node id = CSR row).  ``num_walks`` rounds; each round starts one walk from every node, in a seeded random order (one
  device permutation per round).  A walk holds ``walk_length`` nodes including the start; the first step draws
  P(x | v) ~ w(v, x), later steps from t -> v draw P(x | t, v) ~ w(v, x) * alpha with alpha = 1/p if x = t, 1 if x is a
  neighbour of t, 1/q otherwise (exact rejection sampling, no O(sum deg^2) tables).  A node without neighbours ends its
  walk; the remaining slots hold -1.  ``.walks`` is ``int32[num_walks * n, walk_length]``.
* Skip-gram with negative sampling follows word2vec.c / gensim's Cython path (``sg=1, hs=0``; node2vec 0.4.3 forces
  ``sg=1``): counts per node from the walks (``min_count=1``, -1 is no token), gensim's ``cum_table`` for the negatives,
  gensim's keep probability for ``sample`` (drawn once per token and epoch, before windowing), the reduced window
  ``b = r % window``, word2vec.c's per-pair update with the exact sigmoid, a learning rate decaying linearly per centre
  token, ``syn0 = (u - 0.5) / dim`` and ``syn1neg = 0`` at the start.  The result is ``syn0`` in node order.
* Random numbers come from one stateless counter hash (splitmix64 finaliser of (seed, a, b, c)), so the walks are
  bit-reproducible whatever the launch shape or batching, and a one-warp skip-gram run (``num_warps=1``) can be replayed.
  The default run fills the GPU (Hogwild) and, like gensim with ``workers > 1``, is not bit-reproducible.

Defaults: ``Node2Vec`` takes node2vec 0.4.3's (``dimensions=128, walk_length=80, num_walks=10, p=q=1``) and ``fit`` gensim 4's
(``window=5, negative=5, sample=1e-3, alpha=0.025, min_alpha=1e-4, epochs=5, seed=1``).  The keyword arguments the reference
passes to ``fit(...)`` are not recorded in this repository (SURVEY records the constructor calls only), so none are assumed.
CBOW (``sg=0``), hierarchical softmax (``hs=1``) and ``min_count > 1`` raise ``NotImplementedError``.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _native as N
from .ops import _cuda, _stream

MAX_WALK_LENGTH = 512  # HICGAT_N2V_MAX_WALK_LENGTH: a walk's kept tokens live in shared memory
_CUM_DOMAIN = 2**31 - 1


def _check_walk_args(dimensions, walk_length, num_walks, p, q):
    if not (p > 0 and q > 0 and np.isfinite(p) and np.isfinite(q)):
        raise ValueError(f"Node2Vec: p and q must be finite and > 0 (got p={p}, q={q})")
    if not 1 <= int(walk_length) <= MAX_WALK_LENGTH:
        raise ValueError(f"Node2Vec: walk_length must be in [1, {MAX_WALK_LENGTH}] (got {walk_length})")
    if int(num_walks) < 1:
        raise ValueError(f"Node2Vec: num_walks must be >= 1 (got {num_walks})")
    _check_dim(dimensions)


def _check_dim(dim):
    if int(dim) % 128 or not 128 <= int(dim) <= 1024:
        raise ValueError(f"node2vec: the embedding width must be a multiple of 128 in [128, 1024] (got {dim}); "
                         "the skip-gram kernel spreads a row over the 32 lanes of a warp in 16-byte pieces")


def transition_cdf(graph) -> torch.Tensor:
    """Per-row cumulative edge weight, f32[nnz] (f64 segmented cumsum; the last entry of a row is its total)."""
    v = graph.value.double()
    cs = torch.cumsum(v, 0)
    before = torch.cat((torch.zeros(1, dtype=torch.float64, device=v.device), cs))[graph.rowptr[:-1]]
    return (cs - torch.repeat_interleave(before, graph.rowptr[1:] - graph.rowptr[:-1], output_size=graph.nnz)).float().contiguous()


def random_walks(graph, starts: torch.Tensor, walk_length: int, p: float, q: float, seed: int, walk_id0: int = 0) -> torch.Tensor:
    """``int32[len(starts), walk_length]``: one second-order walk per start; row i is walk id ``walk_id0 + i``."""
    _check_walk_args(128, walk_length, 1, p, q)
    _cuda(starts)
    starts = starts.to(torch.int32).contiguous()
    if starts.numel() and (int(starts.min()) < 0 or int(starts.max()) >= graph.n):
        raise ValueError("random_walks: a start node is outside the graph")
    r32, c32 = graph.i32()
    cdf = graph._get("n2v_cdf", lambda: transition_cdf(graph))
    out = torch.empty(starts.numel(), int(walk_length), dtype=torch.int32, device=starts.device)
    N.check(N.lib().hicgat_node2vec_walks(r32.data_ptr(), c32.data_ptr(), cdf.data_ptr(), starts.data_ptr(), starts.numel(), int(walk_id0),
                                          int(walk_length), float(p), float(q), int(seed) & (2**64 - 1), out.data_ptr(), _stream()),
            "hicgat_node2vec_walks")
    return out


def cum_table(counts: np.ndarray) -> np.ndarray:
    """gensim's ``make_cum_table``: uint32 round(cumsum(count^0.75) / sum * (2^31 - 1)), accumulated in order in f64."""
    pw = np.asarray(counts, dtype=np.float64) ** 0.75
    return np.round(np.cumsum(pw) / pw.sum() * _CUM_DOMAIN).astype(np.uint32)


def keep_thresholds(counts: np.ndarray, sample: float) -> np.ndarray:
    """gensim's ``sample_int``: uint32(p_keep * (2^32 - 1)), p_keep = (sqrt(c / (sample T)) + 1) (sample T) / c capped at 1."""
    c = np.asarray(counts, dtype=np.float64)
    total = c.sum()
    thr = sample * total if sample else total  # gensim: sample = 0 keeps every token
    prob = np.minimum((np.sqrt(c / thr) + 1.0) * (thr / c), 1.0)
    return (prob * (2**32 - 1)).astype(np.uint32)


class KeyedVectors:
    """``model.wv`` look-alike: ``vectors`` (n x dim CUDA f32) indexed by node id, as int or as str(int)."""

    def __init__(self, vectors: torch.Tensor):
        self.vectors = vectors
        self.vector_size = vectors.shape[1]

    def __len__(self):
        return self.vectors.shape[0]

    def __getitem__(self, key):
        if isinstance(key, (list, tuple)):
            return self.vectors[torch.tensor([int(k) for k in key], device=self.vectors.device)]
        return self.vectors[int(key)]


class SkipGram:
    """Skip-gram with negative sampling over a walk corpus: the vocabulary, negative table and keep thresholds of gensim
    (built on the host from the node counts), ``syn0`` / ``syn1neg`` on the GPU, one ``hicgat_sgns_epoch`` launch per
    :meth:`epoch`.  ``num_warps=None`` fills the GPU (Hogwild); ``num_warps=1`` is the serial, replayable order."""

    def __init__(self, walks: torch.Tensor, n: int, vector_size: int = 128, window: int = 5, negative: int = 5, sample: float = 1e-3,
                 alpha: float = 0.025, min_alpha: float = 1e-4, epochs: int = 5, seed: int = 1, num_warps: int | None = None,
                 sg: int = 1, hs: int = 0, min_count: int = 1):
        _check_sg_args(vector_size, window, negative, sample, alpha, min_alpha, epochs, sg, hs, min_count)
        _cuda(walks)
        if walks.dim() != 2 or walks.dtype != torch.int32 or not 1 <= walks.shape[1] <= MAX_WALK_LENGTH:
            raise ValueError(f"SkipGram: walks must be int32[num_walks, walk_length <= {MAX_WALK_LENGTH}]")
        self.walks, self.n, self.dim = walks.contiguous(), int(n), int(vector_size)
        self.window, self.negative, self.sample = int(window), int(negative), float(sample)
        self.alpha, self.min_alpha, self.epochs, self.seed = float(alpha), float(min_alpha), int(epochs), int(seed)
        self.num_warps = 0 if num_warps is None else int(num_warps)
        valid = self.walks >= 0
        counts = torch.bincount(self.walks[valid].long(), minlength=self.n)
        if counts.numel() != self.n:
            raise ValueError("SkipGram: a walk holds a node id >= n")
        lengths = valid.sum(1)
        self.walk_offsets = torch.zeros(self.walks.shape[0] + 1, dtype=torch.int64, device=walks.device)
        torch.cumsum(lengths, 0, out=self.walk_offsets[1:])
        self.counts = counts.cpu().numpy()
        if (self.counts == 0).any():  # every node starts walks in Node2Vec; a bare corpus may miss some
            raise ValueError("SkipGram: every node id in [0, n) must occur in the walks (min_count=1 vocabulary in node order)")
        self.total_tokens = int(self.counts.sum())
        self.cum_table = torch.from_numpy(cum_table(self.counts).view(np.int32)).to(walks.device)
        self.keep_threshold = torch.from_numpy(keep_thresholds(self.counts, self.sample).view(np.int32)).to(walks.device)
        gen = torch.Generator(device=walks.device).manual_seed(self.seed)
        self.syn0 = ((torch.rand(self.n, self.dim, generator=gen, device=walks.device) - 0.5) / self.dim).contiguous()
        self.syn1neg = torch.zeros(self.n, self.dim, dtype=torch.float32, device=walks.device)

    def epoch(self, e: int) -> None:
        N.check(N.lib().hicgat_sgns_epoch(self.walks.data_ptr(), self.walk_offsets.data_ptr(), self.walks.shape[0], self.walks.shape[1],
                                          self.cum_table.data_ptr(), self.keep_threshold.data_ptr(), self.n, self.dim, self.window,
                                          self.negative, self.alpha, self.min_alpha, int(e), self.epochs, self.seed & (2**64 - 1),
                                          self.num_warps, self.syn0.data_ptr(), self.syn1neg.data_ptr(), _stream()), "hicgat_sgns_epoch")

    def train(self) -> "SkipGram":
        for e in range(self.epochs):
            self.epoch(e)
        return self

    @property
    def wv(self) -> KeyedVectors:
        return KeyedVectors(self.syn0)


def _check_sg_args(vector_size, window, negative, sample, alpha, min_alpha, epochs, sg, hs, min_count):
    if sg != 1:
        raise NotImplementedError("node2vec: only skip-gram (sg=1) is implemented; node2vec 0.4.3 forces sg=1")
    if hs != 0:
        raise NotImplementedError("node2vec: hierarchical softmax (hs=1) is not implemented; use negative sampling")
    if min_count != 1:
        raise NotImplementedError("node2vec: min_count > 1 is not implemented (every node keeps its vector)")
    _check_dim(vector_size)
    if int(window) < 1 or not 0 <= int(negative) <= 31 or int(epochs) < 1:
        raise ValueError(f"node2vec: need window >= 1, 0 <= negative <= 31, epochs >= 1 (got {window}, {negative}, {epochs})")
    if not (sample >= 0 and alpha >= 0 and min_alpha >= 0):
        raise ValueError("node2vec: sample, alpha and min_alpha must be >= 0")


class Node2Vec:
    """``node2vec.Node2Vec(graph, dimensions, walk_length, num_walks, p, q, workers, seed)`` on a :class:`CSRGraph`.  The walks
    are generated at construction, as in the package, and kept as ``.walks`` (int32 CUDA tensor).  ``workers`` has no
    effect.  ``seed=None`` draws one from torch's default generator."""

    def __init__(self, graph, dimensions: int = 128, walk_length: int = 80, num_walks: int = 10, p: float = 1, q: float = 1,
                 workers: int = 1, seed: int | None = None):
        _check_walk_args(dimensions, walk_length, num_walks, p, q)
        self.dimensions, self.walk_length, self.num_walks, self.p, self.q, self.workers = int(dimensions), int(walk_length), int(num_walks), p, q, workers
        self.seed = int(torch.randint(0, 2**62, ()).item()) if seed is None else int(seed)
        self.graph = graph
        gen = torch.Generator(device=graph.device).manual_seed(self.seed)
        starts = torch.cat([torch.randperm(graph.n, generator=gen, device=graph.device) for _ in range(self.num_walks)])
        self.walks = random_walks(graph, starts, self.walk_length, p, q, self.seed)

    def fit(self, window: int = 5, negative: int = 5, sample: float = 1e-3, alpha: float = 0.025, min_alpha: float = 1e-4,
            epochs: int = 5, seed: int = 1, vector_size: int | None = None, sg: int = 1, hs: int = 0, min_count: int = 1,
            workers: int | None = None, num_warps: int | None = None) -> SkipGram:
        """gensim ``Word2Vec(walks, ...)``: returns the trained model; ``.wv.vectors`` is the n x dim CUDA tensor and
        ``.wv[i]`` / ``.wv[str(i)]`` a node's vector.  ``num_warps=1`` runs the serial, replayable order."""
        vector_size = self.dimensions if vector_size is None else vector_size
        _check_sg_args(vector_size, window, negative, sample, alpha, min_alpha, epochs, sg, hs, min_count)
        return SkipGram(self.walks, self.graph.n, vector_size, window, negative, sample, alpha, min_alpha, epochs, seed, num_warps).train()
