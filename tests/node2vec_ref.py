"""numpy restatement of the node2vec contract in ``include/hicgat.h`` / ``hic_gnn_b200/node2vec.py``: the counter hash, the
closed-form second-order transition probabilities, gensim's count -> ``cum_table`` / keep-probability rules and a serial
skip-gram replay (the order of ``hicgat_sgns_epoch`` with ``num_warps = 1``)."""
from __future__ import annotations

import numpy as np

_M64 = (1 << 64) - 1


def mix64(z: int) -> int:
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _M64
    return z ^ (z >> 31)


def n2v_hash(seed: int, a: int, b: int, c: int) -> int:
    h = mix64((seed & _M64) ^ 0x9E3779B97F4A7C15)
    h = mix64(h ^ (a & _M64))
    h = mix64(h ^ (b & _M64))
    return mix64(h ^ (c & _M64))


def transition_probs(rowptr, col, w, t: int, v: int, p: float, q: float) -> dict:
    """P(x | t, v) of node2vec over the neighbours x of v (t = -1: the first step, P(x | v) ~ w(v, x))."""
    beg, end = int(rowptr[v]), int(rowptr[v + 1])
    xs, wv = np.asarray(col[beg:end]), np.asarray(w[beg:end], dtype=np.float64)
    if t < 0:
        alpha = np.ones_like(wv)
    else:
        nt = set(np.asarray(col[int(rowptr[t]):int(rowptr[t + 1])]).tolist())
        alpha = np.array([1.0 / p if x == t else (1.0 if x in nt else 1.0 / q) for x in xs.tolist()])
    pr = wv * alpha
    return dict(zip(xs.tolist(), (pr / pr.sum()).tolist()))


def cum_table(counts) -> np.ndarray:
    """gensim ``make_cum_table`` (domain 2^31 - 1), accumulated word by word."""
    pw = [float(c) ** 0.75 for c in counts]
    total = sum(pw)
    out, acc = [], 0.0
    for x in pw:
        acc += x
        out.append(round(acc / total * (2**31 - 1)))
    return np.array(out, dtype=np.uint32)


def keep_probability(counts, sample: float) -> np.ndarray:
    c = np.asarray(counts, dtype=np.float64)
    thr = sample * c.sum() if sample else c.sum()
    return np.minimum((np.sqrt(c / thr) + 1.0) * (thr / c), 1.0)


def keep_thresholds(counts, sample: float) -> np.ndarray:
    return (keep_probability(counts, sample) * (2**32 - 1)).astype(np.uint32)


def _sigmoid_grad(f: np.float32, label: float, a: np.float32) -> np.float32:
    if f > 6:
        return np.float32((label - 1.0) * a)
    if f < -6:
        return np.float32(label * a)
    s = np.float32(1.0) / (np.float32(1.0) + np.exp(np.float32(-f)))
    return np.float32((np.float32(label) - s) * a)


def sgns_replay(walks: np.ndarray, syn0: np.ndarray, n: int, window: int, negative: int, sample: float, alpha: float,
                min_alpha: float, epochs: int, seed: int, epoch_range=None):
    """Serial skip-gram epochs over int32 walks (-1 = padding) from the initial ``syn0``; returns (syn0, syn1neg) f32."""
    walks = np.asarray(walks)
    syn0 = np.array(syn0, dtype=np.float32, copy=True)
    syn1 = np.zeros_like(syn0)
    valid = walks >= 0
    counts = np.bincount(walks[valid].astype(np.int64), minlength=n)
    cum = cum_table(counts).astype(np.int64)
    thr = keep_thresholds(counts, sample).astype(np.int64)
    offsets = np.concatenate(([0], np.cumsum(valid.sum(1))))
    total_t = int(offsets[-1])
    for e in (range(epochs) if epoch_range is None else epoch_range):
        for w in range(walks.shape[0]):
            kept, kpos = [], []
            for i, tok in enumerate(walks[w].tolist()):
                if tok < 0:
                    continue
                rp = int(offsets[w]) + i
                if (n2v_hash(seed, e, rp, 0) >> 32) <= thr[tok]:
                    kept.append(tok)
                    kpos.append(rp)
            nk = len(kept)
            for ci in range(nk):
                c, rp = kept[ci], kpos[ci]
                reach = window - ((n2v_hash(seed, e, rp, 1 << 32) >> 32) % window)
                a = np.float32(max(min_alpha, alpha - (alpha - min_alpha) * (e * total_t + rp) / (epochs * total_t)))
                jj = 0
                for j in range(max(0, ci - reach), min(nk - 1, ci + reach) + 1):
                    if j == ci:
                        continue
                    targets = [(c, 1.0)]
                    for k in range(negative):
                        r = n2v_hash(seed, e, rp, (2 << 32) | (jj * negative + k)) >> 32
                        t = int(np.searchsorted(cum, r % int(cum[-1]), side="left"))
                        if t != c:
                            targets.append((t, 0.0))
                    o = kept[j]
                    l1 = syn0[o].copy()
                    neu1e = np.zeros_like(l1)
                    for t, label in targets:
                        f = np.float32(np.dot(l1, syn1[t]))
                        g = _sigmoid_grad(f, label, a)
                        neu1e += g * syn1[t]
                        syn1[t] += g * l1
                    syn0[o] += neu1e
                    jj += 1
    return syn0, syn1
