#!/usr/bin/env python
"""The reference's pipeline on its own shipped data, end to end on one B200, with the drop-in modules:

    contact list (Data/GM12878_1mb_chr19_list.txt)      utils.convert_to_matrix      utils.py:10-26
    -> KR normalisation                                 kr.kr_norm                   normalize.R / r_utils.R:1-93
    -> graph + wish distances                           utils.load_input / wish_target   utils.py:29-80
    -> GAT net, MSE + Pearson loop until |d loss| <= thresh   train.fit              HiC_GAT_generalize_directly.py:182-260
    -> dSCC                                             metrics.dscc                 HiC-GNN_main.py:135-139

The contact list comes from tests/golden (a copy of the reference's fixture recorded by make_golden.py).  The node
features are seeded random features (``--features random``, default) or node2vec embeddings of the map's own graph with the
reference's parameters (``--features node2vec``: ``Node2Vec(dimensions=512, walk_length=150, num_walks=50, p=1.75, q=0.4,
seed=42).fit()``, HiC_GAT_generalize_directly.py:153-155, on the GPU through hic_gnn_b200.node2vec).

    python examples/chr19_gat_hic.py [--steps 300] [--model gat|net] [--features random|node2vec]
"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np
import torch

from hic_gnn_b200 import kr, metrics, models, node2vec, train, utils


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=300, help="upper bound; the reference's stop rule may end the loop earlier")
    ap.add_argument("--model", default="gat", choices=["gat", "net"])
    ap.add_argument("-lr", type=float, default=1e-3)
    ap.add_argument("-thresh", type=float, default=1e-8)
    ap.add_argument("--features", default="random", choices=["random", "node2vec"])
    args = ap.parse_args()
    contacts = np.load(os.path.join(ROOT, "tests", "golden", "reference_golden.npz"))["1mb_list"]
    raw = utils.convert_to_matrix(contacts)            # dense symmetric counts on the GPU
    raw.fill_diagonal_(0)                               # HiC-GNN_main.py:80
    normed = kr.kr_norm(raw)                            # replaces the Rscript subprocess
    n = normed.shape[0]
    if args.features == "node2vec":
        graph = utils.load_input(normed, torch.zeros(n, 1)).edge_index
        feats = node2vec.Node2Vec(graph, dimensions=512, walk_length=150, num_walks=50, p=1.75, q=0.4, seed=42).fit().wv.vectors
    else:
        feats = 0.25 * torch.randn(n, 512, generator=torch.Generator().manual_seed(42))
    data = utils.load_input(normed, feats)              # CSR graph, bit-exact with the reference
    target = utils.wish_target(data.y, 1.0)             # cont2dist(., 1) as the f32 layout the loss kernel streams
    torch.manual_seed(42)
    model = (models.GATNetSelectiveResidualsUpdated if args.model == "gat" else models.Net)().cuda()
    mode = "mse_pearson" if args.model == "gat" else "mse"
    hist = train.fit(model, data.x.float(), data.edge_index, target, mode=mode, lr=args.lr, thresh=args.thresh, max_steps=args.steps,
                     use_cuda_graph=True, check_every=10)
    with torch.no_grad():
        coords = model.get_model(data.x.float(), data.edge_index)
    print(f"features={args.features} loci={n} nnz={data.edge_index.nnz} steps={len(hist)} loss {hist[0]:.5f} -> {hist[-1]:.5f} dSCC={metrics.dscc(coords, target):.4f}")
    return hist, coords


if __name__ == "__main__":
    main()
