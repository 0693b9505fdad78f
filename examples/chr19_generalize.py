#!/usr/bin/env python
"""BASELINE.json configs[1]: GM12878 chr19 500 kb GAT generalisation from the 1 Mb model
(HiC_GAT_generalize_directly.py), end to end on one B200 with the drop-in modules:

    1 Mb and 500 kb contact lists          utils.convert_to_matrix -> kr.kr_norm         utils.py:10-26, r_utils.R:1-93
    train on the 1 Mb map                  utils.load_input / wish_target / train.fit    HiC_GAT_generalize_directly.py:182-260
    save / reload the weights              state_dict round trip (reference keys)        :282, :312-314
    align the 500 kb embeddings            utils.domain_alignment                        :316, utils.py:83-108
    500 kb structure from the 1 Mb model   utils.load_input + model.get_model            :317-323
    dSCC of the generalised structure      metrics.dscc                                  :335
    PDB file                               utils.WritePDB(coords * 100, ...)             :365

The contact lists come from tests/golden (copies of the reference's Data/ fixtures recorded by make_golden.py).
``--features node2vec`` embeds each resolution's own graph with the reference's node2vec call (``Node2Vec(dimensions=512,
walk_length=150, num_walks=50, p=1.75, q=0.4, seed=42).fit()``, HiC_GAT_generalize_directly.py:153-155, on the GPU through
hic_gnn_b200.node2vec) and aligns the 500 kb embeddings onto the 1 Mb ones with ``domain_alignment``: the reference's flow.
``--features random`` (default) uses seeded stand-ins instead: the 500 kb stand-ins are a rotated, noisy interleaving of the
1 Mb ones, so that the alignment has something to recover.

    python examples/chr19_generalize.py [--steps 300] [--loss mse_pearson|mse_pearson_grad] [--features random|node2vec]
                                        [--track-dscc] [--out /tmp/chr19_500kb_generalized_structure.pdb]

``--loss mse_pearson`` (default) is the reference's loss, whose Pearson term carries no gradient; ``mse_pearson_grad`` trains
on the same total with the gradient of the (1 - r) term as well.  ``--track-dscc`` records the dSCC of every training step on the
device (``fit(dscc_out=...)``), as the reference keeps ``SpRho`` (:242, :189-192), and prints the curve every 50 steps and at the end.
"""
import argparse
import io
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np
import torch

from hic_gnn_b200 import kr, metrics, models, node2vec, train, utils


def normed_map(contacts):
    raw = utils.convert_to_matrix(contacts)
    raw.fill_diagonal_(0)                               # HiC_GAT_generalize_directly.py:118
    return kr.kr_norm(raw)                              # replaces the Rscript subprocess


def node2vec_features(normed):
    graph = utils.load_input(normed, torch.zeros(normed.shape[0], 1)).edge_index
    model = node2vec.Node2Vec(graph, dimensions=512, walk_length=150, num_walks=50, p=1.75, q=0.4, workers=1, seed=42)  # :153-154
    return model.fit().wv.vectors                      # :155


def random_features(n1, n2):
    rng = np.random.default_rng(42)
    emb_trained = 0.25 * rng.standard_normal((n1, 512))
    q, _ = np.linalg.qr(rng.standard_normal((512, 512)))
    emb_untrained = np.repeat(emb_trained, 2, axis=0)[:n2] @ q + 0.01 * rng.standard_normal((min(2 * n1, n2), 512))
    if emb_untrained.shape[0] < n2:
        emb_untrained = np.vstack([emb_untrained, 0.25 * rng.standard_normal((n2 - emb_untrained.shape[0], 512))])
    return emb_trained, emb_untrained


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("-lr", type=float, default=1e-3)
    ap.add_argument("-thresh", type=float, default=1e-8)
    ap.add_argument("-conversion", type=float, default=1.0)
    ap.add_argument("--loss", default="mse_pearson", choices=["mse_pearson", "mse_pearson_grad"])
    ap.add_argument("--features", default="random", choices=["random", "node2vec"])
    ap.add_argument("--track-dscc", action="store_true")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    g = np.load(os.path.join(ROOT, "tests", "golden", "reference_golden.npz"))
    list_trained, list_untrained = g["1mb_list"], g["500kb_list"]
    normed_trained, normed_untrained = normed_map(list_trained), normed_map(list_untrained)
    n1, n2 = normed_trained.shape[0], normed_untrained.shape[0]
    if args.features == "node2vec":
        emb_trained, emb_untrained = node2vec_features(normed_trained), node2vec_features(normed_untrained)
    else:
        emb_trained, emb_untrained = random_features(n1, n2)

    # ---- train on the 1 Mb map
    data = utils.load_input(normed_trained, emb_trained)
    target = utils.wish_target(data.y, args.conversion)
    torch.manual_seed(42)
    model = models.GATNetSelectiveResidualsUpdated().cuda()
    sprho = [] if args.track_dscc else None
    hist = train.fit(model, data.x.float(), data.edge_index, target, mode=args.loss, lr=args.lr, thresh=args.thresh, max_steps=args.steps,
                     use_cuda_graph=True, check_every=10, dscc_out=sprho)
    if sprho is not None:
        for s in list(range(0, len(sprho), 50)) + [len(sprho) - 1]:
            print(f"step {s:4d}: loss {hist[s]:.5f} dSCC {sprho[s]:.4f}")
    with torch.no_grad():
        dscc_trained = metrics.dscc(model.get_model(data.x.float(), data.edge_index), target)
    buf = io.BytesIO()
    torch.save(model.state_dict(), buf)                 # reference: torch.save(model.state_dict(), ..._weights.pt)

    # ---- generalise to the 500 kb map
    model = models.GATNetSelectiveResidualsUpdated().cuda()
    buf.seek(0)
    model.load_state_dict(torch.load(buf))
    model.eval()
    fitembed = utils.domain_alignment(list_trained, list_untrained, emb_trained, emb_untrained)
    data_fit = utils.load_input(normed_untrained, fitembed)
    target_fit = utils.wish_target(data_fit.y, args.conversion)
    with torch.no_grad():
        coords = model.get_model(data_fit.x.float(), data_fit.edge_index)
    dscc_generalised = metrics.dscc(coords, target_fit)
    if args.out:
        utils.WritePDB(coords * 100, args.out)
    print(f"features {args.features}, loss {args.loss}: trained on {n1} loci: steps={len(hist)} loss {hist[0]:.5f} -> {hist[-1]:.5f} dSCC={dscc_trained:.4f}; "
          f"generalised to {n2} loci: dSCC={dscc_generalised:.4f}" + (f"; wrote {args.out}" if args.out else ""))
    return hist, coords, dscc_trained, dscc_generalised


if __name__ == "__main__":
    main()
