#!/usr/bin/env python
"""generate.py -- the reference's inference export (generate.py:33-134) on the B200 kernels.

Loads a pretraining checkpoint (`--load-path`, written by this repo's train.py or by the reference:
same `model` state_dict keys), walks two ego-nets from EVERY node of the target graph in order
(NodeClassificationDataset, graph_dataset.py:279-309), encodes both with the model in eval mode
(BatchNorm running statistics, no dropout) and saves (f(q) + f(k)) / 2 as `<model_folder>/<name>.npy`
(generate.py:48-53,133-134).  The reference batches the whole dataset into ONE batch (:90); here
the nodes go through in `--batch-size` chunks -- eval-mode encoding is per-graph, so the result is
the same.  `--dataset` is an .npz CSR (indptr, indices), `synthetic-<kind>`, or one of the reference's
names whose files are under ./data: the airport / h-index edge lists, the PanTher graphs (kdd, icdm, sigir,
cikm, sigmod, icde; multi-edges collapsed) and the five TU graph-classification sets.

Graph-classification inputs (a TU name, or an .npz with graph_sizes) export ONE embedding per graph
(generate.py:74-81): the eval-mode encoding of the whole graph, seeded at its max-degree node.  Both of
the reference's views are the whole graph, so their mean is that encoding.
"""
import argparse
import os

import numpy as np
import torch

from gcc_b200.datasets import labeled, panther, synthetic
from gcc_b200.datasets.graph_dataset import NodeClassificationDataset
from gcc_b200.models import GraphEncoder

# checkpoint["opt"] attribute -> GraphEncoder keyword (train.py:601-620 builds the model from these)
ENCODER_KWARGS = {
    "positional_embedding_size": "positional_embedding_size", "max_node_freq": "max_node_freq",
    "max_edge_freq": "max_edge_freq", "max_degree": "max_degree",
    "freq_embedding_size": "freq_embedding_size", "degree_embedding_size": "degree_embedding_size",
    "output_dim": "hidden_size", "node_hidden_dim": "hidden_size", "edge_hidden_dim": "hidden_size",
    "num_layers": "num_layer", "num_step_set2set": "set2set_iter",
    "num_layer_set2set": "set2set_lstm_layer", "gnn_model": "model", "norm": "norm",
}


def test_moco(train_loader, model, opt):
    """Embedding of every item: mean of the two views' eval-mode features (generate.py:33-53)."""
    model.eval()
    chunks = []
    with torch.no_grad():
        for view_q, view_k, valid in train_loader:
            pair = torch.stack([model(view_q), model(view_k)])
            if pair.shape[1:] != (view_q.batch_size, opt.hidden_size):
                raise RuntimeError("encoder returned %s" % (tuple(pair.shape),))
            chunks.append(pair.mean(0)[:valid].cpu())        # the last chunk is padded: keep the valid pairs
    return torch.cat(chunks)


def is_graph_dataset(name):
    """A TU name or an .npz of a disjoint union with graph_sizes."""
    if name.endswith(".npz"):
        with np.load(name) as z:
            return "graph_sizes" in z
    return name in labeled.GRAPH_CLASSIFICATION_DSETS


def graph_embeddings(name, encoder, batch_size, positional_embedding_size=32):
    """One eval-mode embedding per whole graph, in dataset order."""
    ds = labeled.GraphClassificationDatasetLabeled(name, positional_embedding_size=positional_embedding_size,
                                                   device=encoder_device(encoder), batch_size=batch_size)
    encoder.eval()
    chunks = []
    with torch.no_grad():
        for graph_q, _ in ds.batches():
            chunks.append(encoder(graph_q).cpu())
    return torch.cat(chunks)


def encoder_device(encoder):
    return next(encoder.parameters()).device


def resolve_graph(name, nodes, edges):
    """`--dataset`: an .npz path is passed through; the reference's node datasets are read from ./data;
    synthetic-chunglu / synthetic-er are generated."""
    if name.endswith(".npz"):
        return name
    if name in labeled._EDGELIST_NAMES:
        e = labeled.Edgelist(*labeled._EDGELIST_NAMES[name])
        return labeled.graph_from_edge_index(e.data.edge_index.numpy())
    if name in panther.PANTHER_NAMES:
        e = panther.SSSingleDataset(panther.PANTHER_ROOT, name)
        return labeled.graph_from_edge_index(e.data.edge_index.numpy())
    if name.endswith("chunglu"):
        return synthetic.chung_lu(nodes, edges, 0.5, seed=0)
    return synthetic.erdos_renyi(nodes, edges, seed=0)


def main(args_test):
    path = args_test.load_path
    if not os.path.isfile(path):
        raise SystemExit("=> no checkpoint found at '{}'".format(path))
    if not torch.cuda.is_available():
        raise SystemExit("generate.py needs a CUDA device (sm_100a); there is no CPU path")
    print("=> loading checkpoint '{}'".format(path))
    ckpt = torch.load(path, map_location="cpu", weights_only=False)
    print("=> loaded successfully '{}' (epoch {})".format(path, ckpt["epoch"]))
    opt = ckpt["opt"]
    gpu = args_test.gpu or 0
    torch.cuda.set_device(gpu)
    opt.device = torch.device("cuda", gpu)

    encoder = GraphEncoder(degree_input=True, **{kw: getattr(opt, attr) for kw, attr in ENCODER_KWARGS.items()})
    encoder.load_state_dict(ckpt["model"])
    encoder = encoder.to(opt.device)
    del ckpt

    if is_graph_dataset(args_test.dataset):
        emb = graph_embeddings(args_test.dataset, encoder, args_test.batch_size, opt.positional_embedding_size)
    else:
        nodes = NodeClassificationDataset(
            dataset=resolve_graph(args_test.dataset, args_test.graph_nodes, args_test.graph_edges),
            rw_hops=opt.rw_hops, subgraph_size=opt.subgraph_size, restart_prob=opt.restart_prob,
            positional_embedding_size=opt.positional_embedding_size, device=opt.device,
            seed=getattr(opt, "seed", 0), batch_size=args_test.batch_size)
        emb = test_moco(nodes, encoder, opt)

    stem = os.path.basename(args_test.dataset)
    stem = stem[:-4] if stem.endswith(".npz") else stem
    out = os.path.join(getattr(opt, "model_folder", "."), stem)
    np.save(out, emb.numpy())
    print("saved {} embeddings of dim {} to {}.npy".format(emb.shape[0], emb.shape[1], out))
    return emb


if __name__ == "__main__":
    ap = argparse.ArgumentParser("inference export: node embeddings from a pretraining checkpoint")
    ap.add_argument("--load-path", type=str, required=True, help="path to load model")
    ap.add_argument("--dataset", type=str, default="synthetic-er",
                    help=".npz CSR file (indptr, indices; graph_sizes + graph_labels for one embedding per graph), "
                         "synthetic-er / synthetic-chunglu, or a dataset name of the reference with its files "
                         "under ./data")
    ap.add_argument("--graph-nodes", type=int, default=2000, help="size of a synthetic target graph")
    ap.add_argument("--graph-edges", type=int, default=10000)
    ap.add_argument("--batch-size", type=int, default=256, help="nodes encoded per launch group")
    ap.add_argument("--gpu", default=None, type=int, help="GPU id to use.")
    main(ap.parse_args())
