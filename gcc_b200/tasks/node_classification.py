"""Node classification of frozen embeddings (reference: gcc/tasks/node_classification.py).

10-fold StratifiedKFold; per fold, one-vs-rest L2 logistic regression (C = 1000) on the training rows and
the top-1 class of the per-class probabilities on the test rows (TopKRanker with one label per node);
prints {"Micro-F1": mean over folds}.  Every fold and class is solved by one launch of gccb_logreg_ovr.
"""
import argparse
import os

import numpy as np

from . import check_model
from .evaluate import N_FOLDS, fold_ids, logreg_ovr, per_fold_accuracy


def load_node_dataset(dataset):
    """(edge_index [2, E] int64, one-hot label matrix [n, C]) of a name of the Edgelist family (files under
    ./data, datasets/labeled.py) or an .npz with y (one-hot [n, C] or int labels [n]) and either edge_index
    or a CSR (indptr, indices)."""
    from ..datasets import labeled
    if isinstance(dataset, str) and dataset.endswith(".npz"):
        z = np.load(dataset)
        if "edge_index" in z:
            ei = z["edge_index"].astype(np.int64)
        else:
            indptr = z["indptr"].astype(np.int64)
            ei = np.stack([np.repeat(np.arange(len(indptr) - 1), np.diff(indptr)), z["indices"].astype(np.int64)])
        y = np.asarray(z["y"])
        if y.ndim == 1:
            y = np.eye(int(y.max()) + 1, dtype=np.float32)[y]
        return ei, y.astype(np.float32)
    if dataset in labeled._EDGELIST_NAMES:
        e = labeled.Edgelist(*labeled._EDGELIST_NAMES[dataset])
        return e.data.edge_index.numpy(), e.data.y.numpy()
    raise NotImplementedError("node classification dataset %r: pass an .npz or one of %s"
                              % (dataset, sorted(labeled._EDGELIST_NAMES)))


class NodeClassification(object):
    """Node classification task."""

    def __init__(self, dataset, model, hidden_size, num_shuffle, seed, emb_path="", **model_args):
        check_model(model, "from_numpy")
        self.edge_index, self.label_matrix = load_node_dataset(dataset)
        self.num_nodes, self.num_classes = self.label_matrix.shape
        self.hidden_size = hidden_size
        self.num_shuffle = num_shuffle
        self.seed = seed
        self.emb = np.load(emb_path)

    def features(self):
        """features_matrix of the reference (:44-48): the embedding of every node that appears in an edge, zeros
        for the others (it is filled from the networkx graph of the edge list)."""
        present = np.zeros(self.num_nodes, dtype=bool)
        present[np.asarray(self.edge_index).reshape(-1)] = True
        feats = np.zeros((self.num_nodes, self.hidden_size), dtype=np.float32)
        feats[present] = self.emb[np.flatnonzero(present)]
        return feats

    def train(self):
        return self._evaluate(self.features(), self.label_matrix, self.num_shuffle)

    def _evaluate(self, features_matrix, label_matrix, num_shuffle):
        label_matrix = np.asarray(label_matrix)
        labels = label_matrix.argmax(axis=1)
        folds = fold_ids(labels, self.seed)
        out = logreg_ovr(features_matrix, labels, folds, label_matrix.shape[1], C=1000.0)
        self.last = dict(out, folds=folds, labels=labels)
        # micro-F1 with one true and one predicted label per row is the accuracy
        return {"Micro-F1": float(np.mean(per_fold_accuracy(out["pred"], labels, folds, N_FOLDS)))}


def parser():
    p = argparse.ArgumentParser()
    p.add_argument("--dataset", type=str, required=True)
    p.add_argument("--model", type=str, required=True)
    p.add_argument("--hidden-size", type=int, required=True)
    p.add_argument("--seed", type=int, default=0)
    p.add_argument("--num-shuffle", type=int, default=10)
    p.add_argument("--emb-path", type=str, default="")
    return p


def main(argv=None):
    args = parser().parse_args(argv)
    check_model(args.model, "from_numpy")
    if not os.path.isfile(args.emb_path):
        raise SystemExit("--emb-path %r: no such file" % args.emb_path)
    task = NodeClassification(args.dataset, args.model, args.hidden_size, args.num_shuffle, args.seed,
                              emb_path=args.emb_path)
    ret = task.train()
    print(ret)
    return ret


if __name__ == "__main__":
    main()
