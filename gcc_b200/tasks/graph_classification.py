"""Graph classification of frozen embeddings (reference: gcc/tasks/graph_classification.py).

10-fold StratifiedKFold; per fold an RBF SVC (C = 100000, gamma='scale', one-vs-one) on the training rows;
prints {"Micro-F1": mean test accuracy over folds}.  Every fold and class pair is solved by one launch of
gccb_svc_ovo.
"""
import argparse
import os

import numpy as np

from . import check_model
from .evaluate import fold_ids, per_fold_accuracy, svc_ovo


def load_graph_labels(dataset):
    """int64 graph labels of a TU name (files under ./data/<NAME>/, numbered like datasets/labeled.py) or of an
    .npz with graph_labels."""
    from ..datasets import labeled
    if isinstance(dataset, str) and dataset.endswith(".npz"):
        return np.asarray(np.load(dataset)["graph_labels"], dtype=np.int64).reshape(-1)
    if dataset in labeled._TU_NAMES:
        name = labeled._TU_NAMES[dataset]
        raw = np.loadtxt(os.path.join("data", name, name + "_graph_labels.txt"), dtype=np.int64).reshape(-1)
        return np.searchsorted(np.unique(raw), raw).astype(np.int64)
    raise NotImplementedError("graph classification dataset %r: pass an .npz or one of %s"
                              % (dataset, labeled.GRAPH_CLASSIFICATION_DSETS))


class GraphClassification(object):
    def __init__(self, dataset, model, hidden_size, num_shuffle, seed, emb_path="", **model_args):
        check_model(model, "from_numpy_graph")
        self.labels = load_graph_labels(dataset)
        self.num_classes = int(self.labels.max()) + 1
        self.hidden_size = hidden_size
        self.num_shuffle = num_shuffle
        self.seed = seed
        self.emb = np.load(emb_path)

    def train(self):
        return self.svc_classify(self.emb, self.labels, False)

    def svc_classify(self, x, y, search):
        if search:
            raise NotImplementedError("the C grid search (search=True) is not implemented; the reference's CLI "
                                      "never enables it")
        y = np.asarray(y, dtype=np.int64)
        folds = fold_ids(y, self.seed)
        out = svc_ovo(x, y, folds, int(y.max()) + 1, C=100000.0)
        self.last = dict(out, folds=folds)
        return {"Micro-F1": float(np.mean(per_fold_accuracy(out["pred"], y, folds)))}


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
    check_model(args.model, "from_numpy_graph")
    if not os.path.isfile(args.emb_path):
        raise SystemExit("--emb-path %r: no such file" % args.emb_path)
    task = GraphClassification(args.dataset, args.model, args.hidden_size, args.num_shuffle, args.seed,
                               emb_path=args.emb_path)
    ret = task.train()
    print(ret)
    return ret


if __name__ == "__main__":
    main()
