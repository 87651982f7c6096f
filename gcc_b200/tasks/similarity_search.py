"""Similarity search between two PanTher graphs (reference: gcc/tasks/similarity_search.py).

For every name present in both .dict files, rank the true match among the embeddings of all shared names of
graph 2 by cosine similarity to the embedding in graph 1; prints {"Recall @ 20": .., "Recall @ 40": ..}.
The ranks come from one launch of gccb_sim_rank: rank = number of candidates scoring strictly higher.
"""
import argparse
import os

import numpy as np

from . import check_model
from .evaluate import sim_rank

K_LIST = (20, 40)


def load_pair(dataset_1, dataset_2):
    """([edge_index_1, edge_index_2], [names_1, names_2]) of two PanTher names (files under ./data/panther)."""
    from ..datasets.panther import PANTHER_ROOT, SSDataset
    data = SSDataset(PANTHER_ROOT, dataset_1, dataset_2).data
    return [d.edge_index.numpy() for d in data], [d.y for d in data]


def load_npz(path):
    """An .npz with keys_1 / ids_1 / keys_2 / ids_2 (the two name -> node id maps); edge lists are optional
    (edge_index_1 / edge_index_2)."""
    z = np.load(path)
    dicts = [dict(zip((str(k) for k in z["keys_%d" % i]), (int(v) for v in z["ids_%d" % i]))) for i in (1, 2)]
    edges = [z["edge_index_%d" % i] if "edge_index_%d" % i in z else None for i in (1, 2)]
    return edges, dicts


class SimilaritySearch(object):
    def __init__(self, dataset_1, dataset_2, model, hidden_size, emb_path_1="", emb_path_2="", **model_args):
        check_model(model, "from_numpy_align")
        if dataset_1.endswith(".npz"):
            self.edges, self.dicts = load_npz(dataset_1)
        else:
            self.edges, self.dicts = load_pair(dataset_1, dataset_2)
        self.hidden_size = hidden_size
        self.embs = [np.load(emb_path_1), np.load(emb_path_2)]

    def _features(self, i):
        """_train_wrap (:27-36): one row per node of the edge list's graph, which must be the embedding's row
        count (FromNumpyAlign); rows of nodes outside every edge stay zero."""
        emb, ei = self.embs[i], self.edges[i]
        if ei is None:
            return np.asarray(emb, dtype=np.float32)
        ei = np.asarray(ei).reshape(-1)
        nodes = np.unique(ei)
        if len(nodes) != emb.shape[0]:
            raise ValueError("embedding %d has %d rows, its graph %d nodes" % (i + 1, emb.shape[0], len(nodes)))
        feats = np.zeros((len(nodes), emb.shape[1]), dtype=np.float32)
        inside = nodes[nodes < len(nodes)]
        feats[inside] = emb[inside]
        return feats

    def train(self):
        return self._evaluate(self._features(0), self._features(1), self.dicts[0], self.dicts[1])

    def _evaluate(self, emb_1, emb_2, dict_1, dict_2):
        # shared names whose ids are rows of both embeddings (a .dict-only node has an id past the graph's)
        shared = sorted(k for k in set(dict_1) & set(dict_2)
                        if dict_1[k] < emb_1.shape[0] and dict_2[k] < emb_2.shape[0])
        idx1 = np.array([dict_1[k] for k in shared], dtype=np.int32)
        idx2 = np.array([dict_2[k] for k in shared], dtype=np.int32)
        rank = sim_rank(emb_1, emb_2, idx1, idx2)
        self.last = dict(rank=rank, keys=shared, idx1=idx1, idx2=idx2)
        return dict(("Recall @ %d" % k, float(np.mean(rank < k))) for k in K_LIST)


def parser():
    p = argparse.ArgumentParser()
    p.add_argument("--dataset", type=str, required=True, help="<name1>_<name2> of data/panther, or an .npz")
    p.add_argument("--model", type=str, required=True)
    p.add_argument("--hidden-size", type=int, required=True)
    p.add_argument("--seed", type=int, default=0)
    p.add_argument("--emb-path-1", type=str, default="")
    p.add_argument("--emb-path-2", type=str, default="")
    return p


def main(argv=None):
    args = parser().parse_args(argv)
    check_model(args.model, "from_numpy_align")
    for p in (args.emb_path_1, args.emb_path_2):
        if not os.path.isfile(p):
            raise SystemExit("embedding %r: no such file" % p)
    if args.dataset.endswith(".npz"):
        d1, d2 = args.dataset, None
    else:
        parts = args.dataset.split("_")
        if len(parts) != 2:
            raise SystemExit("--dataset %r: expected <name1>_<name2>" % args.dataset)
        d1, d2 = parts
    task = SimilaritySearch(d1, d2, args.model, args.hidden_size, emb_path_1=args.emb_path_1,
                            emb_path_2=args.emb_path_2)
    ret = task.train()
    print(ret)
    return ret


if __name__ == "__main__":
    main()
