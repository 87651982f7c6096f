"""PanTher co-author graphs of the similarity-search task (reference: gcc/datasets/data_util.py:111-191).

`<root>/<name>.graph`: a header line, then "x y t" per line (an edge of multiplicity t); `<name>.dict`:
"name<TAB>x" per line.  Node ids are numbered in order of first appearance in the .graph file; a .dict id
missing from the graph gets the next id.  Every edge is listed t times in both directions, like the
reference (graph_from_edge_index collapses the multi-edges for the sampler).
"""
import os

import numpy as np
import torch

from .labeled import Data

PANTHER_NAMES = ("kdd", "icdm", "sigir", "cikm", "sigmod", "icde")
PANTHER_ROOT = "data/panther"


def _read_graph(root, name):
    node2id, edges = {}, []
    with open(os.path.join(root, name + ".graph")) as f:
        f.readline()
        for line in f:
            if not line.strip():
                continue
            x, y, t = (int(v) for v in line.split())
            for v in (x, y):
                if v not in node2id:
                    node2id[v] = len(node2id)
            edges += [(node2id[x], node2id[y]), (node2id[y], node2id[x])] * t
    e = np.asarray(edges, dtype=np.int64).reshape(-1, 2)
    return torch.from_numpy(e.T.copy()), node2id


class SSSingleDataset:
    """data_util.py:111-144: the graph alone (generate.py's input for a PanTher name)."""

    def __init__(self, root, name):
        edge_index, self.node2id = _read_graph(root, name)
        self.data = Data(x=None, edge_index=edge_index, y=None)
        self.transform = None

    def get(self, idx):
        assert idx == 0
        return self.data


class SSDataset:
    """data_util.py:146-191: two graphs; .data[i].y is the {name: node id} map of graph i."""

    def __init__(self, root, name1, name2):
        self.data, self.node2id = [], []
        for name in (name1, name2):
            edge_index, node2id = _read_graph(root, name)
            names = {}
            with open(os.path.join(root, name + ".dict")) as f:
                for line in f:
                    if not line.strip():
                        continue
                    key, sx = line.rstrip("\n").split("\t")
                    x = int(sx)
                    if x not in node2id:
                        node2id[x] = len(node2id)
                    names[key] = node2id[x]
            self.data.append(Data(x=None, edge_index=edge_index, y=names))
            self.node2id.append(node2id)
        self.node2id_1, self.node2id_2 = self.node2id
        self.transform = None

    def get(self, idx):
        assert idx == 0
        return self.data
