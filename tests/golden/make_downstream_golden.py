"""Write tests/golden/downstream_golden.npz: the original project's downstream evaluation on seeded
synthetic embeddings.

It runs the REAL NodeClassification._evaluate, GraphClassification.svc_classify, SimilaritySearch._evaluate
and the PanTher readers (SSSingleDataset, SSDataset) of the original code base (path: argv[1] or $GCC_REF),
with dgl_stub.py standing in for DGL and an empty module for seaborn, which gcc.models.emb imports.
Stored: the inputs, the returned result dicts, and the per-fold predictions of the same sklearn estimators.

    python tests/golden/make_downstream_golden.py /path/to/GCC
"""
import os
import sys
import tempfile
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
REF = sys.argv[1] if len(sys.argv) > 1 else os.environ.get("GCC_REF", "")
import dgl_stub  # noqa: E402

dgl_stub.install()
sys.modules.setdefault("seaborn", types.ModuleType("seaborn"))
sys.path.insert(0, REF)

import torch  # noqa: E402
from sklearn.linear_model import LogisticRegression  # noqa: E402
from sklearn.model_selection import StratifiedKFold  # noqa: E402
from sklearn.svm import SVC  # noqa: E402

from gcc.datasets.data_util import SSDataset, SSSingleDataset  # noqa: E402
from gcc.tasks.graph_classification import GraphClassification  # noqa: E402
from gcc.tasks.node_classification import NodeClassification, TopKRanker  # noqa: E402
from gcc.tasks.similarity_search import SimilaritySearch  # noqa: E402


def blobs(rng, n, d, k, spread):
    """Overlapping Gaussian classes: scores land well below 1."""
    y = rng.integers(0, k, n)
    centers = rng.normal(size=(k, d)) * spread
    return (centers[y] + rng.normal(size=(n, d))).astype(np.float32), y


def main():
    rng = np.random.default_rng(20261017)
    out = {}
    # --- node classification: usa_airport-like 1190 x 64, 4 classes; a few rows far out saturate several classes
    X, y = blobs(rng, 1190, 64, 4, 0.35)
    X[:6] *= 60.0
    Y = np.zeros((len(y), 4), np.float32)
    Y[np.arange(len(y)), y] = 1
    task = NodeClassification.__new__(NodeClassification)
    task.seed = 0
    res = task._evaluate(X.astype(np.float64), torch.Tensor(Y), 10)
    preds = np.full(len(y), -1, np.int64)
    folds = np.full(len(y), -1, np.int64)
    ties = 0
    for f, (tr, te) in enumerate(StratifiedKFold(n_splits=10, shuffle=True, random_state=0).split(np.zeros(len(y)), y)):
        clf = TopKRanker(LogisticRegression(C=1000))
        clf.fit(X[tr].astype(np.float64), torch.Tensor(Y[tr]))
        p = clf.predict(X[te].astype(np.float64), [1] * len(te)).toarray()
        preds[te] = p.argmax(1)
        probs = np.asarray(clf.predict_proba(X[te].astype(np.float64)))
        ties += int(np.sum((probs == 1.0).sum(1) > 1))
        folds[te] = f
    out.update(nc_x=X, nc_y=y, nc_pred=preds, nc_folds=folds, nc_micro_f1=res["Micro-F1"], nc_saturated_ties=ties)
    # --- graph classification: IMDB-MULTI-like 1500 x 64, 3 classes
    X, y = blobs(rng, 1500, 64, 3, 0.3)
    task = GraphClassification.__new__(GraphClassification)
    task.seed = 0
    res = task.svc_classify(X, y, False)
    preds = np.full(len(y), -1, np.int64)
    for tr, te in StratifiedKFold(n_splits=10, shuffle=True, random_state=0).split(X, y):
        preds[te] = SVC(C=100000).fit(X[tr], y[tr]).predict(X[te])
    out.update(gc_x=X, gc_y=y, gc_pred=preds, gc_micro_f1=res["Micro-F1"])
    # --- similarity search: 300 / 320 rows, shared, non-shared and out-of-range keys
    n1, n2, d = 300, 320, 16
    base = rng.normal(size=(400, d))
    e1 = (base[:n1] + 0.8 * rng.normal(size=(n1, d))).astype(np.float32)
    perm = rng.permutation(400)[:n2]
    e2 = (base[perm] + 0.8 * rng.normal(size=(n2, d))).astype(np.float32)
    d1 = {"a%d" % i: i for i in range(n1)}
    d2 = {"a%d" % int(p): j for j, p in enumerate(perm) if p < n1}
    d2.update({"x%d" % j: j for j in range(5)})                  # names only graph 2 has
    d1.update({"a%d" % int(perm[k]): n1 + k for k in range(3) if perm[k] >= n1})
    d2.update({"a%d" % i: n2 + i for i in range(3)})              # id past graph 2's rows
    res = SimilaritySearch._evaluate(None, e1.astype(np.float64), e2.astype(np.float64), dict(d1), dict(d2))
    for i, dd in ((1, d1), (2, d2)):
        out["ss_keys_%d" % i] = np.array(list(dd.keys()))
        out["ss_ids_%d" % i] = np.array(list(dd.values()), np.int64)
    out.update(ss_e1=e1, ss_e2=e2, ss_recall20=res["Recall @ 20"], ss_recall40=res["Recall @ 40"])
    # --- PanTher readers on a small written pair (multi-edges, a .dict name missing from the graph)
    with tempfile.TemporaryDirectory() as tmp:
        g1 = "header\n10 20 1\n20 30 2\n30 10 1\n40 10 3\n"
        g2 = "header\n7 8 2\n8 9 1\n9 7 1\n"
        dict1 = "alice\t20\nbob\t40\ncarol\t99\n"
        dict2 = "alice\t8\nbob\t7\ndave\t55\n"
        for name, txt in (("p1.graph", g1), ("p2.graph", g2), ("p1.dict", dict1), ("p2.dict", dict2)):
            open(os.path.join(tmp, name), "w").write(txt)
        single = SSSingleDataset(tmp, "p1").data
        pair = SSDataset(tmp, "p1", "p2")
        out.update(pt_graph_1=g1, pt_graph_2=g2, pt_dict_1=dict1, pt_dict_2=dict2,
                   pt_single_edge_index=single.edge_index.numpy(),
                   pt_edge_index_1=pair.data[0].edge_index.numpy(), pt_edge_index_2=pair.data[1].edge_index.numpy(),
                   pt_names_1=np.array(sorted(pair.data[0].y)), pt_ids_1=np.array([pair.data[0].y[k] for k in sorted(pair.data[0].y)]),
                   pt_names_2=np.array(sorted(pair.data[1].y)), pt_ids_2=np.array([pair.data[1].y[k] for k in sorted(pair.data[1].y)]))
    np.savez_compressed(os.path.join(HERE, "downstream_golden.npz"), **out)
    print({k: v for k, v in out.items() if np.ndim(v) == 0})


if __name__ == "__main__":
    main()
