"""B200: the downstream kernels (csrc/downstream.cu) against sklearn / numpy and against the original project's
evaluation on the fixture (tests/golden/make_downstream_golden.py), the graph-level export of generate.py and
one run of every task CLI."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gold(golden):
    return golden("downstream_golden")


def test_logreg_weights_match_tight_optimum():
    from sklearn.linear_model import LogisticRegression
    from gcc_b200.tasks.evaluate import fold_ids, logreg_ovr
    rng = np.random.default_rng(7)
    n, d, C = 600, 32, 3
    y = rng.integers(0, C, n)
    X = (rng.normal(size=(C, d))[y] * 0.4 + rng.normal(size=(n, d))).astype(np.float32)
    folds = fold_ids(y, 0)
    out = logreg_ovr(X, y, folds, C, C=1000.0)
    assert np.all(out["status"] == 0), out["status"]
    for f in (0, 5):
        tr = folds != f
        for c in range(C):
            ref = LogisticRegression(C=1000.0, tol=1e-12, max_iter=1000000).fit(X[tr].astype(np.float64), y[tr] == c)
            want = np.concatenate([ref.coef_[0], ref.intercept_])
            got = out["weights"][f, c]
            assert np.linalg.norm(got - want) <= 1e-6 * np.linalg.norm(want), (f, c, np.abs(got - want).max())


def test_node_classification_vs_reference_fixture(gold):
    from gcc_b200.tasks.evaluate import fold_ids, logreg_ovr, per_fold_accuracy
    X, y = gold["nc_x"], gold["nc_y"]
    folds = fold_ids(y, 0)
    assert np.array_equal(folds, gold["nc_folds"])
    out = logreg_ovr(X, y, folds, 4, C=1000.0)
    assert not np.any(out["status"] == 1), out["status"]
    for f in range(10):
        te = folds == f
        assert np.mean(out["pred"][te] == gold["nc_pred"][te]) >= 0.99, f
    f1 = float(np.mean(per_fold_accuracy(out["pred"], y, folds)))
    assert abs(f1 - float(gold["nc_micro_f1"])) <= 0.005, (f1, float(gold["nc_micro_f1"]))
    # rows scaled far out saturate several class probabilities to 1.0 in fp64 (the reference's run had
    # nc_saturated_ties such rows): the tie goes to the highest class, as np.argsort(...)[-1:] returned
    saturated = out["prob"] == 1.0
    tied = np.flatnonzero(saturated.sum(1) > 1)
    assert int(gold["nc_saturated_ties"]) > 0 and len(tied) > 0
    for i in tied:
        assert out["pred"][i] == np.flatnonzero(saturated[i]).max(), (i, out["prob"][i])
        assert out["pred"][i] == gold["nc_pred"][i], (i, out["pred"][i], gold["nc_pred"][i])


def _dual(coef, K):
    return 0.5 * coef @ K @ coef - np.abs(coef).sum()


def test_graph_classification_vs_reference_fixture_and_sklearn_dual(gold):
    from sklearn.svm import SVC
    from gcc_b200.tasks.evaluate import fold_ids, per_fold_accuracy, svc_ovo
    X, y = gold["gc_x"], gold["gc_y"]
    folds = fold_ids(y, 0)
    out = svc_ovo(X, y, folds, 3, C=100000.0)
    assert np.all(out["status"] == 0), out["status"]
    for f in range(10):
        te = folds == f
        mine = int(np.sum(out["pred"][te] == y[te]))
        ref = int(np.sum(gold["gc_pred"][te] == y[te]))
        assert abs(mine - ref) <= 1, (f, mine, ref)
    acc = float(np.mean(per_fold_accuracy(out["pred"], y, folds)))
    assert abs(acc - float(gold["gc_micro_f1"])) <= 0.005, (acc, float(gold["gc_micro_f1"]))
    Xd = X.astype(np.float64)
    sq = (Xd ** 2).sum(1)
    for f in (0, 7):
        tr = folds != f
        assert np.isclose(out["gamma"][f], 1.0 / (X.shape[1] * Xd[tr].var()), rtol=1e-10)
        K = np.exp(-out["gamma"][f] * (sq[:, None] + sq[None] - 2 * Xd @ Xd.T))
        for p, (a, b) in enumerate(((0, 1), (0, 2), (1, 2))):
            rows = np.flatnonzero(tr & ((y == a) | (y == b)))
            sk = SVC(C=100000.0, gamma=out["gamma"][f]).fit(Xd[rows], np.where(y[rows] == a, 1, -1))
            want = np.zeros(len(y))
            want[rows[sk.support_]] = sk.dual_coef_[0]
            ours, ref = _dual(out["coef"][f, p], K), _dual(want, K)
            assert abs(ours - ref) <= 1e-3 * abs(ref), (f, p, ours, ref)


def test_similarity_search_ranks_and_recalls(gold):
    from gcc_b200.tasks.similarity_search import SimilaritySearch
    d1 = dict(zip((str(k) for k in gold["ss_keys_1"]), (int(v) for v in gold["ss_ids_1"])))
    d2 = dict(zip((str(k) for k in gold["ss_keys_2"]), (int(v) for v in gold["ss_ids_2"])))
    task = SimilaritySearch.__new__(SimilaritySearch)
    res = task._evaluate(gold["ss_e1"], gold["ss_e2"], d1, d2)
    assert res == {"Recall @ 20": float(gold["ss_recall20"]), "Recall @ 40": float(gold["ss_recall40"])}
    a = gold["ss_e1"].astype(np.float64)[task.last["idx1"]]
    b = gold["ss_e2"].astype(np.float64)[task.last["idx2"]]
    a /= np.linalg.norm(a, axis=1, keepdims=True)
    b /= np.linalg.norm(b, axis=1, keepdims=True)
    s = a @ b.T
    assert np.array_equal(task.last["rank"], (s > np.diag(s)[:, None]).sum(1))


def test_generate_graph_export_is_the_whole_graph_encoding(tmp_path):
    """generate.py's per-graph export equals the eval-mode encoding of the whole-graph batches that
    test_gpu_finetune checks against the oracle encoder, and does not depend on the batch size."""
    import generate
    from gcc_b200.datasets.labeled import GraphClassificationDatasetLabeled
    from test_gpu_finetune import _encoder, _two_class_graphs
    graphs, labels = _two_class_graphs(14, seed=4)
    ip, ix, sizes, a = [0], [], [], 0
    for g in graphs:
        ip.extend((g.indptr[1:] + ip[-1]).tolist())
        ix.append(g.indices.astype(np.int64) + a)
        sizes.append(g.num_nodes)
        a += g.num_nodes
    path = str(tmp_path / "graphs.npz")
    np.savez(path, indptr=np.array(ip), indices=np.concatenate(ix), graph_sizes=np.array(sizes), graph_labels=labels)
    assert generate.is_graph_dataset(path)
    torch.manual_seed(3)
    model = _encoder(32, 3).cuda().eval()
    e5 = generate.graph_embeddings(path, model, 5).numpy()
    e14 = generate.graph_embeddings(path, model, 14).numpy()
    assert e5.shape == (14, 32)
    assert np.allclose(e5, e14, rtol=1e-3, atol=1e-4)
    ds = GraphClassificationDatasetLabeled((graphs, labels), batch_size=7)
    with torch.no_grad():
        want = torch.cat([model(gq).cpu() for gq, _ in ds.batches()]).numpy()
    assert np.allclose(e5, want, rtol=1e-3, atol=1e-4)


def test_task_clis_end_to_end(gold, tmp_path):
    from gcc_b200.tasks import graph_classification, node_classification, similarity_search
    X, y = gold["nc_x"], gold["nc_y"]
    n = len(y)
    ring = np.stack([np.arange(n), (np.arange(n) + 1) % n])
    np.savez(tmp_path / "nodes.npz", edge_index=ring, y=y)
    np.save(tmp_path / "nodes_emb.npy", X)
    r = node_classification.main(["--dataset", str(tmp_path / "nodes.npz"), "--model", "from_numpy", "--hidden-size",
                                  str(X.shape[1]), "--emb-path", str(tmp_path / "nodes_emb.npy")])
    assert abs(r["Micro-F1"] - float(gold["nc_micro_f1"])) <= 0.005
    np.savez(tmp_path / "graphs.npz", graph_labels=gold["gc_y"])
    np.save(tmp_path / "graphs_emb.npy", gold["gc_x"])
    r = graph_classification.main(["--dataset", str(tmp_path / "graphs.npz"), "--model", "from_numpy_graph",
                                   "--hidden-size", "64", "--emb-path", str(tmp_path / "graphs_emb.npy")])
    assert abs(r["Micro-F1"] - float(gold["gc_micro_f1"])) <= 0.005
    np.savez(tmp_path / "pair.npz", keys_1=gold["ss_keys_1"], ids_1=gold["ss_ids_1"], keys_2=gold["ss_keys_2"],
             ids_2=gold["ss_ids_2"])
    np.save(tmp_path / "e1.npy", gold["ss_e1"])
    np.save(tmp_path / "e2.npy", gold["ss_e2"])
    r = similarity_search.main(["--dataset", str(tmp_path / "pair.npz"), "--model", "from_numpy_align",
                                "--hidden-size", "16", "--emb-path-1", str(tmp_path / "e1.npy"),
                                "--emb-path-2", str(tmp_path / "e2.npy")])
    assert r == {"Recall @ 20": float(gold["ss_recall20"]), "Recall @ 40": float(gold["ss_recall40"])}
