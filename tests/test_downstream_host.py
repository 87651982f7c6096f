"""CPU: the downstream evaluation's readers, folds and CLIs, and the logic of its kernels (csrc/downstream.cu)
under the CPU emulator at toy sizes against numpy / sklearn."""
import os

import numpy as np
import pytest

from emu_util import lib as emu_lib
from emu_util import ptr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def gold(golden):
    return golden("downstream_golden")


def test_panther_readers_match_reference(gold, tmp_path):
    from gcc_b200.datasets.panther import SSDataset, SSSingleDataset
    for name, key in (("p1.graph", "pt_graph_1"), ("p2.graph", "pt_graph_2"), ("p1.dict", "pt_dict_1"),
                      ("p2.dict", "pt_dict_2")):
        (tmp_path / name).write_text(str(gold[key]))
    assert np.array_equal(SSSingleDataset(str(tmp_path), "p1").data.edge_index.numpy(), gold["pt_single_edge_index"])
    pair = SSDataset(str(tmp_path), "p1", "p2")
    for i in (1, 2):
        assert np.array_equal(pair.data[i - 1].edge_index.numpy(), gold["pt_edge_index_%d" % i])
        names = sorted(pair.data[i - 1].y)
        assert names == [str(s) for s in gold["pt_names_%d" % i]]
        assert [pair.data[i - 1].y[k] for k in names] == list(gold["pt_ids_%d" % i])


def test_fold_ids_match_stratified_kfold(gold):
    from sklearn.model_selection import StratifiedKFold
    from gcc_b200.tasks.evaluate import fold_ids
    y = gold["nc_y"]
    f = fold_ids(y, 0)
    assert np.array_equal(f, gold["nc_folds"])
    for k, (_, te) in enumerate(StratifiedKFold(10, shuffle=True, random_state=3).split(np.zeros(len(y)), y)):
        assert np.array_equal(np.flatnonzero(fold_ids(y, 3) == k), te)


def test_cli_arguments_and_unsupported_models(tmp_path):
    from gcc_b200 import tasks
    from gcc_b200.tasks import graph_classification, node_classification, similarity_search
    a = node_classification.parser().parse_args(["--dataset", "x.npz", "--model", "from_numpy", "--hidden-size", "64",
                                                 "--emb-path", "e.npy"])
    assert (a.dataset, a.model, a.hidden_size, a.seed, a.num_shuffle, a.emb_path) == ("x.npz", "from_numpy", 64, 0, 10,
                                                                                      "e.npy")
    a = similarity_search.parser().parse_args(["--dataset", "kdd_icdm", "--model", "from_numpy_align",
                                               "--hidden-size", "64", "--emb-path-1", "a", "--emb-path-2", "b"])
    assert (a.emb_path_1, a.emb_path_2) == ("a", "b")
    for mod, ok in ((node_classification, "from_numpy"), (graph_classification, "from_numpy_graph")):
        for bad in ("prone", "graphwave", "zero", "from_numpy_align"):
            with pytest.raises(NotImplementedError):
                mod.main(["--dataset", "x.npz", "--model", bad, "--hidden-size", "8", "--emb-path", "e.npy"])
        with pytest.raises(SystemExit):                                       # valid model, missing embedding
            mod.main(["--dataset", "x.npz", "--model", ok, "--hidden-size", "8", "--emb-path", str(tmp_path / "no")])
    with pytest.raises(NotImplementedError):
        similarity_search.main(["--dataset", "a_b", "--model", "prone", "--hidden-size", "8"])
    with pytest.raises(NotImplementedError):
        tasks.check_model("from_numpy", "from_numpy_graph")


def test_node_features_zero_rows_outside_edges(tmp_path):
    from gcc_b200.tasks.node_classification import NodeClassification
    emb = np.arange(5 * 3, dtype=np.float32).reshape(5, 3) + 1
    np.save(tmp_path / "e.npy", emb)
    np.savez(tmp_path / "d.npz", edge_index=np.array([[0, 1, 3], [1, 0, 0]]), y=np.array([0, 1, 0, 1, 0]))
    t = NodeClassification(str(tmp_path / "d.npz"), "from_numpy", 3, 10, 0, emb_path=str(tmp_path / "e.npy"))
    f = t.features()
    assert np.array_equal(f[[0, 1, 3]], emb[[0, 1, 3]]) and not f[[2, 4]].any()
    assert t.label_matrix.shape == (5, 2)


def _folds(y, k=3, seed=0):
    from gcc_b200.tasks.evaluate import fold_ids
    return fold_ids(y, seed, n_splits=k)


def test_emu_logreg_matches_tight_sklearn():
    from sklearn.linear_model import LogisticRegression
    lib = emu_lib()
    rng = np.random.default_rng(1)
    n, d, C, K = 60, 8, 3, 3
    y = rng.integers(0, C, n)
    X = (rng.normal(size=(C, d))[y] * 0.6 + rng.normal(size=(n, d))).astype(np.float32)
    folds = _folds(y, K).astype(np.int32)
    yl = y.astype(np.int32)
    W = np.zeros(K * C * (d + 1))
    prob = np.zeros(n * C)
    pred = np.zeros(n, np.int32)
    st = np.zeros(K * C, np.int32)
    wsb = lib.gccb_logreg_ovr_workspace(n, d, C, K)
    ws = np.zeros(wsb // 8 + 1)
    rc = lib.gccb_logreg_ovr(ptr(X), ptr(yl), ptr(folds), n, d, C, K, 10.0, 100, 1e-12, ptr(W), ptr(prob), ptr(pred),
                             ptr(st), ptr(ws), wsb, None)
    assert rc == 0 and np.all(st == 0), st
    W = W.reshape(K, C, d + 1)
    for f in range(K):
        tr = folds != f
        for c in range(C):
            ref = LogisticRegression(C=10.0, tol=1e-12, max_iter=100000).fit(X[tr].astype(np.float64), y[tr] == c)
            want = np.concatenate([ref.coef_[0], ref.intercept_])
            assert np.allclose(W[f, c], want, rtol=1e-5, atol=1e-6), (f, c, W[f, c], want)
    z = np.einsum("nd,ncd->nc", X.astype(np.float64), W[folds, :, :d]) + W[folds, :, d]
    p = 1 / (1 + np.exp(-z))
    assert np.allclose(prob.reshape(n, C), p, rtol=1e-12)
    assert np.array_equal(pred, p.argmax(1))


def test_emu_logreg_absent_class_gets_constant_predictor():
    lib = emu_lib()
    n, d, C, K = 12, 2, 3, 2
    X = np.zeros((n, d), np.float32)
    X[:, 0] = np.arange(n)
    y = np.array([0, 1] * 6, np.int32)                    # class 2 never occurs: constant probability 0
    folds = (np.arange(n) % 4 < 2).astype(np.int32)
    W, prob, pred, st = np.zeros(K * C * (d + 1)), np.zeros(n * C), np.zeros(n, np.int32), np.zeros(K * C, np.int32)
    wsb = lib.gccb_logreg_ovr_workspace(n, d, C, K)
    ws = np.zeros(wsb // 8 + 1)
    assert lib.gccb_logreg_ovr(ptr(X), ptr(y), ptr(folds), n, d, C, K, 1.0, 50, 1e-12, ptr(W), ptr(prob), ptr(pred),
                               ptr(st), ptr(ws), wsb, None) == 0
    assert list(st.reshape(K, C)[:, 2]) == [3, 3] and not prob.reshape(n, C)[:, 2].any()
    assert set(pred) <= {0, 1}


def _svc_emu(X, y, folds, C, K, n_classes):
    lib = emu_lib()
    n, d = X.shape
    P = n_classes * (n_classes - 1) // 2
    gamma, coef, rho, obj = np.zeros(K), np.zeros(K * P * n), np.zeros(K * P), np.zeros(K * P)
    dec, pred, st = np.zeros(n * P), np.zeros(n, np.int32), np.zeros(K * P, np.int32)
    wsb = lib.gccb_svc_ovo_workspace(n, n_classes, K)
    ws = np.zeros(wsb // 8 + 1)
    rc = lib.gccb_svc_ovo(ptr(X), ptr(y), ptr(folds), n, d, n_classes, K, C, 1e-3, 1000000, ptr(gamma), ptr(coef),
                          ptr(rho), ptr(obj), ptr(dec), ptr(pred), ptr(st), ptr(ws), wsb, None)
    assert rc == 0 and np.all(st == 0), st
    return gamma, coef.reshape(K, P, n), rho.reshape(K, P), obj.reshape(K, P), dec.reshape(n, P), pred


def _dual(coef, K):
    return 0.5 * coef @ K @ coef - np.abs(coef).sum()


def test_emu_svc_matches_sklearn():
    from sklearn.svm import SVC
    rng = np.random.default_rng(2)
    n, d, nc, K = 41, 4, 3, 2
    y = rng.integers(0, nc, n).astype(np.int32)
    X = (rng.normal(size=(nc, d))[y] + 0.9 * rng.normal(size=(n, d))).astype(np.float32)
    folds = _folds(y, K).astype(np.int32)
    gamma, coef, rho, obj, dec, pred = _svc_emu(X, y, folds, 10.0, K, nc)
    Xd = X.astype(np.float64)
    pairs = [(a, b) for a in range(nc) for b in range(a + 1, nc)]
    for f in range(K):
        tr = folds != f
        assert np.isclose(gamma[f], 1.0 / (d * Xd[tr].var()), rtol=1e-12)
        sk = SVC(C=10.0).fit(Xd[tr], y[tr])
        Kf = np.exp(-gamma[f] * ((Xd[:, None] - Xd[None]) ** 2).sum(-1))
        for p, (a, b) in enumerate(pairs):
            rows = np.flatnonzero(tr & ((y == a) | (y == b)))
            sub = SVC(C=10.0, gamma=gamma[f], tol=1e-8).fit(Xd[rows], np.where(y[rows] == a, 1, -1))
            want = np.zeros(n)
            want[rows[sub.support_]] = sub.dual_coef_[0]
            # sklearn's binary dual_coef_ is signed for classes_ = [-1, 1]; ours is y * alpha with y(a) = +1
            assert np.isclose(_dual(coef[f, p], Kf), _dual(want, Kf), rtol=1e-3), (f, p)
            assert np.isclose(obj[f, p], _dual(coef[f, p], Kf), rtol=1e-4)
        te = folds == f
        assert np.mean(pred[te] == sk.predict(Xd[te])) >= 0.9


def test_emu_sim_rank_matches_numpy():
    lib = emu_lib()
    rng = np.random.default_rng(3)
    m, d = 30, 16
    E1 = rng.normal(size=(40, d)).astype(np.float32)
    E2 = rng.normal(size=(35, d)).astype(np.float32)
    i1 = rng.permutation(40)[:m].astype(np.int32)
    i2 = rng.permutation(35)[:m].astype(np.int32)
    E2[i2] = (E1[i1] + 2.5 * rng.normal(size=(m, d))).astype(np.float32)
    rank = np.zeros(m, np.int32)
    wsb = lib.gccb_sim_rank_workspace(m, d)
    ws = np.zeros(wsb // 8 + 1)
    assert lib.gccb_sim_rank(ptr(E1), ptr(E2), d, ptr(i1), ptr(i2), m, ptr(rank), ptr(ws), wsb, None) == 0
    a = E1.astype(np.float64)[i1]
    b = E2.astype(np.float64)[i2]
    a /= np.linalg.norm(a, axis=1, keepdims=True)
    b /= np.linalg.norm(b, axis=1, keepdims=True)
    s = a @ b.T
    want = (s > np.diag(s)[:, None]).sum(1)
    assert np.array_equal(rank, want) and rank.min() == 0 and rank.max() > 0
