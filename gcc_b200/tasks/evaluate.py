"""Host side of the downstream kernels (csrc/downstream.cu): fold assignment and one call per task.

The folds are sklearn's StratifiedKFold(n_splits=10, shuffle=True, random_state=seed), exactly as the
reference draws them (node_classification.py:55-60, graph_classification.py:47); every row gets the id of
the fold in which it is a test row, and one launch then solves every fold.
"""
import numpy as np
import torch
from sklearn.model_selection import StratifiedKFold

from .. import _lib

N_FOLDS = 10
STATUS = {0: "converged", 1: "iteration cap reached", 2: "no further decrease at fp64 resolution",
          3: "class absent from the training fold (constant 0)", 4: "only class of the training fold (constant 1)"}


def fold_ids(labels, seed, n_splits=N_FOLDS):
    labels = np.asarray(labels)
    folds = np.empty(len(labels), dtype=np.int32)
    skf = StratifiedKFold(n_splits=n_splits, shuffle=True, random_state=seed)
    for f, (_, test) in enumerate(skf.split(np.zeros(len(labels)), labels)):
        folds[test] = f
    return folds


def _dev(a, dtype):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=dtype)).cuda()


def _ws(nbytes):
    return torch.empty(max(int(nbytes), 8), dtype=torch.uint8, device="cuda")


def _warn(kind, status):
    bad = [(i, int(s)) for i, s in enumerate(status) if s in (1, 2)]
    if bad:
        import sys
        sys.stderr.write("%s: %d problem(s) stopped early: %s\n" % (
            kind, len(bad), ", ".join("#%d %s" % (i, STATUS[s]) for i, s in bad[:5])))


def logreg_ovr(X, labels, folds, n_classes, C=1000.0, max_iter=100, tol=1e-12, n_folds=N_FOLDS):
    """Per fold and class, L2 logistic regression on the training rows; returns dict(pred [n], prob [n, C],
    weights [folds, C, d+1], status [folds*C]) as numpy arrays."""
    lib = _lib.get()
    _lib.require_device()
    X = np.asarray(X, dtype=np.float32)
    n, d = X.shape
    Xd, yd, fd = _dev(X, np.float32), _dev(labels, np.int32), _dev(folds, np.int32)
    W = torch.zeros(n_folds * n_classes * (d + 1), dtype=torch.float64, device="cuda")
    prob = torch.zeros(n * n_classes, dtype=torch.float64, device="cuda")
    pred = torch.zeros(n, dtype=torch.int32, device="cuda")
    status = torch.zeros(n_folds * n_classes, dtype=torch.int32, device="cuda")
    wsb = lib.gccb_logreg_ovr_workspace(n, d, n_classes, n_folds)
    ws = _ws(wsb)
    rc = lib.gccb_logreg_ovr(_lib.dptr(Xd), _lib.dptr(yd), _lib.dptr(fd), n, d, n_classes, n_folds, float(C),
                             int(max_iter), float(tol), _lib.dptr(W), _lib.dptr(prob), _lib.dptr(pred),
                             _lib.dptr(status), _lib.dptr(ws), wsb, _lib.stream_ptr())
    _lib.check(rc, "gccb_logreg_ovr")
    out = dict(pred=pred.cpu().numpy(), prob=prob.cpu().numpy().reshape(n, n_classes),
               weights=W.cpu().numpy().reshape(n_folds, n_classes, d + 1), status=status.cpu().numpy())
    _warn("logistic regression", out["status"])
    return out


def svc_ovo(X, labels, folds, n_classes, C=100000.0, eps=1e-3, max_iter=10_000_000, n_folds=N_FOLDS):
    """Per fold, RBF C-SVC one-vs-one on the training rows; returns dict(pred [n], gamma [folds],
    coef [folds, pairs, n], rho / obj / status [folds, pairs], dec [n, pairs])."""
    lib = _lib.get()
    _lib.require_device()
    X = np.asarray(X, dtype=np.float32)
    n, d = X.shape
    P = n_classes * (n_classes - 1) // 2
    Xd, yd, fd = _dev(X, np.float32), _dev(labels, np.int32), _dev(folds, np.int32)
    f64 = lambda k: torch.zeros(k, dtype=torch.float64, device="cuda")
    gamma, coef, rho, obj, dec = f64(n_folds), f64(n_folds * P * n), f64(n_folds * P), f64(n_folds * P), f64(n * P)
    pred = torch.zeros(n, dtype=torch.int32, device="cuda")
    status = torch.zeros(n_folds * P, dtype=torch.int32, device="cuda")
    wsb = lib.gccb_svc_ovo_workspace(n, n_classes, n_folds)
    ws = _ws(wsb)
    rc = lib.gccb_svc_ovo(_lib.dptr(Xd), _lib.dptr(yd), _lib.dptr(fd), n, d, n_classes, n_folds, float(C),
                          float(eps), int(max_iter), _lib.dptr(gamma), _lib.dptr(coef), _lib.dptr(rho),
                          _lib.dptr(obj), _lib.dptr(dec), _lib.dptr(pred), _lib.dptr(status), _lib.dptr(ws), wsb,
                          _lib.stream_ptr())
    _lib.check(rc, "gccb_svc_ovo")
    out = dict(pred=pred.cpu().numpy(), gamma=gamma.cpu().numpy(), coef=coef.cpu().numpy().reshape(n_folds, P, n),
               rho=rho.cpu().numpy().reshape(n_folds, P), obj=obj.cpu().numpy().reshape(n_folds, P),
               status=status.cpu().numpy().reshape(n_folds, P), dec=dec.cpu().numpy().reshape(n, P))
    _warn("SVC", out["status"].reshape(-1))
    return out


def sim_rank(E1, E2, idx1, idx2):
    """rank[q] = number of shared candidates scoring strictly above the true match of query q."""
    lib = _lib.get()
    _lib.require_device()
    E1, E2 = np.asarray(E1, dtype=np.float32), np.asarray(E2, dtype=np.float32)
    m, d = len(idx1), E1.shape[1]
    r = torch.zeros(m, dtype=torch.int32, device="cuda")
    wsb = lib.gccb_sim_rank_workspace(m, d)
    ws = _ws(wsb)
    a, b = _dev(E1, np.float32), _dev(E2, np.float32)
    i1, i2 = _dev(idx1, np.int32), _dev(idx2, np.int32)
    rc = lib.gccb_sim_rank(_lib.dptr(a), _lib.dptr(b), d, _lib.dptr(i1), _lib.dptr(i2), m, _lib.dptr(r),
                           _lib.dptr(ws), wsb, _lib.stream_ptr())
    _lib.check(rc, "gccb_sim_rank")
    return r.cpu().numpy()


def per_fold_accuracy(pred, labels, folds, n_folds=N_FOLDS):
    pred, labels, folds = np.asarray(pred), np.asarray(labels), np.asarray(folds)
    return np.array([np.mean(pred[folds == f] == labels[folds == f]) for f in range(n_folds)])
