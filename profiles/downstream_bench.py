#!/usr/bin/env python
"""Time the frozen-embedding evaluation (csrc/downstream.cu) on the GPU against sklearn on the host cores of the
same machine, at dataset-like sizes, on seeded synthetic embeddings with overlapping classes.

    python profiles/downstream_bench.py --out downstream_bench.json [--sk-folds 1]

GPU: wall time of one call that solves all 10 folds (ends in a device synchronise), after one warm-up call
of the same shape.  sklearn: the reference's estimators (OneVsRest LogisticRegression(C=1000),
SVC(C=100000)) on `--sk-folds` folds, scaled to 10.  Both scores are recorded.  The card's name and power
limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def blobs(rng, n, d, k, spread):
    y = rng.integers(0, k, n)
    return (rng.normal(size=(k, d))[y] * spread + rng.normal(size=(n, d))).astype(np.float32), y


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (s.strip() for s in out.split(","))
        return dict(gpu=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:          # the measurement still stands; say that the card was not read
        return dict(gpu="unknown (%s)" % e)


def timed(fn):
    import torch
    torch.cuda.synchronize()
    t = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="downstream_bench.json")
    ap.add_argument("--sk-folds", type=int, default=1)
    args = ap.parse_args()
    import torch
    from sklearn.linear_model import LogisticRegression
    from sklearn.multiclass import OneVsRestClassifier
    from sklearn.svm import SVC
    from gcc_b200.tasks.evaluate import fold_ids, logreg_ovr, per_fold_accuracy, sim_rank, svc_ovo
    torch.cuda.set_device(0)
    rng = np.random.default_rng(0)
    res = dict(card(), host_cpus=os.cpu_count(), sk_folds=args.sk_folds, runs=[])
    configs = [("node", "h-index-like", 5000, 64, 2, 0.25), ("node", "h-index-like", 5000, 256, 2, 0.12),
               ("graph", "COLLAB-like", 5000, 64, 3, 0.3), ("graph", "REDDIT-MULTI-5K-like", 4999, 64, 5, 0.3),
               ("graph", "REDDIT-MULTI-5K-like", 4999, 256, 5, 0.15), ("sim", "panther-like", 3000, 64, 0, 0.0),
               ("sim", "panther-like", 3000, 256, 0, 0.0)]
    for task, name, n, d, k, spread in configs:
        run = dict(task=task, like=name, n=n, d=d, classes=k)
        if task == "sim":
            base = rng.normal(size=(n, d))
            e1 = (base + 0.8 * rng.normal(size=(n, d))).astype(np.float32)
            e2 = (base + 0.8 * rng.normal(size=(n, d))).astype(np.float32)
            idx = np.arange(n, dtype=np.int32)
            sim_rank(e1, e2, idx, idx)
            t, rank = timed(lambda: sim_rank(e1, e2, idx, idx))
            a = e1 / np.linalg.norm(e1.astype(np.float64), axis=1, keepdims=True)
            b = e2 / np.linalg.norm(e2.astype(np.float64), axis=1, keepdims=True)
            t0 = time.perf_counter()
            s = a @ b.T
            want = (s > np.diag(s)[:, None]).sum(1)
            run.update(gpu_s=t, numpy_s=time.perf_counter() - t0, ranks_equal=bool(np.array_equal(rank, want)),
                       recall20=float(np.mean(rank < 20)))
        else:
            X, y = blobs(rng, n, d, k, spread)
            folds = fold_ids(y, 0)
            if task == "node":
                call = lambda: logreg_ovr(X, y, folds, k, C=1000.0)
            else:
                call = lambda: svc_ovo(X, y, folds, k, C=100000.0)
            call()
            t, out = timed(call)
            acc = per_fold_accuracy(out["pred"], y, folds)
            sk_t, sk_acc = 0.0, []
            for f in range(args.sk_folds):
                tr, te = folds != f, folds == f
                t0 = time.perf_counter()
                if task == "node":
                    Y = np.eye(k)[y[tr]]
                    clf = OneVsRestClassifier(LogisticRegression(C=1000)).fit(X[tr].astype(np.float64), Y)
                    p = np.asarray(clf.predict_proba(X[te].astype(np.float64)))
                    pred = k - 1 - p[:, ::-1].argmax(1)          # ties to the highest class, like TopKRanker
                else:
                    pred = SVC(C=100000).fit(X[tr], y[tr]).predict(X[te])
                sk_t += time.perf_counter() - t0
                sk_acc.append(float(np.mean(pred == y[te])))
            run.update(gpu_s_10_folds=t, sklearn_s_per_fold=sk_t / args.sk_folds,
                       sklearn_s_10_folds_est=10 * sk_t / args.sk_folds, gpu_acc_folds=acc.tolist(),
                       sklearn_acc_folds=sk_acc, status_counts=np.bincount(np.asarray(out["status"]).reshape(-1)).tolist())
        res["runs"].append(run)
        print(json.dumps(run), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(dict((k, v) for k, v in res.items() if k != "runs")))


if __name__ == "__main__":
    main()
