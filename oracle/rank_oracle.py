"""Test oracle of the relation evaluation (gcgcn_b200/evaluate.py): the DocRED baseline evaluation of
config/Config.py:480-545 and the Ign F1 of config/Config_bert.py:626-650, restated from the definition in
include/gcgcn_b200.h ("relation evaluation").

A document is ``(score, correct, intrain)``: float32 ``[n, n, R]`` sigmoid scores, bool ``[n, n, R]`` facts and an
optional bool ``[n, n, R]`` in-train mask.  Scores, not logits, are the input, so the oracle can be fed the evaluator's
own float32 scores.  ``literal`` is the reference's loop (tuples, ``list.sort(reverse=True)``, appends, float32 arrays,
``np.trapezoid``); ``vectorised`` computes the same with a stable argsort and cumulative sums, for large inputs.
Both return a dict with the fields of ``RelationEvaluator.result`` plus ``auc_f64`` / ``ign_auc_f64`` (the float32
trapezoid terms summed in float64) and ``order`` (candidate ids in ranked order).
"""
from __future__ import annotations

import numpy as np


def candidates(docs):
    """Flat candidate arrays in insertion order (documents, then i, j != i, r >= 1): score, correct, intrain, doc, row,
    col, relation."""
    cols = [[] for _ in range(7)]
    for d, (score, correct, intrain) in enumerate(docs):
        n, _, R = score.shape
        i, j, r = np.meshgrid(np.arange(n), np.arange(n), np.arange(1, R), indexing="ij")
        keep = (i != j).reshape(-1)
        i, j, r = i.reshape(-1)[keep], j.reshape(-1)[keep], r.reshape(-1)[keep]
        it = np.zeros(len(i), bool) if intrain is None else np.asarray(intrain, bool)[i, j, r]
        for c, v in zip(cols, (np.asarray(score, np.float32)[i, j, r], np.asarray(correct, bool)[i, j, r], it,
                               np.full(len(i), d), i, j, r)):
            c.append(v)
    return [np.concatenate(c) if c else np.zeros(0) for c in cols]


def _finish(pr_x, pr_y, pr_yi, ranked_scores, order, T, input_theta, has_intrain):
    f1_arr = 2 * pr_x * pr_y / (pr_x + pr_y + 1e-20)
    best = int(f1_arr.argmax())
    if input_theta == -1:
        w = best
    else:
        above = np.nonzero(ranked_scores.astype(np.float64) > input_theta)[0]
        w = int(above[-1]) if above.size else 0

    def terms(y):
        return (np.diff(pr_x) * (y[1:] + y[:-1]) / 2.0).astype(np.float32)

    out = {"count": len(order), "total_recall": T, "f1": float(f1_arr[best]), "theta": float(ranked_scores[best]),
           "best_pos": best, "auc": float(np.trapezoid(x=pr_x, y=pr_y)),
           "auc_f64": float(terms(pr_y).astype(np.float64).sum()), "w": w, "f1_at_w": float(f1_arr[w]),
           "precision_at_w": float(pr_y[w]), "recall_at_w": float(pr_x[w]), "ign_f1": None, "ign_auc": None,
           "ign_auc_f64": None, "ign_f1_at_w": None, "order": order}
    if has_intrain:
        f1_ign = 2 * pr_x * pr_yi / (pr_x + pr_yi + 1e-20)
        out.update(ign_f1=float(f1_ign.max()), ign_auc=float(np.trapezoid(x=pr_x, y=pr_yi)),
                   ign_auc_f64=float(terms(pr_yi).astype(np.float64).sum()), ign_f1_at_w=float(f1_ign[w]))
    return out


def literal(docs, input_theta=-1.0, total_recall=None):
    """The reference's evaluation loop, candidate by candidate."""
    test_result = []
    cid = 0
    for score, correct, intrain in docs:
        n, _, R = score.shape
        for i in range(n):
            for j in range(n):
                if i == j:
                    continue
                for r in range(1, R):
                    it = False if intrain is None else bool(intrain[i, j, r])
                    test_result.append((bool(correct[i, j, r]), float(score[i, j, r]), it, cid))
                    cid += 1
    test_result.sort(key=lambda x: x[1], reverse=True)
    T = sum(1 for x in test_result if x[0]) if total_recall is None else total_recall
    if T == 0:
        T = 1
    pr_x, pr_y, pr_yi = [], [], []
    correct = in_train = 0
    for i, item in enumerate(test_result):
        correct += item[0]
        in_train += item[0] and item[2]
        pr_y.append(float(correct) / (i + 1))
        pr_x.append(float(correct) / T)
        pr_yi.append(0.0 if in_train == correct else float(correct - in_train) / (i + 1 - in_train))
    has_intrain = any(d[2] is not None for d in docs)
    return _finish(np.asarray(pr_x, dtype="float32"), np.asarray(pr_y, dtype="float32"),
                   np.asarray(pr_yi, dtype="float32"), np.asarray([x[1] for x in test_result], dtype=np.float32),
                   np.asarray([x[3] for x in test_result], dtype=np.int64), T, input_theta, has_intrain)


def vectorised(score, correct, intrain=None, input_theta=-1.0, total_recall=None):
    """The same from flat candidate arrays in insertion order (``candidates(docs)[:3]``)."""
    score = np.asarray(score, np.float32)
    correct = np.asarray(correct, bool)
    order = np.argsort(-score, kind="stable")
    T = int(correct.sum()) if total_recall is None else int(total_recall)
    if T == 0:
        T = 1
    c = np.cumsum(correct[order], dtype=np.int64)
    k1 = np.arange(1, len(order) + 1, dtype=np.int64)
    pr_x = (c / T).astype(np.float32)
    pr_y = (c / k1).astype(np.float32)
    if intrain is not None:
        t = np.cumsum((correct & np.asarray(intrain, bool))[order], dtype=np.int64)
        den = np.where(t == c, 1, k1 - t)
        pr_yi = np.where(t == c, 0.0, (c - t) / den).astype(np.float32)
    else:
        pr_yi = None
    return _finish(pr_x, pr_y, pr_yi, score[order], order.astype(np.int64), T, input_theta, intrain is not None)
