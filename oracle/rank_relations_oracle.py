"""Test oracle of the per-relation evaluation (RelationEvaluator.per_relation, result_at, predictions_at in
gcgcn_b200/evaluate.py), restated from the definitions in include/gcgcn_b200.h ("relation evaluation per relation")
on top of the whole-set oracle (oracle/rank_oracle.py): a relation's evaluation is the whole-set evaluation of its
candidates alone, and the selection is a mask over the stable ranking."""
from __future__ import annotations

import numpy as np

from .rank_oracle import candidates, literal, vectorised


def per_relation(docs, input_theta=-1.0, total_recall=None, loop=False):
    """Entry r - 1: the evaluation of relation r's candidates alone, i.e. ``vectorised`` (``literal`` with
    ``loop=True``) on every document's relation slice ``[..., [0, r]]`` (relation 0 is not a candidate).
    ``input_theta``: a scalar or one value per relation; ``total_recall``: None or one value per relation."""
    R = docs[0][0].shape[2]
    theta = np.broadcast_to(np.asarray(input_theta, np.float64), (R - 1,))
    out = []
    for r in range(1, R):
        sl = [(s[..., [0, r]], c[..., [0, r]], None if it is None else it[..., [0, r]]) for s, c, it in docs]
        tr = None if total_recall is None else int(total_recall[r - 1])
        if loop:
            out.append(literal(sl, input_theta=float(theta[r - 1]), total_recall=tr))
        else:
            s, c, it = candidates(sl)[:3]
            has = any(d[2] is not None for d in docs)
            out.append(vectorised(s, c, it if has else None, input_theta=float(theta[r - 1]), total_recall=tr))
    return out


def select(score, correct, relation, theta, intrain=None, total_recall=None):
    """The candidates whose score > theta[relation - 1], in ranked order (stable, by score descending), from flat
    candidate arrays in insertion order (``candidates(docs)``: score, correct, intrain and relation).  Returns
    ``order`` (their ids), ``count_selected``, ``correct``, ``precision``, ``recall``, ``f1`` and ``ign_f1`` (None
    without intrain), in float32 as the curve rounds them."""
    score = np.asarray(score, np.float32)
    correct = np.asarray(correct, bool)
    theta = np.asarray(theta, np.float32)
    order = np.argsort(-score, kind="stable")
    keep = score[order] > theta[np.asarray(relation, np.int64)[order] - 1]
    sel = order[keep]
    m, c = int(sel.size), int(correct[sel].sum())
    T = int(correct.sum()) if total_recall is None else int(total_recall)
    T = max(T, 1)
    f32 = np.float32

    def f1(x, y):
        return f32(f32(f32(2) * x) * y) / f32(f32(x + y) + f32(1e-20))

    precision = f32(c / m) if m else f32(0)
    recall = f32(c / T)
    out = {"order": sel.astype(np.int64), "count_selected": m, "correct": c, "precision": float(precision),
           "recall": float(recall), "f1": float(f1(recall, precision)), "ign_f1": None}
    if intrain is not None:
        t = int((correct & np.asarray(intrain, bool))[sel].sum())
        out["ign_f1"] = float(f1(recall, f32(0) if t == c else f32((c - t) / (m - t))))
    return out
