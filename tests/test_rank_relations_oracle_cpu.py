"""The per-relation oracle (oracle/rank_relations_oracle.py) on the host, on small tie-heavy sets: per_relation agrees
with the reference's literal loop on each relation's candidates, and select with a candidate-by-candidate loop and,
at one threshold for every relation, with the literal loop's values at that threshold.  No GPU needed."""
import numpy as np
import pytest

from oracle import rank_oracle as RO
from oracle import rank_relations_oracle as RR
from test_rank_oracle_cpu import FIELDS, assert_same, random_docs


@pytest.mark.parametrize("seed", range(4))
@pytest.mark.parametrize("with_intrain", [True, False])
def test_per_relation_equals_the_literal_loop(seed, with_intrain):
    R = 3 + seed
    docs = random_docs(seed, [0, 1, 2, 3, 5][: 2 + seed % 4] + [4], R=R, with_intrain=with_intrain)
    theta = np.where(np.arange(R - 1) % 2 == 0, -1.0, 0.5)
    tr = np.arange(R - 1) * 2                                       # 0 counts as 1
    for kw in ({}, {"input_theta": 0.25}, {"input_theta": theta, "total_recall": tr}):
        vec, lit = RR.per_relation(docs, **kw), RR.per_relation(docs, loop=True, **kw)
        assert len(vec) == len(lit) == R - 1
        for a, b in zip(vec, lit):
            assert_same(a, b)
    # relation r alone: the candidates of the flat list whose relation is r, ranked on their own
    s, c, it, _, _, _, rel = RO.candidates(docs)
    for r, got in enumerate(RR.per_relation(docs, loop=True), start=1):
        m = rel == r
        ref = RO.vectorised(s[m], c[m], it[m] if with_intrain else None)
        for k in FIELDS:
            assert got[k] == ref[k], (r, k)


def test_two_relations_are_the_whole_set():
    docs = random_docs(9, [3, 4, 2], R=2)
    assert_same(RR.per_relation(docs, loop=True)[0], RO.literal(docs))


def select_loop(docs, theta, total_recall=None):
    items = []                                                      # (score, correct, intrain, id, relation)
    cid = 0
    for score, correct, intrain in docs:
        n, _, R = score.shape
        for i in range(n):
            for j in range(n):
                if i == j:
                    continue
                for r in range(1, R):
                    items.append((float(score[i, j, r]), bool(correct[i, j, r]),
                                  intrain is not None and bool(intrain[i, j, r]), cid, r))
                    cid += 1
    items.sort(key=lambda x: x[0], reverse=True)
    picked = [x for x in items if x[0] > float(np.float32(theta[x[4] - 1]))]
    T = sum(x[1] for x in items) if total_recall is None else total_recall
    return [x[3] for x in picked], len(picked), sum(x[1] for x in picked), sum(x[1] and x[2] for x in picked), max(T, 1)


@pytest.mark.parametrize("seed", range(4))
def test_select_equals_a_candidate_loop(seed):
    R = 4 + seed
    docs = random_docs(20 + seed, [2, 5, 3, 0, 4], R=R)
    s, c, it, _, _, _, rel = RO.candidates(docs)
    theta = np.random.RandomState(seed).choice(np.asarray([0.0, 0.25, 0.5, 0.999, 1.0], np.float32), R - 1)
    for tr in (None, 9):
        got = RR.select(s, c, rel, theta, intrain=it, total_recall=tr)
        ids, m, cc, t, T = select_loop(docs, theta, tr)
        np.testing.assert_array_equal(got["order"], ids)
        assert (got["count_selected"], got["correct"]) == (m, cc)
        assert got["precision"] == (float(np.float32(cc / m)) if m else 0.0)
        assert got["recall"] == float(np.float32(cc / T))
        assert (got["ign_f1"] is None) is False


@pytest.mark.parametrize("theta", [0.0, 0.25, 0.5, 0.999])
def test_uniform_select_equals_the_literal_loop_at_theta(theta):
    R = 6
    docs = random_docs(31, [3, 4, 5], R=R)
    s, c, it, _, _, _, rel = RO.candidates(docs)
    theta = float(np.float32(theta))                                # the thresholds are float32
    lit = RO.literal(docs, input_theta=theta)
    got = RR.select(s, c, rel, np.full(R - 1, theta, np.float32), intrain=it)
    assert got["count_selected"] == lit["w"] + 1 > 0
    np.testing.assert_array_equal(got["order"], lit["order"][:lit["w"] + 1])
    assert (got["precision"], got["recall"], got["f1"], got["ign_f1"]) == (
        lit["precision_at_w"], lit["recall_at_w"], lit["f1_at_w"], lit["ign_f1_at_w"])


def test_threshold_above_every_score_selects_nothing():
    docs = random_docs(3, [3, 4], R=5)
    s, c, it, _, _, _, rel = RO.candidates(docs)
    got = RR.select(s, c, rel, np.full(4, 2.0, np.float32), intrain=it)
    assert got["order"].size == 0
    assert (got["count_selected"], got["correct"], got["precision"], got["recall"], got["f1"], got["ign_f1"]) == (
        0, 0, 0.0, 0.0, 0.0, 0.0)
