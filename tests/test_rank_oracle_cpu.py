"""The relation-evaluation oracle (oracle/rank_oracle.py) on the host: the vectorised restatement equals the literal
reference loop on tie-heavy inputs, a hand-worked example pins the definition, and the evaluation kernels compile for
sm_100a without local memory.  No GPU needed."""
import os
import re
import subprocess

import numpy as np
import pytest

from oracle import rank_oracle as RO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LEVELS = np.asarray([0.0, 1.0, 0.5, 0.25, 1e-30, 0.999], dtype=np.float32)
FIELDS = ("count", "total_recall", "f1", "theta", "best_pos", "auc", "auc_f64", "w", "f1_at_w", "precision_at_w",
          "recall_at_w", "ign_f1", "ign_auc", "ign_auc_f64", "ign_f1_at_w")


def random_docs(seed, sizes, R=6, p_true=0.2, with_intrain=True):
    rng = np.random.RandomState(seed)
    docs = []
    for n in sizes:
        s = rng.rand(n, n, R).astype(np.float32)
        tie = rng.rand(n, n, R) < 0.6                          # most scores on a handful of levels, exact 0 and 1 among them
        s[tie] = LEVELS[rng.randint(len(LEVELS), size=int(tie.sum()))]
        correct = rng.rand(n, n, R) < p_true
        intrain = (rng.rand(n, n, R) < 0.5) if with_intrain else None
        docs.append((s, correct, intrain))
    return docs


def assert_same(a, b):
    for k in FIELDS:
        assert a[k] == b[k], (k, a[k], b[k])
    np.testing.assert_array_equal(a["order"], b["order"])


def vectorised_of(docs, **kw):
    s, c, it = RO.candidates(docs)[:3]
    return RO.vectorised(s, c, it if any(d[2] is not None for d in docs) else None, **kw)


@pytest.mark.parametrize("seed", range(6))
@pytest.mark.parametrize("theta", [-1.0, 0.5, 0.25, 2.0, -0.5])
def test_vectorised_equals_the_literal_loop(seed, theta):
    docs = random_docs(seed, [0, 1, 2, 3, 5][: 2 + seed % 4] + [4])
    lit = RO.literal(docs, input_theta=theta)
    assert_same(lit, vectorised_of(docs, input_theta=theta))
    if theta == 2.0:
        assert lit["w"] == 0                                    # no score above: position 0
    if theta == -0.5:
        assert lit["w"] == lit["count"] - 1                     # every score above


@pytest.mark.parametrize("total_recall", [None, 0, 7, 1000])
def test_total_recall_override_and_no_positives(total_recall):
    docs = random_docs(11, [3, 4], p_true=0.0 if total_recall in (None, 0) else 0.2)
    lit = RO.literal(docs, total_recall=total_recall)
    assert_same(lit, vectorised_of(docs, total_recall=total_recall))
    if total_recall in (None, 0):
        assert lit["total_recall"] == 1 and lit["f1"] == 0.0 and lit["best_pos"] == 0 and lit["auc"] == 0.0


def test_without_intrain_the_ign_fields_are_none():
    docs = random_docs(3, [4, 3], with_intrain=False)
    lit = RO.literal(docs)
    assert lit["ign_f1"] is None and lit["ign_auc"] is None and lit["ign_f1_at_w"] is None
    assert_same(lit, vectorised_of(docs))


def test_hand_worked_example():
    # one document, n = 2, R = 3: candidates (0,1,1) (0,1,2) (1,0,1) (1,0,2) with ids 0..3
    s = np.zeros((2, 2, 3), np.float32)
    c = np.zeros((2, 2, 3), bool)
    it = np.zeros((2, 2, 3), bool)
    s[0, 1, 1], s[0, 1, 2], s[1, 0, 1], s[1, 0, 2] = 0.9, 0.5, 0.9, 0.1
    c[0, 1, 1] = c[1, 0, 2] = True
    it[0, 1, 1] = True
    r = RO.literal([(s, c, it)], input_theta=0.5)
    np.testing.assert_array_equal(r["order"], [0, 2, 1, 3])     # stable: the two 0.9 keep id order
    # c_k = 1 1 1 2, T = 2: x = .5 .5 .5 1, y = 1 .5 1/3 .5; f1 = 2/3 .5 .4 2/3 -> the first maximum
    assert r["best_pos"] == 0 and r["theta"] == np.float32(0.9) and r["f1"] == np.float32(2 / 3)
    assert r["w"] == 1 and r["precision_at_w"] == 0.5 and r["recall_at_w"] == 0.5   # last score > 0.5 is position 1
    # Ign: the first fact is in train -> t_k = c_k for k < 3, yi = 0 0 0 (2-1)/(4-1)
    assert r["ign_f1_at_w"] == 0.0
    assert r["ign_f1"] == np.float32(2 * np.float32(1.0) * np.float32(1 / 3)) / np.float32(np.float32(4 / 3) + np.float32(1e-20))
    # trapezoid: x steps only between positions 2 and 3: (1 - .5) (.5 + 1/3) / 2
    assert abs(r["auc"] - 0.5 * (0.5 + 1 / 3) / 2) < 1e-7
    assert_same(r, vectorised_of([(s, c, it)], input_theta=0.5))


def test_ign_is_zero_while_every_fact_so_far_was_in_train():
    docs = random_docs(5, [4])
    s, c, it = docs[0]
    it[...] = c                                                # every fact seen in training
    r = RO.literal([(s, c, it)])
    assert r["ign_f1"] == 0.0 and r["ign_auc"] == 0.0 and r["ign_f1_at_w"] == 0.0
    assert_same(r, vectorised_of([(s, c, it)]))


def test_single_candidate_has_zero_auc():
    s = np.full((2, 2, 2), 0.3, np.float32)
    c = np.zeros((2, 2, 2), bool)
    c[0, 1, 1] = True
    r = RO.literal([(s[:1, :1], c[:1, :1], None), (s, c, None)])
    assert r["count"] == 2
    r1 = RO.vectorised(np.asarray([0.3], np.float32), np.asarray([True]))
    assert r1["auc"] == 0.0 and r1["f1"] == 1.0 and r1["w"] == 0


def test_rank_kernels_compile_without_local_memory():
    """-Xptxas -v: no stack frame and no spills in any kernel of csrc/rank.cu."""
    src = os.path.join(ROOT, "gcgcn_b200", "csrc", "rank.cu")
    out = subprocess.run([os.environ.get("NVCC", "nvcc"), "-gencode", "arch=compute_100a,code=sm_100a", "-O3",
                          "-std=c++17", "-I", os.path.join(ROOT, "include"), "-Xptxas", "-v", "-c", "-o", os.devnull,
                          src], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    frames = re.findall(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", out.stderr)
    assert len(frames) >= 10
    assert all(f == ("0", "0", "0") for f in frames), frames
