"""-m gpu: relation evaluation per relation (RelationEvaluator.per_relation, result_at, predictions_at; csrc/rank.cu,
gcgcn_rank_by_relation / gcgcn_rank_curve_relations / gcgcn_rank_select) against the NumPy oracle
(oracle/rank_relations_oracle.py) fed the evaluator's own float32 scores, and against the whole-set evaluation of the
same evaluator (relations = 2, columns [0, r], uniform thresholds, merged parts)."""
import numpy as np
import pytest
import torch

from oracle import rank_oracle as RO
from oracle import rank_relations_oracle as RR
from test_gpu_rank_eval import candidate_mask
from gcgcn_b200 import _lib
from gcgcn_b200.batch import RaggedBatch
from gcgcn_b200.evaluate import MAX_RELATIONS, SORT_TILE, RelationEvaluator
from gcgcn_b200.functional import _p, _stream

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
EXACT = ("count", "total_recall", "f1", "theta", "best_pos", "w", "f1_at_w", "precision_at_w", "recall_at_w", "ign_f1",
         "ign_f1_at_w")
PRED = ("doc", "row", "col", "relation", "score")
SMALL = [0, 1, 2, 5, 9, 13, 21, 3]            # 676 candidates per relation: every segment shorter than one tile
SPANNING = [60, 70, 13]                       # 8526 per relation: three tiles per segment, the last one partial
LARGE = [100, 100, 50, 20]                    # 22630 per relation: 2.17 M candidates at R = 97


def make_inputs(sizes, R, seed, scale=8.0, p_true=0.05, p_train=0.5):
    gen = torch.Generator(device=DEV).manual_seed(seed)
    P = int(sum(n * n for n in sizes))
    z = torch.randn(P, R, generator=gen, device=DEV) * scale          # saturates to exact 0 and 1 often: many ties
    z[torch.rand(P, R, generator=gen, device=DEV) < 0.2] = 3.0        # and a repeated mid value
    labels = (torch.rand(P, R, generator=gen, device=DEV) < p_true).float()
    intrain = (torch.rand(P, R, generator=gen, device=DEV) < p_train) & (labels > 0.5)
    return z, labels, intrain


def evaluator(sizes, R, data, with_intrain=True):
    z, labels, intrain = data
    ev = RelationEvaluator(R, DEV)
    ev.add(z, labels, RaggedBatch(sizes, DEV), intrain=intrain if with_intrain else None)
    return ev


def flat(ev, sizes, R, data, with_intrain=True):
    """score, correct, intrain (None without) and relation of every candidate, in id order, on the host."""
    _, labels, intrain = data
    keep = candidate_mask(sizes, R).to(DEV)
    s = ev.scores.cpu().numpy()
    c = (labels[keep] > 0.5).cpu().numpy()
    it = intrain[keep].cpu().numpy() if with_intrain else None
    rel = np.arange(s.size) % (R - 1) + 1
    return s, c, it, rel


def docs_of(ev, sizes, R, data, with_intrain=True):
    """The oracle's documents ([n, n, R] score, correct, intrain) holding the evaluator's own scores."""
    _, labels, intrain = data
    keep = candidate_mask(sizes, R)
    full = torch.zeros(keep.shape, dtype=torch.float32)
    full[keep] = ev.scores.cpu()
    lab = labels.cpu() > 0.5
    it = intrain.cpu()
    docs, p0 = [], 0
    for n in sizes:
        sl = slice(p0, p0 + n * n)
        docs.append((full[sl].reshape(n, n, R).numpy(), lab[sl].reshape(n, n, R).numpy(),
                     it[sl].reshape(n, n, R).numpy() if with_intrain else None))
        p0 += n * n
    return docs


def oracle_flat(s, c, it, rel, R, input_theta=-1.0, total_recall=None):
    """RO.vectorised on each relation's candidates (a mask over the flat arrays, not the documents' slices)."""
    theta = np.broadcast_to(np.asarray(input_theta, np.float64), (R - 1,))
    out = []
    for r in range(1, R):
        m = rel == r
        out.append(RO.vectorised(s[m], c[m], None if it is None else it[m], input_theta=float(theta[r - 1]),
                                 total_recall=None if total_recall is None else int(total_recall[r - 1])))
    return out


def check_relations(res, refs):
    assert len(res["relation"]) == len(refs)
    np.testing.assert_array_equal(res["relation"], np.arange(1, len(refs) + 1))
    for i, ref in enumerate(refs):
        for k in EXACT:
            got = None if res[k] is None else res[k][i]
            assert got == ref[k], (i + 1, k, got, ref[k])
        assert abs(res["auc"][i] - ref["auc"]) <= 1e-5 * max(abs(ref["auc"]), 1e-30) + 1e-12, i + 1
        assert abs(res["auc"][i] - ref["auc_f64"]) <= 1e-9, i + 1
        if ref["ign_auc"] is None:
            assert res["ign_auc"] is None
        else:
            assert abs(res["ign_auc"][i] - ref["ign_auc"]) <= 1e-5 * max(abs(ref["ign_auc"]), 1e-30) + 1e-12, i + 1
            assert abs(res["ign_auc"][i] - ref["ign_auc_f64"]) <= 1e-9, i + 1


def same_relations(a, b):
    assert a.keys() == b.keys()
    for k in a:
        if a[k] is None or b[k] is None:
            assert a[k] is None and b[k] is None, k
        else:
            np.testing.assert_array_equal(a[k], b[k], err_msg=k)


# ------------------------------------------------------------------------------------------------ per-relation curve
@pytest.mark.parametrize("sizes,R", [([2], 97), (SMALL, 3), (SMALL, 97), (SPANNING, 5), ([2, 3], MAX_RELATIONS)])
@pytest.mark.parametrize("with_intrain", [True, False])
def test_per_relation_matches_the_oracle(sizes, R, with_intrain):
    data = make_inputs(sizes, R, 7 * R + len(sizes), p_true=0.2)
    ev = evaluator(sizes, R, data, with_intrain)
    docs = docs_of(ev, sizes, R, data, with_intrain)
    check_relations(ev.per_relation(), RR.per_relation(docs))
    theta = np.linspace(-0.5, 1.5, R - 1)                       # -1 on some relations, values inside and outside (0, 1)
    theta[::3] = -1.0
    tr = np.arange(R - 1) % 7 * 3                               # 0 counts as 1
    check_relations(ev.per_relation(input_theta=theta, total_recall=tr),
                    RR.per_relation(docs, input_theta=theta, total_recall=tr))
    check_relations(ev.per_relation(input_theta=0.5), RR.per_relation(docs, input_theta=0.5))


def test_per_relation_matches_the_literal_loop():
    sizes, R = [3, 4, 2], 6
    data = make_inputs(sizes, R, 5, p_true=0.3)
    ev = evaluator(sizes, R, data)
    docs = docs_of(ev, sizes, R, data)
    res = ev.per_relation()
    check_relations(res, RR.per_relation(docs, loop=True))
    check_relations(ev.per_relation(input_theta=res["theta"]), RR.per_relation(docs, input_theta=res["theta"], loop=True))


@pytest.mark.parametrize("sizes", [SPANNING, LARGE])
def test_per_relation_at_size(sizes):
    R = 97
    data = make_inputs(sizes, R, 17, scale=6.0, p_true=0.02)
    ev = evaluator(sizes, R, data)
    assert ev.count // (R - 1) > SORT_TILE
    s, c, it, rel = flat(ev, sizes, R, data)
    check_relations(ev.per_relation(), oracle_flat(s, c, it, rel, R))
    theta = np.full(R - 1, 0.9)
    tr = np.full(R - 1, 50)
    check_relations(ev.per_relation(input_theta=theta, total_recall=tr),
                    oracle_flat(s, c, it, rel, R, input_theta=theta, total_recall=tr))


# ----------------------------------------------------------------------------------------------------- consistency
@pytest.mark.parametrize("theta", [-1.0, 0.5, 0.95, 2.0])
@pytest.mark.parametrize("total_recall", [None, 1000])
def test_two_relations_equal_result(theta, total_recall):
    data = make_inputs(SPANNING, 2, 3, p_true=0.1)
    ev = evaluator(SPANNING, 2, data)
    per = ev.per_relation(input_theta=theta, total_recall=None if total_recall is None else [total_recall])
    whole = ev.result(input_theta=theta, total_recall=total_recall)
    for k, v in whole.items():
        assert per[k][0] == v, k
    ev2 = evaluator(SPANNING, 2, data, with_intrain=False)
    assert ev2.per_relation()["ign_f1"] is None and ev2.result()["ign_f1"] is None


def test_each_relation_equals_an_evaluator_of_its_columns():
    sizes, R = SMALL + [30], 9
    data = make_inputs(sizes, R, 11, p_true=0.1)
    z, labels, intrain = data
    ev = evaluator(sizes, R, data)
    theta = np.where(np.arange(R - 1) % 2 == 0, -1.0, 0.75)
    tr = np.arange(1, R) * 5
    per = ev.per_relation(input_theta=theta, total_recall=tr)
    for r in range(1, R):
        cols = [0, r]
        one = RelationEvaluator(2, DEV)
        one.add(z[:, cols].contiguous(), labels[:, cols].contiguous(), RaggedBatch(sizes, DEV),
                intrain=intrain[:, cols].contiguous())
        whole = one.result(input_theta=float(theta[r - 1]), total_recall=int(tr[r - 1]))
        for k, v in whole.items():
            assert per[k][r - 1] == v, (r, k)


def _parts(sizes, R, data, groups):
    z, labels, intrain = data
    ptr = np.concatenate([[0], np.cumsum(np.asarray(sizes, np.int64) ** 2)])
    evs = []
    for docs in groups:
        ev = RelationEvaluator(R, DEV, doc_sizes=sizes)
        rows = torch.from_numpy(np.concatenate([np.arange(ptr[g], ptr[g + 1]) for g in docs] +
                                               [np.zeros(0, np.int64)])).to(DEV)
        ev.add(z[rows], labels[rows], RaggedBatch([sizes[g] for g in docs], DEV), intrain=intrain[rows],
               doc_index=list(docs))
        evs.append(ev)
    return evs


@pytest.mark.parametrize("groups", [[[0, 2, 4, 6], [1, 3, 5, 7, 8]], [[0, 1, 2], [3, 4, 5], [6, 7, 8]]])
def test_merged_parts_equal_one_evaluator(groups):
    sizes, R = SMALL + [30], 97
    data = make_inputs(sizes, R, 13, p_true=0.1)
    merged = RelationEvaluator.merged(_parts(sizes, R, data, groups))
    one = _parts(sizes, R, data, [list(range(len(sizes)))])[0]
    same_relations(merged.per_relation(), one.per_relation())
    theta = merged.per_relation()["theta"]
    same_relations(merged.per_relation(input_theta=0.5), one.per_relation(input_theta=0.5))
    assert merged.result_at(theta) == one.result_at(theta)
    pa, pb = merged.predictions_at(theta), one.predictions_at(theta)
    for k in PRED:
        assert torch.equal(pa[k], pb[k]), k


# ---------------------------------------------------------------------------------------------- selection, decoding
@pytest.mark.parametrize("sizes,R", [(SMALL, 97), (SPANNING, 5), (LARGE, 97)])
def test_selection_equals_a_mask_over_the_ranking(sizes, R):
    data = make_inputs(sizes, R, 19, p_true=0.05)
    ev = evaluator(sizes, R, data)
    rng = np.random.RandomState(R)
    theta = rng.choice(np.asarray([0.0, 0.5, 0.9, 0.999, 1.0, 0.25], np.float32), R - 1)
    key, pay = (t.cpu().numpy().view(np.uint32) for t in ev.ranked)
    score, ids = (~key).view(np.float32), (pay >> 2).astype(np.int64)
    mask = score > theta[ids % (R - 1)]
    s, c, it, rel = flat(ev, sizes, R, data)
    ref = RR.select(s, c, rel, theta, intrain=it)
    np.testing.assert_array_equal(ref["order"], ids[mask])
    got = ev.result_at(theta)
    for k in ("count_selected", "correct", "precision", "recall", "f1", "ign_f1"):
        assert got[k] == ref[k], (k, got[k], ref[k])
    assert got["count_selected"] == int(mask.sum()) and got["correct"] == int((pay[mask] & 1).sum())
    pred = ev.predictions_at(theta)
    np.testing.assert_array_equal(pred["score"].cpu().numpy(), score[mask])
    n = np.asarray(sizes, np.int64)
    first = np.concatenate([[0], np.cumsum((n * n - n) * (R - 1))])
    doc = pred["doc"].cpu().numpy().astype(np.int64)
    i, j, r = (pred[k].cpu().numpy().astype(np.int64) for k in ("row", "col", "relation"))
    np.testing.assert_array_equal(first[doc] + (i * (n[doc] - 1) + j - (j > i)) * (R - 1) + r - 1, ids[mask])
    got, ref = ev.result_at(theta, total_recall=7), RR.select(s, c, rel, theta, intrain=it, total_recall=7)
    for k in ("count_selected", "correct", "precision", "recall", "f1", "ign_f1"):
        assert got[k] == ref[k], (k, got[k], ref[k])


@pytest.mark.parametrize("theta", [0.0, 0.5, 0.95, 0.999])
def test_uniform_threshold_equals_result_and_predictions(theta):
    R = 97
    data = make_inputs(SPANNING, R, 23, p_true=0.05)
    ev = evaluator(SPANNING, R, data)
    theta = float(np.float32(theta))                            # the thresholds are float32
    whole = ev.result(input_theta=theta)
    assert bool((ev.scores > theta).any())
    at = ev.result_at(np.full(R - 1, theta, np.float32))
    assert at["count_selected"] == whole["w"] + 1
    assert (at["precision"], at["recall"], at["f1"], at["ign_f1"]) == (
        whole["precision_at_w"], whole["recall_at_w"], whole["f1_at_w"], whole["ign_f1_at_w"])
    pa, pb = ev.predictions_at(np.full(R - 1, theta, np.float32)), ev.predictions(theta)
    for k in PRED:
        assert torch.equal(pa[k], pb[k]), k


def test_threshold_above_every_score_selects_nothing():
    R = 97
    data = make_inputs(SMALL, R, 29)
    ev = evaluator(SMALL, R, data)
    at = ev.result_at(np.full(R - 1, 2.0, np.float32))
    assert at == {"count_selected": 0, "correct": 0, "precision": 0.0, "recall": 0.0, "f1": 0.0, "ign_f1": 0.0}
    pred = ev.predictions_at(np.full(R - 1, 2.0, np.float32))
    assert set(pred) == set(PRED)
    for k in PRED:
        assert pred[k].numel() == 0 and pred[k].device == DEV
    assert pred["score"].dtype == torch.float32 and pred["doc"].dtype == torch.int32


def test_dev_thresholds_decode_an_unlabeled_set():
    R = 97
    dev_data = make_inputs(SMALL, R, 31, p_true=0.2)
    theta = evaluator(SMALL, R, dev_data).per_relation()["theta"]
    z, _, _ = make_inputs(SPANNING, R, 37)
    test = RelationEvaluator(R, DEV)
    test.add(z, None, RaggedBatch(SPANNING, DEV))
    with pytest.raises(_lib.GcgcnError, match="without labels"):
        test.per_relation()
    with pytest.raises(_lib.GcgcnError, match="without labels"):
        test.result_at(theta)
    pred = test.predictions_at(theta)
    key, pay = (t.cpu().numpy().view(np.uint32) for t in test.ranked)
    score, ids = (~key).view(np.float32), (pay >> 2).astype(np.int64)
    mask = score > theta[ids % (R - 1)]
    assert pred["score"].numel() == int(mask.sum()) > 0
    np.testing.assert_array_equal(pred["relation"].cpu().numpy(), ids[mask] % (R - 1) + 1)
    np.testing.assert_array_equal(pred["score"].cpu().numpy(), score[mask])


# ----------------------------------------------------------------------------------------------------------- errors
def test_errors():
    R = 97
    z, labels, _ = make_inputs([4, 3], R, 41)
    ev = evaluator([4, 3], R, (z, labels, None), with_intrain=False)
    with pytest.raises(_lib.GcgcnError, match="relations - 1"):
        ev.per_relation(input_theta=[0.5] * (R - 2))
    with pytest.raises(_lib.GcgcnError, match="relations - 1"):
        ev.per_relation(total_recall=5)
    with pytest.raises(_lib.GcgcnError, match="relations - 1"):
        ev.result_at(0.5)                                        # one threshold per relation
    bad = z.clone()
    bad[1, 7] = float("nan")
    ev = evaluator([4, 3], R, (bad, labels, None), with_intrain=False)
    for call in (lambda: ev.per_relation(), lambda: ev.result_at(np.full(R - 1, 0.5, np.float32)),
                 lambda: ev.predictions_at(np.full(R - 1, 0.5, np.float32))):
        with pytest.raises(_lib.GcgcnError, match="NaN"):
            call()
    R = MAX_RELATIONS + 1
    z, labels, _ = make_inputs([3], R, 43)
    ev = evaluator([3], R, (z, labels, None), with_intrain=False)
    ev.result()                                                  # the whole-set evaluation has no such limit
    with pytest.raises(_lib.GcgcnError, match="at most 256"):
        ev.per_relation()
    with pytest.raises(_lib.GcgcnError, match="at most 256"):
        ev.predictions_at(np.full(R - 1, 0.5, np.float32))
    key, pay = evaluator([2], 4, make_inputs([2], 4, 47)).ranked
    lib = _lib.load()
    ws = torch.empty(int(lib.gcgcn_rank_relations_ws_bytes(6, 4)), dtype=torch.uint8, device=DEV)
    out_key, out_pay = torch.empty_like(key), torch.empty_like(pay)
    with pytest.raises(_lib.GcgcnError, match="multiple"):      # 5 candidates cannot be 3 relations' equal shares
        _lib.call("gcgcn_rank_by_relation", _p(key), _p(pay), 5, 4, _p(out_key), _p(out_pay), _p(ws), ws.numel(),
                  _stream(DEV))
    with pytest.raises(_lib.GcgcnError, match="ws_bytes"):
        _lib.call("gcgcn_rank_by_relation", _p(key), _p(pay), 6, 4, _p(out_key), _p(out_pay), _p(ws), 16,
                  _stream(DEV))
