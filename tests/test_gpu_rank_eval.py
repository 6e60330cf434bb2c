"""-m gpu: relation evaluation on the device (gcgcn_b200/evaluate.py, csrc/rank.cu) against the NumPy oracle
(oracle/rank_oracle.py) fed the evaluator's own float32 scores, and against torch.sort at the bench-shard size."""
import numpy as np
import pytest
import torch

from helpers import head_labels, head_state
from oracle import rank_oracle as RO
from gcgcn_b200 import _lib, synthetic as S
from gcgcn_b200.batch import RaggedBatch
from gcgcn_b200.evaluate import MAX_CANDIDATES, RESULT_BYTES, SORT_TILE, RelationEvaluator
from gcgcn_b200.functional import _p, _stream

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
R = 97
EXACT = ("count", "total_recall", "f1", "theta", "best_pos", "w", "f1_at_w", "precision_at_w", "recall_at_w", "ign_f1",
         "ign_f1_at_w")


def sort_direct(score):
    """gcgcn_rank_sort on scores with payload = id << 2 | id & 3 (the flags must travel with the id)."""
    n = score.numel()
    ids = torch.arange(n, dtype=torch.int64, device=DEV)
    pay = ((ids << 2) | (ids & 3)).to(torch.int32)
    ws = torch.empty(int(_lib.load().gcgcn_rank_ws_bytes(n)), dtype=torch.uint8, device=DEV)
    key, spay = torch.empty_like(pay), torch.empty_like(pay)
    _lib.call("gcgcn_rank_sort", _p(score), _p(pay), n, _p(key), _p(spay), _p(ws), ws.numel(), _stream(DEV))
    return key, spay


def tie_heavy(n, seed):
    rng = np.random.RandomState(seed)
    s = rng.rand(n).astype(np.float32)
    tie = rng.rand(n) < 0.7
    levels = np.asarray([0.0, 1.0, 0.5, 1e-30, 0.75, np.float32(2.0 ** -126)], np.float32)
    s[tie] = levels[rng.randint(len(levels), size=int(tie.sum()))]
    return s


def candidate_mask(sizes, R=R):
    """[total_pairs, R] bool: True at the candidates (off-diagonal pairs, r >= 1); boolean indexing with it lists them
    in id order."""
    bt = RaggedBatch(sizes, "cpu")
    keep = torch.ones(bt.total_pairs, R, dtype=torch.bool)
    keep[:, 0] = False
    diag = np.concatenate([bt.pair_ptr_host[b] + np.arange(n) * (n + 1) for b, n in enumerate(sizes)] or [np.zeros(0)])
    keep[torch.from_numpy(diag.astype(np.int64))] = False
    return keep


def make_inputs(sizes, seed, scale=8.0, p_true=0.05, p_train=0.5):
    gen = torch.Generator(device=DEV).manual_seed(seed)
    P = int(sum(n * n for n in sizes))
    z = torch.randn(P, R, generator=gen, device=DEV) * scale          # saturates to exact 0 and 1 often: many ties
    z[torch.rand(P, R, generator=gen, device=DEV) < 0.2] = 3.0        # and a repeated mid value
    labels = (torch.rand(P, R, generator=gen, device=DEV) < p_true).float()
    intrain = (torch.rand(P, R, generator=gen, device=DEV) < p_train) & (labels > 0.5)
    return z, labels, intrain


def oracle_for(ev, sizes, labels, intrain, **kw):
    keep = candidate_mask(sizes).to(DEV)
    s = ev.scores.cpu().numpy()
    c = (labels[keep] > 0.5).cpu().numpy()
    it = None if intrain is None else intrain[keep].cpu().numpy()
    return RO.vectorised(s, c, it, **kw)


def check_against(res, ref):
    for k in EXACT:
        assert res[k] == ref[k], (k, res[k], ref[k])
    assert abs(res["auc"] - ref["auc"]) <= 1e-5 * max(abs(ref["auc"]), 1e-30) + 1e-12
    assert abs(res["auc"] - ref["auc_f64"]) <= 1e-9
    if ref["ign_auc"] is not None:
        assert abs(res["ign_auc"] - ref["ign_auc"]) <= 1e-5 * max(abs(ref["ign_auc"]), 1e-30) + 1e-12
        assert abs(res["ign_auc"] - ref["ign_auc_f64"]) <= 1e-9


# ------------------------------------------------------------------------------------------------------------- sort
@pytest.mark.parametrize("count", [1, 2, SORT_TILE - 1, SORT_TILE, SORT_TILE + 1, 100_000])
def test_sort_is_stable_and_exact(count):
    s = tie_heavy(count, count)
    key, pay = sort_direct(torch.from_numpy(s).to(DEV))
    order = np.argsort(-s, kind="stable")
    key, pay = key.cpu().numpy().view(np.uint32), pay.cpu().numpy().view(np.uint32)
    np.testing.assert_array_equal(pay >> 2, order)
    np.testing.assert_array_equal(pay & 3, order & 3)
    np.testing.assert_array_equal(~key, s[order].view(np.uint32))


def shard_scores(num_docs, seed):
    sizes = S.shard_doc_sizes(num_docs)
    bt = RaggedBatch(sizes, DEV)
    gen = torch.Generator(device=DEV).manual_seed(seed)
    z = torch.randn(bt.total_pairs, R, generator=gen, device=DEV) * 8.0
    ev = RelationEvaluator(R, DEV)
    ev.add(z, None, bt)
    return ev, z, sizes


@pytest.mark.parametrize("num_docs", [175, 6144])      # 1.0e7 candidates; the 6144-document bench shard (2.9e8)
def test_sort_matches_torch_stable_sort(num_docs):
    ev, z, sizes = shard_scores(num_docs, 7)
    s = ev.scores
    ref = torch.sort(s, descending=True, stable=True)
    key, pay = ev.ranked
    assert torch.equal((pay.long() & 0xFFFFFFFF) >> 2, ref.indices)
    assert torch.equal(torch.bitwise_not(key), ref.values.view(torch.int32))


def test_scores_within_one_ulp_of_torch_sigmoid():
    sizes = [5, 0, 1, 9, 42]
    z, _, _ = make_inputs(sizes, 3)
    ev = RelationEvaluator(R, DEV)
    ev.add(z, None, RaggedBatch(sizes, DEV))
    ref = torch.sigmoid(z)[candidate_mask(sizes).to(DEV)]
    got = ev.scores
    assert got.shape == ref.shape
    assert int((got.view(torch.int32) - ref.view(torch.int32)).abs().max()) <= 1


# ------------------------------------------------------------------------------------------------------------ curve
SIZES = [0, 1, 2, 5, 9, 13, 21, 3]


@pytest.mark.parametrize("theta", [-1.0, 0.5, 0.95, 2.0, -0.5])
@pytest.mark.parametrize("total_recall", [None, 1000])
def test_curve_matches_the_oracle(theta, total_recall):
    z, labels, intrain = make_inputs(SIZES, 11)
    ev = RelationEvaluator(R, DEV)
    ev.add(z, labels, RaggedBatch(SIZES, DEV), intrain=intrain)
    res = ev.result(input_theta=theta, total_recall=total_recall)
    ref = oracle_for(ev, SIZES, labels, intrain, input_theta=theta, total_recall=total_recall)
    check_against(res, ref)
    pay = ev.ranked[1].cpu().numpy().view(np.uint32)
    np.testing.assert_array_equal(pay >> 2, ref["order"])


def test_curve_matches_the_literal_loop_and_theta_roundtrip():
    sizes = [3, 4, 2]
    z, labels, intrain = make_inputs(sizes, 5, p_true=0.2)
    ev = RelationEvaluator(R, DEV)
    ev.add(z, labels, RaggedBatch(sizes, DEV), intrain=intrain)
    s = ev.scores.cpu().numpy()
    cand = RO.candidates([(np.zeros((n, n, R), np.float32), np.zeros((n, n, R), bool), None) for n in sizes])
    lab = labels.cpu().numpy().reshape(-1, R) > 0.5
    it = intrain.cpu().numpy().reshape(-1, R)
    bt = RaggedBatch(sizes, "cpu")
    docs = []
    for b, n in enumerate(sizes):
        p0 = int(bt.pair_ptr_host[b])
        sc = np.zeros((n, n, R), np.float32)
        m = cand[3] == b
        sc[cand[4][m], cand[5][m], cand[6][m]] = s[m]
        docs.append((sc, lab[p0:p0 + n * n].reshape(n, n, R), it[p0:p0 + n * n].reshape(n, n, R)))
    res = ev.result()
    check_against(res, RO.literal(docs))
    check_against(ev.result(input_theta=res["theta"]), RO.literal(docs, input_theta=res["theta"]))


def test_no_intrain_and_no_positives():
    z, labels, _ = make_inputs(SIZES, 2)
    ev = RelationEvaluator(R, DEV)
    ev.add(z, torch.zeros_like(labels), RaggedBatch(SIZES, DEV))
    res = ev.result()
    assert res["ign_f1"] is None and res["ign_auc"] is None and res["ign_f1_at_w"] is None
    assert res["total_recall"] == 1 and res["f1"] == 0.0 and res["best_pos"] == 0 and res["auc"] == 0.0
    check_against(res, oracle_for(ev, SIZES, torch.zeros_like(labels), None))


def test_curve_at_bench_shard_size_against_a_torch_restatement():
    sizes = S.shard_doc_sizes(6144)
    bt = RaggedBatch(sizes, DEV)
    z, labels, intrain = make_inputs(list(sizes), 13, scale=6.0, p_true=0.02)
    ev = RelationEvaluator(R, DEV)
    ev.add(z, labels, bt, intrain=intrain)
    theta = 0.9
    res, res_t = ev.result(), ev.result(input_theta=theta)
    keep = candidate_mask(list(sizes)).to(DEV)
    s = ev.scores
    assert int((s.view(torch.int32) - torch.sigmoid(z[keep]).view(torch.int32)).abs().max()) <= 1
    corr = labels[keep] > 0.5
    intr = intrain[keep]
    del z, labels, intrain, keep
    order = torch.sort(s, descending=True, stable=True).indices
    c = torch.cumsum(corr[order], 0)
    t = torch.cumsum((corr & intr)[order], 0)
    del corr, intr
    N = s.numel()
    T = int(c[-1])
    k1 = torch.arange(1, N + 1, device=DEV, dtype=torch.float64)
    x = (c.double() / T).float()
    y = (c.double() / k1).float()
    f1 = 2 * x * y / (x + y + 1e-20)
    yi = torch.where(t == c, torch.zeros((), device=DEV, dtype=torch.float64),
                     (c - t).double() / (k1 - t.double()).clamp(min=1.0)).float()
    f1i = 2 * x * yi / (x + yi + 1e-20)
    best = int(torch.argmax(f1))
    w_t = int((s > theta).sum()) - 1
    assert res["count"] == N and res["total_recall"] == T
    assert res["best_pos"] == best and res["f1"] == float(f1[best]) and res["theta"] == float(s[order[best]])
    assert res["ign_f1"] == float(f1i.max()) and res["ign_f1_at_w"] == float(f1i[best])
    assert res_t["w"] == w_t and res_t["f1_at_w"] == float(f1[w_t]) and res_t["ign_f1_at_w"] == float(f1i[w_t])
    assert res_t["precision_at_w"] == float(y[w_t]) and res_t["recall_at_w"] == float(x[w_t])
    auc = float(((x[1:] - x[:-1]) * (y[1:] + y[:-1]) / 2).double().sum())
    iauc = float(((x[1:] - x[:-1]) * (yi[1:] + yi[:-1]) / 2).double().sum())
    assert abs(res["auc"] - auc) <= 1e-9 and abs(res["ign_auc"] - iauc) <= 1e-9


# ------------------------------------------------------------------------------------------------------- candidates
def test_batches_split_across_adds_give_the_same_result_bit_for_bit():
    z, labels, intrain = make_inputs(SIZES, 17)
    one = RelationEvaluator(R, DEV)
    one.add(z, labels, RaggedBatch(SIZES, DEV), intrain=intrain)
    many = RelationEvaluator(R, DEV)
    bt = RaggedBatch(SIZES, "cpu")
    for lo, hi in ((0, 3), (3, 4), (4, 4), (4, len(SIZES))):
        p0, p1 = int(bt.pair_ptr_host[lo]), int(bt.pair_ptr_host[hi])
        many.add(z[p0:p1], labels[p0:p1], RaggedBatch(SIZES[lo:hi], DEV), intrain=intrain[p0:p1])
    assert torch.equal(one.scores, many.scores)
    a, b = one.result(), many.result()
    assert a == b and a == one.result()                    # and two calls on the same evaluator agree
    for x, y in zip(one.ranked, many.ranked):
        assert torch.equal(x, y)
    pa, pb = one.predictions(), many.predictions()
    for k in pa:
        assert torch.equal(pa[k], pb[k])


def test_add_after_result_reranks():
    z, labels, intrain = make_inputs(SIZES, 19)
    ev = RelationEvaluator(R, DEV)
    ev.add(z, labels, RaggedBatch(SIZES, DEV), intrain=intrain)
    first = ev.result()
    ev.add(z, labels, RaggedBatch(SIZES, DEV), intrain=intrain)
    both = ev.result()
    assert both["count"] == 2 * first["count"]
    s = ev.scores.cpu().numpy()
    keep = candidate_mask(SIZES).to(DEV)
    c = np.concatenate([(labels[keep] > 0.5).cpu().numpy()] * 2)
    it = np.concatenate([intrain[keep].cpu().numpy()] * 2)
    check_against(both, RO.vectorised(s, c, it))


# ------------------------------------------------------------------------------------------------------- end to end
def test_graph_head_end_to_end():
    from gcgcn_b200.featurize import wire_from_record
    from gcgcn_b200.head import GraphHead, HeadBatch
    seeds = list(range(12))
    wires = [wire_from_record(S.make_record(sd, n=S.DOC_N[sd], L=S.DOC_L[sd], S=S.DOC_S[sd])) for sd in seeds]
    head = GraphHead()
    head.load_state_dict(head_state(0), strict=True)
    head = head.to(DEV).eval()
    hb = HeadBatch(wires, DEV)
    sizes = [w.n for w in wires]
    gen = torch.Generator(device=DEV).manual_seed(0)
    ctx = torch.randn(hb.total_tokens, 128, generator=gen, device=DEV)
    labels = torch.cat([head_labels(sd, w.n).view(-1, R) for sd, w in zip(seeds, wires)]).to(DEV)
    with torch.no_grad():
        logits = head(ctx, hb)["logits"]
    ev = RelationEvaluator(R, DEV)
    ev.add(logits, labels, hb.batch)
    res = ev.result()
    check_against(res, oracle_for(ev, sizes, labels, None))
    pred = ev.predictions(res["theta"])
    rows = pred["score"].numel()
    assert rows == ev.result(input_theta=res["theta"])["w"] + 1
    doc, i, j, r = (pred[k].long().cpu() for k in ("doc", "row", "col", "relation"))
    n = torch.tensor(sizes)[doc]
    pair_ptr = torch.from_numpy(hb.batch.pair_ptr_host)[doc]
    assert bool((i != j).all()) and bool((r >= 1).all()) and bool((i < n).all()) and bool((j < n).all())
    z = logits[(pair_ptr + i * n + j).to(DEV), r.to(DEV)]
    bits = pred["score"].view(torch.int32)
    assert int((bits - torch.sigmoid(z).view(torch.int32)).abs().max()) <= 1
    # the id the candidate kernel gave that (doc, row, col, relation) holds exactly that score
    off = torch.from_numpy(np.concatenate([[0], np.cumsum([(m * m - m) * (R - 1) for m in sizes])]))[doc]
    ids = off + (i * (n - 1) + j - (j > i).long()) * (R - 1) + r - 1
    assert torch.equal(ev.scores.cpu()[ids], pred["score"].cpu())
    assert torch.equal(((ev.ranked[1][:rows].long() & 0xFFFFFFFF) >> 2).cpu(), ids)
    if bool((ev.scores > res["theta"]).any()):
        assert bool((pred["score"].cpu() > res["theta"]).all())       # the list the reference dumps


# ----------------------------------------------------------------------------------------------------------- errors
def test_errors():
    sizes = [4, 3]
    z, labels, _ = make_inputs(sizes, 23)
    bt = RaggedBatch(sizes, DEV)
    count = sum(n * n - n for n in sizes) * (R - 1)
    score = torch.empty(count, device=DEV)
    pay = torch.empty(count, dtype=torch.int32, device=DEV)
    ctr = torch.zeros(2, dtype=torch.int64, device=DEV)
    with pytest.raises(_lib.GcgcnError, match="2\\^30"):
        _lib.call("gcgcn_rank_candidates", bt.ref, _p(z), R, _p(labels), None, MAX_CANDIDATES - count, _p(score), _p(pay),
                  _p(ctr), _stream(DEV))
    ev = RelationEvaluator(R, DEV)
    ev.count = MAX_CANDIDATES - 1                           # as if nearly 2^30 candidates had been added
    with pytest.raises(_lib.GcgcnError, match="2\\^30"):
        ev.add(z, labels, bt)

    bad = z.clone()
    bad[1, 7] = float("nan")                                # pair (0, 1) of the first document
    ev = RelationEvaluator(R, DEV)
    ev.add(bad, labels, bt)
    with pytest.raises(_lib.GcgcnError, match="NaN"):
        ev.result()

    ev = RelationEvaluator(R, DEV)
    ev.add(z, None, bt)
    with pytest.raises(_lib.GcgcnError, match="without labels"):
        ev.result()
    with pytest.raises(_lib.GcgcnError):
        ev.predictions()
    pred = ev.predictions(0.5)                              # unlabeled sets still list their predictions
    assert pred["score"].numel() == int((ev.scores > 0.5).sum())

    ev = RelationEvaluator(R, DEV)
    with pytest.raises(_lib.GcgcnError):
        ev.add(z[:-1], labels[:-1], bt)                     # logits not [total_pairs, R]
    with pytest.raises(_lib.GcgcnError):
        ev.add(z, labels[:, :-1], bt)
    with pytest.raises(_lib.GcgcnError):
        ev.add(z, labels, bt, intrain=labels[:-1] > 0)
    with pytest.raises(_lib.GcgcnError):
        RelationEvaluator(R, DEV).add(z[:, :-1], None, bt)  # relations differ from the evaluator's
    with pytest.raises(_lib.GcgcnError):
        ev.result()                                         # nothing added
    ev.add(torch.zeros(1, R, device=DEV), None, RaggedBatch([1], DEV))
    with pytest.raises(_lib.GcgcnError, match="no candidates"):
        ev.predictions(0.5)


def test_unaligned_workspace_and_decode_bounds():
    """The workspace may have any alignment (the library aligns inside it); decode refuses rows beyond the ranking."""
    z, labels, intrain = make_inputs(SIZES, 29)
    ev = RelationEvaluator(R, DEV)
    ev.add(z, labels, RaggedBatch(SIZES, DEV), intrain=intrain)
    ref = ev.result()
    key0, pay0 = ev.ranked
    n = ev.count
    nbytes = int(_lib.load().gcgcn_rank_ws_bytes(n))
    raw = torch.empty(nbytes + 64, dtype=torch.uint8, device=DEV)
    ws = raw[4:4 + nbytes]                                  # 4 bytes past a 512-byte boundary
    key, pay = torch.empty_like(key0), torch.empty_like(pay0)
    score, payload = ev._chunks[0]
    _lib.call("gcgcn_rank_sort", _p(score), _p(payload), n, _p(key), _p(pay), _p(ws), nbytes, _stream(DEV))
    assert torch.equal(key, key0) and torch.equal(pay, pay0)
    out = torch.empty(RESULT_BYTES, dtype=torch.uint8, device=DEV)
    _lib.call("gcgcn_rank_curve", _p(key), _p(pay), n, ref["total_recall"], 1, -1.0, _p(out), _p(ws), nbytes,
              _stream(DEV))
    r = _lib.RankResult.from_buffer_copy(out.cpu().numpy().tobytes())
    assert (r.best_pos, r.w, r.f1, r.auc, r.ign_f1, r.ign_auc) == (ref["best_pos"], ref["w"], ref["f1"], ref["auc"],
                                                                  ref["ign_f1"], ref["ign_auc"])
    doc_off = torch.zeros(len(SIZES) + 1, dtype=torch.int64, device=DEV)
    doc_n = torch.tensor(SIZES, dtype=torch.int32, device=DEV)
    cols = [torch.empty(n + 1, dtype=torch.int32, device=DEV) for _ in range(4)]
    sc = torch.empty(n + 1, device=DEV)
    with pytest.raises(_lib.GcgcnError, match="rows"):
        _lib.call("gcgcn_rank_decode", _p(key), _p(pay), n + 1, n, _p(doc_off), _p(doc_n), len(SIZES), R,
                  *[_p(c) for c in cols], _p(sc), _stream(DEV))
