"""-m gpu: relation evaluation of a document set held in shards (gcgcn_b200/evaluate.py, csrc/rank.cu): global
candidate ids, the merge of sorted rankings, RelationEvaluator.merged / all_gather and the curve points.  The merged
evaluator must equal, bit for bit, one evaluator fed the union of the documents in ascending global order; that one is
tied to the local-id evaluator and to the NumPy oracle (oracle/rank_oracle.py)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import rank_oracle as RO
from test_gpu_rank_eval import candidate_mask, check_against, make_inputs, tie_heavy
from gcgcn_b200 import _lib
from gcgcn_b200.batch import RaggedBatch, shard_documents
from gcgcn_b200.evaluate import MAX_CANDIDATES, SORT_TILE, RelationEvaluator
from gcgcn_b200.functional import _p, _stream
from gcgcn_b200.sharding import local_documents

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
R = 97
# 16 documents, 89 088 candidates (22 sort tiles); documents 0, 1, 9 and 13 have no candidate
SIZES = [0, 1, 2, 5, 9, 13, 21, 3, 7, 1, 4, 11, 6, 0, 8, 2]


# ------------------------------------------------------------------------------------------------------------ helpers
def _pair_rows(sizes, docs):
    ptr = np.concatenate([[0], np.cumsum(np.asarray(sizes, np.int64) ** 2)])
    rows = [np.arange(ptr[g], ptr[g + 1]) for g in docs]
    return torch.from_numpy(np.concatenate(rows + [np.zeros(0, np.int64)]).astype(np.int64))


def feed(ev, sizes, data, docs, dev=DEV, batches=2, doc_index=True):
    """add() the documents `docs` (ascending global indices) in `batches` consecutive batches."""
    z, labels, intrain = data
    for chunk in np.array_split(np.asarray(docs, np.int64), batches):
        if chunk.size == 0:
            continue
        rows = _pair_rows(sizes, chunk).to(z.device)
        ev.add(z[rows].to(dev), None if labels is None else labels[rows].to(dev),
               RaggedBatch([sizes[g] for g in chunk], dev), intrain=None if intrain is None else intrain[rows].to(dev),
               doc_index=chunk.tolist() if doc_index else None)
    return ev


def inputs(seed, with_intrain=True):
    z, labels, intrain = make_inputs(SIZES, seed)
    return z, labels, intrain if with_intrain else None


def assert_same_evaluation(a, b):
    """ranked arrays, result at two thresholds, predictions and curve of a and b are bit-identical."""
    for x, y in zip(a.ranked, b.ranked):
        assert torch.equal(x, y)
    for theta in (-1.0, 0.5):
        assert a.result(input_theta=theta) == b.result(input_theta=theta)
    res = a.result()
    pa, pb = a.predictions(res["theta"]), b.predictions(res["theta"])
    assert pa.keys() == pb.keys()
    for k in pa:
        assert torch.equal(pa[k], pb[k]), k
    for total_recall in (None, 1000):
        ca, cb = a.curve(total_recall), b.curve(total_recall)
        for k in ("x", "y", "y_ign"):
            assert (ca[k] is None) == (cb[k] is None), k
            if ca[k] is not None:
                assert torch.equal(ca[k], cb[k]), k


def contiguous_split(n_docs, parts, seed):
    """`parts` contiguous runs of uneven length (empty ones included)."""
    cuts = np.sort(np.random.RandomState(seed).randint(0, n_docs + 1, size=parts - 1))
    bounds = np.concatenate([[0], cuts, [n_docs]])
    return [list(range(bounds[k], bounds[k + 1])) for k in range(parts)]


def global_ids(sizes, docs):
    n = np.asarray(sizes, np.int64)
    first = np.concatenate([[0], np.cumsum((n * n - n) * (R - 1))])
    return np.concatenate([np.arange(first[g], first[g + 1]) for g in docs])


def oracle_curve(score, correct, intrain, total_recall=None):
    """pr_x, pr_y, pr_yi as RO.vectorised forms them (restated: the oracle returns only the scalars)."""
    order = np.argsort(-score, kind="stable")
    T = int(correct.sum()) if total_recall is None else int(total_recall)
    T = max(T, 1)
    c = np.cumsum(correct[order], dtype=np.int64)
    k1 = np.arange(1, len(order) + 1, dtype=np.int64)
    pr_x, pr_y = (c / T).astype(np.float32), (c / k1).astype(np.float32)
    if intrain is None:
        return pr_x, pr_y, None
    t = np.cumsum((correct & intrain)[order], dtype=np.int64)
    pr_yi = np.where(t == c, 0.0, (c - t) / np.where(t == c, 1, k1 - t)).astype(np.float32)
    return pr_x, pr_y, pr_yi


# ------------------------------------------------------------------------------------------------------- the kernel
def merge_direct(ka, pa, kb, pb, ws_offset=0):
    na, nb = ka.numel(), kb.numel()
    nbytes = int(_lib.load().gcgcn_rank_merge_ws_bytes(na + nb))
    raw = torch.empty(nbytes + 64, dtype=torch.uint8, device=DEV)
    ws = raw[ws_offset:ws_offset + nbytes]
    key = torch.empty(na + nb, dtype=torch.int32, device=DEV)
    pay = torch.empty_like(key)
    _lib.call("gcgcn_rank_merge", _p(ka), _p(pa), na, _p(kb), _p(pb), nb, _p(key), _p(pay), _p(ws), nbytes,
              _stream(DEV))
    return key, pay


def composite(key, pay):
    """(key, payload) as one int64 whose signed order is the unsigned 64-bit order of key << 32 | payload."""
    return (((key.long() & 0xFFFFFFFF) - (1 << 31)) << 32) | (pay.long() & 0xFFFFFFFF)


def sorted_run(n, seed, all_equal=False):
    """A run ascending by (key, payload): keys tie-heavy (70 % on six levels, exact 0 and 1 among them), payloads
    random 32-bit values."""
    gen = torch.Generator(device=DEV).manual_seed(seed)
    if n <= 1 << 20:
        key = torch.from_numpy(~tie_heavy(n, seed).view(np.uint32)).view(torch.int32).to(DEV)
    else:
        levels = torch.from_numpy(~tie_heavy(64, seed).view(np.uint32)).view(torch.int32).to(DEV)
        key = torch.randint(-2 ** 31, 2 ** 31, (n,), generator=gen, device=DEV, dtype=torch.int64).to(torch.int32)
        tie = torch.rand(n, generator=gen, device=DEV) < 0.7
        key = torch.where(tie, levels[torch.randint(0, 64, (n,), generator=gen, device=DEV)], key)
    if all_equal:
        key = torch.full((n,), -1082130433, dtype=torch.int32, device=DEV)      # ~bits(1.0)
    pay = torch.randint(-2 ** 31, 2 ** 31, (n,), generator=gen, device=DEV, dtype=torch.int64).to(torch.int32)
    order = torch.sort(composite(key, pay), stable=True).indices
    return key[order], pay[order]


def check_merge(na, nb, seed, all_equal=False, ws_offset=0):
    ka, pa = sorted_run(na, seed, all_equal)
    kb, pb = sorted_run(nb, seed + 1, all_equal)
    key, pay = merge_direct(ka, pa, kb, pb, ws_offset)
    ck = torch.cat([ka, kb])
    cp = torch.cat([pa, pb])
    order = torch.sort(composite(ck, cp), stable=True).indices
    assert torch.equal(key, ck[order]) and torch.equal(pay, cp[order])


T = SORT_TILE


@pytest.mark.parametrize("na,nb", [(0, 1), (1, 0), (0, T), (T, 0), (1, 1), (T // 2 - 1, T // 2), (T // 2, T // 2),
                                   (T // 2, T // 2 + 1), (T - 1, T + 1), (2 * T - 1, 1), (3 * T + 1, 2),
                                   (100_000, 37), (250_000, 260_001)])
def test_merge_is_the_stable_sort_of_the_concatenation(na, nb):
    check_merge(na, nb, 3 * na + nb)


@pytest.mark.parametrize("na,nb", [(T, T), (5000, 70_000)])
def test_merge_all_equal_keys(na, nb):
    check_merge(na, nb, 5, all_equal=True)


def test_merge_two_runs_of_150m():
    check_merge(150_000_000, 150_000_007, 11)


def test_merge_misaligned_workspace_and_argument_errors():
    check_merge(30_000, 9_000, 13, ws_offset=4)
    ka, pa = sorted_run(1000, 1)
    kb, pb = sorted_run(1000, 2)
    nbytes = int(_lib.load().gcgcn_rank_merge_ws_bytes(2000))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    out = torch.empty(2 * 2000 + 4, dtype=torch.int32, device=DEV)
    with pytest.raises(_lib.GcgcnError, match="aligned"):
        _lib.call("gcgcn_rank_merge", _p(ka), _p(pa), 1000, _p(kb), _p(pb), 1000, _p(out[1:]), _p(out[2004:]), _p(ws),
                  nbytes, _stream(DEV))
    with pytest.raises(_lib.GcgcnError, match="ws_bytes"):
        _lib.call("gcgcn_rank_merge", _p(ka), _p(pa), 1000, _p(kb), _p(pb), 1000, _p(out), _p(out[2000:]), _p(ws),
                  nbytes - 1, _stream(DEV))
    with pytest.raises(_lib.GcgcnError, match="2\\^30"):          # checked before any pointer is read
        _lib.call("gcgcn_rank_merge", _p(ka), _p(pa), MAX_CANDIDATES // 2, _p(kb), _p(pb), MAX_CANDIDATES // 2,
                  _p(out), _p(out[2000:]), _p(ws), nbytes, _stream(DEV))


# ------------------------------------------------------------------------------------------------- single process
SPLITS = [(parts, kind) for parts in (1, 2, 3, 5, 8) for kind in ("shard", "contiguous")]


@pytest.mark.parametrize("parts,kind", SPLITS)
def test_merged_parts_equal_one_evaluator_over_the_union(parts, kind):
    data = inputs(31 + parts)
    shards = shard_documents(SIZES, parts) if kind == "shard" else contiguous_split(len(SIZES), parts, parts)
    evs = [feed(RelationEvaluator(R, DEV, doc_sizes=SIZES), SIZES, data, docs) for docs in shards]
    merged = RelationEvaluator.merged(evs)
    one = feed(RelationEvaluator(R, DEV, doc_sizes=SIZES), SIZES, data, range(len(SIZES)), batches=1)
    assert merged.count == one.count
    assert_same_evaluation(merged, one)


def test_zero_candidate_and_empty_parts_merge_away():
    data = inputs(41)
    docs = [d for d in range(len(SIZES)) if d not in (0, 1, 9, 13)]
    evs = [feed(RelationEvaluator(R, DEV, doc_sizes=SIZES), SIZES, data, [0, 1, 9]),       # no candidates
           RelationEvaluator(R, DEV, doc_sizes=SIZES),                                       # no add() at all
           feed(RelationEvaluator(R, DEV, doc_sizes=SIZES), SIZES, data, docs)]
    one = feed(RelationEvaluator(R, DEV, doc_sizes=SIZES), SIZES, data, range(len(SIZES)))
    assert_same_evaluation(RelationEvaluator.merged(evs), one)
    assert_same_evaluation(RelationEvaluator.merged([evs[2]]), one)


@pytest.mark.parametrize("with_intrain", [True, False])
def test_global_ids_over_every_document_equal_local_ids(with_intrain):
    data = inputs(43, with_intrain)
    glob = feed(RelationEvaluator(R, DEV, doc_sizes=SIZES), SIZES, data, range(len(SIZES)), batches=3)
    loc = feed(RelationEvaluator(R, DEV), SIZES, data, range(len(SIZES)), batches=3, doc_index=False)
    assert torch.equal(glob.scores, loc.scores)
    assert_same_evaluation(glob, loc)
    # and the all_gather of a process without a process group is merged([ev])
    assert_same_evaluation(glob.all_gather(), loc)


@pytest.mark.parametrize("with_intrain", [True, False])
def test_subset_with_gaps_matches_the_oracle(with_intrain):
    data = inputs(47, with_intrain)
    z, labels, intrain = data
    subset = [2, 3, 5, 6, 8, 10, 11, 14, 15]
    parts = [subset[0::3], subset[1::3], subset[2::3]]
    merged = RelationEvaluator.merged([feed(RelationEvaluator(R, DEV, doc_sizes=SIZES), SIZES, data, p)
                                       for p in parts])
    # the oracle on the union in global order, fed the scores of the candidate kernel
    scores = feed(RelationEvaluator(R, DEV), SIZES, data, subset, batches=1, doc_index=False).scores.cpu().numpy()
    rows = _pair_rows(SIZES, subset).to(DEV)
    keep = candidate_mask([SIZES[g] for g in subset]).to(DEV)
    correct = (labels[rows][keep] > 0.5).cpu().numpy()
    it = None if intrain is None else intrain[rows][keep].cpu().numpy()
    ids = global_ids(SIZES, subset)
    for theta in (-1.0, 0.5):
        ref = RO.vectorised(scores, correct, it, input_theta=theta)
        check_against(merged.result(input_theta=theta), ref)
        pay = merged.ranked[1].cpu().numpy().view(np.uint32)
        np.testing.assert_array_equal(pay >> 2, ids[ref["order"]])
    for total_recall in (None, 1000):
        x, y, yi = oracle_curve(scores, correct, it, total_recall)
        c = merged.curve(total_recall)
        np.testing.assert_array_equal(c["x"].cpu().numpy().view(np.uint32), x.view(np.uint32))
        np.testing.assert_array_equal(c["y"].cpu().numpy().view(np.uint32), y.view(np.uint32))
        if yi is None:
            assert c["y_ign"] is None
        else:
            np.testing.assert_array_equal(c["y_ign"].cpu().numpy().view(np.uint32), yi.view(np.uint32))
    pred = merged.predictions(merged.result()["theta"])
    assert set(pred["doc"].cpu().tolist()) <= set(subset)         # global document indices


def test_curve_points_of_the_local_evaluator_match_the_oracle():
    z, labels, intrain = make_inputs(SIZES, 53)
    ev = RelationEvaluator(R, DEV)
    ev.add(z, labels, RaggedBatch(SIZES, DEV), intrain=intrain)
    keep = candidate_mask(SIZES).to(DEV)
    x, y, yi = oracle_curve(ev.scores.cpu().numpy(), (labels[keep] > 0.5).cpu().numpy(), intrain[keep].cpu().numpy())
    c = ev.curve()
    assert c["x"].dtype == torch.float32 and c["x"].numel() == ev.count
    for got, ref in ((c["x"], x), (c["y"], y), (c["y_ign"], yi)):
        np.testing.assert_array_equal(got.cpu().numpy().view(np.uint32), ref.view(np.uint32))
    res = ev.result()
    assert float(c["x"][res["best_pos"]]) == res["recall_at_w"] and float(c["y"][res["best_pos"]]) == res["precision_at_w"]


# ----------------------------------------------------------------------------------------------------------- errors
def test_errors():
    data = inputs(59)
    z, labels, _ = data
    with pytest.raises(_lib.GcgcnError, match="2\\^30"):
        RelationEvaluator(R, DEV, doc_sizes=[3, 1 << 13, 5])         # (2^26 - 2^13) 96 candidates: nothing allocated
    ev = RelationEvaluator(R, DEV, doc_sizes=SIZES)
    with pytest.raises(_lib.GcgcnError, match="needs doc_index"):
        feed(ev, SIZES, data, [2, 3], batches=1, doc_index=False)
    with pytest.raises(_lib.GcgcnError, match="doc_index needs"):
        feed(RelationEvaluator(R, DEV), SIZES, data, [2, 3], batches=1)
    rows = _pair_rows(SIZES, [2, 3]).to(DEV)
    bt = RaggedBatch([SIZES[2], SIZES[3]], DEV)
    for bad in ([2], [2, 3, 4], [2, 16], [-1, 3], [3, 2], [2, 2], [3, 4]):   # length, range, order, entity counts
        with pytest.raises(_lib.GcgcnError):
            ev.add(z[rows], labels[rows], bt, doc_index=bad)
    ev.add(z[rows], labels[rows], bt, doc_index=[2, 3])
    rows4 = _pair_rows(SIZES, [3]).to(DEV)
    with pytest.raises(_lib.GcgcnError, match="increase"):
        ev.add(z[rows4], labels[rows4], RaggedBatch([SIZES[3]], DEV), doc_index=[3])    # not after the last one
    assert ev._docs == [2, 3]

    def part(docs, **kw):
        return feed(RelationEvaluator(R, DEV, **kw), SIZES, data, docs, batches=1, doc_index="doc_sizes" in kw)

    a = part([2, 3], doc_sizes=SIZES)
    with pytest.raises(_lib.GcgcnError, match="doc_sizes"):
        RelationEvaluator.merged([a, part([5])])                      # a part without global ids
    with pytest.raises(_lib.GcgcnError, match="doc_sizes"):
        part([5]).all_gather()
    with pytest.raises(_lib.GcgcnError, match="relations"):
        RelationEvaluator.merged([a, RelationEvaluator(5, DEV, doc_sizes=SIZES)])
    with pytest.raises(_lib.GcgcnError, match="doc_sizes differ"):
        RelationEvaluator.merged([a, RelationEvaluator(R, DEV, doc_sizes=SIZES[:-1])])
    with pytest.raises(_lib.GcgcnError, match="share documents"):
        RelationEvaluator.merged([a, part([3, 5], doc_sizes=SIZES)])
    big = [RelationEvaluator(R, DEV, doc_sizes=SIZES) for _ in range(2)]
    for b in big:
        b.count = MAX_CANDIDATES // 2                                 # as if 2^29 candidates each had been added
    with pytest.raises(_lib.GcgcnError, match="2\\^30"):
        RelationEvaluator.merged(big)
    with pytest.raises(_lib.GcgcnError, match="no candidates"):
        RelationEvaluator.merged([part([0, 1], doc_sizes=SIZES), part([9, 13], doc_sizes=SIZES)])
    with pytest.raises(_lib.GcgcnError):
        RelationEvaluator.merged([])
    if torch.cuda.device_count() > 1:
        with pytest.raises(_lib.GcgcnError, match="parts on"):
            RelationEvaluator.merged([a, RelationEvaluator(R, torch.device("cuda:1"), doc_sizes=SIZES)])
    m = RelationEvaluator.merged([a])
    with pytest.raises(_lib.GcgcnError, match="final"):
        m.add(z[rows], labels[rows], bt, doc_index=[2, 3])
    with pytest.raises(_lib.GcgcnError, match="ranking only"):
        m.scores
    unlabeled = part([5], doc_sizes=SIZES)
    unlabeled._labeled = False
    with pytest.raises(_lib.GcgcnError, match="without labels"):
        RelationEvaluator.merged([a, unlabeled]).result()
    with pytest.raises(_lib.GcgcnError, match="without labels"):
        RelationEvaluator.merged([a, unlabeled]).curve()


# ---------------------------------------------------------------------------------------------------- several ranks
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _gather_worker(rank, world, port, backend, in_path, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = torch.device("cuda", rank if backend == "nccl" else 0)
    torch.cuda.set_device(dev)
    dist.init_process_group(backend, rank=rank, world_size=world)
    try:
        data = torch.load(in_path)
        ev = RelationEvaluator(R, dev, doc_sizes=SIZES)
        feed(ev, SIZES, data, local_documents(SIZES, rank, world), dev=dev)
        m = ev.all_gather()
        res = m.result()
        out = {"result": res, "result_05": m.result(input_theta=0.5), "ranked": [t.cpu() for t in m.ranked],
               "pred": {k: v.cpu() for k, v in m.predictions(res["theta"]).items()},
               "curve": {k: (None if v is None else v.cpu()) for k, v in m.curve().items()}}
        torch.save(out, os.path.join(out_dir, f"rank{rank}.pt"))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def _run_ranks(tmp_path, world, backend):
    data = inputs(61)
    in_path = str(tmp_path / "inputs.pt")
    torch.save([t.cpu() for t in data], in_path)
    mp.spawn(_gather_worker, args=(world, _free_port(), backend, in_path, str(tmp_path)), nprocs=world, join=True)
    one = feed(RelationEvaluator(R, DEV, doc_sizes=SIZES), SIZES, data, range(len(SIZES)), batches=1)
    res = one.result()
    ref = {"result": res, "result_05": one.result(input_theta=0.5), "ranked": [t.cpu() for t in one.ranked],
           "pred": {k: v.cpu() for k, v in one.predictions(res["theta"]).items()},
           "curve": {k: (None if v is None else v.cpu()) for k, v in one.curve().items()}}
    for r in range(world):
        got = torch.load(tmp_path / f"rank{r}.pt")
        assert got["result"] == ref["result"] and got["result_05"] == ref["result_05"], r
        for a, b in zip(got["ranked"], ref["ranked"]):
            assert torch.equal(a, b), r
        for k in ref["pred"]:
            assert torch.equal(got["pred"][k], ref["pred"][k]), (r, k)
        for k in ref["curve"]:
            assert torch.equal(got["curve"][k], ref["curve"][k]), (r, k)


def test_all_gather_two_ranks_on_one_gpu_through_gloo(tmp_path):
    _run_ranks(tmp_path, 2, "gloo")


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_all_gather_nccl_two_ranks(tmp_path):
    _run_ranks(tmp_path, 2, "nccl")


@pytest.mark.skipif(torch.cuda.device_count() < 3, reason="needs more than 2 GPUs")
def test_all_gather_nccl_every_gpu(tmp_path):
    _run_ranks(tmp_path, torch.cuda.device_count(), "nccl")
