"""Relation evaluation on the GPU: the DocRED baseline evaluation of ``Config.test`` (config/Config.py:432-561) and the
Ign F1 of ``Config_bert`` (config/Config_bert.py:626-650), from the logits ``GraphHead`` returns.

Every (document, row i, column j != i, relation r >= 1) is a candidate scored with sigmoid.  The candidates are ranked by
score, descending and stable (equal scores keep insertion order, as the reference's ``list.sort(reverse=True)``), and
the precision/recall curve over the ranking gives the best F1, the threshold where it is reached, the AUC and the F1 at
a given threshold (include/gcgcn_b200.h, "relation evaluation", has the exact definitions).  Scoring, the device-wide
radix sort, the curve and the decoding of predictions are this package's kernels (csrc/rank.cu); the host receives
one small result struct.  No CPU path.

    ev = RelationEvaluator(relations=97, device="cuda")
    for hb, context, labels in dev_batches:
        out = head(context, hb)                                  # GraphHead, eval mode, no_grad
        ev.add(out["logits"], labels, hb.batch)                  # labels / intrain: [total_pairs, R]
    res = ev.result(input_theta=-1.0)
    pred = ev.predictions(res["theta"])

``per_relation`` evaluates every relation's candidates alone (the same fields as ``result``, one entry per relation),
and ``result_at`` / ``predictions_at`` score and list the candidates above one threshold per relation, e.g. the θ_r a
dev set's ``per_relation`` found, applied to a test set.

A set evaluated in shards numbers its candidates globally: ``doc_sizes`` (the entity counts of every document of the
set, in its order) fixes each document's first candidate id, and ``add(..., doc_index=...)`` names the documents of a
batch.  Each shard is ranked alone; ``merged`` (one device) or ``all_gather`` (one shard per rank) merges the sorted
runs into the ranking of the whole set, so every rank computes the result one evaluator over all documents would.
"""
from __future__ import annotations

import ctypes
import hashlib
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from .batch import RaggedBatch
from .functional import _cuda, _p, _stream

SORT_TILE = 4096                # GCGCN_RANK_TILE of include/gcgcn_b200.h
MAX_CANDIDATES = 1 << 30        # one evaluator, or one globally numbered set, holds fewer (payload: id << 2 | flags)
RESULT_BYTES = ctypes.sizeof(_lib.RankResult)
MAX_RELATIONS = 257             # per_relation / result_at / predictions_at: relations 1 .. 256 (one 8-bit digit)
_RESULT_DTYPE = np.dtype([(name, np.int64 if ctype is ctypes.c_int64 else np.float64 if ctype is ctypes.c_double
                           else np.float32) for name, ctype in _lib.RankResult._fields_])


class RelationEvaluator:
    """Accumulates the candidates of any number of batches (``add``), ranks them once, lazily, and evaluates the ranking
    (``result``, ``curve``) or lists its head (``predictions``).  Candidate ids, and so the order of equal scores,
    follow the order of ``add`` calls and of the documents inside each batch.

    With ``doc_sizes`` (entity counts of every document of the evaluated set, in global order) ids are global instead:
    document g's candidates start at sum over g' < g of (n_g'^2 - n_g')(relations - 1), ``add`` takes the global
    indices of its batch's documents, and they must increase strictly across all ``add`` calls.  Evaluators of
    disjoint document sets of one ``doc_sizes`` combine with ``merged`` or ``all_gather`` into the evaluator of their
    union, bit for bit."""

    def __init__(self, relations: int = 97, device="cuda", doc_sizes: Optional[Sequence[int]] = None):
        self.relations = int(relations)
        if self.relations < 2:
            raise _lib.GcgcnError("RelationEvaluator: relations must be >= 2 (relation 0 is not a candidate)")
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.GcgcnError("RelationEvaluator runs on CUDA only (no CPU fallback)")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        _lib.load()
        self._doc_sizes = None          # global mode: entity count of every document of the set
        self._doc_first = None          # global mode: first candidate id of every document, [G + 1]
        if doc_sizes is not None:
            n = np.asarray(doc_sizes, dtype=np.int64).reshape(-1)
            if (n < 0).any():
                raise _lib.GcgcnError("RelationEvaluator: doc_sizes must be >= 0")
            first = np.zeros(n.size + 1, dtype=np.int64)
            np.cumsum((n * n - n) * (self.relations - 1), out=first[1:])
            if first[-1] >= MAX_CANDIDATES:
                raise _lib.GcgcnError(f"RelationEvaluator: doc_sizes hold {int(first[-1])} candidates, one evaluated "
                                      "set holds fewer than 2^30")
            self._doc_sizes, self._doc_first = n, first
        self.count = 0
        self._chunks = []               # (score f32, payload) of every add() in order
        self._doc_n = []                # entity count of every document, add() order
        self._docs = []                 # global mode: global index of every document added, ascending
        self._labeled = True
        self._has_intrain = False
        self._merged = False            # the result of merged() / all_gather(): ranked, holds no scores
        self._counters = torch.zeros(2, dtype=torch.int64, device=self.device)   # correct candidates, NaN scores
        self._host_counters = None
        self._ranked = None             # (sorted_key, sorted_payload, ws) while no add() follows
        self._by_relation = None        # the ranking partitioned by relation (per_relation), while no add() follows

    # ---------------------------------------------------------------------------------------------------------------
    def add(self, logits: torch.Tensor, labels: Optional[torch.Tensor], batch: RaggedBatch,
            intrain: Optional[torch.Tensor] = None, doc_index: Optional[Sequence[int]] = None) -> None:
        """Score the candidates of one batch.  logits, labels (multi-hot; > 0.5 is a fact) and intrain (non-zero = the
        fact was seen in training) are ``[batch.total_pairs, relations]``; labels None for an unlabeled set.
        ``doc_index`` (with ``doc_sizes`` only, and then required): the global index of each document of the batch."""
        if self._merged:
            raise _lib.GcgcnError("RelationEvaluator.add: a merged evaluator is final")
        doc_first = self._global_doc_first(batch, doc_index)
        shape = (batch.total_pairs, self.relations)
        logits = _cuda(logits.detach(), "logits")
        if tuple(logits.shape) != shape:
            raise _lib.GcgcnError(f"add: logits must be {list(shape)}, got {list(logits.shape)}")
        if labels is not None:
            labels = _cuda(labels.detach(), "labels")
            if tuple(labels.shape) != shape:
                raise _lib.GcgcnError(f"add: labels must be {list(shape)}, got {list(labels.shape)}")
        if intrain is not None:
            intrain = _cuda(intrain.detach(), "intrain", dtype=None)
            if tuple(intrain.shape) != shape:
                raise _lib.GcgcnError(f"add: intrain must be {list(shape)}, got {list(intrain.shape)}")
            if intrain.dtype == torch.bool:
                intrain = intrain.view(torch.uint8)
            elif intrain.dtype != torch.uint8:
                intrain = (intrain != 0).view(torch.uint8)
        for t in (labels, intrain):
            if t is not None and t.device != logits.device:
                raise _lib.GcgcnError("add: logits, labels and intrain must be on one device")
        if logits.device != self.device or batch.device != self.device:
            raise _lib.GcgcnError(f"add: tensors on {logits.device}, batch on {batch.device}, evaluator on {self.device}")
        n = batch.sizes.astype(np.int64)
        count = int(((n * n - n).sum())) * (self.relations - 1)
        score = torch.empty(count, dtype=torch.float32, device=self.device)
        payload = torch.empty(count, dtype=torch.int32, device=self.device)
        if doc_first is None:
            _lib.call("gcgcn_rank_candidates", batch.ref, _p(logits), self.relations, _p(labels), _p(intrain),
                      self.count, _p(score), _p(payload), _p(self._counters), _stream(self.device))
        else:
            _lib.call("gcgcn_rank_candidates_at", batch.ref, _p(logits), self.relations, _p(labels), _p(intrain),
                      _p(doc_first), _p(score), _p(payload), _p(self._counters), _stream(self.device))
            self._docs.extend(int(g) for g in doc_index)
        self._chunks.append((score, payload))
        self._doc_n.extend(int(v) for v in n)
        self.count += count
        self._labeled &= labels is not None
        self._has_intrain |= intrain is not None
        self._host_counters = None
        self._ranked = None
        self._by_relation = None

    def _global_doc_first(self, batch: RaggedBatch, doc_index) -> Optional[torch.Tensor]:
        """Check doc_index against doc_sizes; the batch documents' first global ids on the device (None: local ids)."""
        if self._doc_sizes is None:
            if doc_index is not None:
                raise _lib.GcgcnError("add: doc_index needs an evaluator built with doc_sizes")
            return None
        if doc_index is None:
            raise _lib.GcgcnError("add: an evaluator built with doc_sizes needs doc_index")
        idx = np.asarray(doc_index, dtype=np.int64).reshape(-1)
        if idx.size != batch.num_docs:
            raise _lib.GcgcnError(f"add: doc_index has {idx.size} entries, the batch {batch.num_docs} documents")
        if idx.size == 0:
            return torch.zeros(0, dtype=torch.int64, device=self.device)
        if idx.min() < 0 or idx.max() >= self._doc_sizes.size:
            raise _lib.GcgcnError(f"add: doc_index outside [0, {self._doc_sizes.size})")
        prev = self._docs[-1] if self._docs else -1
        if idx[0] <= prev or (np.diff(idx) <= 0).any():
            raise _lib.GcgcnError("add: doc_index must increase strictly across all add() calls")
        if not np.array_equal(self._doc_sizes[idx], np.asarray(batch.sizes, dtype=np.int64)):
            raise _lib.GcgcnError("add: the batch's entity counts differ from doc_sizes[doc_index]")
        return torch.from_numpy(self._doc_first[idx]).to(self.device)

    def rank(self) -> None:
        """Sort every candidate added so far (``result`` and ``predictions`` do this when they need it)."""
        if self._ranked is not None:
            return
        if self.count == 0:
            raise _lib.GcgcnError("RelationEvaluator: no candidates (every document has fewer than 2 entities)")
        score = self.scores
        payload = self._chunks[0][1]
        lib = _lib.load()
        ws = torch.empty(int(lib.gcgcn_rank_ws_bytes(self.count)), dtype=torch.uint8, device=self.device)
        key = torch.empty(self.count, dtype=torch.int32, device=self.device)
        pay = torch.empty(self.count, dtype=torch.int32, device=self.device)
        _lib.call("gcgcn_rank_sort", _p(score), _p(payload), self.count, _p(key), _p(pay), _p(ws), ws.numel(),
                  _stream(self.device))
        self._ranked = (key, pay, ws)

    @property
    def scores(self) -> torch.Tensor:
        """float32 score of every candidate added so far, in insertion order."""
        if self._merged:
            raise _lib.GcgcnError("RelationEvaluator.scores: a merged evaluator holds its ranking only")
        if len(self._chunks) > 1:
            self._chunks = [(torch.cat([c[0] for c in self._chunks]), torch.cat([c[1] for c in self._chunks]))]
        return self._chunks[0][0] if self._chunks else torch.zeros(0, device=self.device)

    @property
    def ranked(self):
        """(sorted_key, sorted_payload) int32 views of the ranking: key = ~bits(score), payload = id << 2 |
        intrain << 1 | correct."""
        self.rank()
        return self._ranked[0], self._ranked[1]

    def _counts(self):
        if self._host_counters is None:
            self._host_counters = [int(v) for v in self._counters.cpu()]
        return self._host_counters

    def _total_recall(self, total_recall: Optional[int]) -> int:
        self.rank()
        positives, nans = self._counts()
        if nans:
            raise _lib.GcgcnError(f"RelationEvaluator: {nans} NaN scores (NaN logits)")
        return positives if total_recall is None else int(total_recall)

    def _curve(self, input_theta: float, total_recall: Optional[int]) -> _lib.RankResult:
        T = self._total_recall(total_recall)
        key, pay, ws = self._ranked
        out = torch.empty(RESULT_BYTES, dtype=torch.uint8, device=self.device)
        _lib.call("gcgcn_rank_curve", _p(key), _p(pay), self.count, T, int(self._has_intrain), float(input_theta),
                  _p(out), _p(ws), ws.numel(), _stream(self.device))
        return _lib.RankResult.from_buffer_copy(out.cpu().numpy().tobytes())

    def result(self, input_theta: float = -1.0, total_recall: Optional[int] = None) -> dict:
        """Best F1 over the ranking, its threshold ``theta`` and position, the AUC, and F1 / precision / recall at the
        position ``w`` that ``input_theta`` selects (-1: the best-F1 position; otherwise the last score above it).
        ``total_recall`` (default: the number of correct candidates; 0 counts as 1) is the recall denominator; the
        reference counts the gold facts of the records.  Ign fields are None unless some ``add`` passed intrain."""
        if not self._labeled:
            raise _lib.GcgcnError("RelationEvaluator.result: a batch was added without labels")
        r = self._curve(input_theta, total_recall)
        ign = self._has_intrain
        return {"count": int(r.count), "total_recall": int(r.total_recall), "f1": float(r.f1), "theta": float(r.theta),
                "best_pos": int(r.best_pos), "auc": float(r.auc), "w": int(r.w), "f1_at_w": float(r.f1_at_w),
                "precision_at_w": float(r.precision_at_w), "recall_at_w": float(r.recall_at_w),
                "ign_f1": float(r.ign_f1) if ign else None, "ign_auc": float(r.ign_auc) if ign else None,
                "ign_f1_at_w": float(r.ign_f1_at_w) if ign else None}

    def curve(self, total_recall: Optional[int] = None) -> dict:
        """The precision/recall curve at every ranked position (the reference's ``pr_x``, ``pr_y`` and, with intrain,
        the Ign ``pr_y``): float32 device tensors ``x``, ``y`` and ``y_ign`` (None unless some ``add`` passed
        intrain) of length ``count``.  ``total_recall`` as in ``result``."""
        if not self._labeled:
            raise _lib.GcgcnError("RelationEvaluator.curve: a batch was added without labels")
        T = self._total_recall(total_recall)
        _, pay, ws = self._ranked
        x = torch.empty(self.count, dtype=torch.float32, device=self.device)
        y = torch.empty_like(x)
        y_ign = torch.empty_like(x) if self._has_intrain else None
        _lib.call("gcgcn_rank_curve_points", _p(pay), self.count, T, int(self._has_intrain), _p(x), _p(y), _p(y_ign),
                  _p(ws), ws.numel(), _stream(self.device))
        return {"x": x, "y": y, "y_ign": y_ign}

    def predictions(self, input_theta: float = -1.0, total_recall: Optional[int] = None) -> dict:
        """The first w + 1 ranked candidates (the list the reference dumps, C:551-554) as int32 tensors ``doc`` (index of
        the document in add() order; its global index with ``doc_sizes``), ``row``, ``col``, ``relation`` and float32
        ``score``, on the device."""
        if input_theta == -1.0 and not self._labeled:
            raise _lib.GcgcnError("RelationEvaluator.predictions: the best-F1 threshold needs labels; pass input_theta")
        r = self._curve(input_theta, total_recall)
        key, pay, _ = self._ranked
        return self._decode(key, pay, int(r.w) + 1, self.count)

    def _decode(self, key, pay, rows, count) -> dict:
        """The first ``rows`` candidates of the run (key, pay) of length ``count`` as ``predictions`` lists them."""
        if self._doc_sizes is None:
            n = np.asarray(self._doc_n, dtype=np.int64)
            off = np.zeros(n.size + 1, dtype=np.int64)
            np.cumsum((n * n - n) * (self.relations - 1), out=off[1:])
        else:
            n, off = self._doc_sizes, self._doc_first
        doc_off = torch.from_numpy(off).to(self.device)
        doc_n = torch.from_numpy(n.astype(np.int32)).to(self.device)
        out = {k: torch.empty(rows, dtype=torch.int32, device=self.device) for k in ("doc", "row", "col", "relation")}
        out["score"] = torch.empty(rows, dtype=torch.float32, device=self.device)
        _lib.call("gcgcn_rank_decode", _p(key), _p(pay), rows, count, _p(doc_off), _p(doc_n), int(n.size), self.relations,
                  _p(out["doc"]), _p(out["row"]), _p(out["col"]), _p(out["relation"]), _p(out["score"]),
                  _stream(self.device))
        return out

    # ------------------------------------------------------------------------------------------------- per relation
    def _per_relation_values(self, values, dtype, what, scalar_ok=False) -> np.ndarray:
        """``values`` as one host value per relation r >= 1 (a scalar stands for all of them if ``scalar_ok``)."""
        v = np.asarray(values, dtype=dtype)
        if v.ndim == 0 and scalar_ok:
            v = np.full(self.relations - 1, v, dtype=dtype)
        if v.shape != (self.relations - 1,):
            raise _lib.GcgcnError(f"RelationEvaluator: {what} must hold relations - 1 = {self.relations - 1} values, "
                                  f"got shape {list(v.shape)}")
        return v

    def _relation_ws(self) -> torch.Tensor:
        """The ranking's workspace when it is large enough for the per-relation entry points, else a new one."""
        need = int(_lib.load().gcgcn_rank_relations_ws_bytes(self.count, self.relations))
        ws = self._ranked[2]
        return ws if ws.numel() >= need else torch.empty(need, dtype=torch.uint8, device=self.device)

    def per_relation(self, input_theta=-1.0, total_recall: Optional[Sequence[int]] = None) -> dict:
        """``result`` for every relation r >= 1 on its own: relation r's candidates, in their order in the ranking (the
        stable ranking of those candidates alone).  Host NumPy arrays of length relations - 1, entry r - 1 for
        relation r: the fields of ``result`` (Ign fields None unless some ``add`` passed intrain) and ``relation``.
        ``input_theta``: a scalar or one value per relation (-1: the relation's best-F1 position; otherwise its last
        score above the value).  ``total_recall``: None (each relation's correct candidates) or one value per
        relation.  At most 256 relations r >= 1."""
        if not self._labeled:
            raise _lib.GcgcnError("RelationEvaluator.per_relation: a batch was added without labels")
        self._total_recall(None)                            # ranks; raises on NaN scores
        theta = self._per_relation_values(input_theta, np.float64, "input_theta", scalar_ok=True)
        tr = None if total_recall is None else self._per_relation_values(total_recall, np.int64, "total_recall")
        key, pay, _ = self._ranked
        ws = self._relation_ws()
        st = _stream(self.device)
        if self._by_relation is None:
            rel_key, rel_pay = torch.empty_like(key), torch.empty_like(pay)
            _lib.call("gcgcn_rank_by_relation", _p(key), _p(pay), self.count, self.relations, _p(rel_key), _p(rel_pay),
                      _p(ws), ws.numel(), st)
            self._by_relation = (rel_key, rel_pay)
        rel_key, rel_pay = self._by_relation
        theta_d = torch.from_numpy(theta).to(self.device)
        tr_d = None if tr is None else torch.from_numpy(tr).to(self.device)
        out = torch.empty((self.relations - 1) * RESULT_BYTES, dtype=torch.uint8, device=self.device)
        _lib.call("gcgcn_rank_curve_relations", _p(rel_key), _p(rel_pay), self.count, self.relations, _p(tr_d),
                  int(self._has_intrain), _p(theta_d), _p(out), _p(ws), ws.numel(), st)
        r = out.cpu().numpy().view(_RESULT_DTYPE)
        ign = self._has_intrain
        res = {k: r[k].copy() for k in ("count", "total_recall", "f1", "theta", "best_pos", "auc", "w", "f1_at_w",
                                         "precision_at_w", "recall_at_w")}
        for k in ("ign_f1", "ign_auc", "ign_f1_at_w"):
            res[k] = r[k].copy() if ign else None
        res["relation"] = np.arange(1, self.relations, dtype=np.int64)
        return res

    def _select(self, theta):
        """The candidates above theta[relation - 1], in ranked order: (key, payload) runs of length m, and (m, c, t)."""
        self._total_recall(None)                            # ranks; raises on NaN scores
        theta = self._per_relation_values(theta, np.float32, "theta")
        key, pay, _ = self._ranked
        ws = self._relation_ws()
        out_key, out_pay = torch.empty_like(key), torch.empty_like(pay)
        counts = torch.empty(3, dtype=torch.int64, device=self.device)
        _lib.call("gcgcn_rank_select", _p(key), _p(pay), self.count, self.relations,
                  _p(torch.from_numpy(theta).to(self.device)), _p(out_key), _p(out_pay), _p(counts), _p(ws), ws.numel(),
                  _stream(self.device))
        m, c, t = (int(v) for v in counts.cpu())
        return out_key, out_pay, m, c, t

    def result_at(self, theta, total_recall: Optional[int] = None) -> dict:
        """Precision, recall, F1 and Ign F1 of the candidates whose score is above ``theta[relation - 1]`` (one float32
        threshold per relation r >= 1, e.g. ``per_relation()["theta"]`` of a dev set): ``count_selected`` (m),
        ``correct`` (c), precision = c / m (0 when m = 0), recall = c / total_recall (default: the correct candidates;
        < 1 counts as 1), f1 and ``ign_f1`` (None unless some ``add`` passed intrain), rounded as ``result``."""
        if not self._labeled:
            raise _lib.GcgcnError("RelationEvaluator.result_at: a batch was added without labels")
        T = max(self._total_recall(total_recall), 1)
        _, _, m, c, t = self._select(theta)
        f32 = np.float32

        def f1(x, y):                                       # float32, every operation rounded (rank.cu, curve_f1)
            return f32(f32(f32(2) * x) * y) / f32(f32(x + y) + f32(1e-20))

        precision = f32(c / m) if m else f32(0)
        recall = f32(c / T)
        out = {"count_selected": m, "correct": c, "precision": float(precision), "recall": float(recall),
               "f1": float(f1(recall, precision)), "ign_f1": None}
        if self._has_intrain:
            ign = f32(0) if t == c else f32((c - t) / (m - t))
            out["ign_f1"] = float(f1(recall, ign))
        return out

    def predictions_at(self, theta) -> dict:
        """``predictions`` for the candidates whose score is above ``theta[relation - 1]`` (one float32 threshold per
        relation r >= 1), in ranked order.  Needs no labels: dev-set thresholds applied to a test set."""
        key, pay, m, _, _ = self._select(theta)
        return self._decode(key, pay, m, m)

    # --------------------------------------------------------------------------------------------------- sharded sets
    @classmethod
    def merged(cls, parts: Sequence["RelationEvaluator"]) -> "RelationEvaluator":
        """The evaluator of the union of ``parts``: evaluators on one device with the same ``relations`` and
        ``doc_sizes`` and disjoint documents.  Each part is ranked, then the sorted runs merge pairwise in a fixed
        tree order (csrc/rank.cu, ``gcgcn_rank_merge``).  ``result``, ``curve``, ``predictions`` and ``ranked`` of
        the result are bit-identical to those of one evaluator fed the union in ascending global order.  The result
        is final: ``add`` and ``scores`` raise."""
        parts = list(parts)
        if not parts:
            raise _lib.GcgcnError("RelationEvaluator.merged: no parts")
        head = parts[0]
        for p in parts:
            if p._doc_sizes is None:
                raise _lib.GcgcnError("RelationEvaluator.merged: every part needs doc_sizes (global candidate ids)")
            if p.relations != head.relations:
                raise _lib.GcgcnError(f"RelationEvaluator.merged: relations {p.relations} != {head.relations}")
            if p.device != head.device:
                raise _lib.GcgcnError(f"RelationEvaluator.merged: parts on {p.device} and {head.device}")
            if not np.array_equal(p._doc_sizes, head._doc_sizes):
                raise _lib.GcgcnError("RelationEvaluator.merged: the parts' doc_sizes differ")
        total = sum(p.count for p in parts)
        if total >= MAX_CANDIDATES:
            raise _lib.GcgcnError(f"RelationEvaluator.merged: {total} candidates, one evaluated set holds fewer than 2^30")
        runs = [p.ranked for p in parts if p.count > 0]
        counters = torch.stack([p._counters for p in parts]).sum(0)
        return cls._from_runs(head, runs, counters, [p._docs for p in parts], all(p._labeled for p in parts),
                              any(p._has_intrain for p in parts))

    def all_gather(self, group=None) -> "RelationEvaluator":
        """The evaluator of the documents of every rank of ``group`` (default: the world), on every rank.  Each rank
        ranks its own candidates; the ranks exchange their sorted runs and a few counts with all_gather_into_tensor
        (on the device under NCCL, through the host under other backends), and every rank merges the runs in rank
        order.  So every rank holds the same bits and reaches the same threshold and checkpoint decisions.  Without a
        process group, or with one rank, this is ``merged([self])``.  Errors are raised on every rank alike."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
            return type(self).merged([self])
        world = dist.get_world_size(group)
        comm = self.device if dist.get_backend(group) == "nccl" else torch.device("cpu")
        if self.count > 0:
            self.rank()

        def gather(t):                           # 1-D t -> [world, t.numel()], rank r's t in row r
            out = torch.empty(world * t.numel(), dtype=t.dtype, device=comm)
            dist.all_gather_into_tensor(out, t.to(comm).contiguous(), group=group)
            return out.view(world, -1)

        # metadata first, so that every rank sees the same inconsistency and raises the same error
        sizes = self._doc_sizes
        digest = 0 if sizes is None else int.from_bytes(hashlib.blake2b(sizes.tobytes(), digest_size=7).digest(), "little")
        meta = torch.tensor([self.count, int(sizes is not None), 0 if sizes is None else sizes.size, digest,
                             self.relations, int(self._labeled), int(self._has_intrain), len(self._docs)],
                            dtype=torch.int64)
        m = gather(torch.cat([meta.to(self.device), self._counters])).cpu()
        if not bool((m[:, 1] == 1).all()):
            raise _lib.GcgcnError("RelationEvaluator.all_gather: every rank's evaluator needs doc_sizes")
        if not bool((m[:, 4] == m[0, 4]).all()):
            raise _lib.GcgcnError("RelationEvaluator.all_gather: the ranks' relations differ")
        if not bool((m[:, 2:4] == m[0, 2:4]).all()):
            raise _lib.GcgcnError("RelationEvaluator.all_gather: the ranks' doc_sizes differ")
        counts = [int(c) for c in m[:, 0]]
        if sum(counts) >= MAX_CANDIDATES:
            raise _lib.GcgcnError(f"RelationEvaluator.all_gather: {sum(counts)} candidates, one evaluated set holds "
                                  "fewer than 2^30")
        ndocs = [int(d) for d in m[:, 7]]
        docs = torch.full((max(max(ndocs), 1),), -1, dtype=torch.int64)
        docs[:len(self._docs)] = torch.tensor(self._docs, dtype=torch.int64)
        d = gather(docs).cpu().numpy()
        doc_lists = [d[r, :ndocs[r]].tolist() for r in range(world)]
        # the runs, padded to the longest (a multiple of 4: every rank's payload run starts 16-byte aligned)
        maxc = (max(counts) + 3) // 4 * 4
        runs = []
        if maxc > 0:
            send = torch.zeros(2 * maxc, dtype=torch.int32, device=self.device)
            if self.count > 0:
                key, pay = self.ranked
                send[:self.count] = key
                send[maxc:maxc + self.count] = pay
            recv = gather(send).to(self.device)
            runs = [(recv[r, :c], recv[r, maxc:maxc + c]) for r, c in enumerate(counts) if c > 0]
        counters = m[:, 8:10].sum(0).to(self.device)
        return type(self)._from_runs(self, runs, counters, doc_lists, bool((m[:, 5] == 1).all()),
                                     bool((m[:, 6] == 1).any()))

    @classmethod
    def _from_runs(cls, like, runs, counters, doc_lists, labeled, has_intrain) -> "RelationEvaluator":
        """The merged evaluator over sorted (key, payload) runs of disjoint documents of ``like``'s doc_sizes."""
        docs = np.concatenate([np.asarray(d, dtype=np.int64) for d in doc_lists])
        if np.unique(docs).size != docs.size:
            raise _lib.GcgcnError("RelationEvaluator: the parts share documents")
        if not runs:
            raise _lib.GcgcnError("RelationEvaluator: no candidates (every document has fewer than 2 entities)")
        out = cls(like.relations, like.device, doc_sizes=like._doc_sizes)
        dev, st = out.device, _stream(out.device)
        lib = _lib.load()
        total = sum(int(k.numel()) for k, _ in runs)
        ws = torch.empty(int(lib.gcgcn_rank_merge_ws_bytes(total)), dtype=torch.uint8, device=dev)
        while len(runs) > 1:                     # pairwise rounds: (0, 1), (2, 3), ...; an odd last run moves up
            nxt = []
            for (ka, pa), (kb, pb) in zip(runs[0::2], runs[1::2]):
                n = ka.numel() + kb.numel()
                key = torch.empty(n, dtype=torch.int32, device=dev)
                pay = torch.empty(n, dtype=torch.int32, device=dev)
                _lib.call("gcgcn_rank_merge", _p(ka), _p(pa), ka.numel(), _p(kb), _p(pb), kb.numel(), _p(key), _p(pay),
                          _p(ws), ws.numel(), st)
                nxt.append((key, pay))
            if len(runs) % 2:
                nxt.append(runs[-1])
            runs = nxt
        key, pay = runs[0]
        out.count = total
        out._ranked = (key, pay, torch.empty(int(lib.gcgcn_rank_ws_bytes(total)), dtype=torch.uint8, device=dev))
        out._counters = counters
        out._docs = np.sort(docs).tolist()
        out._labeled = labeled
        out._has_intrain = has_intrain
        out._merged = True
        return out
