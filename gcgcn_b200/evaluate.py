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
"""
from __future__ import annotations

import ctypes
from typing import Optional

import numpy as np
import torch

from . import _lib
from .batch import RaggedBatch
from .functional import _cuda, _p, _stream

SORT_TILE = 4096                # GCGCN_RANK_TILE of include/gcgcn_b200.h
MAX_CANDIDATES = 1 << 30        # one evaluator holds fewer (the payload packs id << 2 | flags)
RESULT_BYTES = ctypes.sizeof(_lib.RankResult)


class RelationEvaluator:
    """Accumulates the candidates of any number of batches (``add``), ranks them once, lazily, and evaluates the ranking
    (``result``) or lists its head (``predictions``).  Candidate ids, and so the order of equal scores, follow the
    order of ``add`` calls and of the documents inside each batch."""

    def __init__(self, relations: int = 97, device="cuda"):
        self.relations = int(relations)
        if self.relations < 2:
            raise _lib.GcgcnError("RelationEvaluator: relations must be >= 2 (relation 0 is not a candidate)")
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.GcgcnError("RelationEvaluator runs on CUDA only (no CPU fallback)")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        _lib.load()
        self.count = 0
        self._chunks = []               # (score f32, payload) of every add() in order
        self._doc_n = []                # entity count of every document, add() order
        self._labeled = True
        self._has_intrain = False
        self._counters = torch.zeros(2, dtype=torch.int64, device=self.device)   # correct candidates, NaN scores
        self._host_counters = None
        self._ranked = None             # (sorted_key, sorted_payload, ws) while no add() follows

    # ---------------------------------------------------------------------------------------------------------------
    def add(self, logits: torch.Tensor, labels: Optional[torch.Tensor], batch: RaggedBatch,
            intrain: Optional[torch.Tensor] = None) -> None:
        """Score the candidates of one batch.  logits, labels (multi-hot; > 0.5 is a fact) and intrain (non-zero = the
        fact was seen in training) are ``[batch.total_pairs, relations]``; labels None for an unlabeled set."""
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
        _lib.call("gcgcn_rank_candidates", batch.ref, _p(logits), self.relations, _p(labels), _p(intrain), self.count,
                  _p(score), _p(payload), _p(self._counters), _stream(self.device))
        self._chunks.append((score, payload))
        self._doc_n.extend(int(v) for v in n)
        self.count += count
        self._labeled &= labels is not None
        self._has_intrain |= intrain is not None
        self._host_counters = None
        self._ranked = None

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
        """float32 score of every candidate added so far, in id (insertion) order."""
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

    def _curve(self, input_theta: float, total_recall: Optional[int]) -> _lib.RankResult:
        self.rank()
        positives, nans = self._counts()
        if nans:
            raise _lib.GcgcnError(f"RelationEvaluator: {nans} NaN scores (NaN logits)")
        T = positives if total_recall is None else int(total_recall)
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

    def predictions(self, input_theta: float = -1.0, total_recall: Optional[int] = None) -> dict:
        """The first w + 1 ranked candidates (the list the reference dumps, C:551-554) as int32 tensors ``doc`` (index of
        the document in add() order), ``row``, ``col``, ``relation`` and float32 ``score``, on the device."""
        if input_theta == -1.0 and not self._labeled:
            raise _lib.GcgcnError("RelationEvaluator.predictions: the best-F1 threshold needs labels; pass input_theta")
        r = self._curve(input_theta, total_recall)
        rows = int(r.w) + 1
        n = np.asarray(self._doc_n, dtype=np.int64)
        off = np.zeros(n.size + 1, dtype=np.int64)
        np.cumsum((n * n - n) * (self.relations - 1), out=off[1:])
        doc_off = torch.from_numpy(off).to(self.device)
        doc_n = torch.from_numpy(n.astype(np.int32)).to(self.device)
        out = {k: torch.empty(rows, dtype=torch.int32, device=self.device) for k in ("doc", "row", "col", "relation")}
        out["score"] = torch.empty(rows, dtype=torch.float32, device=self.device)
        key, pay, _ = self._ranked
        _lib.call("gcgcn_rank_decode", _p(key), _p(pay), rows, self.count, _p(doc_off), _p(doc_n), int(n.size), self.relations,
                  _p(out["doc"]), _p(out["row"]), _p(out["col"]), _p(out["relation"]), _p(out["score"]),
                  _stream(self.device))
        return out
