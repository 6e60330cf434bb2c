"""Relation classifier and loss of GCGCN on the GPU (SURVEY.md section 8f row 2, second half).

``logits = bili_layer_01(h, t) + classification_layer_01(cat[h, t])`` (/root/reference/models/GCGCN_glove.py:275-276,
356-358) over every pair of a ragged batch, and the trainer's loss (config/Config.py:355-364).  ``h``, ``t`` are
``entity_feature_h`` / ``entity_feature_t`` ``[total_pairs, 128]`` (``modules.pair_dense``).  The bilinear form is the
one dense n^2-scale contraction of the model (2 * 128 * 128 * 97 flop per pair): it runs on this package's tcgen05 GEMM
with ``W'`` the ``[R, 128, 128]`` weight viewed as ``[128, R*128]``, in fp32 (3xTF32) or, with
``relation_logits(..., dtype=torch.bfloat16)``, on bf16-rounded operands (one ``kind::f16`` tensor-core pass, fp32
accumulation; parameters, inputs and gradients stay fp32).  ``h W'`` is contracted with ``t`` in the GEMM's epilogue and
never stored.  No CPU path.
"""
from __future__ import annotations

import torch
from torch import nn
from torch.autograd import Function

from . import _lib
from .batch import RaggedBatch
from .functional import D, LinearFn, _cuda, _p, _stream, workspace

FUSED_CHUNK_PAIRS = 1 << 18  # pairs per backward call (workspace: 1 KB of pre-split h + 1.6 KB of split-K partials per pair)
DTYPES = {torch.float32: _lib.F32, torch.bfloat16: _lib.BF16}


def _wmat(W: torch.Tensor) -> torch.Tensor:
    """[R, 128(a), 128(b)] -> [128(a), R*128 (r, b)]."""
    R = W.shape[0]
    return W.permute(1, 0, 2).reshape(D, R * D).contiguous()


class BilinearFn(Function):
    """out[p, r] = sum_{a,b} h[p,a] W[r,a,b] t[p,b] + bias[r]   (torch.nn.Bilinear, G:275, 358), with the operand type
    ``dtype`` (torch.float32 or torch.bfloat16; include/gcgcn_b200.h, gcgcn_bilinear_fwd, gives both numerics).  h, t, W,
    bias and every gradient are fp32.  The forward is one call; the backward makes host calls of at most
    FUSED_CHUNK_PAIRS pairs that accumulate dW' through beta = 1."""

    @staticmethod
    def forward(ctx, h, t, W, bias, dtype):
        h, t, W, bias = _cuda(h, "h"), _cuda(t, "t"), _cuda(W, "weight"), _cuda(bias, "bias")
        P, R, dev, code = h.shape[0], W.shape[0], h.device, DTYPES[dtype]
        if W.shape[1:] != (D, D) or h.shape[1] != D or t.shape != h.shape:
            raise _lib.GcgcnError(f"bilinear: expected h, t [P, {D}] and weight [R, {D}, {D}]")
        Wm = _wmat(W)
        out = torch.empty(P, R, device=dev)
        if P > 0:
            # one tensor-core pass: the accumulator tiles of h W' are contracted with t in the GEMM's epilogue
            ws = workspace(dev, int(_lib.load().gcgcn_bilinear_ws_bytes(P, R, code)))
            _lib.call("gcgcn_bilinear_fwd", _p(h), _p(t), _p(Wm), _p(bias), P, R, code, 0, _p(out), R, ws.data_ptr(),
                      ws.numel(), _stream(dev))
        ctx.save_for_backward(h, t, Wm)
        ctx.R, ctx.code = R, code
        return out

    @staticmethod
    def backward(ctx, dout):
        h, t, Wm = ctx.saved_tensors
        R, code, dev, P = ctx.R, ctx.code, h.device, h.shape[0]
        dout = _cuda(dout, "dout")
        dh, dt = torch.empty_like(h), torch.empty_like(t)
        dWm = torch.zeros_like(Wm)
        # three tensor-core passes per call, nothing of size [pairs, R*128] is ever stored: dt and dh through the
        # row-accumulate epilogue, dW' with its Khatri-Rao operand generated in the GEMM's producers
        Wm2 = Wm.view(D, R, D).permute(2, 1, 0).reshape(D, R * D).contiguous()       # W viewed as [b][(r, a)]
        lib = _lib.load()
        for p0 in range(0, P, FUSED_CHUNK_PAIRS):
            p1 = min(P, p0 + FUSED_CHUNK_PAIRS)
            rows = p1 - p0
            ws = workspace(dev, int(lib.gcgcn_bilinear_bwd_ws_bytes(rows, R, code)))
            _lib.call("gcgcn_bilinear_bwd", _p(h[p0:p1]), _p(t[p0:p1]), _p(Wm), _p(Wm2), _p(dout[p0:p1]), rows, R, code,
                      1.0, _p(dh[p0:p1]), _p(dt[p0:p1]), _p(dWm), ws.data_ptr(), ws.numel(), _stream(dev))
        dbias = torch.empty(R, device=dev)
        ws = workspace(dev, 8 << 20)
        _lib.call("gcgcn_colsum", _p(dout), P, R, R, _p(dbias), ws.data_ptr(), ws.numel(), _stream(dev))
        dW = dWm.view(D, R, D).permute(1, 0, 2).contiguous()
        return dh, dt, dW, dbias, None


class PairBceFn(Function):
    """Per-document loss of config/Config.py:355-364 from logits and multi-hot labels [total_pairs, R]."""

    @staticmethod
    def forward(ctx, logits, labels, batch: RaggedBatch):
        logits, labels = _cuda(logits, "logits"), _cuda(labels, "labels")
        if logits.shape != labels.shape or logits.shape[0] != batch.total_pairs:
            raise _lib.GcgcnError("pair_bce: logits and labels must both be [total_pairs, R]")
        loss = torch.empty(batch.num_docs, device=logits.device)
        _lib.call("gcgcn_pair_bce_fwd", batch.ref, _p(logits), _p(labels), logits.shape[1], _p(loss), _stream(logits.device))
        ctx.save_for_backward(logits, labels)
        ctx.batch = batch
        return loss

    @staticmethod
    def backward(ctx, dloss):
        logits, labels = ctx.saved_tensors
        dloss = _cuda(dloss, "dloss")
        dz = torch.empty_like(logits)
        _lib.call("gcgcn_pair_bce_bwd", ctx.batch.ref, _p(logits), _p(labels), logits.shape[1], _p(dloss), _p(dz),
                  _stream(logits.device))
        return dz, None, None


class DocBiasFn(Function):
    """z + v[doc of pair]: the BERT variant's ``cls_feature`` (B:346-347) broadcast over each document's pair grid."""

    @staticmethod
    def forward(ctx, z, v, batch: RaggedBatch):
        z, v = _cuda(z, "logits"), _cuda(v, "cls_feature")
        if v.shape != (batch.num_docs, z.shape[1]):
            raise _lib.GcgcnError(f"cls_feature must be [{batch.num_docs}, {z.shape[1]}], got {tuple(v.shape)}")
        out = z.clone()
        _lib.call("gcgcn_doc_bias_fwd", batch.ref, _p(v), z.shape[1], _p(out), _stream(z.device))
        ctx.batch = batch
        return out

    @staticmethod
    def backward(ctx, dz):
        dz = _cuda(dz, "dlogits")
        dv = torch.empty(ctx.batch.num_docs, dz.shape[1], device=dz.device)
        _lib.call("gcgcn_doc_bias_bwd", ctx.batch.ref, _p(dz), dz.shape[1], _p(dv), _stream(dz.device))
        return dz, dv, None


def relation_logits(h: torch.Tensor, t: torch.Tensor, bili: nn.Bilinear, cls: nn.Linear, cls_feature=None,
                    batch: RaggedBatch = None, dtype=torch.float32) -> torch.Tensor:
    """G:356-358: ``bili(h, t) + cls(cat[h, t])`` without forming the concatenation (the linear layer is split by
    input columns into its h and t halves).  ``cls_feature`` [num_docs, R] (with ``batch``) adds the BERT variant's
    per-document term, B:346-347.  ``dtype`` is the operand type of the bilinear form: torch.float32 (3xTF32, fp32
    parity) or torch.bfloat16; the linear layer, the logits and every gradient are fp32 either way."""
    if dtype not in DTYPES:
        raise _lib.GcgcnError(f"relation_logits: dtype must be torch.float32 or torch.bfloat16, got {dtype}")
    w = cls.weight
    lin = LinearFn.apply(h, w[:, :D], cls.bias) + LinearFn.apply(t, w[:, D:], None)
    z = BilinearFn.apply(h, t, bili.weight, bili.bias, dtype) + lin
    return z if cls_feature is None else DocBiasFn.apply(z, cls_feature, batch)


def pair_bce_loss(logits: torch.Tensor, labels: torch.Tensor, batch: RaggedBatch) -> torch.Tensor:
    """[num_docs] losses exactly as the reference trainer forms them per document (C:355-364)."""
    return PairBceFn.apply(logits, labels, batch)
