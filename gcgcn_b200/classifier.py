"""Relation classifier and loss of GCGCN on the GPU (SURVEY.md section 8f row 2, second half).

``logits = bili_layer_01(h, t) + classification_layer_01(cat[h, t])`` (/root/reference/models/GCGCN_glove.py:275-276,
356-358) over every pair of a ragged batch, and the trainer's loss (config/Config.py:355-364).  ``h``, ``t`` are
``entity_feature_h`` / ``entity_feature_t`` ``[total_pairs, 128]`` (``modules.pair_dense``).  The bilinear form is the
one dense n^2-scale contraction of the model (2 * 128 * 128 * 97 flop per pair): it runs on this package's tcgen05 GEMM
(3xTF32) as ``Y = h W'`` with ``W'`` the ``[R, 128, 128]`` weight viewed as ``[128, R*128]``, then a row-wise reduction
against ``t``; the pairs are walked in chunks so that ``Y`` (R*128 floats per pair) stays inside a fixed workspace.
``relation_logits(..., dtype=torch.bfloat16)`` runs the bilinear form on bf16-rounded operands instead (``BilinearBf16Fn``:
one ``kind::f16`` tensor-core pass, fp32 accumulation; parameters, inputs and gradients stay fp32).  No CPU path.
"""
from __future__ import annotations

import torch
from torch import nn
from torch.autograd import Function

from . import _lib
from .batch import RaggedBatch
from .functional import D, LinearFn, _cuda, _p, _stream, gemm, workspace

CHUNK_PAIRS = 8192          # 8192 pairs x 97 x 128 floats = 407 MB of Y per chunk
FUSED_BACKWARD = True       # False: the backward materialises Y / dY chunk by chunk (test hook; also the path below 8192 pairs)
FUSED_MIN_PAIRS = 8192      # the generated-operand weight-gradient GEMM needs K >= 8192
FUSED_CHUNK_PAIRS = 1 << 18  # pairs per fused backward call (workspace: 1 KB of pre-split h + 1.6 KB of split-K partials per pair)
FUSED_FORWARD = True        # False: the forward materialises Y = h W' chunk by chunk like the backward does (test hook)


def _wmat(W: torch.Tensor) -> torch.Tensor:
    """[R, 128(a), 128(b)] -> [128(a), R*128 (r, b)]."""
    R = W.shape[0]
    return W.permute(1, 0, 2).reshape(D, R * D).contiguous()


class BilinearFn(Function):
    """out[p, r] = sum_{a,b} h[p,a] W[r,a,b] t[p,b] + bias[r]   (torch.nn.Bilinear, G:275, 358)."""

    @staticmethod
    def forward(ctx, h, t, W, bias):
        h, t, W, bias = _cuda(h, "h"), _cuda(t, "t"), _cuda(W, "weight"), _cuda(bias, "bias")
        P, R, dev = h.shape[0], W.shape[0], h.device
        if W.shape[1:] != (D, D) or h.shape[1] != D or t.shape != h.shape:
            raise _lib.GcgcnError(f"bilinear: expected h, t [P, {D}] and weight [R, {D}, {D}]")
        Wm = _wmat(W)
        out = torch.empty(P, R, device=dev)
        if FUSED_FORWARD and P > 0:
            # one tensor-core pass: the accumulator tiles of h W' are contracted with t in the GEMM's epilogue
            ws = workspace(dev, int(_lib.load().gcgcn_bilinear_ws_bytes(P, R)))
            _lib.call("gcgcn_bilinear_fwd", _p(h), _p(t), _p(Wm), _p(bias), P, R, 0, _p(out), R, ws.data_ptr(), ws.numel(),
                      _stream(dev))
        else:
            for p0 in range(0, P, CHUNK_PAIRS):
                p1 = min(P, p0 + CHUNK_PAIRS)
                Y = gemm(h[p0:p1], Wm)
                _lib.call("gcgcn_bilinear_reduce_fwd", _p(Y), _p(t[p0:p1]), _p(bias), p1 - p0, R, 0, _p(out[p0:p1]), R,
                          _stream(dev))
                del Y
        ctx.save_for_backward(h, t, Wm)
        ctx.R = R
        return out

    @staticmethod
    def backward(ctx, dout):
        h, t, Wm = ctx.saved_tensors
        R, dev, P = ctx.R, h.device, h.shape[0]
        dout = _cuda(dout, "dout")
        dh, dt = torch.empty_like(h), torch.empty_like(t)
        dWm = torch.zeros_like(Wm)
        p_done = 0
        if FUSED_BACKWARD and P >= FUSED_MIN_PAIRS:
            # three tensor-core passes per chunk, nothing of size [pairs, R*128] is ever stored: dt and dh through the
            # row-accumulate epilogue, dW' with its Khatri-Rao operand generated in the GEMM's producers
            Wm2 = Wm.view(D, R, D).permute(2, 1, 0).reshape(D, R * D).contiguous()       # W viewed as [b][(r, a)]
            lib = _lib.load()
            while P - p_done >= FUSED_MIN_PAIRS:
                p1 = P if P - p_done <= FUSED_CHUNK_PAIRS + FUSED_MIN_PAIRS else p_done + FUSED_CHUNK_PAIRS
                rows = p1 - p_done
                ws = workspace(dev, int(lib.gcgcn_bilinear_bwd_ws_bytes(rows, R)))
                _lib.call("gcgcn_bilinear_bwd", _p(h[p_done:p1]), _p(t[p_done:p1]), _p(Wm), _p(Wm2), _p(dout[p_done:p1]), rows,
                          R, 1.0, _p(dh[p_done:p1]), _p(dt[p_done:p1]), _p(dWm), ws.data_ptr(), ws.numel(), _stream(dev))
                p_done = p1
        for p0 in range(p_done, P, CHUNK_PAIRS):
            p1 = min(P, p0 + CHUNK_PAIRS)
            rows = p1 - p0
            Y = gemm(h[p0:p1], Wm)                                               # recomputed, not saved
            _lib.call("gcgcn_bilinear_dt_bwd", _p(dout[p0:p1]), R, _p(Y), rows, R, _p(dt[p0:p1]), _stream(dev))
            dY = Y                                                               # same storage
            _lib.call("gcgcn_bilinear_outer_bwd", _p(dout[p0:p1]), R, _p(t[p0:p1]), rows, R, _p(dY), _stream(dev))
            gemm(dY, Wm, trans_b=True, out=dh[p0:p1])                            # dh = dY W'^T
            gemm(h[p0:p1], dY, trans_a=True, out=dWm, beta=1.0)                  # dW' += h^T dY
            del Y, dY
        dbias = torch.empty(R, device=dev)
        ws = workspace(dev, 8 << 20)
        _lib.call("gcgcn_colsum", _p(dout), P, R, R, _p(dbias), ws.data_ptr(), ws.numel(), _stream(dev))
        dW = dWm.view(D, R, D).permute(1, 0, 2).contiguous()
        return dh, dt, dW, dbias


class BilinearBf16Fn(Function):
    """The bilinear form with bf16 operands and fp32 accumulation (include/gcgcn_b200.h, gcgcn_bilinear_bf16_fwd):
    out[p, r] = sum_b (sum_a bf16(h[p,a]) bf16(W[r,a,b])) t[p,b] + bias[r].  h, t, W, bias and every gradient are fp32;
    dW[r,a,b] = sum_p bf16(h[p,a]) bf16(dout[p,r] t[p,b]).  The fused kernels take any number of pairs: the backward makes
    host calls of at most FUSED_CHUNK_PAIRS pairs that accumulate dW' through beta = 1, and has no chunked path."""

    @staticmethod
    def forward(ctx, h, t, W, bias):
        h, t, W, bias = _cuda(h, "h"), _cuda(t, "t"), _cuda(W, "weight"), _cuda(bias, "bias")
        P, R, dev = h.shape[0], W.shape[0], h.device
        if W.shape[1:] != (D, D) or h.shape[1] != D or t.shape != h.shape:
            raise _lib.GcgcnError(f"bilinear: expected h, t [P, {D}] and weight [R, {D}, {D}]")
        Wm = _wmat(W)
        out = torch.empty(P, R, device=dev)
        if P > 0:
            ws = workspace(dev, int(_lib.load().gcgcn_bilinear_bf16_ws_bytes(P, R)))
            _lib.call("gcgcn_bilinear_bf16_fwd", _p(h), _p(t), _p(Wm), _p(bias), P, R, 0, _p(out), R, ws.data_ptr(),
                      ws.numel(), _stream(dev))
        ctx.save_for_backward(h, t, Wm)
        ctx.R = R
        return out

    @staticmethod
    def backward(ctx, dout):
        h, t, Wm = ctx.saved_tensors
        R, dev, P = ctx.R, h.device, h.shape[0]
        dout = _cuda(dout, "dout")
        dh, dt = torch.empty_like(h), torch.empty_like(t)
        dWm = torch.zeros_like(Wm)
        Wm2 = Wm.view(D, R, D).permute(2, 1, 0).reshape(D, R * D).contiguous()       # W viewed as [b][(r, a)]
        lib = _lib.load()
        for p0 in range(0, P, FUSED_CHUNK_PAIRS):
            p1 = min(P, p0 + FUSED_CHUNK_PAIRS)
            rows = p1 - p0
            ws = workspace(dev, int(lib.gcgcn_bilinear_bf16_bwd_ws_bytes(rows, R)))
            _lib.call("gcgcn_bilinear_bf16_bwd", _p(h[p0:p1]), _p(t[p0:p1]), _p(Wm), _p(Wm2), _p(dout[p0:p1]), rows, R,
                      1.0, _p(dh[p0:p1]), _p(dt[p0:p1]), _p(dWm), ws.data_ptr(), ws.numel(), _stream(dev))
        dbias = torch.empty(R, device=dev)
        ws = workspace(dev, 8 << 20)
        _lib.call("gcgcn_colsum", _p(dout), P, R, R, _p(dbias), ws.data_ptr(), ws.numel(), _stream(dev))
        dW = dWm.view(D, R, D).permute(1, 0, 2).contiguous()
        return dh, dt, dW, dbias


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
    parity) or torch.bfloat16 (BilinearBf16Fn); the linear layer, the logits and every gradient are fp32 either way."""
    if dtype not in (torch.float32, torch.bfloat16):
        raise _lib.GcgcnError(f"relation_logits: dtype must be torch.float32 or torch.bfloat16, got {dtype}")
    w = cls.weight
    lin = LinearFn.apply(h, w[:, :D], cls.bias) + LinearFn.apply(t, w[:, D:], None)
    bilinear = BilinearBf16Fn if dtype == torch.bfloat16 else BilinearFn
    z = bilinear.apply(h, t, bili.weight, bili.bias) + lin
    return z if cls_feature is None else DocBiasFn.apply(z, cls_feature, batch)


def pair_bce_loss(logits: torch.Tensor, labels: torch.Tensor, batch: RaggedBatch) -> torch.Tensor:
    """[num_docs] losses exactly as the reference trainer forms them per document (C:355-364)."""
    return PairBceFn.apply(logits, labels, batch)
