"""Float64 test oracle of the relation classifier and the trainer's loss (gcgcn_b200/classifier.py, csrc/classifier.cu),
restated from the definitions in include/gcgcn_b200.h in plain torch, on whichever device its inputs live:

  bilinear   out[p, r] = sum_{a,b} h[p, a] W[r, a, b] t[p, b] + bias[r]                (torch.nn.Bilinear, G:275, 358)
  pair_bce   loss[b] = sum over the ordered pairs i != j of document b of mean_r BCE(sigmoid(z), y), / (n_b^2 - n_b)
  doc_bias   z[p] + v[document of pair p]                                                (B:346-347)

Everything is computed in float64 without the clamps of torch's fp32 BCE (log at -100), so compare the loss with it
only where the logits do not saturate.  The bilinear form is walked in row chunks: at 532 k pairs its [pairs, R*128]
intermediate h W' would be 50 GB in float64.
"""
from __future__ import annotations

import torch

D = 128
CHUNK_ROWS = 16384            # [16384, 97 * 128] float64 = 1.6 GB per intermediate


def wprime(W: torch.Tensor) -> torch.Tensor:
    """W [R, 128 (a), 128 (b)] -> W' [128 (a), R*128 (r, b)] with W'[a][r*128 + b] = W[r][a][b]."""
    R, A, B = W.shape
    out = W.new_empty(A, R * B)
    for r in range(R):
        out[:, r * B:(r + 1) * B] = W[r]
    return out


def wsecond(W: torch.Tensor) -> torch.Tensor:
    """W [R, 128 (a), 128 (b)] -> W'' [128 (b), R*128 (r, a)] with W''[b][r*128 + a] = W[r][a][b]."""
    R, A, B = W.shape
    out = W.new_empty(B, R * A)
    for r in range(R):
        out[:, r * A:(r + 1) * A] = W[r].t()
    return out


def bilinear(h, t, W, bias=None, dout=None, chunk=CHUNK_ROWS):
    """out [P, R]; with dout [P, R] also (dh, dt, dW [R, 128, 128], dbias [R]), all float64:
    dt[p, b] = sum_r dout[p, r] (h W')[p, r*128 + b],  dh[p, a] = sum_r dout[p, r] (t W'')[p, r*128 + a],
    dW'[a][r*128 + b] = sum_p h[p, a] dout[p, r] t[p, b],  dbias[r] = sum_p dout[p, r]."""
    h, t, W = h.double(), t.double(), W.double()
    P, R = h.shape[0], W.shape[0]
    Wp, Wpp = wprime(W), wsecond(W)
    out = h.new_empty(P, R)
    grads = dout is not None
    if grads:
        dout = dout.double()
        dh, dt = torch.empty_like(h), torch.empty_like(t)
        dWp = h.new_zeros(D, R * D)
    for p0 in range(0, P, chunk):
        sl = slice(p0, min(P, p0 + chunk))
        hc, tc = h[sl], t[sl]
        Y = (hc @ Wp).view(-1, R, D)
        out[sl] = torch.einsum("prb,pb->pr", Y, tc)
        if grads:
            dc = dout[sl]
            dt[sl] = torch.einsum("pr,prb->pb", dc, Y)
            del Y
            Z = (tc @ Wpp).view(-1, R, D)
            dh[sl] = torch.einsum("pr,pra->pa", dc, Z)
            del Z
            dWp += hc.t() @ (dc[:, :, None] * tc[:, None, :]).reshape(-1, R * D)
        else:
            del Y
    if bias is not None:
        out += bias.double()
    if not grads:
        return out
    dW = torch.stack([dWp[:, r * D:(r + 1) * D] for r in range(R)])
    return out, dh, dt, dW, dout.sum(0)


def pair_bce(z, y, sizes, dloss=None):
    """Per-document loss [num_docs] of logits z and labels y [total_pairs, R] over documents of `sizes` entities
    (pairs document-major, i-major); with dloss [num_docs] also d(sum_b dloss[b] loss[b]) / dz.  A document of one
    entity has no pair i != j: loss 0, gradient 0."""
    z, y = z.double(), y.double()
    R = z.shape[1]
    loss = z.new_zeros(len(sizes))
    dz = None if dloss is None else torch.zeros_like(z)
    lo = 0
    for b, n in enumerate(sizes):
        zz, yy = z[lo:lo + n * n].view(n, n, R), y[lo:lo + n * n].view(n, n, R)
        if n > 1:
            off = ~torch.eye(n, dtype=torch.bool, device=z.device)
            bce = torch.logaddexp(torch.zeros_like(zz), zz) - yy * zz          # BCE(sigmoid(z), y), no clamp
            loss[b] = bce.mean(-1)[off].sum() / (n * n - n)
            if dloss is not None:
                g = (torch.sigmoid(zz) - yy) * (float(dloss[b]) / ((n * n - n) * R))
                g[~off] = 0.0
                dz[lo:lo + n * n] = g.view(n * n, R)
        lo += n * n
    return loss if dloss is None else (loss, dz)


def doc_bias_fwd(z, v, sizes):
    """z [total_pairs, R] + v[document of the pair], float64."""
    counts = torch.tensor([n * n for n in sizes], device=v.device)
    return z.double() + v.double().repeat_interleave(counts, dim=0)


def doc_bias_bwd(dz, sizes):
    """dv[b] = sum of dz over the n_b^2 pairs of document b (its diagonal pairs included), float64."""
    dz = dz.double()
    out, lo = [], 0
    for n in sizes:
        out.append(dz[lo:lo + n * n].sum(0))
        lo += n * n
    return torch.stack(out)
